"""Host-side mirror of the reference's interface for the hot path, on top of the C ABI.

Names follow /root/reference/src/core: Fusion::parse_csv (fusion.rs:23-91), FastaReader (fasta_reader.rs),
FastqReader / FastqReaderPair (fastq_reader.rs:75-147), Indexer::make_index (indexer.rs:122-177),
FusionMapper (fusion_mapper.rs:23-87, 253-275, 379-392), PairEndScanner::scan_pair_end (pescanner.rs:427-518),
SingleEndScanner::scan_single_end (sescanner.rs:183-205).  Everything that computes runs in the CUDA library;
this file only loads inputs, owns buffers and regroups records — there is no CPU fallback.
"""
import ctypes as C
import gzip
import os

import numpy as np

from ._abi import (GF_E_CAPACITY, GF_E_REF_PANIC, GF_OK, gf_alignable_result, gf_break_job, gf_break_out, gf_break_ref,
                   gf_fastq_read_pair, gf_index_info, gf_lookup, gf_map_stats, gf_match, gf_merge_info, gf_gene_span, gf_params, gf_ref_contig,
                   gf_reference_info, load_library)
from .batch import ReadBatch


class GeneFuseError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__(f"genefuse_b200 error {code}: {msg}")
        self.code = code


def _check(lib, rc, allow=()):
    if rc != GF_OK and rc not in allow:
        raise GeneFuseError(rc, lib.gf_last_error().decode(errors="replace"))
    return rc


# ---------------------------------------------------------------------------------------------- loaders
class Gene:
    """src/core/gene.rs: name, chr, [start, end), exons; reversed iff exon[0].start > exon[1].start (:98-107)."""

    def __init__(self, name, chrom, start, end):
        self.name, self.chr, self.start, self.end = name, chrom, start, end
        self.exons = []
        self.reversed = False

    def add_exon(self, eid, start, end):
        self.exons.append((eid, start, end))
        if len(self.exons) > 1 and self.exons[0][1] > self.exons[1][1]:
            self.reversed = True

    def valid(self):
        # gene.rs:40-42
        return self.name != "invalid" and self.start != 0 and self.end != 0

    def is_reversed(self):
        return self.reversed


class Fusion:
    def __init__(self, gene):
        self.gene = gene

    def is_reversed(self):
        return self.gene.reversed

    @staticmethod
    def parse_csv(path):
        """fusion.rs:23-91: '>NAME,chr:start-end' gene lines, 'id,start,end' exon lines, '#' comments."""
        fusions = []
        cur = None
        with open(path, "r") as f:
            for raw in f:
                line = raw.strip()
                sp = line.split(",")
                if len(sp) < 2 or sp[0].startswith("#"):
                    continue
                if sp[0].startswith(">"):
                    if cur is not None and cur.valid():
                        fusions.append(Fusion(cur))
                    name = sp[0][1:].strip()
                    chrom, rng = sp[1].split(":")
                    a, b = rng.split("-")
                    cur = Gene(name, chrom.strip(), int(a), int(b))
                    continue
                if len(sp) < 3 or cur is None:
                    continue
                cur.add_exon(int(sp[0]), int(sp[1]), int(sp[2]))
        if cur is not None and cur.valid():
            fusions.append(Fusion(cur))
        return fusions


def _open_maybe_gz(path):
    return gzip.open(path, "rb") if path.endswith(".gz") else open(path, "rb")


class FastaReader:
    """fasta_reader.rs:121-201: name = header up to the first space or newline; everything after a space on
    the header line is filtered into the sequence like any other line (:155-178); contigs sorted by name."""

    def __init__(self, path):
        self.m_fasta_file = path
        self.m_all_contigs = {}

    def read_all(self):
        contigs = {}
        with _open_maybe_gz(self.m_fasta_file) as f:
            data = f.read()
        for rec in data.split(b">")[1:]:
            cut = len(rec)
            for ch in (b"\n", b" "):
                k = rec.find(ch)
                if k >= 0:
                    cut = min(cut, k)
            name = rec[:cut].decode()
            body = rec[cut:]
            # the reference keeps every byte that is not whitespace/CR (:155-178)
            seq = bytes(c for c in body if c not in b"\n\r \t")
            contigs[name] = seq
        self.m_all_contigs = dict(sorted(contigs.items()))
        return self


class FastqReader:
    """fastq_reader.rs:75-147: four lines per record, one trailing '\\n' stripped (no '\\r' strip)."""

    def __init__(self, path):
        self.path = path

    def read_all(self):
        with _open_maybe_gz(self.path) as f:
            lines = f.read().split(b"\n")
        names, reads = [], []
        for i in range(0, len(lines) - 3, 4):
            if not lines[i]:
                break
            names.append(lines[i])
            reads.append((lines[i + 1], lines[i + 3]))
        return names, reads


class FastqReaderPair:
    def __init__(self, path1, path2):
        self.left, self.right = FastqReader(path1), FastqReader(path2)

    def read_all(self):
        n1, r1 = self.left.read_all()
        n2, r2 = self.right.read_all()
        n = min(len(r1), len(r2))
        return (n1[:n], n2[:n]), ReadBatch.from_reads(r1[:n], r2[:n])


# ---------------------------------------------------------------------------------------------- index
def resolve_gene_spans(reference, fusions):
    """Indexer::make_index's host half (indexer.rs:136-159): chromosome-name resolution (exact, 'chr'+name,
    name without 'chr'), slice contig[m_start..m_end], upper-case.  Unresolved -> empty gene that keeps its id."""
    contigs = reference.m_all_contigs
    spans = []
    for fu in fusions:
        g = fu.gene
        chrom = g.chr
        if chrom not in contigs:
            if ("chr" + chrom) in contigs:
                chrom = "chr" + chrom
            elif chrom.replace("chr", "") in contigs:
                chrom = chrom.replace("chr", "")
            else:
                spans.append((b"", g.reversed))
                continue
        seq = contigs[chrom]
        if g.start > g.end or g.end > len(seq):
            # the reference's `.get(start..end).unwrap()` panics here (indexer.rs:154-158)
            raise GeneFuseError(-1, f"gene {g.name}: span {g.start}..{g.end} outside contig {chrom} (reference panics)")
        spans.append((seq[g.start:g.end].upper(), g.reversed))
    return spans


class Indexer:
    """Device index handle (replaces Indexer::{m_kmer_pos, m_dupe_list, m_bloom_filter})."""

    def __init__(self, gene_spans, params=None, device=0):
        self.lib = load_library()
        self.params = params or gf_params.default()
        self.device = device
        self.m_fusion_seq = [s for s, _ in gene_spans]   # kept on the host like the reference (cluster_matches)
        self.reversed = [bool(r) for _, r in gene_spans]
        arr = (gf_gene_span * max(1, len(gene_spans)))()
        keep = []
        for i, (seq, rev) in enumerate(gene_spans):
            buf = C.create_string_buffer(seq, len(seq)) if len(seq) else None
            keep.append(buf)
            arr[i].seq = C.cast(buf, C.c_void_p).value if buf is not None else None
            arr[i].len = len(seq)
            arr[i].reversed = 1 if rev else 0
        h = C.c_void_p()
        _check(self.lib, self.lib.gf_index_create(arr, len(gene_spans), C.byref(self.params), device, C.byref(h)))
        self.h = h

    @classmethod
    def make_index(cls, reference, fusions, params=None, device=0):
        return cls(resolve_gene_spans(reference, fusions), params, device)

    def info(self):
        out = gf_index_info()
        _check(self.lib, self.lib.gf_index_get_info(self.h, C.byref(out)))
        return out

    def lookup(self, kmers):
        kmers = np.ascontiguousarray(kmers, dtype=np.uint32)
        out = (gf_lookup * max(1, len(kmers)))()
        _check(self.lib, self.lib.gf_index_lookup(self.h, kmers.ctypes.data, len(kmers), out))
        return [(o.kind, o.n_sites, tuple((o.contig[j], o.position[j]) for j in range(o.n_sites)))
                for o in out[:len(kmers)]]

    def close(self):
        if getattr(self, "h", None):
            self.lib.gf_index_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


# ---------------------------------------------------------------------------------------------- mapper
class FusionMapper:
    """fusion_mapper.rs:23-87.  Owns the index and the n_genes^2 match buckets."""

    def __init__(self, indexer, fusion_list=None):
        self.m_indexer = indexer
        self.lib = indexer.lib
        self.fusion_list = fusion_list
        self.n_genes = len(indexer.m_fusion_seq)
        self.fusion_matches = {}   # bucket index -> [gf_match]; sparse form of the n_genes^2 Vec (:47-49)
        self.last_rc = GF_OK

    @classmethod
    def from_ref_and_fusion_files(cls, ref_file, fusion_file, params=None, device=0):
        fusions = Fusion.parse_csv(fusion_file)
        ref = FastaReader(ref_file).read_all()
        return cls(Indexer.make_index(ref, fusions, params, device), fusions)

    @classmethod
    def from_fasta_reader_and_fusion_files(cls, fasta_reader, fusion_file, params=None, device=0):
        fusions = Fusion.parse_csv(fusion_file)
        return cls(Indexer.make_index(fasta_reader, fusions, params, device), fusions)

    @classmethod
    def from_gene_spans(cls, gene_spans, params=None, device=0):
        return cls(Indexer(gene_spans, params, device))

    # -- the batch calls that replace the per-pack loops
    def _map(self, batch, cap=None):
        cap = cap or max(4096, batch.n // 64)   # matches are << 1 % of pairs; grown on GF_E_CAPACITY
        st = batch.as_struct()
        while True:
            out = (gf_match * cap)()
            n = C.c_uint64(0)
            rc = self.lib.gf_map_pairs(self.m_indexer.h, C.byref(st), out, cap, C.byref(n))
            if rc == GF_E_CAPACITY:
                cap = int(n.value)
                continue
            _check(self.lib, rc, allow=(GF_E_REF_PANIC,))
            self.last_rc = rc
            return [out[i] for i in range(n.value)]

    def scan_pair_end(self, batch):
        """PairEndScanner::scan_pair_end over a whole batch; records sorted by (pair_idx, source)."""
        assert batch.paired
        return self._map(batch)

    def scan_single_end(self, batch):
        assert not batch.paired
        return self._map(batch)

    def scan_fastq(self, fq1, fq2=None):
        """raw FASTQ text (bytes) -> matches; the records are split on the device (gf_map_fastq)"""
        cap = 4096
        while True:
            out = (gf_match * cap)()
            n, nrec = C.c_uint64(0), C.c_uint64(0)
            rc = self.lib.gf_map_fastq(self.m_indexer.h, fq1, len(fq1), fq2, len(fq2) if fq2 is not None else 0, out, cap,
                                       C.byref(n), C.byref(nrec))
            if rc == GF_E_CAPACITY:
                cap = int(n.value)
                continue
            _check(self.lib, rc, allow=(GF_E_REF_PANIC,))
            self.last_rc = rc
            return [out[i] for i in range(n.value)], int(nrec.value)

    def fast_merge(self, batch):
        out = (gf_merge_info * max(1, batch.n))()
        st = batch.as_struct()
        _check(self.lib, self.lib.gf_fast_merge(self.m_indexer.h, C.byref(st), out))
        return [(o.merged, o.olen, o.diff, o.merged_len) for o in out[:batch.n]]

    def set_output_mode(self, mode):
        """GF_OUT_DROP_FILTERED | GF_OUT_BUCKET_ORDER: the per-record filters of filter_matches and the bucket / sort_matches
        key order are applied on the device (include/genefuse_gpu.h); finish_order() then settles the read-name ties."""
        _check(self.lib, self.lib.gf_index_set_output_mode(self.m_indexer.h, mode))

    def finish_order(self, records, read_name_of):
        """records in GF_OUT_BUCKET_ORDER order -> the reference's final order: inside every run of equal
        gf_match_order_key (same bucket, read_break and read length) sort by read name descending, stable
        (read_match.rs:228, fusion_mapper.rs:384)."""
        from ._abi import gf_match_order_key
        out, i = [], 0
        while i < len(records):
            k = gf_match_order_key(self.n_genes, records[i])
            j = i
            while j < len(records) and gf_match_order_key(self.n_genes, records[j]) == k:
                j += 1
            run = records[i:j]
            if j - i > 1:
                sort_read_matches(run, read_name_of)
            out.extend(run)
            i = j
        return out

    def map_stats(self):
        out = gf_map_stats()
        _check(self.lib, self.lib.gf_get_map_stats(self.m_indexer.h, C.byref(out)), allow=(GF_E_REF_PANIC,))
        return out

    def adjust_fusion_break(self, results):
        """FusionResult::adjust_fusion_break (fusion_result.rs:299-397) for clustered matches.
        `results` = [(m_left_ref, m_right_ref, [(m_read.m_seq, m_read_break), ...]), ...] (bytes; the two reference strings
        are what make_reference builds, :242-297).  Returns, per result, [(shift, m_left_distance, m_right_distance, status),
        ...]; the caller adds `shift` to m_read_break and to both gene positions (:317-319).  status is gf_break_out.status:
        1 = a shifted break leaves the read, 2 = a distance over more than 640 columns, where the reference panics; then
        self.last_rc is GF_E_REF_PANIC."""
        arena = bytearray()
        refs = (gf_break_ref * max(1, len(results)))()
        jobs_l = []
        for r, (lref, rref, matches) in enumerate(results):
            refs[r].left_off, refs[r].left_len = len(arena), len(lref)
            arena += lref
            refs[r].right_off, refs[r].right_len = len(arena), len(rref)
            arena += rref
            for seq, rb in matches:
                jobs_l.append((len(arena), len(seq), rb, r))
                arena += seq
        jobs = (gf_break_job * max(1, len(jobs_l)))()
        for j, (off, ln, rb, r) in enumerate(jobs_l):
            jobs[j].seq_off, jobs[j].seq_len, jobs[j].read_break, jobs[j].result = off, ln, rb, r
        out = (gf_break_out * max(1, len(jobs_l)))()
        rc = self.lib.gf_adjust_fusion_break(self.m_indexer.h, bytes(arena), len(arena), refs, len(results), jobs, len(jobs_l), out)
        _check(self.lib, rc, allow=(GF_E_REF_PANIC,))
        self.last_rc = rc
        res, j = [], 0
        for _l, _r, matches in results:
            res.append([(out[j + k].shift, out[j + k].left_distance, out[j + k].right_distance, out[j + k].status)
                        for k in range(len(matches))])
            j += len(matches)
        return res

    # -- fusion_mapper.rs:253-275 / 379-392
    def add_match(self, m):
        self.fusion_matches.setdefault(fusion_bucket(self.n_genes, m), []).append(m)

    def sort_matches(self, read_name_of):
        """sort_by(|a, b| b.partial_cmp(a)) with ReadMatch's order (read_match.rs:203-229): read_break desc,
        read length asc, read name desc; stable.  `read_name_of(m)` supplies m_read.m_name."""
        for v in self.fusion_matches.values():
            sort_read_matches(v, read_name_of)

    def close(self):
        self.m_indexer.close()


def fusion_bucket(n_genes, m):
    """FusionMapper::add_match (fusion_mapper.rs:253-275): index of the n_genes x n_genes bucket a match goes to"""
    return n_genes * m.r_contig + m.l_contig


def sort_read_matches(matches, read_name_of):
    """FusionMapper::sort_matches (fusion_mapper.rs:379-385) = sort_by(|a, b| b.partial_cmp(a)) with ReadMatch's order
    (read_match.rs:203-229): read_break descending, read length ascending, read name descending; stable, so exact ties
    keep the push order ((pair_idx, source) = the reference's order at -t 1)."""
    import functools

    def cmp(a, b):
        # partial_cmp(self=b, other=a): break asc on (b, a) -> desc on (a, b); len compared other-vs-self
        if a.read_break != b.read_break:
            return -1 if b.read_break < a.read_break else 1
        if a.seq_len != b.seq_len:
            return -1 if a.seq_len < b.seq_len else 1
        na, nb = read_name_of(a), read_name_of(b)
        if na != nb:
            return -1 if nb < na else 1
        return 0

    matches.sort(key=functools.cmp_to_key(cmp))


class PackStream:
    """The batched shim (gf_stream_*): packs of reads in — as lists of (seq, qual) byte strings, the shape of the reference's
    ReadPairPack (pescanner.rs:350-425) — large batches to the device; records come back numbered by the caller."""

    def __init__(self, mapper, paired=True, batch_pairs=0):
        self.lib, self.mapper, self.paired = mapper.lib, mapper, paired
        h = C.c_void_p()
        _check(self.lib, self.lib.gf_stream_create(mapper.m_indexer.h, 1 if paired else 0, batch_pairs, C.byref(h)))
        self.h = h

    def push(self, first_pair, r1, r2=None):
        n = len(r1)

        def arrays(reads):
            ptrs = (C.c_char_p * n)(*[s for s, _ in reads])
            qptr = (C.c_char_p * n)(*[q for _, q in reads])
            lens = (C.c_uint32 * n)(*[len(s) for s, _ in reads])
            return ptrs, qptr, lens
        a1 = arrays(r1)
        a2 = arrays(r2) if r2 is not None else (None, None, None)
        _check(self.lib, self.lib.gf_stream_push(self.h, first_pair, n, a1[0], a1[1], a1[2], a2[0], a2[1], a2[2]))

    def flush(self):
        _check(self.lib, self.lib.gf_stream_flush(self.h))

    def take(self):
        cap = 4096
        while True:
            out = (gf_match * cap)()
            n = C.c_uint64(0)
            rc = self.lib.gf_stream_take(self.h, out, cap, C.byref(n))
            if rc == GF_E_CAPACITY:
                cap = int(n.value)
                continue
            _check(self.lib, rc, allow=(GF_E_REF_PANIC,))
            return [out[i] for i in range(n.value)]

    def counts(self):
        a, b = C.c_uint64(0), C.c_uint64(0)
        _check(self.lib, self.lib.gf_stream_get_counts(self.h, C.byref(a), C.byref(b)))
        return int(a.value), int(b.value)

    def close(self):
        if getattr(self, "h", None):
            self.lib.gf_stream_destroy(self.h)
            self.h = None


def bgzf_compress(data, block=65280, level=1):
    """`data` as BGZF (blocked gzip, what bgzip / bcl2fastq write): gzip members of <= 64 KB that carry their compressed size in
    a 'BC' extra field, closed by the empty EOF member.  Harness utility for the tests and the bench."""
    import struct
    import zlib
    out = []
    for p in list(range(0, len(data), block)) + [None]:
        raw = b"" if p is None else data[p:p + block]
        co = zlib.compressobj(level, zlib.DEFLATED, -15)
        body = co.compress(raw) + co.flush()
        out.append(b"\x1f\x8b\x08\x04\x00\x00\x00\x00\x00\xff\x06\x00BC\x02\x00" + struct.pack("<H", len(body) + 25) + body +
                   struct.pack("<II", zlib.crc32(raw) & 0xFFFFFFFF, len(raw)))
    return b"".join(out)


class FastqStream:
    """FastqReader / FastqReaderPair as a byte stream (gf_fastq_stream_*): feed raw file bytes (plain or gzip, pieces may end
    anywhere), whole records are split and mapped on the device; records are numbered from the start of the files."""

    def __init__(self, mapper, paired=True, gz=False, chunk_bytes=0, keep_reads=False):
        """mapper: one FusionMapper, or a list of them (list mode: every chunk is inflated, split and converted once and mapped
        against each; collect mapper k's records with take(k) / take_reads(k)).
        keep_reads: gather the FASTQ lines of every pair that has a record on the device (collect them with take_reads)"""
        mappers = list(mapper) if isinstance(mapper, (list, tuple)) else [mapper]
        self.lib = mappers[0].lib
        h = C.c_void_p()
        handles = (C.c_void_p * len(mappers))(*[m.m_indexer.h for m in mappers])
        _check(self.lib, self.lib.gf_fastq_stream_create_list(handles, len(mappers), 1 if paired else 0, 1 if gz else 0, chunk_bytes,
                                                              C.byref(h)))
        self.h = h
        self.paired = paired
        if keep_reads:
            _check(self.lib, self.lib.gf_fastq_stream_keep_reads(self.h))

    def feed(self, fq1=b"", fq2=b""):
        _check(self.lib, self.lib.gf_fastq_stream_feed(self.h, fq1 if fq1 else None, len(fq1), fq2 if fq2 else None, len(fq2)))

    def finish(self):
        _check(self.lib, self.lib.gf_fastq_stream_finish(self.h))

    def take(self, index=0):
        """the records of mapper `index` (of the list the stream was made with) mapped since its last take"""
        cap = 4096
        while True:
            out = (gf_match * cap)()
            n = C.c_uint64(0)
            rc = self.lib.gf_fastq_stream_take_index(self.h, index, out, cap, C.byref(n))
            if rc == GF_E_CAPACITY:
                cap = int(n.value)
                continue
            _check(self.lib, rc, allow=(GF_E_REF_PANIC,))
            return [out[i] for i in range(n.value)]

    def take_reads(self, index=0):
        """(records, {pair_idx: ((name, seq, strand, qual) of mate 1, the same of mate 2 or None)}) of mapper `index` on a
        stream that keeps reads: the lines exactly as FastqReader::read yields them, of that mapper's records' pairs"""
        caps = [4096, 4096, 1 << 20]
        while True:
            out = (gf_match * caps[0])()
            pairs = (gf_fastq_read_pair * caps[1])()
            text = (C.c_uint8 * caps[2])()
            n, npair, ntext = C.c_uint64(0), C.c_uint64(0), C.c_uint64(0)
            rc = self.lib.gf_fastq_stream_take_reads_index(self.h, index, out, caps[0], C.byref(n), pairs, caps[1], C.byref(npair),
                                                           text, caps[2], C.byref(ntext))
            if rc == GF_E_CAPACITY:
                caps = [max(caps[0], int(n.value)), max(caps[1], int(npair.value)), max(caps[2], int(ntext.value))]
                continue
            _check(self.lib, rc, allow=(GF_E_REF_PANIC,))
            buf = bytes(text)[:ntext.value]
            reads = {}
            for i in range(npair.value):
                p = pairs[i]
                pos = p.text_off
                mates = []
                for m in range(2):
                    lines = []
                    for ln in p.len[m]:
                        lines.append(buf[pos:pos + ln])
                        pos += ln
                    mates.append(tuple(lines))
                reads[int(p.pair_idx)] = (mates[0], mates[1] if self.paired else None)
            return [out[i] for i in range(n.value)], reads

    def counts(self):
        a, b, c = C.c_uint64(0), C.c_uint64(0), C.c_uint64(0)
        _check(self.lib, self.lib.gf_fastq_stream_get_counts(self.h, C.byref(a), C.byref(b), C.byref(c)))
        return int(a.value), int(b.value), int(c.value)

    @classmethod
    def scan_files(cls, mapper, path1, path2=None, piece=8 << 20, chunk_bytes=0):
        """the whole FastqReaderPair loop: format by file extension (fastq_reader.rs:149-166), files read in `piece`-byte
        reads and fed as they come"""
        gz = path1.endswith(".gz")
        st = cls(mapper, paired=path2 is not None, gz=gz, chunk_bytes=chunk_bytes)
        f1 = open(path1, "rb")
        f2 = open(path2, "rb") if path2 else None
        try:
            while True:
                a = f1.read(piece)
                b = f2.read(piece) if f2 else b""
                if not a and not b:
                    break
                st.feed(a, b)
            st.finish()
            return st.take(), st.counts()
        finally:
            f1.close()
            if f2:
                f2.close()
            st.close()

    def close(self):
        if getattr(self, "h", None):
            self.lib.gf_fastq_stream_destroy(self.h)
            self.h = None


class Matcher:
    """matcher.rs as FusionMapper::remove_alignables uses it (fusion_mapper.rs:488-542): built ONCE per reference (the
    reference streams through the GPU scan once, gf_reference_create), then asked per set of surviving read sequences."""

    def __init__(self, contigs, device=0):
        """contigs: FastaReader.m_all_contigs (dict name -> bytes; iterated in ascending name order like the BTreeMap), or
        a list of bytes / numpy uint8 arrays already in that order, or (device_pointer, length) tuples."""
        self.lib = load_library()
        if isinstance(contigs, dict):
            contigs = [contigs[k] for k in sorted(contigs)]
        arr = (gf_ref_contig * max(1, len(contigs)))()
        self._keep = []
        for i, c in enumerate(contigs):
            if isinstance(c, tuple):
                arr[i].seq, arr[i].len = c
                continue
            a = np.frombuffer(c, dtype=np.uint8) if isinstance(c, (bytes, bytearray)) else np.ascontiguousarray(c, dtype=np.uint8)
            self._keep.append(a)
            arr[i].seq = a.ctypes.data if len(a) else None
            arr[i].len = len(a)
        h = C.c_void_p()
        _check(self.lib, self.lib.gf_reference_create(arr, len(contigs), device, C.byref(h)))
        self.h = h
        self._keep = []

    def info(self):
        out = gf_reference_info()
        _check(self.lib, self.lib.gf_reference_get_info(self.h, C.byref(out)))
        return out

    def remove_alignables(self, seqs):
        """seqs: list of bytes (ReadMatch::get_read().m_seq in bucket order).  Returns (alignable flags, result struct, rc);
        rc is GF_E_REF_PANIC where the reference's Matcher would abort the run."""
        off = np.zeros(len(seqs) + 1, dtype=np.uint64)
        if seqs:
            np.cumsum([len(s) for s in seqs], out=off[1:])
        arena = np.frombuffer(b"".join(seqs), dtype=np.uint8) if seqs else np.zeros(0, np.uint8)
        flags = np.zeros(max(1, len(seqs)), dtype=np.uint8)
        res = gf_alignable_result()
        rc = self.lib.gf_alignable_filter(self.h, arena.ctypes.data if len(arena) else None, off.ctypes.data, len(seqs),
                                          flags.ctypes.data, C.byref(res))
        _check(self.lib, rc, allow=(GF_E_REF_PANIC,))
        return flags[:len(seqs)], res, rc

    def close(self):
        if getattr(self, "h", None):
            self.lib.gf_reference_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class PairEndScanner:
    """pescanner.rs: scan() = build mapper, map all pairs, push matches into the mapper's buckets."""

    def __init__(self, fusion_file, ref_file, read1, read2, device=0):
        self.fusion_file, self.ref_file, self.read1, self.read2, self.device = fusion_file, ref_file, read1, read2, device
        self.mapper = None

    def scan(self):
        self.mapper = FusionMapper.from_ref_and_fusion_files(self.ref_file, self.fusion_file, device=self.device)
        (names1, _names2), batch = FastqReaderPair(self.read1, self.read2).read_all()
        matches = self.mapper.scan_pair_end(batch)
        for m in matches:
            self.mapper.add_match(m)
        return matches


class MultiGpuMapper:
    """One process, several GPUs (gf_multi_*): index replicated, every batch sharded by pairs, records gathered on the
    host in (pair_idx, source) order — the same answer as FusionMapper on one device."""

    def __init__(self, gene_spans, devices, params=None):
        self.lib = load_library()
        self.params = params or gf_params.default()
        arr = (gf_gene_span * max(1, len(gene_spans)))()
        keep = []
        for i, (seq, rev) in enumerate(gene_spans):
            buf = C.create_string_buffer(seq, len(seq)) if len(seq) else None
            keep.append(buf)
            arr[i].seq = C.cast(buf, C.c_void_p).value if buf is not None else None
            arr[i].len = len(seq)
            arr[i].reversed = 1 if rev else 0
        devs = (C.c_int * len(devices))(*devices)
        h = C.c_void_p()
        _check(self.lib, self.lib.gf_multi_create(arr, len(gene_spans), C.byref(self.params), devs, len(devices), C.byref(h)))
        self.h = h

    def scan(self, batch):
        cap = max(4096, batch.n // 64)
        st = batch.as_struct()
        while True:
            out = (gf_match * cap)()
            n = C.c_uint64(0)
            rc = self.lib.gf_multi_map_pairs(self.h, C.byref(st), out, cap, C.byref(n))
            if rc == GF_E_CAPACITY:
                cap = int(n.value)
                continue
            _check(self.lib, rc, allow=(GF_E_REF_PANIC,))
            return [out[i] for i in range(n.value)]

    def close(self):
        if getattr(self, "h", None):
            self.lib.gf_multi_destroy(self.h)
            self.h = None


def scan_list(mappers, batch):
    """List mode (fusion_scan.rs:62-188): the same reads against several FusionMappers (one per fusion CSV, all on one
    device) in ONE call — the batch is uploaded and converted once, then mapped per index (gf_list_map_pairs).
    Returns one record list per mapper, each identical to mapper.scan_pair_end(batch) / scan_single_end(batch)."""
    lib = mappers[0].lib
    n = len(mappers)
    hs = (C.c_void_p * n)(*[m.m_indexer.h.value for m in mappers])
    caps = [max(4096, batch.n // 64)] * n
    st = batch.as_struct()
    while True:
        bufs = [(gf_match * c)() for c in caps]
        outs = (C.POINTER(gf_match) * n)(*[C.cast(b, C.POINTER(gf_match)) for b in bufs])
        ccaps = (C.c_uint64 * n)(*caps)
        nout = (C.c_uint64 * n)()
        rc = lib.gf_list_map_pairs(hs, n, C.byref(st), outs, ccaps, nout)
        if rc == GF_E_CAPACITY:
            caps = [max(c, int(k)) for c, k in zip(caps, nout)]
            continue
        _check(lib, rc, allow=(GF_E_REF_PANIC,))
        for m in mappers:
            m.last_rc = rc
        return [[bufs[h][i] for i in range(nout[h])] for h in range(n)]
