"""gf_fastq_stream_keep_reads / take_reads: the FASTQ lines of every matched pair, gathered on the device from the chunk's text.

Every line that comes back is checked against a restatement of FastqReader::read on the same files, in every input format
(plain, multi-member gzip, BGZF inflated on the device and on the host threads), paired and single end, in 4096-byte chunks fed
in uneven pieces (records carried across chunk tails, BGZF members cut by a piece) and in one chunk.  The end-to-end test builds
every ReadMatch of a report from take_reads alone and compares the report bytes with the in-memory pipeline's.
"""
import ctypes as C
import gzip
import os
import random

import numpy as np
import pytest

import _oracle as orc
import report_port as rp
from genefuserust_b200 import ReadBatch, synth
from genefuserust_b200._abi import (GF_E_CAPACITY, GF_E_INVALID, GF_OK, GF_OUT_BUCKET_ORDER, GF_OUT_DROP_FILTERED,
                                    gf_fastq_read_pair, gf_match)

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def test_read_pair_layout():
    assert C.sizeof(gf_fastq_read_pair) == 48
    assert gf_fastq_read_pair.pair_idx.offset == 0
    assert gf_fastq_read_pair.text_off.offset == 8
    assert gf_fastq_read_pair.len.offset == 16 and gf_fastq_read_pair.len.size == 32


def fastq_records(text):
    """FastqReader::read restated (src/core/fastq_reader.rs:75-147): four read_line calls per record, each line loses one
    trailing '\\n' ('\\r' stays); a record is returned only if all four reads returned > 0 bytes"""
    recs, pos = [], 0

    def read_line():
        nonlocal pos
        if pos >= len(text):
            return None
        k = text.find(b"\n", pos)
        line = text[pos:] if k < 0 else text[pos:k + 1]
        pos += len(line)
        return line[:-1] if line.endswith(b"\n") else line
    while True:
        four = tuple(read_line() for _ in range(4))
        if any(x is None for x in four):
            return recs
        recs.append(four)


def odd_fastq(batch, mate, rng, final_newline=True, extra_tail=b""):
    """records with CRLF line ends, names with spaces and empty name lines mixed in"""
    out = []
    for i in range(batch.n):
        s, q = batch.read(i, mate)
        name = b"@SYN:%d:%d %d:N:0:ACGT" % (i, rng.randint(0, 99999), mate)
        r = rng.random()
        if r < 0.03:
            name = b""
        eol = b"\r\n" if r > 0.97 else b"\n"
        out.append(name + eol + s + eol + b"+" + eol + q + eol)
    text = b"".join(out)
    if not final_newline:
        text = text[:-1]
    return text + extra_tail


def encode(host, data, fmt, rng):
    if fmt == "plain":
        return data
    if fmt == "gzip":                 # several members, cut anywhere
        cuts = sorted(rng.sample(range(1, len(data)), 3))
        return b"".join(gzip.compress(data[a:c], compresslevel=1) for a, c in zip([0] + cuts, cuts + [len(data)]))
    return host.bgzf_compress(data, block=4000)


def run_stream(host, m, e1, e2, gz, chunk_bytes, keep, rng=None, take_prob=0.0):
    """feed e1 / e2 (e2 None: single end) in uneven pieces when rng is given, else whole; takes at random when take_prob > 0"""
    st = host.FastqStream(m, paired=e2 is not None, gz=gz, chunk_bytes=chunk_bytes, keep_reads=keep)
    recs, reads = [], {}

    def take():
        if keep:
            r, d = st.take_reads()
            assert not set(d) & set(reads)
            reads.update(d)
            recs.extend(r)
        else:
            recs.extend(st.take())
    try:
        if rng is None:
            st.feed(e1, e2 or b"")
        else:
            p1 = p2 = 0
            while p1 < len(e1) or (e2 is not None and p2 < len(e2)):
                a = rng.randint(1, 12000)          # (both mates alike: one far ahead of the other makes the chunks grow)
                st.feed(e1[p1:p1 + a], e2[p2:p2 + a] if e2 is not None else b"")
                p1 += a
                p2 += a
                if rng.random() < take_prob:
                    take()
        st.finish()
        take()
        counts = st.counts()
    finally:
        st.close()
    return recs, reads, counts


@pytest.fixture(scope="module")
def host():
    import __graft_entry__ as ge
    ge.build()
    from genefuserust_b200 import host as h
    return h


@pytest.fixture(scope="module")
def panel():
    return synth.make_panel(scale=0.02)


@pytest.fixture(scope="module")
def mapper(host, panel):
    m = host.FusionMapper.from_gene_spans(panel.genes(), device=0)
    yield m
    m.close()


@pytest.fixture(scope="module")
def inputs(panel):
    """two FASTQ files of synthetic pairs with many fusions; mate 1 ends without a newline, mate 2 with an incomplete record"""
    rng = random.Random(23)
    b = synth.generate_pairs(panel, 8000, read_len=150, seed=77, p_fusion=0.15)
    fq1 = odd_fastq(b, 1, rng, final_newline=False)
    fq2 = odd_fastq(b, 2, rng, extra_tail=b"@incomplete\nACGT\n+\n")
    m1, m2 = fastq_records(fq1), fastq_records(fq2)
    assert len(m1) == len(m2) == b.n
    o = orc.OracleIndex(panel.genes())
    want_pe = o.scan(ReadBatch.from_reads([(r[1], r[3]) for r in m1], [(r[1], r[3]) for r in m2]), threads=8)
    want_se = o.scan(ReadBatch.from_reads([(r[1], r[3]) for r in m1]), threads=8)
    o.close()
    return {"fq": (fq1, fq2), "model": (m1, m2), "want": (want_pe, want_se)}


def check_reads(recs, reads, model, paired):
    assert set(reads) == {r.pair_idx for r in recs}
    for i, (r1, r2) in reads.items():
        assert r1 == model[0][i], i
        assert r2 == (model[1][i] if paired else None), i


@pytest.mark.gpu
@pytest.mark.parametrize("paired", [True, False], ids=["pe", "se"])
@pytest.mark.parametrize("fmt", ["plain", "gzip", "bgzf", "bgzf_host"])
def test_reads_equal_the_reader_model(host, mapper, inputs, fmt, paired, monkeypatch):
    rng = random.Random(f"{fmt}-{paired}")
    if fmt == "bgzf_host":
        monkeypatch.setenv("GF_BGZF_DEVICE", "0")
    fq1, fq2 = inputs["fq"]
    e1 = encode(host, fq1, fmt, rng)
    e2 = encode(host, fq2, fmt, rng) if paired else None
    want = inputs["want"][0 if paired else 1]
    gz = fmt != "plain"
    for chunk_bytes in (4096, 0):
        piece_rng = random.Random(5) if chunk_bytes else None
        plain_recs, _, _ = run_stream(host, mapper, e1, e2, gz, chunk_bytes, False, random.Random(5) if chunk_bytes else None)
        recs, reads, (n_rec, _tb, calls) = run_stream(host, mapper, e1, e2, gz, chunk_bytes, True, piece_rng)
        assert [r.astuple() for r in recs] == [r.astuple() for r in plain_recs] == want, (fmt, chunk_bytes)
        check_reads(recs, reads, inputs["model"], paired)
        assert len(reads) >= 300, len(reads)
        if chunk_bytes:
            assert calls > 100, calls
        assert n_rec == len(inputs["model"][0])


@pytest.mark.gpu
@pytest.mark.parametrize("paired", [True, False], ids=["pe", "se"])
def test_arena_grows_to_the_lines(host, panel, paired):
    """the device arena for the lines starts small and grows when a chunk's lines do not fit: the first chunk on a fresh index
    takes one more launch (the gather again, into the grown arena); the same chunk again fits and takes none"""
    rng = random.Random(41)
    b = synth.generate_pairs(panel, 20000, read_len=150, seed=91, p_fusion=0.15)
    fq1, fq2 = odd_fastq(b, 1, rng), odd_fastq(b, 2, rng)
    model = (fastq_records(fq1), fastq_records(fq2))
    m = host.FusionMapper.from_gene_spans(panel.genes(), device=0)
    try:
        got = []
        for _ in range(2):
            recs, reads, (_n, _tb, calls) = run_stream(host, m, fq1, fq2 if paired else None, False, 0, True)
            assert calls == 1
            check_reads(recs, reads, model, paired)
            nbytes = sum(sum(len(x) for x in r1) + (sum(len(x) for x in r2) if r2 else 0) for r1, r2 in reads.values())
            got.append((recs, reads, nbytes, int(m.map_stats().kernel_launches)))
    finally:
        m.close()
    (r0, d0, nb, l0), (r1, d1, _, l1) = got
    assert nb > 300 << 10, nb                 # more than the arena's first size (256 KiB)
    assert [r.astuple() for r in r0] == [r.astuple() for r in r1] and d0 == d1
    assert l0 == l1 + 1, (l0, l1)


def _mode_run(host, mapper, e1, e2, mode):
    mapper.set_output_mode(mode)
    try:
        return run_stream(host, mapper, e1, e2, False, 1 << 16, True, random.Random(8))
    finally:
        mapper.set_output_mode(0)


@pytest.mark.gpu
def test_output_modes(host, mapper, inputs):
    fq1, fq2 = inputs["fq"]
    recs, reads, _ = _mode_run(host, mapper, fq1, fq2, 0)
    check_reads(recs, reads, inputs["model"], True)
    # GF_OUT_DROP_FILTERED: exactly the pairs of the surviving records
    drec, dreads, _ = _mode_run(host, mapper, fq1, fq2, GF_OUT_DROP_FILTERED)
    kept = [r.astuple() for r in recs if r.filter_flags == 0]
    assert sorted(r.astuple() for r in drec) == kept
    assert set(dreads) == {r.pair_idx for r in drec}
    assert all(dreads[p] == reads[p] for p in dreads)
    assert len(set(reads) - set(dreads)) >= 1           # pairs whose every record is filtered really occur
    # GF_OUT_BUCKET_ORDER: other order, the same reads
    brec, breads, _ = _mode_run(host, mapper, fq1, fq2, GF_OUT_BUCKET_ORDER)
    assert sorted(r.astuple() for r in brec) == [r.astuple() for r in recs]
    assert breads == reads


def _raw_take(lib, st, caps):
    out = (gf_match * max(1, caps[0]))()
    pairs = (gf_fastq_read_pair * max(1, caps[1]))()
    text = (C.c_uint8 * max(1, caps[2]))()
    n = [C.c_uint64(0) for _ in range(3)]
    rc = lib.gf_fastq_stream_take_reads(st.h, out, caps[0], C.byref(n[0]), pairs, caps[1], C.byref(n[1]), text, caps[2],
                                        C.byref(n[2]))
    cnt = tuple(int(x.value) for x in n)
    if rc != GF_OK:
        return rc, cnt, None
    return rc, cnt, ([out[i].astuple() for i in range(cnt[0])], [(p.pair_idx, p.text_off, tuple(tuple(x) for x in p.len))
                                                                   for p in pairs[:cnt[1]]], bytes(text)[:cnt[2]])


@pytest.mark.gpu
def test_capacity_protocol_and_misuse(host, mapper, inputs):
    fq1, fq2 = inputs["fq"]
    lib = mapper.lib

    def filled():
        st = host.FastqStream(mapper, paired=True, chunk_bytes=1 << 16, keep_reads=True)
        st.feed(fq1, fq2)
        st.finish()
        return st
    st = filled()
    rc, need, full = _raw_take(lib, st, (1 << 20, 1 << 20, 1 << 26))
    st.close()
    assert rc == GF_OK and need[0] > 300 and need[1] >= 300
    for k in range(3):                  # each capacity too small in turn: all counts set, nothing consumed
        st = filled()
        caps = list(need)
        caps[k] -= 1
        rc, cnt, _ = _raw_take(lib, st, caps)
        assert rc == GF_E_CAPACITY and cnt == need, (k, cnt)
        rc, cnt, again = _raw_take(lib, st, need)
        assert rc == GF_OK and cnt == need and again == full, k
        rc, cnt, _ = _raw_take(lib, st, need)
        assert rc == GF_OK and cnt == (0, 0, 0)
        st.close()
    # takes interleaved at random with the feeds add up to one final take
    recs, reads, _ = run_stream(host, mapper, fq1, fq2, False, 4096, True, random.Random(3), take_prob=0.2)
    frecs, freads, _ = run_stream(host, mapper, fq1, fq2, False, 4096, True, random.Random(3))
    assert sorted(r.astuple() for r in recs) == [r.astuple() for r in frecs] and reads == freads
    # misuse: keep_reads after a feed, take on a stream that keeps reads, take_reads on one that does not
    st = host.FastqStream(mapper, paired=True)
    st.feed(fq1[:1000], fq2[:1000])
    assert lib.gf_fastq_stream_keep_reads(st.h) == GF_E_INVALID
    rc, _, _ = _raw_take(lib, st, (10, 10, 10))
    assert rc == GF_E_INVALID
    st.close()
    st = host.FastqStream(mapper, paired=True, keep_reads=True)
    st.feed(fq1, fq2)
    st.finish()
    n = C.c_uint64(0)
    out = (gf_match * 100000)()
    assert lib.gf_fastq_stream_take(st.h, out, 100000, C.byref(n)) == GF_E_INVALID
    rc, cnt, _ = _raw_take(lib, st, need)
    assert rc == GF_OK and cnt == need         # nothing was dropped by the refused take
    st.close()


# ------------------------------------------------------------------------------------------------ end to end: the report
def report_case(tmp_path, n_pairs=120_000, seed=31):
    """testdata/fusions.csv rebased onto synthetic contigs with planted fusions between its four genes and N gaps in the
    spacers; groups of 3 pairs share a read name (sort_matches' name tie-break)"""
    genes = rp.parse_csv(os.path.join(GOLD, "testdata", "fusions.csv"))
    by_chr = {}
    for g in genes:
        by_chr.setdefault(g.m_chr, []).append(g)
    rng = np.random.RandomState(seed)
    contigs, new_genes, csv_lines = {}, {}, []
    for ci, (chrom, gl) in enumerate(sorted(by_chr.items())):
        cur, layout = 10_000, []
        for g in gl:
            layout.append((g, cur - g.m_start))
            cur += (g.m_end - g.m_start) + 10_000
        seq = synth.random_bases(seed * 131 + ci, cur).copy()
        for g, delta in layout:
            s0 = g.m_start + delta - 10_000
            for k in range(150):
                p = s0 + 20 + 60 * k
                seq[p:p + int(rng.randint(1, 4))] = ord("N")
        contigs[chrom] = seq
        for g, delta in layout:
            new_genes[g.m_name] = delta
    for g in genes:
        delta = new_genes[g.m_name]
        csv_lines.append(f">{g.m_name}_ENST,{g.m_chr}:{g.m_start + delta}-{g.m_end + delta}")
        csv_lines += [f"{e.id},{e.start + delta},{e.end + delta}" for e in g.m_exons]
    csv_path = os.path.join(tmp_path, "fusions.synth.csv")
    open(csv_path, "w").write("\n".join(csv_lines) + "\n")
    fa_path = os.path.join(tmp_path, "ref.synth.fa")
    with open(fa_path, "wb") as f:
        for chrom, seq in contigs.items():
            b = seq.tobytes()
            f.write(b">" + chrom.encode() + b"\n" + b"\n".join(b[i:i + 60] for i in range(0, len(b), 60)) + b"\n")
    from genefuserust_b200 import host
    ref = host.FastaReader(fa_path).read_all()
    spans = host.resolve_gene_spans(ref, host.Fusion.parse_csv(csv_path))
    rgenes = rp.parse_csv(csv_path)
    ng = len(spans)
    planted = []
    for k in range(8):
        ga, gb = k % ng, (k + 1 + k // ng) % ng
        la, lb = len(spans[ga][0]), len(spans[gb][0])
        planted.append((ga, int(rng.randint(la // 4, 3 * la // 4)), 1 if (k & 1) == 0 else -1,
                        gb, int(rng.randint(lb // 4, 3 * lb // 4)), 1 if (k & 2) == 0 else -1))
    panel = synth.Panel([g.m_name for g in rgenes], [np.frombuffer(s, dtype=np.uint8).copy() for s, _ in spans],
                        [int(r) for _, r in spans], planted)
    batch = synth.generate_pairs(panel, n_pairs, read_len=150, seed=seed, p_fusion=0.03, threads=8)
    n1 = [b"@SYN:%d:%d 1:N:0:ACGT" % (seed, i // 3) for i in range(batch.n)]
    n2 = [b"@SYN:%d:%d 2:N:0:ACGT" % (seed, i // 3) for i in range(batch.n)]
    return {"spans": spans, "rgenes": rgenes, "batch": batch, "names": (n1, n2),
            "contigs": [ref.m_all_contigs[k] for k in sorted(ref.m_all_contigs)]}


class ReadsOfStream:
    """what read_of_record needs (batch.read(i, mate)), from take_reads alone"""

    def __init__(self, reads):
        self.reads = reads

    def read(self, i, mate):
        _name, seq, _strand, qual = self.reads[i][mate - 1]
        return seq, qual


def device_report(host, m, case, recs, batch, names):
    """records in GF_OUT_DROP_FILTERED | GF_OUT_BUCKET_ORDER order -> ReadMatches -> Matcher -> clusters -> JSON report"""
    spans = case["spans"]
    reads = {(r.pair_idx, r.source): rp.read_of_record(r, batch, names, orc.fast_merge) for r in recs}
    recs = m.finish_order(recs, lambda r: reads[(r.pair_idx, r.source)].m_name)
    rms = [rp.make_read_match(r, reads[(r.pair_idx, r.source)]) for r in recs]
    fm = {}
    for rm in rms:
        fm.setdefault(len(spans) * rm.m_right_gp.contig + rm.m_left_gp.contig, []).append(rm)
    push = [rm for b in sorted(fm) for rm in sorted(fm[b], key=lambda x: x.push_key)]
    mt = host.Matcher(case["contigs"], device=0)
    flags, res, rc = mt.remove_alignables([rm.m_read.m_seq for rm in push])
    mt.close()
    assert rc == 0 and not flags.any()

    def gpu_adjust(batch_of_results):
        return [[(s, ld, rd) for (s, ld, rd, _status) in r] for r in m.adjust_fusion_break(batch_of_results)]
    results = rp.cluster_matches(fm, len(spans) ** 2, case["rgenes"], [s for s, _ in spans], orc.edit_distance, gpu_adjust)
    return rp.json_report(results), results


@pytest.mark.gpu
def test_report_from_streamed_bgzf_reads(host, tmp_path):
    case = report_case(str(tmp_path))
    batch, names = case["batch"], case["names"]
    texts = []
    for mate in (1, 2):
        rows = []
        for i in range(batch.n):
            s, q = batch.read(i, mate)
            rows.append(names[mate - 1][i] + b"\n" + s + b"\n+\n" + q + b"\n")
        texts.append(host.bgzf_compress(b"".join(rows)))
    paths = [str(tmp_path / f"case_R{k}.fq.gz") for k in (1, 2)]
    for p, t in zip(paths, texts):
        open(p, "wb").write(t)
    m = host.FusionMapper.from_gene_spans(case["spans"], device=0)
    m.set_output_mode(GF_OUT_DROP_FILTERED | GF_OUT_BUCKET_ORDER)
    try:
        want_body, want_res = device_report(host, m, case, m.scan_pair_end(batch), batch, names)
        st = host.FastqStream(m, paired=True, gz=True, chunk_bytes=8 << 20, keep_reads=True)
        files = [open(p, "rb") for p in paths]
        try:
            while True:
                a, b = files[0].read(3 << 20), files[1].read(1 << 20)
                if not a and not b:
                    break
                st.feed(a, b)
            st.finish()
            recs, reads = st.take_reads()
            _n, _tb, calls = st.counts()
        finally:
            for f in files:
                f.close()
            st.close()
        assert calls > 3
        snames = ({i: r[0][0] for i, r in reads.items()}, {i: r[1][0] for i, r in reads.items()})
        body, res = device_report(host, m, case, recs, ReadsOfStream(reads), snames)
    finally:
        m.close()
    assert [(r.m_title, r.m_unique, len(r.m_matches)) for r in res] == [(r.m_title, r.m_unique, len(r.m_matches)) for r in want_res]
    assert body == want_body
    assert len(res) >= 4 and len(body) > 10_000
