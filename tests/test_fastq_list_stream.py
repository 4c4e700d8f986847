"""gf_fastq_stream_create_list: one FASTQ stream mapped against several indices (list mode on FASTQ input).

Each chunk is copied, inflated, split and converted once; every index screens and verifies it into its own records, and the
lines of the union of the matched pairs are gathered once with a per-pair mask of the indices that matched them.  The contract
is that index h of a list stream returns exactly what a stream over idx[h] alone returns, fed the same pieces with takes at the
same points: records, descriptors (text_off included), text bytes and the GF_E_REF_PANIC return.  So every test compares the
list stream with single-index streams over the same bytes, through the raw C ABI, and the records with the oracle.

The handles: the small panel, a subset of it (pairs that the full panel matches and the subset does not really occur: asserted),
and a panel of unrelated genes that matches nothing.
"""
import ctypes as C
import random
import threading

import pytest

import _oracle as orc
from genefuserust_b200 import ReadBatch, synth
from genefuserust_b200._abi import (GF_E_CAPACITY, GF_E_INVALID, GF_E_LIMIT, GF_E_REF_PANIC, GF_FQ_GZIP, GF_FQ_PLAIN, GF_OK,
                                    GF_OUT_BUCKET_ORDER, GF_OUT_DROP_FILTERED, gf_fastq_read_pair, gf_match)
from test_fastq_reads import encode, fastq_records, odd_fastq

FORMATS = ["plain", "gzip", "bgzf", "bgzf_host"]


@pytest.fixture(scope="module")
def host():
    import __graft_entry__ as ge
    ge.build()
    from genefuserust_b200 import host as h
    return h


@pytest.fixture(scope="module")
def panel():
    return synth.make_panel(scale=0.02)


def panel_genes(panel):
    """full panel, a subset, unrelated genes (a different seed: no 16-mer in common with the reads)"""
    g = panel.genes()
    return [g, g[:40], synth.make_panel(seed=991, scale=0.01, max_genes=12, plant=False).genes()]


@pytest.fixture(scope="module")
def mappers(host, panel):
    ms = [host.FusionMapper.from_gene_spans(g, device=0) for g in panel_genes(panel)]
    yield ms
    for m in ms:
        m.close()


@pytest.fixture(scope="module")
def inputs(panel):
    """as test_fastq_reads: two FASTQ files with CRLF records, empty names, mate 1 without a final newline, mate 2 with an
    incomplete trailing record; the oracle's records of every distinct panel, paired and single end"""
    rng = random.Random(23)
    b = synth.generate_pairs(panel, 8000, read_len=150, seed=77, p_fusion=0.15)
    fq1 = odd_fastq(b, 1, rng, final_newline=False)
    fq2 = odd_fastq(b, 2, rng, extra_tail=b"@incomplete\nACGT\n+\n")
    m1, m2 = fastq_records(fq1), fastq_records(fq2)
    assert len(m1) == len(m2) == b.n
    want = []
    for genes in panel_genes(panel):
        o = orc.OracleIndex(genes)
        want.append((o.scan(ReadBatch.from_reads([(r[1], r[3]) for r in m1], [(r[1], r[3]) for r in m2]), threads=8),
                     o.scan(ReadBatch.from_reads([(r[1], r[3]) for r in m1]), threads=8)))
        o.close()
    return {"fq": (fq1, fq2), "model": (m1, m2), "want": want}


# ------------------------------------------------------------------------------------------------ the raw ABI
def handles(ms):
    return [m.m_indexer.h for m in ms]


def create(lib, hs, paired, gz, chunk_bytes, keep, single_api=False):
    sh = C.c_void_p()
    fmt = GF_FQ_GZIP if gz else GF_FQ_PLAIN
    if single_api:
        assert len(hs) == 1
        rc = lib.gf_fastq_stream_create(hs[0], 1 if paired else 0, fmt, chunk_bytes, C.byref(sh))
    else:
        rc = lib.gf_fastq_stream_create_list((C.c_void_p * len(hs))(*hs), len(hs), 1 if paired else 0, fmt, chunk_bytes, C.byref(sh))
    assert rc == GF_OK, lib.gf_last_error()
    if keep:
        assert lib.gf_fastq_stream_keep_reads(sh) == GF_OK
    return sh


def raw_take(lib, sh, index, keep, single_api=False, caps=(64, 64, 1024)):
    """(rc, records, descriptors, text) with the capacity protocol; single_api: gf_fastq_stream_take / take_reads"""
    caps = list(caps)
    while True:
        out = (gf_match * max(1, caps[0]))()
        pairs = (gf_fastq_read_pair * max(1, caps[1]))()
        text = (C.c_uint8 * max(1, caps[2]))()
        n = [C.c_uint64(0) for _ in range(3)]
        if keep and single_api:
            rc = lib.gf_fastq_stream_take_reads(sh, out, caps[0], C.byref(n[0]), pairs, caps[1], C.byref(n[1]), text, caps[2],
                                                C.byref(n[2]))
        elif keep:
            rc = lib.gf_fastq_stream_take_reads_index(sh, index, out, caps[0], C.byref(n[0]), pairs, caps[1], C.byref(n[1]), text,
                                                      caps[2], C.byref(n[2]))
        elif single_api:
            rc = lib.gf_fastq_stream_take(sh, out, caps[0], C.byref(n[0]))
        else:
            rc = lib.gf_fastq_stream_take_index(sh, index, out, caps[0], C.byref(n[0]))
        cnt = [int(x.value) for x in n]
        if rc == GF_E_CAPACITY:
            caps = [max(c, k) for c, k in zip(caps, cnt)]
            continue
        assert rc in (GF_OK, GF_E_REF_PANIC), (rc, lib.gf_last_error())
        return (rc, [out[i].astuple() for i in range(cnt[0])],
                [(p.pair_idx, p.text_off, tuple(tuple(x) for x in p.len)) for p in pairs[:cnt[1]]], bytes(text)[:cnt[2]])


def counts(lib, sh):
    v = [C.c_uint64(0) for _ in range(3)]
    assert lib.gf_fastq_stream_get_counts(sh, *[C.byref(x) for x in v]) == GF_OK
    return tuple(int(x.value) for x in v)


def feed_all(lib, sh, e1, e2, piece_seed, on_piece=None):
    """e1 / e2 in uneven pieces (piece_seed None: whole), on_piece(i) after piece i"""
    def feed(a, b):
        assert lib.gf_fastq_stream_feed(sh, a or None, len(a), b or None, len(b)) == GF_OK, lib.gf_last_error()
    if piece_seed is None:
        feed(e1, e2 or b"")
        if on_piece:
            on_piece(0)
    else:
        rng = random.Random(piece_seed)
        p1 = p2 = i = 0
        while p1 < len(e1) or (e2 is not None and p2 < len(e2)):
            a = rng.randint(1, 12000)
            feed(e1[p1:p1 + a], e2[p2:p2 + a] if e2 is not None else b"")
            p1 += a
            p2 += a
            if on_piece:
                on_piece(i)
            i += 1
    assert lib.gf_fastq_stream_finish(sh) == GF_OK, lib.gf_last_error()


def take_at(i, h, take_prob):
    """the same take schedule for the list stream and the single streams"""
    return take_prob > 0 and random.Random(f"{i}-{h}").random() < take_prob


def run(lib, hs, e1, e2, gz, chunk_bytes, keep, piece_seed, take_prob=0.0, single_api=False):
    """[per handle: list of takes], counts"""
    sh = create(lib, hs, e2 is not None, gz, chunk_bytes, keep, single_api)
    takes = [[] for _ in hs]
    try:
        def on_piece(i):
            for h in range(len(hs)):
                if take_at(i, h, take_prob):
                    takes[h].append(raw_take(lib, sh, h, keep, single_api))
        feed_all(lib, sh, e1, e2, piece_seed, on_piece)
        for h in range(len(hs)):
            takes[h].append(raw_take(lib, sh, h, keep, single_api))
        return takes, counts(lib, sh)
    finally:
        lib.gf_fastq_stream_destroy(sh)


def run_singles(lib, hs, e1, e2, gz, chunk_bytes, keep, piece_seed, take_prob=0.0):
    """each handle in a stream of its own (the old entry points), fed the same pieces with takes at the same points"""
    takes, cnts = [], []
    for h, x in enumerate(hs):
        sh = create(lib, [x], e2 is not None, gz, chunk_bytes, keep, single_api=True)
        t = []
        try:
            def on_piece(i):
                if take_at(i, h, take_prob):
                    t.append(raw_take(lib, sh, 0, keep, single_api=True))
            feed_all(lib, sh, e1, e2, piece_seed, on_piece)
            t.append(raw_take(lib, sh, 0, keep, single_api=True))
            cnts.append(counts(lib, sh))
        finally:
            lib.gf_fastq_stream_destroy(sh)
        takes.append(t)
    return takes, cnts


def decode(descs, text, paired):
    """{pair_idx: (mate-1 lines, mate-2 lines or None)} of one take"""
    out = {}
    for pair_idx, off, lens in descs:
        mates = []
        for m in range(2):
            lines = []
            for ln in lens[m]:
                lines.append(text[off:off + ln])
                off += ln
            mates.append(tuple(lines))
        out[pair_idx] = (mates[0], mates[1] if paired else None)
    return out


def check_lines(takes, model, paired):
    """every take: its pairs are exactly its records' pairs, every line as FastqReader::read yields it"""
    seen = set()
    for _rc, recs, descs, text in takes:
        reads = decode(descs, text, paired)
        assert set(reads) == {r[0] for r in recs}
        assert not set(reads) & seen
        seen |= set(reads)
        for i, (r1, r2) in reads.items():
            assert r1 == model[0][i], i
            assert r2 == (model[1][i] if paired else None), i
    return seen


# ------------------------------------------------------------------------------------------------ tests
def test_list_stream_exports(host):
    from genefuserust_b200._abi import EXPORTS, load_library
    lib = load_library()
    for name in ("gf_fastq_stream_create_list", "gf_fastq_stream_take_index", "gf_fastq_stream_take_reads_index"):
        assert name in EXPORTS
        getattr(lib, name)


@pytest.mark.gpu
@pytest.mark.parametrize("paired", [True, False], ids=["pe", "se"])
@pytest.mark.parametrize("fmt", FORMATS)
def test_identical_to_single_index_streams(host, mappers, inputs, fmt, paired, monkeypatch):
    rng = random.Random(f"{fmt}-{paired}")
    if fmt == "bgzf_host":
        monkeypatch.setenv("GF_BGZF_DEVICE", "0")
    lib = mappers[0].lib
    hs = handles(mappers)
    fq1, fq2 = inputs["fq"]
    e1 = encode(host, fq1, fmt, rng)
    e2 = encode(host, fq2, fmt, rng) if paired else None
    gz = fmt != "plain"
    for chunk_bytes in (4096, 0):
        seed = 5 if chunk_bytes else None
        for keep in (True, False):
            got, (n_rec, _tb, calls) = run(lib, hs, e1, e2, gz, chunk_bytes, keep, seed)
            want, single_counts = run_singles(lib, hs, e1, e2, gz, chunk_bytes, keep, seed)
            assert got == want, (fmt, chunk_bytes, keep)
            assert all(c == (n_rec, _tb, calls) for c in single_counts)
            assert n_rec == len(inputs["model"][0])
            if chunk_bytes:
                assert calls > 100, calls
            for h in range(len(hs)):      # the records of every distinct panel are the oracle's
                (rc, recs, _d, _t), = got[h]
                assert rc == GF_OK
                assert recs == inputs["want"][h][0 if paired else 1], (h, fmt, chunk_bytes)
            if keep:
                pairs = [check_lines(got[h], inputs["model"], paired) for h in range(len(hs))]
                # coverage: the full panel matches pairs the subset does not; the unrelated panel matches nothing
                assert len(pairs[0]) >= 300 and len(pairs[1]) >= 1 and not pairs[2], [len(p) for p in pairs]
                assert pairs[0] - pairs[1]


@pytest.mark.gpu
def test_mixed_output_modes(host, panel, mappers, inputs):
    """three output modes in one stream: each handle gets its own mode's records and the pairs of its surviving records"""
    full2 = host.FusionMapper.from_gene_spans(panel.genes(), device=0)
    ms = [mappers[0], mappers[1], full2]
    modes = [0, GF_OUT_DROP_FILTERED | GF_OUT_BUCKET_ORDER, GF_OUT_DROP_FILTERED]
    lib = ms[0].lib
    fq1, fq2 = inputs["fq"]
    try:
        for m, mode in zip(ms, modes):
            m.set_output_mode(mode)
        e1, e2 = host.bgzf_compress(fq1, block=4000), host.bgzf_compress(fq2, block=4000)
        got, _ = run(lib, handles(ms), e1, e2, True, 4096, True, 8)
        want, _ = run_singles(lib, handles(ms), e1, e2, True, 4096, True, 8)
    finally:
        for m in ms:
            m.set_output_mode(0)
        full2.close()
    assert got == want
    for h in range(3):
        check_lines(got[h], inputs["model"], True)
    base = [r for _rc, r, _d, _t in got[0]][0]
    kept = sorted(r for r in base if r[-1] == 0)        # filter_flags is the last field of astuple
    drop = [r for _rc, r, _d, _t in got[2]][0]
    assert drop == kept and len(kept) < len(base)
    assert {d[0] for d in got[2][0][2]} < {d[0] for d in got[0][0][2]}   # pairs whose every record is filtered: gone


@pytest.mark.gpu
@pytest.mark.parametrize("keep", [True, False], ids=["reads", "records"])
def test_one_index_list_equals_create(host, mappers, inputs, keep):
    lib = mappers[0].lib
    x = mappers[0].m_indexer.h
    fq1, fq2 = inputs["fq"]
    e1, e2 = host.bgzf_compress(fq1, block=4000), host.bgzf_compress(fq2, block=4000)
    out = []
    for single_api in (False, True):
        takes, cnt = run(lib, [x], e1, e2, True, 4096, keep, 13, take_prob=0.1, single_api=single_api)
        out.append((takes, cnt, int(mappers[0].map_stats().kernel_launches)))
    assert out[0] == out[1]
    assert out[0][1][2] > 100 and len(out[0][0][0]) > 5


@pytest.mark.gpu
@pytest.mark.parametrize("paired", [True, False], ids=["pe", "se"])
def test_union_arena_grows(host, panel, paired):
    """the union's arena (idx[0]'s) starts small: the first chunk on fresh handles takes one more launch on idx[0] (the
    gather again, into the grown arena); the same chunk again takes none; the lines are the same both times"""
    rng = random.Random(41)
    b = synth.generate_pairs(panel, 20000, read_len=150, seed=91, p_fusion=0.15)
    fq1, fq2 = odd_fastq(b, 1, rng), odd_fastq(b, 2, rng)
    model = (fastq_records(fq1), fastq_records(fq2))
    ms = [host.FusionMapper.from_gene_spans(g, device=0) for g in panel_genes(panel)]
    lib = ms[0].lib
    try:
        got = []
        for _ in range(2):
            takes, (_n, _tb, calls) = run(lib, handles(ms), fq1, fq2 if paired else None, False, 0, True, None)
            assert calls == 1
            got.append((takes, [int(m.map_stats().kernel_launches) for m in ms]))
    finally:
        for m in ms:
            m.close()
    (t0, l0), (t1, l1) = got
    assert t0 == t1
    nbytes = sum(len(t[0][3]) for t in t0[:2])
    assert nbytes > 300 << 10, nbytes        # more than the arena's first size (256 KiB)
    for h in range(3):
        check_lines(t0[h], model, paired)
    assert l0[0] == l1[0] + 1 and l0[1:] == l1[1:], (l0, l1)


@pytest.mark.gpu
def test_takes_while_feeding(host, mappers, inputs):
    """takes interleaved per handle while feeding: each equals the single stream's take at the same point, and a take on one
    handle leaves the others' records and lines in place (they add up to one final take)"""
    lib = mappers[0].lib
    hs = handles(mappers)
    fq1, fq2 = inputs["fq"]
    e1, e2 = host.bgzf_compress(fq1, block=4000), host.bgzf_compress(fq2, block=4000)
    got, _ = run(lib, hs, e1, e2, True, 4096, True, 3, take_prob=0.15)
    want, _ = run_singles(lib, hs, e1, e2, True, 4096, True, 3, take_prob=0.15)
    assert got == want
    once, _ = run(lib, hs, e1, e2, True, 4096, True, 3)
    for h in range(3):
        assert len(got[h]) > 10
        recs = sorted(r for t in got[h] for r in t[1])
        assert recs == once[h][0][1]
        lines = {}
        for _rc, _r, d, t in got[h]:
            lines.update(decode(d, t, True))
        assert lines == decode(once[h][0][2], once[h][0][3], True)
        check_lines(got[h], inputs["model"], True)


@pytest.mark.gpu
def test_capacity_per_index_and_misuse(host, panel, mappers, inputs):
    lib = mappers[0].lib
    hs = handles(mappers)
    fq1, fq2 = inputs["fq"]

    def filled(keep=True):
        sh = create(lib, hs, True, False, 1 << 16, keep)
        feed_all(lib, sh, fq1, fq2, None)
        return sh
    sh = filled()
    full = [raw_take(lib, sh, h, True, caps=(1 << 20, 1 << 20, 1 << 26)) for h in range(3)]
    lib.gf_fastq_stream_destroy(sh)
    need = (len(full[1][1]), len(full[1][2]), len(full[1][3]))
    assert min(need) >= 1 and len(full[0][1]) > len(full[1][1]) and not full[2][1]
    for k in range(3):                  # index 1's capacities too small in turn: all counts set, nothing consumed anywhere
        sh = filled()
        caps = list(need)
        caps[k] -= 1
        out = (gf_match * caps[0])()
        pairs = (gf_fastq_read_pair * caps[1])()
        text = (C.c_uint8 * caps[2])()
        n = [C.c_uint64(0) for _ in range(3)]
        rc = lib.gf_fastq_stream_take_reads_index(sh, 1, out, caps[0], C.byref(n[0]), pairs, caps[1], C.byref(n[1]), text, caps[2],
                                                  C.byref(n[2]))
        assert rc == GF_E_CAPACITY and tuple(int(x.value) for x in n) == need, k
        assert [raw_take(lib, sh, h, True) for h in (2, 1, 0)] == [full[2], full[1], full[0]]
        assert [raw_take(lib, sh, h, True)[1:] for h in range(3)] == [([], [], b"")] * 3
        lib.gf_fastq_stream_destroy(sh)
    sh = filled(keep=False)             # records only: the same per index
    n = C.c_uint64(0)
    out = (gf_match * 1)()
    assert lib.gf_fastq_stream_take_index(sh, 0, out, 1, C.byref(n)) == GF_E_CAPACITY and n.value == len(full[0][1])
    assert raw_take(lib, sh, 0, False)[1] == full[0][1]
    # misuse on a stream of three: plain take / take_reads, index out of range, reads from a stream that does not keep them
    assert lib.gf_fastq_stream_take(sh, out, 1, C.byref(n)) == GF_E_INVALID
    assert lib.gf_fastq_stream_take_index(sh, 3, out, 1, C.byref(n)) == GF_E_INVALID
    pairs = (gf_fastq_read_pair * 1)()
    text = (C.c_uint8 * 1)()
    n2, n3 = C.c_uint64(0), C.c_uint64(0)
    assert lib.gf_fastq_stream_take_reads_index(sh, 0, out, 1, C.byref(n), pairs, 1, C.byref(n2), text, 1, C.byref(n3)) == GF_E_INVALID
    assert raw_take(lib, sh, 1, False)[1] == full[1][1]      # nothing was consumed by the refused calls
    lib.gf_fastq_stream_destroy(sh)
    sh = filled()
    assert lib.gf_fastq_stream_take_reads(sh, out, 1, C.byref(n), pairs, 1, C.byref(n2), text, 1, C.byref(n3)) == GF_E_INVALID
    assert lib.gf_fastq_stream_take_reads_index(sh, 3, out, 1, C.byref(n), pairs, 1, C.byref(n2), text, 1, C.byref(n3)) == GF_E_INVALID
    assert lib.gf_fastq_stream_take_index(sh, 0, out, 1, C.byref(n)) == GF_E_INVALID
    assert [raw_take(lib, sh, h, True) for h in range(3)] == full
    lib.gf_fastq_stream_destroy(sh)
    # the list itself: duplicate, NULL, empty, more than 64
    bad = C.c_void_p()

    def create_rc(lst, n_idx=None):
        arr = (C.c_void_p * max(1, len(lst)))(*lst)
        return lib.gf_fastq_stream_create_list(arr, len(lst) if n_idx is None else n_idx, 1, GF_FQ_PLAIN, 0, C.byref(bad))
    assert create_rc([hs[0], hs[1], hs[0]]) == GF_E_INVALID
    assert create_rc([hs[0], None]) == GF_E_INVALID
    assert create_rc([], 0) == GF_E_INVALID
    assert lib.gf_fastq_stream_create_list(None, 1, 1, GF_FQ_PLAIN, 0, C.byref(bad)) == GF_E_INVALID
    assert lib.gf_fastq_stream_create(None, 1, GF_FQ_PLAIN, 0, C.byref(bad)) == GF_E_INVALID
    tiny = synth.make_panel(seed=5, scale=0.002, max_genes=2, plant=False).genes()
    many = [host.FusionMapper.from_gene_spans(tiny, device=0) for _ in range(65)]
    try:
        assert create_rc(handles(many)) == GF_E_LIMIT
        assert create_rc(handles(many[:64])) == GF_OK
        lib.gf_fastq_stream_destroy(bad)
    finally:
        for m in many:
            m.close()


@pytest.mark.gpu
def test_other_calls_on_idx0_while_streaming(host, panel, mappers, inputs):
    """a thread maps pairs and adjusts fusion breaks on idx[0] while a BGZF list stream is fed in small chunks (the unconsumed
    BGZF tail is copied back inside the locked mapping call, so these calls cannot overwrite it first); every result is
    compared with the same work done alone"""
    lib = mappers[0].lib
    hs = handles(mappers)
    fq1, fq2 = inputs["fq"]
    e1, e2 = host.bgzf_compress(fq1, block=4000), host.bgzf_compress(fq2, block=4000)
    want, _ = run(lib, hs, e1, e2, True, 4096, True, 21)
    m = mappers[0]
    batch = synth.generate_pairs(panel, 3000, read_len=150, seed=5, p_fusion=0.2)
    a, b = sorted((s for s, _r in panel.genes()), key=len)[-2:]
    jobs = [(a[:400], b[:400], [(a[300 - k:400] + b[:100 + k], 100 - k) for k in range(0, 60, 7)])]
    want_map = [r.astuple() for r in m.scan_pair_end(batch)]
    want_adj = m.adjust_fusion_break(jobs)
    assert len(want_map) > 100
    stop, errors, rounds = threading.Event(), [], [0]

    def other():
        try:
            while not stop.is_set():
                assert [r.astuple() for r in m.scan_pair_end(batch)] == want_map
                assert m.adjust_fusion_break(jobs) == want_adj
                rounds[0] += 1
        except BaseException as e:  # (reported by the main thread)
            errors.append(e)
    t = threading.Thread(target=other)
    t.start()
    try:
        got, _ = run(lib, hs, e1, e2, True, 4096, True, 21)
    finally:
        stop.set()
        t.join()
    assert not errors, errors
    assert got == want
    assert rounds[0] >= 1
