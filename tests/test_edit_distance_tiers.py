"""Edit distances of the device against a plain O(mn) Levenshtein DP (orc.levenshtein_dp), where the kernels go wrong.

Every distance the library reports comes from one systolic bit-parallel routine in csrc/gf_map.cu: a block of 64 columns per
lane, carries passed from lane to lane.  warp_edit_distance runs one job on the whole warp (1..32 blocks, up to 2048
columns) and group_edit_distance<G> runs 32 / G jobs side by side.  k_verify picks its tier from the longest of the 8 jobs of
its 4 candidates (<= 256 columns: G = 4, <= 512: G = 8, <= 1024: G = 16, longer: whole warp); k_adjust_break always uses the
whole warp.  The jobs here sit at every block count, on both sides of the lane and tier edges, with partial last blocks and
with the pattern bytes that are not ACGTN (the slow match path)."""
import random
from collections import namedtuple

import pytest

import _oracle as orc
from genefuserust_b200 import ReadBatch, synth

PANIC_COLS = 640   # the reference's edit_distance panics on more than 10 blocks of 64 columns on both sides
COMP = bytes.maketrans(b"ACGTacgt", b"TGCAtgca")
ODD = b"NnacgtRYSWKMBDHV\x00\xff"   # pattern bytes that take the device's slow path, or its N mask
GF_E_REF_PANIC = -5


def dp(a, b):
    return orc.levenshtein_dp(a, b)


def bases(rng, n, alphabet=b"ACGT"):
    return bytes(rng.choice(alphabet) for _ in range(n))


def revcomp(s):
    return s[::-1].translate(COMP)


# ---------------------------------------------------------------------------------------------------------------------
# 1. adjust_fusion_break restated

Adjust = namedtuple("Adjust", "shift left right wrap panic cols")


def adjust_ref(seq, read_break, lref, rref):
    """FusionResult::adjust_fusion_break (fusion_result.rs:299-397), restated from the oracle's fr_calc_ed and its 7-shift
    loop with levenshtein_dp as the distance.
    shift: the first (most negative) shift whose 20 bases on either side of the break are closest to the references;
    left / right: that shift's full-length distances; wrap: a shift puts the break outside the read; panic: a shift's
    full-length comparison is longer than 640 columns (the reference computes them for every shift, winning or not);
    cols: the column counts of the winning shift's two full-length comparisons."""
    nl, nr = len(lref), len(rref)
    best = None
    wrap = panic = False
    for s in range(-3, 4):
        left_len = read_break + s + 1
        right_len = len(seq) - left_len
        if left_len < 0 or right_len < 0:
            wrap = True
            break
        lc2, rc2 = min(left_len, nl), min(right_len, nr)
        panic |= lc2 > PANIC_COLS or rc2 > PANIC_COLS
        lc, rc = min(lc2, 20), min(rc2, 20)
        total = dp(seq[left_len - lc:left_len], lref[nl - lc:]) + dp(seq[left_len:left_len + rc], rref[:rc])
        if best is None or total < best[0]:
            best = (total, s, left_len, lc2, rc2)
    if wrap:
        return Adjust(0, 0, 0, True, panic, (0, 0))
    _total, s, left_len, lc2, rc2 = best
    left = dp(seq[left_len - lc2:left_len], lref[nl - lc2:])
    right = dp(seq[left_len:left_len + rc2], rref[:rc2])
    return Adjust(s, left, right, False, panic, (lc2, rc2))


def _noisy(rng, s, n_edits):
    s = bytearray(s)
    for _ in range(n_edits):
        if not s:
            break
        k = rng.randrange(len(s))
        op = rng.random()
        if op < 0.6:
            s[k] = rng.choice(b"ACGT")
        elif op < 0.8:
            del s[k]
        else:
            s.insert(k, rng.choice(b"ACGT"))
    return bytes(s)


def _random_adjust_job(rng):
    """a read around a break and two references cut from it near the break (or not at all), with noise; lengths on both
    sides of 640 columns, breaks the shifts push outside the read"""
    n = rng.choice((rng.randint(0, 40), rng.randint(20, 400), rng.randint(20, 400), rng.randint(600, 1000),
                    rng.randint(600, 1000)))
    seq = bytearray(bases(rng, n))
    for _ in range(rng.randint(0, 3)):
        if n:
            seq[rng.randrange(n)] = rng.choice(ODD)
    seq = bytes(seq)
    u = rng.random()
    if n >= 700 and u < 0.5:
        rb = rng.randint(634, 646)           # a left comparison that crosses 640 columns inside the 7 shifts
    elif u < 0.15:
        rb = rng.choice((-4, -1, 0, 1, 2, n - 4, n - 3, n - 2, n, n + 2))
    else:
        rb = rng.randint(0, max(0, n - 1))
    cut = min(max(rb + 1 + rng.randint(-3, 3), 0), n)
    left, right = seq[:cut], seq[cut:]

    def ref(part, far_end_first):
        k = rng.random()
        if k < 0.1:
            return bases(rng, rng.randint(0, 60))
        if k < 0.4:                            # longer than the read's side
            extra = bases(rng, rng.randint(1, 700))
            part = extra + part if far_end_first else part + extra
        elif k < 0.6:                          # shorter
            m = rng.randint(0, len(part))
            part = part[len(part) - m:] if far_end_first else part[:m]
        return _noisy(rng, part, rng.randint(0, 3))
    return seq, rb, ref(left, True), ref(right, False)


def test_adjust_ref_equals_oracle():
    """adjust_ref is the oracle's adjust_fusion_break: the same tuple where neither flag is set, status 1 (the reference
    panics) exactly where one is"""
    rng = random.Random(20261022)
    jobs = [_random_adjust_job(rng) for _ in range(3000)]
    # the reference's own edge: a 641-column left comparison panics, 600 and 640 do not
    for nl in (600, 640, 641):
        lref, rref = bases(rng, nl), bases(rng, 200)
        jobs.append((lref + rref, 640, lref, rref))
    n = {"plain": 0, "wrap": 0, "panic": 0, "shifted": 0}
    for seq, rb, lref, rref in jobs:
        want = adjust_ref(seq, rb, lref, rref)
        got = orc.adjust_fusion_break(seq, rb, lref, rref)
        if want.wrap or want.panic:
            assert got == (0, 0, 0, 1), (len(seq), rb, len(lref), len(rref), want)
            n["wrap" if want.wrap else "panic"] += 1
        else:
            assert got == (want.shift, want.left, want.right, 0), (len(seq), rb, len(lref), len(rref), want)
            n["plain"] += 1
            n["shifted"] += want.shift != 0
    assert [adjust_ref(*j).panic for j in jobs[-3:]] == [False, False, True]
    assert n["plain"] > 1500 and n["wrap"] > 100 and n["panic"] > 300 and n["shifted"] > 200, n


# ---------------------------------------------------------------------------------------------------------------------
# device fixtures

@pytest.fixture(scope="module")
def host():
    import __graft_entry__ as ge
    ge.build()
    from genefuserust_b200 import host as h
    return h


@pytest.fixture(scope="module")
def tier_genes():
    """12 genes of 8-12 kb, every third one reversed"""
    return [(synth.random_bases(7100 + g, 8000 + 367 * g).tobytes(), g % 3 == 1) for g in range(12)]


@pytest.fixture(scope="module")
def tier_mappers(host, tier_genes):
    m = host.FusionMapper.from_gene_spans(tier_genes, device=0)
    o = orc.OracleIndex(tier_genes)
    yield m, o
    m.close()
    o.close()


# ---------------------------------------------------------------------------------------------------------------------
# 2. + 3. warp_edit_distance at every block count, through gf_adjust_fusion_break

LENGTHS = sorted({x for b in range(1, 33) for x in (64 * b - 1, 64 * b, 64 * b + 1) if x <= 2048} | {1, 2, 19, 20, 21})
REGIMES = ("identical", "subs", "indel", "random", "a_vs_c", "odd_bytes")
EDGE_COLS = (62, 63, 64, 65, 66, 126, 127, 128, 129, 130)


def _comparison(rng, L, regime, k):
    """(read bytes, reference bytes), both L long, of one full-length comparison"""
    t = bases(rng, L)
    if regime == "identical":
        return t, t
    if regime == "subs":
        p = bytearray(t)
        for q in rng.sample(range(L), min(L, rng.randint(1, 4))):
            p[q] = rng.choice(b"ACGT".replace(bytes([p[q]]), b""))
        return bytes(p), t
    if regime == "indel":                    # one insertion or deletion across the edge of the first or second block
        c = EDGE_COLS[k % len(EDGE_COLS)]
        c = c if c < L else L // 2
        if k % 2:
            return t[:c] + t[c + 1:] + bases(rng, 1), t
        return (t[:c] + bases(rng, 1) + t[c:])[:L], t
    if regime == "random":
        return bases(rng, L), t
    if regime == "a_vs_c":
        return b"A" * L, b"C" * L
    t = bases(rng, L, b"ACGTACGTACGTNRYKM")   # odd_bytes: the reference holds N and IUPAC letters too
    p = bytearray(t)
    for _ in range(L // 8 + 1):
        p[rng.randrange(L)] = rng.choice(ODD)
    return bytes(p), t


def _block_job(rng, L, regime, long_left, k):
    """(seq, read_break, lref, rref) whose left (long_left) or right full-length comparison is the L-column one.  Up to 2042
    columns the read has 3 spare bases beyond that side (repeats of the comparison's outer byte, so that A..A against C..C
    costs L columns at every shift), and every shift compares L columns; the other side is short and identical to its
    reference.  2047 and 2048 columns fill the whole read: L columns at the outermost shift only, which a
    reference of bytes the read never holds (every column of it costs 1) makes the best one."""
    p, t = _comparison(rng, L, regime, k)
    if L + 6 <= 2048:
        o = bases(rng, rng.randint(3, min(40, 2045 - L)))
        if long_left:
            return p[:1] * 3 + p + o, 3 + L - 1, t, o
        return o + p + p[-1:] * 3, len(o) - 1, o, t
    rest, z = bases(rng, 2048 - L), b"Z" * 20
    if long_left:
        return p + rest, L - 4, t, z
    return rest + p, len(rest) + 2, z, t


@pytest.mark.gpu
def test_adjust_break_every_block_count(tier_mappers):
    """all jobs in one call, shuffled, so that neighbouring warps run different lengths: the device equals adjust_ref
    field for field (distances over 640 columns too, where the job is flagged with status 2), and the oracle where
    nothing is flagged"""
    m, _ = tier_mappers
    rng = random.Random(64)
    jobs = [(L, regime, long_left) + _block_job(rng, L, regime, long_left, k)
            for k, (L, regime, long_left) in enumerate((L, r, s) for L in LENGTHS for r in REGIMES for s in (True, False))]
    rng.shuffle(jobs)
    got = m.adjust_fusion_break([(lref, rref, [(seq, rb)]) for _L, _r, _s, seq, rb, lref, rref in jobs])
    hit = set()
    n_flagged = n_nonzero = 0
    for (L, regime, long_left, seq, rb, lref, rref), [g] in zip(jobs, got):
        want = adjust_ref(seq, rb, lref, rref)
        ctx = (L, regime, long_left, want)
        assert not want.wrap
        assert g == (want.shift, want.left, want.right, 2 if want.panic else 0), (g, ctx)
        if not want.panic:
            assert g == orc.adjust_fusion_break(seq, rb, lref, rref), ctx
        cols = want.cols[0 if long_left else 1]
        if L + 6 <= 2048:
            assert cols == L, ctx                          # the construction holds
        if cols == L:
            hit.add(L)
            dist = want.left if long_left else want.right
            if regime == "a_vs_c" and want.shift == 0:
                assert dist == L, ctx
            n_nonzero += dist > 0
        n_flagged += want.panic
    assert hit == set(LENGTHS), sorted(set(LENGTHS) - hit)
    assert n_flagged > 500 and n_nonzero > 600
    assert m.last_rc == GF_E_REF_PANIC


@pytest.mark.gpu
def test_adjust_break_reports_reference_panic(tier_mappers):
    """status 1 where a shift leaves the read, else status 2 where a shift compares more than 640 columns (winning or
    not), and GF_E_REF_PANIC from the call iff a job is flagged"""
    m, _ = tier_mappers
    rng = random.Random(641)
    cases = []
    for nl in (600, 640, 641):                 # 641 columns on the left at shifts 0..3
        lref, rref = bases(rng, nl), bases(rng, 200)
        cases.append((lref + rref, 640, lref, rref))
    seq = bases(rng, 1000)                     # 641 columns only at shift +3; shift 0 (638 columns) wins
    cases.append((seq, 637, bases(rng, 5) + seq[:638], seq[638:]))
    seq = bases(rng, 900)                      # 700 columns on the right
    cases.append((seq, 199, seq[:200], seq[200:]))
    seq = bases(rng, 1239)                     # 641 columns on the right at shift -3 only
    cases.append((seq, 600, seq[:601], seq[601:] + bases(rng, 10)))
    seq = bases(rng, 300)
    cases += [(seq, 1, seq[:2], seq[2:]), (seq, 297, seq[:298], seq[298:]), (seq, 150, seq[:151], seq[151:])]
    seq = bases(rng, 1500)                     # over 640 columns at shift -3, outside the read at shift +2
    cases.append((seq, 1498, seq[:1499], seq[1499:]))
    want = [adjust_ref(*c) for c in cases]
    status = [1 if w.wrap else 2 if w.panic else 0 for w in want]
    assert status == [0, 0, 2, 2, 2, 2, 1, 1, 0, 1]
    assert want[3].shift == 0 and want[3].cols[0] == 638

    def run(sel):
        got = m.adjust_fusion_break([(cases[i][2], cases[i][3], [(cases[i][0], cases[i][1])]) for i in sel])
        for i, [g] in zip(sel, got):
            w = want[i]
            assert g == ((0, 0, 0, 1) if w.wrap else (w.shift, w.left, w.right, status[i])), (i, g, w)
            assert orc.adjust_fusion_break(*cases[i])[3] == (1 if status[i] else 0), i
        return m.last_rc
    assert run(range(len(cases))) == GF_E_REF_PANIC
    assert run([i for i, s in enumerate(status) if s == 0]) == 0
    assert run([2]) == GF_E_REF_PANIC          # a distance over 640 columns alone
    assert run([6]) == GF_E_REF_PANIC


# ---------------------------------------------------------------------------------------------------------------------
# 4. k_verify's tiers through the mapping path

def _piece(gene, start, n, fwd):
    s = gene[start:start + n]
    return s if fwd else revcomp(s)


def _fragment(rng, genes, lens):
    """consecutive pieces of different genes, `lens` bases each, either strand; now and then the first piece starts at its
    gene's first base or the last one ends at its gene's end and a few foreign bases follow (calc_ed's -1 / -2 sentinels)"""
    gs = rng.sample(range(len(genes)), len(lens))
    edge = rng.random()
    out = b""
    for i, (g, n) in enumerate(zip(gs, lens)):
        seq = genes[g][0]
        if i == 0 and edge < 0.07:
            start = 0
        elif i == len(lens) - 1 and edge > 0.93:
            start = len(seq) - n + 3
        else:
            start = rng.randint(0, len(seq) - n)
        piece = _piece(seq, start, n, rng.random() < 0.6)
        out += piece + bases(rng, n - len(piece))
    return out


def _noise(rng, frag, zone):
    """up to 3 substitutions and one single-base indel inside frag[16:-16], and (in `zone`, a range of frag positions) up
    to 2 bytes that are N, lower case or IUPAC: few enough mismatches for the records to survive"""
    f = bytearray(frag)
    for _ in range(rng.choice((0, 1, 2, 3))):
        k = rng.randrange(16, len(f) - 16)
        f[k] = rng.choice(b"ACGT".replace(bytes([f[k]]), b""))
    if rng.random() < 0.3:
        k = rng.randrange(16, len(f) - 16)
        if rng.random() < 0.5:
            del f[k]
            f.insert(len(f) - 16, rng.choice(b"ACGT"))
        else:
            f.insert(k, rng.choice(b"ACGT"))
            del f[len(f) - 16]
    if zone[1] - zone[0] > 40 and rng.random() < 0.3:
        for _ in range(rng.randint(1, 2)):
            f[rng.randrange(zone[0] + 16, zone[1] - 16)] = rng.choice(b"NnacgtRYKM")
    return bytes(f)


def _split(rng, longer, n):
    """(left, right) lengths of an n-base read whose longer part is `longer`, on a random side"""
    return (longer, n - longer) if rng.random() < 0.5 else (n - longer, longer)


def _pair(frag, read_len):
    q = b"E" * read_len
    return (frag[:read_len], q[:min(read_len, len(frag))]), (revcomp(frag)[:read_len], q[:min(read_len, len(frag))])


def _long_batch(rng, genes):
    """max_len = 1000: 2x1000 pairs whose 1000-1970-base fragments merge, the longer part near the 512 / 640 / 1024 tier
    and panic edges and up to ~1900; 2x300 pairs that merge to 316-570 bases, the longer part near 256 / 257; 2x1000 pairs
    that do not merge, one break in each mate.  All shuffled together, so that a warp's 4 candidates mix tiers."""
    pairs = []
    for t in (511, 512, 513, 514, 639, 640, 641, 642, 1023, 1024, 1025, 1026, 1300, 1600, 1900):
        for _ in range(20):
            longer = t + rng.randint(-1, 1)
            lo = max(60, 1000 - longer)
            n = longer + rng.randint(lo, max(lo, min(460, 1970 - longer)))
            frag = _noise(rng, _fragment(rng, genes, _split(rng, longer, n)), (0, n - 1000))
            pairs.append(_pair(frag, 1000))
    for t in (250, 255, 256, 257, 258, 262, 400, 500):
        for _ in range(14):
            longer = t + rng.randint(-1, 1)
            n = longer + rng.randint(60, min(300, 570 - longer))
            frag = _noise(rng, _fragment(rng, genes, _split(rng, longer, n)), (0, n - 300))
            pairs.append(_pair(frag, 300))
    for _ in range(60):
        j1, z = rng.randint(100, 900), rng.randint(100, 900)
        frag = _noise(rng, _fragment(rng, genes, (j1, 2300 - j1 - z, z)), (0, 2300))
        pairs.append(_pair(frag, 1000))
    rng.shuffle(pairs)
    return ReadBatch.from_reads([p[0] for p in pairs], [p[1] for p in pairs])


def _single_end_batch(rng, genes):
    reads = []
    for t in (255, 256, 257, 258, 511, 512, 513, 514, 639, 640, 641, 642, 800, 930):
        for _ in range(10):
            longer = t + rng.randint(-1, 1)
            n = rng.randint(longer + 60, 1000)
            frag = _noise(rng, _fragment(rng, genes, _split(rng, longer, n)), (0, n))
            reads.append((frag, b"E" * n))
    rng.shuffle(reads)
    return ReadBatch.from_reads(reads)


def _small_batch(rng, genes):
    """max_len = 256: 2x256 pairs that merge to 440-482 bases with the break near one end (the G = 8 tier of k_verify's
    small instance), mixed with pairs that do not merge (G = 4)"""
    pairs = []
    for _ in range(220):
        n = rng.randint(440, 482)
        frag = _noise(rng, _fragment(rng, genes, _split(rng, n - rng.randint(50, 80), n)), (0, n - 256))
        pairs.append(_pair(frag, 256))
    for _ in range(100):
        j1, z = rng.randint(60, 196), rng.randint(60, 196)
        frag = _noise(rng, _fragment(rng, genes, (j1, 700 - j1 - z, z)), (0, 700))
        pairs.append(_pair(frag, 256))
    rng.shuffle(pairs)
    return ReadBatch.from_reads([p[0] for p in pairs], [p[1] for p in pairs])


def _record_seq(batch, r):
    """the sequence a record was matched on: the merged read, R1 or R2, reverse-complemented when used_rc"""
    pair, source, used_rc = r[0], r[1], r[2]
    s1, q1 = batch.read(pair, 1)
    if source == 0:
        seq = orc.fast_merge(s1, q1, *batch.read(pair, 2))[0]
    else:
        seq = s1 if source == 1 else batch.read(pair, 2)[0]
    return orc.reverse_complement(seq) if used_rc else seq


def _calc_ed(part, gene, start, end):
    """FusionMapper::calc_ed (fusion_mapper.rs:224-251) with levenshtein_dp: (distance, verified columns, reverse strand)"""
    if (start >= 0 and end <= 0) or (start <= 0 and end >= 0):
        return -1, 0, False
    if abs(start) >= len(gene) or abs(end) >= len(gene):
        return -2, 0, False
    rc = start < 0
    if rc:
        part, start, end = orc.reverse_complement(part), -end, -start
    return dp(part, gene[start:end + 1]), len(part), rc


def _low_complexity(s):
    return len(s) < 20 or sum(a != b for a, b in zip(s, s[1:])) < 7


def _recompute(batch, records, genes, stats):
    """every record's l_dist / r_dist / filter_flags from its own fields and the gene bytes"""
    for r in records:
        _pair_idx, _src, _urc, _rev, rb, lc, lp, rc_, rp, _gap, l_dist, r_dist, seq_len, _ol, _od, ff = r
        seq = _record_seq(batch, r)
        assert len(seq) == seq_len, r
        left, right = seq[:rb + 1], seq[rb + 1:]
        ld, lcols, lrc = _calc_ed(left, genes[lc][0], lp - len(left) + 1, lp)
        rd, rcols, rrc = _calc_ed(right, genes[rc_][0], rp, rp + len(right) - 1)
        assert (l_dist, r_dist) == (ld, rd), r
        want_ff = (1 if _low_complexity(left) or _low_complexity(right) else 0) | (2 if ld + rd >= 5 else 0) | \
                  (4 if lc == rc_ and abs(lp - rp) < 50 else 0)
        assert ff == want_ff, r
        longest = max(lcols, rcols)
        band = 0 if longest <= 256 else 1 if longest <= 512 else 2 if longest <= 1024 else 3
        if longest:
            stats["band"][band] += 1
            stats["band_nonzero"][band] += max(ld, rd) > 0
        stats["sentinel"] |= {d for d in (ld, rd) if d < 0}
        stats["rc"] += lrc + rrc
        stats["le640"] += 0 < lcols <= PANIC_COLS or 0 < rcols <= PANIC_COLS
        stats["gt640"] += lcols > PANIC_COLS or rcols > PANIC_COLS


def _new_stats():
    return {"band": [0] * 4, "band_nonzero": [0] * 4, "sentinel": set(), "rc": 0, "le640": 0, "gt640": 0}


def _check_coverage(stats):
    print("coverage:", stats)
    assert all(n >= 30 for n in stats["band"]), stats
    assert all(n > 0 for n in stats["band_nonzero"]), stats
    assert stats["sentinel"] == {-1, -2}, stats
    assert stats["rc"] > 0 and stats["le640"] > 0 and stats["gt640"] > 0, stats


@pytest.mark.gpu
def test_verify_tiers_mapping_path(tier_mappers, tier_genes):
    """k_verify at every tier: records equal the oracle's, every distance equals the DP's, and the batches reach what
    they are for"""
    m, o = tier_mappers
    rng = random.Random(1025)
    stats = _new_stats()
    batches = [("long", _long_batch(rng, tier_genes)), ("single", _single_end_batch(rng, tier_genes)),
               ("small", _small_batch(rng, tier_genes))]
    assert [b.max_len for _n, b in batches] == [1000, 1000, 256]
    for name, b in batches:
        got = [r.astuple() for r in (m.scan_pair_end(b) if b.paired else m.scan_single_end(b))]
        want = o.scan(b, threads=8)
        assert got == want, (name, len(got), len(want), sorted(set(got) ^ set(want))[:4])
        panics = o.counters()["n_panic"]
        assert (m.last_rc == GF_E_REF_PANIC) == (panics > 0), (name, m.last_rc, panics)
        assert (panics > 0) == (name != "small")
        _recompute(b, got, tier_genes, stats)
    _check_coverage(stats)
