/*
 * gf_map.cu — per-read fusion matching on the GPU.
 *
 * Replaces, for a whole batch of read pairs (paths relative to /root/reference):
 *   PairEndScanner::scan_pair_end   src/core/pescanner.rs:427-518   (per-pair policy, rc retry)
 *   SingleEndScanner::scan_single_end src/core/sescanner.rs:183-205
 *   SequenceReadPair::fast_merge    src/core/read.rs:313-440
 *   FusionMapper::map_read / make_match / calc_distance / calc_ed   src/core/fusion_mapper.rs:93-251
 *   Indexer::map_read / in_required_direction / segment_mask       src/core/indexer.rs:252-679
 *   edit_distance                   src/core/edit_distance.rs:12-197
 *
 * Kernels:
 *   screen    every pair: fast_merge decision + a CONSERVATIVE form of map_read's first pass.  Reads <= 256 bases: the
 *             split pipeline k_prep -> k_seed -> k_diag / k_scan of gf_screen_split.cuh (thread per pair / per sequence,
 *             bit-planes, L2-resident filter + gene planes; the bound is documented there).  Longer reads (up to 1024
 *             bases): k_screen (warp per pair, same structures).
 *             A sequence is dropped only when it provably fails the vote gate of indexer.rs:353-360:
 *                 T = sum of sites voted, c_d = votes of unique keys on one diagonal d (any d)
 *                 count1 >= c_d and count1 + count2 <= T   =>   count2 <= T - c_d
 *             so "T < ceil(major/2)+ceil(minor/2)  or  T - c_d < ceil(minor/2)" can never pass the gate.
 *             Everything else goes to the survivor list.
 *   k_exact   (warp per survivor)           the literal algorithm: exact vote table, top-2 in BTreeMap order,
 *             gate, second pass mask, mismatch gate, segment_mask, direction gate, make_match, and the
 *             reverse-complement retry of scan_pair_end.  Emits candidate records.
 *   k_verify  (warp per 4 candidates)       calc_distance/calc_ed: bit-parallel (Myers/Hyyro) Levenshtein with
 *             one 64-column block per lane, carries passed lane to lane in a systolic pipeline; the 8 distances of 4
 *             candidates run side by side in groups of 4 lanes (8 / 16 lanes for longer parts); exact for any distance,
 *             so the -1/-2 sentinels and the ">= 5" filter downstream see the reference's values.  Also sets the
 *             post-filter flags.
 *   k_adjust_break (warp per clustered match)  FusionResult::adjust_fusion_break, src/core/fusion_result.rs:299-397.
 */
#include <climits>
#include <cstdlib>
#include <cstdio>

#include "gf_internal.h"
#include "gf_swar.cuh"

namespace {

#define FULL 0xFFFFFFFFu
using swar::zero_bytes;

__device__ __forceinline__ uint32_t fsr(const uint32_t* plane, uint32_t bitpos) {
    uint32_t w = bitpos >> 5;
    return __funnelshift_r(plane[w], plane[w + 1], bitpos & 31u);
}
__device__ __forceinline__ uint32_t lowmask(int nbits) { /* nbits >= 1 */
    return nbits >= 32 ? 0xFFFFFFFFu : ((1u << nbits) - 1u);
}
/* record [s, e) of an arena (offsets relative to `base`, `bytes` readable; 0 = extent unknown, not checked) lies inside the
 * arena and is at most max_len long — offsets that are not ascending or wrap fail here */
__device__ __forceinline__ bool record_ok(uint64_t s, uint64_t e, uint64_t base, uint64_t bytes, int max_len) {
    if (e < s || e - s > (uint64_t)max_len || s < base) return false;
    return bytes == 0 || (s - base <= bytes && e - s <= bytes - (s - base));
}

/* ------------------------------------------------------------------------------------------------ */
/* per-warp shared state of the screen kernel: bit-planes, one bit per base                          */
template <int MAXW>
struct ScreenWarp {
    /* R1 forward */
    uint32_t r1lo[MAXW + 1], r1hi[MAXW + 1], r1v[MAXW + 1], r1n[MAXW + 1], q1hi[MAXW + 1], q1lo[MAXW + 1];
    /* reverse complement of R2 (read.rs:314) and its reversed qualities */
    uint32_t c2lo[MAXW + 1], c2hi[MAXW + 1], c2v[MAXW + 1], c2n[MAXW + 1], q2hi[MAXW + 1], q2lo[MAXW + 1];
    /* overlap-resolved rc(R2) (x*) and the sequence that is mapped (m*) */
    uint32_t xlo[MAXW + 1], xhi[MAXW + 1], xv[MAXW + 1];
    uint32_t mlo[2 * MAXW + 2], mhi[2 * MAXW + 2], mv[2 * MAXW + 2];
    /* screen v2: reverse-complement planes of the mapped sequence, gene planes along the seed diagonal,
     * per-chunk equality / hit words and the list of offsets that still need a filter probe */
    uint32_t rlo[2 * MAXW + 2], rhi[2 * MAXW + 2], rv[2 * MAXW + 2];
    uint32_t glo[2 * MAXW + 3], ghi[2 * MAXW + 3], gv[2 * MAXW + 3], gc[3][2 * MAXW + 3];
    uint32_t eq[2 * MAXW + 2], hit[2 * MAXW + 2];
    uint16_t others[32 * MAXW + 32];
    /* forward planes of R2 (mapped when the pair does not merge) */
    uint32_t f2lo[MAXW + 1], f2hi[MAXW + 1], f2v[MAXW + 1];
    /* SWAR scratch: 6 byte-granular planes, bit (p + a) of plane j <-> base p of the read being converted,
     * a = misalignment (0..7) of the read's first byte w.r.t. the 8-byte loads */
    uint32_t sp[6][MAXW + 4];
};

/* ---- SWAR plane construction: 8 ASCII bytes per lane and load --------------------------------------- */
__device__ __forceinline__ uint32_t gather4(uint32_t t) { /* bits 0,8,16,24 -> bits 0..3 */
    return ((t * 0x01020408u) >> 24) & 0xFu;
}
/* 4 bases -> 4-bit masks: code bits (A0 T1 C2 G3), valid = one of ACGT (upper case, or either case when ci) */
__device__ __forceinline__ void classify4(uint32_t x, bool ci, uint32_t* lo, uint32_t* hi, uint32_t* v) {
    const uint32_t xu = ci ? (x & 0xDFDFDFDFu) : x;
    const uint32_t t = (xu >> 1) & 0x03030303u; /* A0 C1 T2 G3 per byte */
    const uint32_t u = t | (t >> 4);
    const uint32_t sel = (u & 0xFFu) | ((u >> 8) & 0xFF00u);
    const uint32_t expect = __byte_perm(0x47544341u, 0u, sel); /* 'A','C','T','G' */
    /* common case: all four bytes are ACGT -> one compare instead of the per-byte zero test */
    const uint32_t vv = xu == expect ? 0xFu : gather4(zero_bytes(xu ^ expect) >> 7);
    *v = vv;
    *lo = gather4((xu >> 2) & 0x01010101u) & vv;
    *hi = gather4((xu >> 1) & 0x01010101u) & vv;
}
__device__ __forceinline__ uint32_t ge4(uint32_t q, uint32_t thr4) { /* per byte: (q & 0x7F) >= thr */
    return gather4((((q | 0x80808080u) - thr4) & 0x80808080u) >> 7);
}
/* 8 bytes at the 8-aligned address `p`; bytes outside [lo, hi) read as 0 (never touches memory outside) */
__device__ __forceinline__ uint2 load8_guarded(const uint8_t* p, const uint8_t* lo, const uint8_t* hi) {
    if (p >= lo && p + 8 <= hi) return __ldg(reinterpret_cast<const uint2*>(p));
    uint32_t w[2] = {0u, 0u};
    for (int t = 0; t < 8; t++)
        if (p + t >= lo && p + t < hi) w[t >> 2] |= (uint32_t)__ldg(p + t) << (8 * (t & 3));
    return make_uint2(w[0], w[1]);
}
/* Converts one read into the 6 scratch planes S.sp[0..5] (byte L of each plane = bases 8L-a .. 8L-a+7):
 *   0 lo, 1 hi, 2 valid (case-insensitive when ci), 3 extra (R1: is 'N'; R2: valid upper-case only), 4 q>='?', 5 q<='0'
 * Returns the bit shifts (a_seq, a_qual) to apply when reading the scratch planes. */
template <int MAXW>
__device__ __forceinline__ void swar_convert(ScreenWarp<MAXW>& S, const uint8_t* seq, const uint8_t* qual, int len,
                                             const uint8_t* seq_lo, const uint8_t* seq_hi, const uint8_t* qual_lo,
                                             const uint8_t* qual_hi, bool is_r2, int* a_seq, int* a_qual) {
    const uint32_t lane = gf_lane();
    const int as = (int)((uintptr_t)seq & 7u), aq = (int)((uintptr_t)qual & 7u);
    const uint8_t* s0 = seq - as;
    const uint8_t* q0 = qual - aq;
    uint8_t* b0 = reinterpret_cast<uint8_t*>(S.sp[0]);
    uint8_t* b1 = reinterpret_cast<uint8_t*>(S.sp[1]);
    uint8_t* b2 = reinterpret_cast<uint8_t*>(S.sp[2]);
    uint8_t* b3 = reinterpret_cast<uint8_t*>(S.sp[3]);
    uint8_t* b4 = reinterpret_cast<uint8_t*>(S.sp[4]);
    uint8_t* b5 = reinterpret_cast<uint8_t*>(S.sp[5]);
    const int nbytes = 4 * (((len + 31) >> 5) + 3); /* scratch bytes that later reads may touch */
    for (int L = (int)lane; L < nbytes; L += 32) {
        uint32_t lo = 0, hi = 0, v = 0, ex = 0, qh = 0, ql = 0;
        /* sequence planes: base p = 8L - as + t */
        {
            int p0 = 8 * L - as;
            if (p0 < len && p0 + 8 > 0) {
                uint2 x = load8_guarded(s0 + 8 * L, seq_lo, seq_hi);
                uint32_t l0, h0, v0, l1, h1, v1;
                classify4(x.x, is_r2, &l0, &h0, &v0);
                classify4(x.y, is_r2, &l1, &h1, &v1);
                lo = l0 | (l1 << 4); hi = h0 | (h1 << 4); v = v0 | (v1 << 4);
                if (is_r2) {
                    uint32_t c0, c1, c2, c3, c4, c5;
                    classify4(x.x, false, &c0, &c1, &c2);
                    classify4(x.y, false, &c3, &c4, &c5);
                    ex = c2 | (c5 << 4);
                } else {
                    ex = gather4(zero_bytes(x.x ^ 0x4E4E4E4Eu) >> 7) | (gather4(zero_bytes(x.y ^ 0x4E4E4E4Eu) >> 7) << 4);
                }
                int tlo = max(0, -p0), thi = min(8, len - p0);
                uint32_t pm = ((1u << thi) - 1u) & ~((1u << tlo) - 1u);
                lo &= pm; hi &= pm; v &= pm; ex &= pm;
            }
        }
        if (qual) {
            int p0 = 8 * L - aq;
            if (p0 < len && p0 + 8 > 0) {
                uint2 q = load8_guarded(q0 + 8 * L, qual_lo, qual_hi);
                qh = ge4(q.x, 0x3F3F3F3Fu) | (ge4(q.y, 0x3F3F3F3Fu) << 4);               /* >= '?' */
                ql = (~(ge4(q.x, 0x31313131u) | (ge4(q.y, 0x31313131u) << 4))) & 0xFFu;  /* <= '0' */
                int tlo = max(0, -p0), thi = min(8, len - p0);
                uint32_t pm = ((1u << thi) - 1u) & ~((1u << tlo) - 1u);
                qh &= pm; ql &= pm;
            }
        }
        b0[L] = (uint8_t)lo; b1[L] = (uint8_t)hi; b2[L] = (uint8_t)v; b3[L] = (uint8_t)ex;
        b4[L] = (uint8_t)qh; b5[L] = (uint8_t)ql;
    }
    *a_seq = as;
    *a_qual = aq;
    __syncwarp();
}
/* 32 bits of a scratch plane starting at (possibly negative) bit position pos */
__device__ __forceinline__ uint32_t win32(const uint32_t* pl, int pos) {
    if (pos >= 0) return fsr(pl, (uint32_t)pos);
    if (pos > -32) return pl[0] << (-pos);
    return 0u;
}
/* R1 planes (forward) from the scratch */
template <int MAXW>
__device__ __forceinline__ void planes_r1(ScreenWarp<MAXW>& S, const uint8_t* seq, const uint8_t* qual, int len,
                                          const uint8_t* slo, const uint8_t* shi, const uint8_t* qlo, const uint8_t* qhi) {
    int as, aq;
    swar_convert<MAXW>(S, seq, qual, len, slo, shi, qlo, qhi, false, &as, &aq);
    const int nw = (len + 31) >> 5;
    for (int k = (int)gf_lane(); k <= nw; k += 32) {
        const bool in = k < nw;
        S.r1lo[k] = in ? fsr(S.sp[0], (uint32_t)(32 * k + as)) : 0u;
        S.r1hi[k] = in ? fsr(S.sp[1], (uint32_t)(32 * k + as)) : 0u;
        S.r1v[k] = in ? fsr(S.sp[2], (uint32_t)(32 * k + as)) : 0u;
        S.r1n[k] = in ? fsr(S.sp[3], (uint32_t)(32 * k + as)) : 0u;
        S.q1hi[k] = in ? fsr(S.sp[4], (uint32_t)(32 * k + aq)) : 0u;
        S.q1lo[k] = in ? fsr(S.sp[5], (uint32_t)(32 * k + aq)) : 0u;
    }
    __syncwarp();
}
/* R2: forward planes (f2*, upper-case validity) and the planes of reverse_complement(R2) (c2*, sequence.rs:22-60:
 * case-insensitive, everything else 'N') with reversed qualities */
template <int MAXW>
__device__ __forceinline__ void planes_r2(ScreenWarp<MAXW>& S, const uint8_t* seq, const uint8_t* qual, int len,
                                          const uint8_t* slo, const uint8_t* shi, const uint8_t* qlo, const uint8_t* qhi) {
    int as, aq;
    swar_convert<MAXW>(S, seq, qual, len, slo, shi, qlo, qhi, true, &as, &aq);
    const int nw = (len + 31) >> 5;
    for (int k = (int)gf_lane(); k <= nw; k += 32) {
        const bool in = k < nw;
        uint32_t fv = in ? fsr(S.sp[3], (uint32_t)(32 * k + as)) : 0u;
        S.f2v[k] = fv;
        S.f2lo[k] = in ? (fsr(S.sp[0], (uint32_t)(32 * k + as)) & fv) : 0u;
        S.f2hi[k] = in ? (fsr(S.sp[1], (uint32_t)(32 * k + as)) & fv) : 0u;
        uint32_t clo = 0, chi = 0, cv = 0, cn = 0, cqh = 0, cql = 0;
        if (in) {
            const int pos = len - 32 * k - 32; /* out bit b = src[len-1-(32k+b)] */
            cv = __brev(win32(S.sp[2], pos + as));
            clo = ~__brev(win32(S.sp[0], pos + as)) & cv; /* complement = code ^ 1 */
            chi = __brev(win32(S.sp[1], pos + as));
            cn = lowmask(len - 32 * k) & ~cv;
            cqh = __brev(win32(S.sp[4], pos + aq));
            cql = __brev(win32(S.sp[5], pos + aq));
        }
        S.c2lo[k] = clo; S.c2hi[k] = chi; S.c2v[k] = cv; S.c2n[k] = cn; S.q2hi[k] = cqh; S.q2lo[k] = cql;
    }
    __syncwarp();
}

/* fast_merge's inner loop for one overlap length (read.rs:339-367), 32 bases per step.
 * passes <=> every mismatch is a "low quality diff" and there are at most 2 of them. */
template <int MAXW>
__device__ __forceinline__ bool overlap_ok(const ScreenWarp<MAXW>& S, int len1, int olen, int* diff) {
    const int offset = len1 - olen;
    int cnt = 0;
    for (int k = 0; 32 * k < olen; k++) {
        uint32_t bp = (uint32_t)(offset + 32 * k);
        uint32_t alo = fsr(S.r1lo, bp), ahi = fsr(S.r1hi, bp), an = fsr(S.r1n, bp), av = fsr(S.r1v, bp);
        uint32_t m = lowmask(olen - 32 * k);
        uint32_t mism = ((alo ^ S.c2lo[k]) | (ahi ^ S.c2hi[k]) | (an ^ S.c2n[k]) | (~av & ~an)) & m;
        if (mism) {
            cnt += __popc(mism);
            if (cnt > 2) return false;
            uint32_t lowq = (fsr(S.q1hi, bp) & S.q2lo[k]) | (fsr(S.q1lo, bp) & S.q2hi[k]);
            if (mism & ~lowq) return false;
        }
    }
    *diff = cnt;
    return true;
}
/* smallest passing overlap length >= 30 (read.rs:323-367); -1 when the pair does not merge */
template <int MAXW>
__device__ __forceinline__ int find_overlap(const ScreenWarp<MAXW>& S, int len1, int len2, int* diff_out) {
    const int minlen = min(len1, len2);
    const uint32_t lane = gf_lane();
    for (int base = 30; base <= minlen; base += 32) {
        int o = base + (int)lane;
        int diff = 0;
        bool ok = o <= minlen && overlap_ok<MAXW>(S, len1, o, &diff);
        uint32_t b = __ballot_sync(FULL, ok);
        if (b) {
            int first = __ffs(b) - 1;
            *diff_out = __shfl_sync(FULL, diff, first);
            return base + first;
        }
    }
    *diff_out = 0;
    return -1;
}
/* merged sequence planes (read.rs:369-428): R1[..offset] ++ rc(R2), overlap mismatches take the R1 base
 * iff q1 >= '?' and q2 <= '0'.  Returns the merged length. */
template <int MAXW>
__device__ __forceinline__ int build_merged(ScreenWarp<MAXW>& S, int len1, int len2, int olen) {
    const uint32_t lane = gf_lane();
    const int offset = len1 - olen;
    const int nw2 = (len2 + 31) >> 5;
    for (int k = (int)lane; k <= nw2; k += 32) {
        uint32_t lo = S.c2lo[k], hi = S.c2hi[k], v = S.c2v[k];
        if (k < nw2 && 32 * k < olen) {
            uint32_t bp = (uint32_t)(offset + 32 * k);
            uint32_t alo = fsr(S.r1lo, bp), ahi = fsr(S.r1hi, bp), an = fsr(S.r1n, bp), av = fsr(S.r1v, bp);
            uint32_t m = lowmask(olen - 32 * k);
            uint32_t mism = ((alo ^ lo) | (ahi ^ hi) | (an ^ S.c2n[k]) | (~av & ~an)) & m;
            uint32_t sel = mism & fsr(S.q1hi, bp) & S.q2lo[k];
            lo = (lo & ~sel) | (alo & sel);
            hi = (hi & ~sel) | (ahi & sel);
            v = (v & ~sel) | (av & sel);
        }
        S.xlo[k] = lo; S.xhi[k] = hi; S.xv[k] = v;
    }
    __syncwarp();
    const int mlen = offset + len2;
    const int nwm = (mlen + 31) >> 5;
    for (int w = (int)lane; w <= nwm; w += 32) {
        uint32_t lo = 0, hi = 0, v = 0;
        if (w < nwm) {
            int pos0 = 32 * w;
            if (pos0 < offset) {
                uint32_t m = lowmask(offset - pos0);
                lo = S.r1lo[w] & m; hi = S.r1hi[w] & m; v = S.r1v[w] & m;
            }
            int j0 = pos0 - offset;
            if (j0 > -32) {
                if (j0 < 0) {
                    lo |= S.xlo[0] << (-j0); hi |= S.xhi[0] << (-j0); v |= S.xv[0] << (-j0);
                } else {
                    lo |= fsr(S.xlo, (uint32_t)j0); hi |= fsr(S.xhi, (uint32_t)j0); v |= fsr(S.xv, (uint32_t)j0);
                }
            }
        }
        S.mlo[w] = lo; S.mhi[w] = hi; S.mv[w] = v;
    }
    __syncwarp();
    return mlen;
}

struct ScreenParams {
    GfDevIndex ix;
    GfDevBatch b;
    uint2* survivors;
    uint32_t survivors_cap;
    GfMapCounters* counters;
    int need_total, need_minor;
};

/* ---- warp-per-pair screen (reads longer than 256 bases): L2-resident working set ---------------------
 * Same conservative bound as screen_sequence (count2 <= T - c_d), but T and c_d are obtained without
 * touching the HBM table for every k-mer:
 *   1. seed: up to 8 spread k-mers are tested in the Bloom filter (L2); the first present one is looked up
 *      in the HBM table; a UNIQUE key gives a site, i.e. a diagonal d of the read against one gene strand.
 *   2. the whole read is compared with the 2-bit gene planes along d (32 bases per xor), a 16-wide run
 *      detector yields every offset whose 16-mer equals the gene window; where that window is an indexed
 *      voting site (count bits of the interleaved gene entries g_if / g_ir) the votes are known exactly: +nsites to T, +1 to c_d.
 *   3. every other valid even offset is probed in the filter: contributes an UPPER bound of its votes to T.
 * No false negatives anywhere => T_ub >= T and c_d <= true votes on d => the drop rule stays safe. */
__device__ __forceinline__ uint32_t run16(uint32_t w0, uint32_t w1) {
    /* bit b set <=> bits [b, b+16) of the 64-bit concatenation are all ones */
    unsigned long long x = (unsigned long long)w0 | ((unsigned long long)w1 << 32);
    x &= x >> 1;
    x &= x >> 2;
    x &= x >> 4;
    x &= x >> 8;
    return (uint32_t)x;
}
/* L2 residency: filter and gene planes are loaded with an evict_last policy, so the 6 GB of reads that stream
 * through the same L2 do not push them out */
__device__ __forceinline__ unsigned long long make_policy_keep() {
    unsigned long long pol;
    asm volatile("createpolicy.fractional.L2::evict_last.b64 %0, 1.0;" : "=l"(pol));
    return pol;
}
__device__ __forceinline__ unsigned long long ldg_filter(const unsigned long long* p, unsigned long long pol) {
    unsigned long long v;
    asm volatile("ld.global.nc.L1::no_allocate.L2::cache_hint.u64 %0, [%1], %2;" : "=l"(v) : "l"(p), "l"(pol));
    return v;
}

template <int MAXW>
__device__ __forceinline__ bool screen_sequence2(const GfDevIndex& ix, ScreenWarp<MAXW>& S, const uint32_t* lo,
                                                 const uint32_t* hi, const uint32_t* v, int len, int need_total,
                                                 int need_minor, unsigned long long* probes) {
    const uint32_t lane = gf_lane();
    const int nprobe = len >= 16 ? ((len - 16) >> 1) + 1 : 0;
    *probes += (unsigned long long)nprobe;
    if (need_total <= 0 || need_minor <= 0) return nprobe > 0 || need_total <= 0; /* degenerate params: keep */
    if (nprobe == 0) return false;
    const int nch = (len + 31) >> 5;
    const unsigned long long pol = make_policy_keep();

    /* 1. seed */
    uint32_t seed_val = GF_EMPTY_VAL;
    int seed_i = 0;
    {
        int i = (int)(((long long)(lane & 7u) * nprobe) >> 3) * 2;
        bool ok = lane < 8 && (fsr(v, (uint32_t)i) & 0xFFFFu) == 0xFFFFu;
        uint32_t key = ((fsr(hi, (uint32_t)i) & 0xFFFFu) << 16) | (fsr(lo, (uint32_t)i) & 0xFFFFu);
        bool present = false;
        if (ok) present = gf_filter_sites(ix, ldg_filter(ix.filter + gf_filter_word(key, ix.filter_words), pol), key, 2u) == 1u;
        uint32_t pm = __ballot_sync(FULL, present);
        while (pm) {
            int src = __ffs(pm) - 1;
            pm &= pm - 1;
            uint32_t k = __shfl_sync(FULL, key, src);
            uint32_t val = gf_table_find(ix, k);
            if (val != GF_EMPTY_VAL && (val >> 30) == GF_KIND_UNIQUE) {
                seed_val = val;
                seed_i = __shfl_sync(FULL, i, src);
                break;
            }
        }
    }

    int T = 0, c_d = 0;
    const uint32_t *plo = lo, *phi = hi, *pv = v; /* planes the "other" offsets are enumerated on */
    bool rc = false;
    uint32_t parity = 0x55555555u;
    if (seed_val != GF_EMPTY_VAL) {
        rc = (seed_val & GF_SITE_STRAND) != 0;
        const uint32_t goff = seed_val & GF_SITE_GOFF_MASK;
        uint32_t D;
        if (!rc) {
            D = goff - (uint32_t)seed_i;
        } else {
            /* compare revcomp(read) with the forward gene: read'[y] = comp(read[len-1-y]) */
            for (int k = (int)lane; k <= nch; k += 32) {
                uint32_t a = 0, b = 0, c = 0;
                if (k < nch) {
                    int pos = len - 32 * k - 32;
                    if (pos >= 0) { a = fsr(lo, (uint32_t)pos); b = fsr(hi, (uint32_t)pos); c = fsr(v, (uint32_t)pos); }
                    else if (pos > -32) { a = lo[0] << (-pos); b = hi[0] << (-pos); c = v[0] << (-pos); }
                    a = __brev(a); b = __brev(b); c = __brev(c);
                    a = (a ^ c) & c; /* complement = code ^ 1 on valid bases */
                }
                S.rlo[k] = a; S.rhi[k] = b; S.rv[k] = c;
            }
            plo = S.rlo; phi = S.rhi; pv = S.rv;
            D = goff + (uint32_t)seed_i - (uint32_t)len + 1u;
            if (len & 1) parity = 0xAAAAAAAAu; /* i' = len-16-i: even i <=> i' has the parity of len */
            __syncwarp();
        }
        /* 2. gene planes along the diagonal: one interleaved 32-byte entry {lo, hi, valid, count bits 0..2} per 32 positions */
        const uint32_t wbase = D >> 5, sh = D & 31u;
        const uint4* gi = reinterpret_cast<const uint4*>(rc ? ix.g_ir : ix.g_if);
        for (int k = (int)lane; k <= nch + 1; k += 32) {
            const uint4 a = __ldg(gi + 2ull * (wbase + k)), b = __ldg(gi + 2ull * (wbase + k) + 1);
            S.glo[k] = a.x; S.ghi[k] = a.y; S.gv[k] = a.z;
            S.gc[0][k] = a.w; S.gc[1][k] = b.x; S.gc[2][k] = b.y;
        }
        __syncwarp();
        for (int k = (int)lane; k <= nch; k += 32) {
            uint32_t e = 0;
            if (k < nch) {
                uint32_t glo = __funnelshift_r(S.glo[k], S.glo[k + 1], sh);
                uint32_t ghi = __funnelshift_r(S.ghi[k], S.ghi[k + 1], sh);
                uint32_t gvv = __funnelshift_r(S.gv[k], S.gv[k + 1], sh);
                e = ~((plo[k] ^ glo) | (phi[k] ^ ghi)) & pv[k] & gvv;
            }
            S.eq[k] = e;
        }
        __syncwarp();
        int c = 0, t = 0;
        for (int k = (int)lane; k < nch; k += 32) {
            uint32_t m = run16(S.eq[k], S.eq[k + 1]) & parity;
            uint32_t c0 = __funnelshift_r(S.gc[0][k], S.gc[0][k + 1], sh) & m;
            uint32_t c1 = __funnelshift_r(S.gc[1][k], S.gc[1][k + 1], sh) & m;
            uint32_t c2 = __funnelshift_r(S.gc[2][k], S.gc[2][k + 1], sh) & m;
            uint32_t h = c0 | c1 | c2; /* equal to an indexed, voting window: votes are known exactly */
            S.hit[k] = h;
            c += __popc(h);
            t += __popc(c0) + 2 * __popc(c1) + 4 * __popc(c2);
        }
        c_d = (int)__reduce_add_sync(FULL, (unsigned)c);
        T = (int)__reduce_add_sync(FULL, (unsigned)t);
    }
    __syncwarp();

    /* 3. every other valid even offset -> filter probe (upper bound of its votes) */
    int t_local = 0;
    if (seed_val == GF_EMPTY_VAL) {
        /* no diagonal: all even offsets, straight from the planes */
        for (int j0 = 0; j0 < nprobe; j0 += 64) {
            uint32_t key[2];
            unsigned long long w[2];
            bool ok[2];
#pragma unroll
            for (int u = 0; u < 2; u++) {
                int j = j0 + 32 * u + (int)lane;
                uint32_t off = 2u * (uint32_t)min(j, nprobe - 1);
                ok[u] = j < nprobe && (fsr(pv, off) & 0xFFFFu) == 0xFFFFu;
                key[u] = ((fsr(phi, off) & 0xFFFFu) << 16) | (fsr(plo, off) & 0xFFFFu);
                w[u] = 0;
                if (ok[u]) w[u] = ldg_filter(ix.filter + gf_filter_word(key[u], ix.filter_words), pol);
            }
#pragma unroll
            for (int u = 0; u < 2; u++)
                if (ok[u]) t_local += (int)gf_filter_sites(ix, w[u], key[u], ix.max_sites);
        }
    } else {
        /* offsets not explained by the diagonal: compact them into a list, then spread over the lanes */
        int total = 0;
        for (int k0 = 0; k0 < nch; k0 += 32) {
            int k = k0 + (int)lane;
            uint32_t om = 0;
            if (k < nch) om = run16(pv[k], pv[k + 1]) & parity & ~S.hit[k];
            if (__ballot_sync(FULL, om != 0u) == 0u) continue;
            int cnt = __popc(om);
            int incl = cnt;
            for (int o = 1; o < 32; o <<= 1) {
                int t = __shfl_up_sync(FULL, incl, o);
                if ((int)lane >= o) incl += t;
            }
            int pos = total + incl - cnt;
            while (om) {
                int b = __ffs(om) - 1;
                om &= om - 1;
                S.others[pos++] = (uint16_t)(32 * k + b);
            }
            total += __shfl_sync(FULL, incl, 31);
        }
        __syncwarp();
        for (int j = (int)lane; j - (int)lane < total; j += 32) {
            if (j < total) {
                uint32_t off = S.others[j];
                uint32_t kk = ((fsr(phi, off) & 0xFFFFu) << 16) | (fsr(plo, off) & 0xFFFFu);
                uint32_t key = rc ? gf_key_revcomp(kk) : kk;
                t_local += (int)gf_filter_sites(ix, ldg_filter(ix.filter + gf_filter_word(key, ix.filter_words), pol), key,
                                                ix.max_sites);
            }
        }
    }
    T += (int)__reduce_add_sync(FULL, (unsigned)t_local);
    return T >= need_total && (T - c_d) >= need_minor;
}

#include "gf_screen_tpp.cuh"
#include "gf_screen_split.cuh"

template <int MAXW, bool PAIRED>
__global__ void __launch_bounds__(256, 3) k_screen(ScreenParams P) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    ScreenWarp<MAXW>* Sall = reinterpret_cast<ScreenWarp<MAXW>*>(smem_raw);
    const uint32_t lane = gf_lane();
    const uint32_t warp_in_block = threadIdx.x >> 5;
    ScreenWarp<MAXW>& S = Sall[warp_in_block];
    const uint64_t n_warps = (uint64_t)gridDim.x * (blockDim.x >> 5);
    const uint64_t gwarp = (uint64_t)blockIdx.x * (blockDim.x >> 5) + warp_in_block;
    const GfDevBatch& B = P.b;

    unsigned long long c_seq = 0, c_probes = 0, c_bytes = 0, c_merged = 0;
    uint32_t err = 0;
    const uint8_t* const NOBOUND = reinterpret_cast<const uint8_t*>(~(uintptr_t)0);
    const uint8_t* bound1 = B.bytes1 ? B.seq1 + B.bytes1 : NOBOUND;
    const uint8_t* qbound1 = B.bytes1 ? B.qual1 + B.bytes1 : NOBOUND;
    const uint8_t* bound2 = (PAIRED && B.bytes2) ? B.seq2 + B.bytes2 : NOBOUND;
    const uint8_t* qbound2 = (PAIRED && B.bytes2) ? B.qual2 + B.bytes2 : NOBOUND;

    for (uint64_t p = gwarp; p < B.n; p += n_warps) {
        const uint64_t o1 = __ldg(B.s1 + p), e1 = __ldg(B.e1 + p);
        const int len1 = (int)(e1 - o1);
        const uint8_t* s1 = B.seq1 + (o1 - B.base1);
        const uint8_t* q1 = B.qual1 + (B.qs1[p] - B.base1);
        int len2 = 0;
        const uint8_t *s2 = nullptr, *q2 = nullptr;
        if (PAIRED) {
            const uint64_t o2 = __ldg(B.s2 + p), e2 = __ldg(B.e2 + p);
            len2 = (int)(e2 - o2);
            s2 = B.seq2 + (o2 - B.base2);
            q2 = B.qual2 + (B.qs2[p] - B.base2);
        }
        if (!record_ok(o1, e1, B.base1, B.bytes1, 32 * MAXW) ||
            (PAIRED && !record_ok(__ldg(B.s2 + p), __ldg(B.e2 + p), B.base2, B.bytes2, 32 * MAXW))) {
            err |= 1u;
            continue;
        }
        __syncwarp();
        planes_r1<MAXW>(S, s1, q1, len1, B.seq1, bound1, B.qual1, qbound1);
        int olen = -1, diff = 0;
        if (PAIRED) {
            planes_r2<MAXW>(S, s2, q2, len2, B.seq2, bound2, B.qual2, qbound2);
            olen = find_overlap<MAXW>(S, len1, len2, &diff);
        }
        __syncwarp();
        /* merged: only the merged read is searched (pescanner.rs:446-470); else R1, then R2 (:472-514) */
        int mlen = 0;
        if (olen >= 0) {
            mlen = build_merged<MAXW>(S, len1, len2, olen);
            c_merged++;
        }
        const int nseq = olen >= 0 ? 1 : (PAIRED ? 2 : 1);
        for (int sq = 0; sq < nseq; sq++) {
            const uint32_t *plo = S.mlo, *phi = S.mhi, *pv = S.mv;
            int len = mlen;
            uint32_t meta = 0u | ((uint32_t)max(olen, 0) << 2) | ((uint32_t)diff << 14);
            if (olen < 0) {
                if (sq == 0) {
                    plo = S.r1lo; phi = S.r1hi; pv = S.r1v;
                    len = len1;
                    meta = 1u;
                } else {
                    plo = S.f2lo; phi = S.f2hi; pv = S.f2v;
                    len = len2;
                    meta = 2u;
                }
            }
            c_seq++;
            c_bytes += (unsigned long long)len;
            const bool sv = screen_sequence2<MAXW>(P.ix, S, plo, phi, pv, len, P.need_total, P.need_minor, &c_probes);
            if (sv && lane == 0) {
                uint32_t slot = atomicAdd(&P.counters->n_survivors, 1u);
                if (slot < P.survivors_cap) P.survivors[slot] = make_uint2((uint32_t)p, meta);
                else err |= 2u;
            }
        }
    }
    if (lane == 0) {
        if (c_seq) atomicAdd(&P.counters->n_sequences, c_seq);
        if (c_probes) atomicAdd(&P.counters->n_probes, c_probes);
        if (c_bytes) atomicAdd(&P.counters->seq_bytes, c_bytes);
        if (c_merged) atomicAdd(&P.counters->n_merged, c_merged);
    }
    err = __reduce_or_sync(FULL, err);
    if (err && lane == 0) atomicOr(&P.counters->error_flags, err);
}

/* parity hook: fast_merge only */
template <int MAXW>
__global__ void __launch_bounds__(256) k_merge_only(GfDevBatch B, gf_merge_info* __restrict__ out, GfMapCounters* counters) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    ScreenWarp<MAXW>* Sall = reinterpret_cast<ScreenWarp<MAXW>*>(smem_raw);
    const uint32_t lane = gf_lane();
    ScreenWarp<MAXW>& S = Sall[threadIdx.x >> 5];
    const uint64_t n_warps = (uint64_t)gridDim.x * (blockDim.x >> 5);
    for (uint64_t p = (uint64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5); p < B.n; p += n_warps) {
        const uint64_t o1 = B.s1[p], o2 = B.s2[p];
        const int len1 = (int)(B.e1[p] - o1), len2 = (int)(B.e2[p] - o2);
        if (len1 > 32 * MAXW || len2 > 32 * MAXW) {
            if (lane == 0) atomicOr(&counters->error_flags, 1u);
            continue;
        }
        __syncwarp();
        planes_r1<MAXW>(S, B.seq1 + (o1 - B.base1), B.qual1 + (B.qs1[p] - B.base1), len1, B.seq1, B.seq1 + B.bytes1, B.qual1,
                        B.qual1 + B.bytes1);
        planes_r2<MAXW>(S, B.seq2 + (o2 - B.base2), B.qual2 + (B.qs2[p] - B.base2), len2, B.seq2, B.seq2 + B.bytes2, B.qual2,
                        B.qual2 + B.bytes2);
        __syncwarp();
        int diff = 0;
        int olen = find_overlap<MAXW>(S, len1, len2, &diff);
        if (lane == 0) {
            gf_merge_info mi;
            mi.merged = olen >= 0;
            mi.olen = olen >= 0 ? olen : 0;
            mi.diff = diff;
            mi.merged_len = olen >= 0 ? len1 - olen + len2 : 0;
            out[p] = mi;
        }
    }
}

/* ------------------------------------------------------------------------------------------------ */
/* raw (ASCII) sequence reconstruction for the exact / verify kernels                                */

/* Loads the sequence a survivor stands for into `seq` (shared memory, `cap` bytes), returns its length, or -1 without
 * writing anything when the record offsets are inconsistent (outside the arena, negative or longer than the buffer).
 * source 0 = merged read (literal read.rs:369-428 given the overlap length), 1 = R1, 2 = R2. */
__device__ int load_sequence(const GfDevBatch& B, uint32_t pair, uint32_t source, int olen, uint8_t* seq, int cap) {
    const uint32_t lane = gf_lane();
    const uint64_t o1 = B.s1[pair], e1 = B.e1[pair];
    if (!record_ok(o1, e1, B.base1, B.bytes1, cap)) return -1;
    const int len1 = (int)(e1 - o1);
    const uint8_t* s1 = B.seq1 + (o1 - B.base1);
    int len;
    if (source == 1) {
        for (int j = (int)lane; j < len1; j += 32) seq[j] = s1[j];
        len = len1;
    } else {
        if (!B.seq2) return -1;
        const uint64_t o2 = B.s2[pair], e2 = B.e2[pair];
        if (!record_ok(o2, e2, B.base2, B.bytes2, cap)) return -1;
        const int len2 = (int)(e2 - o2);
        const uint8_t* s2 = B.seq2 + (o2 - B.base2);
        if (source == 2) {
            for (int j = (int)lane; j < len2; j += 32) seq[j] = s2[j];
            len = len2;
        } else {
            const int offset = len1 - olen;
            if (olen < 0 || offset < 0 || olen > len2 || offset + len2 > cap) return -1;
            const uint8_t* q1 = B.qual1 + (B.qs1[pair] - B.base1);
            const uint8_t* q2 = B.qual2 + (B.qs2[pair] - B.base2);
            for (int j = (int)lane; j < offset; j += 32) seq[j] = s1[j];
            for (int i = (int)lane; i < len2; i += 32) {
                uint8_t c2 = gf_complement_ascii(s2[len2 - 1 - i]);
                uint8_t ch = c2;
                if (i < olen) {
                    uint8_t c1 = s1[offset + i];
                    if (c1 != c2 && q1[offset + i] >= '?' && q2[len2 - 1 - i] <= '0') ch = c1;
                }
                seq[offset + i] = ch;
            }
            len = offset + len2;
        }
    }
    __syncwarp();
    return len;
}
/* SequenceRead::reverse_complement (read.rs:243-261) in place */
__device__ void revcomp_inplace(uint8_t* seq, int len) {
    const uint32_t lane = gf_lane();
    for (int j = (int)lane; 2 * j < len; j += 32) {
        int k = len - 1 - j;
        uint8_t a = seq[j], b = seq[k];
        seq[j] = gf_complement_ascii(b);
        if (k != j) seq[k] = gf_complement_ascii(a);
    }
    __syncwarp();
}

/* ------------------------------------------------------------------------------------------------ */
/* k_exact                                                                                           */
constexpr int EX_SEQ_CAP = 2048 + 64;
constexpr int EX_WARPS = 4;
constexpr long long EX_EMPTY_KEY = LLONG_MIN;

/* per-warp state of the exact path.  Two sizes: reads of up to 256 bases (merged <= 482) use a 256-slot vote table and
 * 544-byte sequence buffers, 4.7 KB per warp, so that 40+ warps are resident per SM (the kernel is a chain of dependent
 * HBM / shared-memory round trips: throughput = survivors in flight); longer reads use 1024 slots and 2112 bytes.  A read
 * whose votes do not fit the shared table (distinct diagonals > 3/4 of the slots: repeats) redoes pass 1 with the warp's
 * table in global memory (GT slots >= the most votes a read of that class can cast). */
template <int TBL, int CAP, int GT>
struct ExactWarpT {
    static constexpr int TBL_SLOTS = TBL, SEQ_CAP = CAP, GLOBAL_SLOTS = GT;
    long long tkeys[TBL];
    int tcnt[TBL];
    uint8_t seq[CAP];
    uint8_t flag[CAP];
    uint32_t plo[CAP / 32 + 2], phi[CAP / 32 + 2], pv[CAP / 32 + 2]; /* the sequence as code / validity bit-planes */
    uint32_t m3[CAP / 32 + 2], m2[CAP / 32 + 2];                     /* mask == MATCH_TOP / == MATCH_SECOND per position */
    int distinct;  /* keys in the shared table */
    int overflow;  /* the shared table is too small for this read */
};
using ExactWarpSmall = ExactWarpT<256, 544, 2048>;
using ExactWarpLarge = ExactWarpT<1024, EX_SEQ_CAP, 8192>;

struct ExactParams {
    GfDevIndex ix;
    GfDevBatch b;
    const uint2* survivors;
    uint32_t survivors_cap;
    GfMapCounters* counters;
    gf_match* out;
    unsigned long long out_cap;
    unsigned long long* n_out;
    long long* gtbl_keys; /* [n_warps_total][GLOBAL_SLOTS] */
    int* gtbl_cnt;
};

struct Top2 { long long k1, k2; int c1, c2; };

/* "better" in the order the reference's ascending BTreeMap scan with strict '>' produces
 * (indexer.rs:336-346): higher count first, ties -> smaller key */
__device__ __forceinline__ bool vote_better(int ca, long long ka, int cb, long long kb) {
    return ca > cb || (ca == cb && ca > 0 && ka < kb);
}
__device__ __forceinline__ void vote_insert(long long* tk, int* tc, uint32_t tmask, long long g, int* distinct, int limit,
                                            int* overflow) {
    if (g == 0) return; /* key 0 is the "no hit" bucket and is never a candidate (k != 0, indexer.rs:337) */
    uint32_t h = (uint32_t)(((unsigned long long)g * 0x9E3779B97F4A7C15ull) >> 40) & tmask;
    for (uint32_t tries = 0; tries <= tmask; tries++) {
        long long old = (long long)atomicCAS((unsigned long long*)&tk[h], (unsigned long long)EX_EMPTY_KEY,
                                             (unsigned long long)g);
        if (old == EX_EMPTY_KEY || old == g) {
            atomicAdd(&tc[h], 1);
            if (old == EX_EMPTY_KEY && atomicAdd(distinct, 1) >= limit) *overflow = 1;
            return;
        }
        h = (h + 1) & tmask;
    }
    *overflow = 1; /* table full */
}
/* W.seq (ASCII, len bytes) -> bit-planes: one ballot per plane and 32 bases (make_kmer_bytes: upper-case ACGT only,
 * indexer.rs:888-904); one zero word behind the last base */
template <class EW>
__device__ void exact_planes(EW& W, int len) {
    const uint32_t lane = gf_lane();
    const int nw = (len + 31) >> 5;
    for (int w = 0; w <= nw; w++) {
        const int j = 32 * w + (int)lane;
        const uint32_t c = j < len ? W.seq[j] : 0u;
        const bool ok = gf_is_acgt_upper(c);
        const uint32_t v = __ballot_sync(FULL, ok), lo = __ballot_sync(FULL, ok && gf_code_lo(c)), hi = __ballot_sync(FULL, ok && gf_code_hi(c));
        if (lane == 0) { W.pv[w] = v; W.plo[w] = lo; W.phi[w] = hi; }
    }
    __syncwarp();
}
/* ask for the table bucket of the k-mer at offset i (L2 prefetch): the lookups of one read are independent of each other, the
 * loop that makes them is a chain of dependent loads per offset (bucket -> dupe list -> site decode) with side effects, so the
 * compiler cannot overlap them — all buckets of a pass are requested up front instead */
template <class EW>
__device__ __forceinline__ void prefetch_site_bucket(const GfDevIndex& ix, const EW& W, int i) {
    const uint32_t bp = (uint32_t)i;
    if ((fsr(W.pv, bp) & 0xFFFFu) != 0xFFFFu) return;
    const uint32_t key = ((fsr(W.phi, bp) & 0xFFFFu) << 16) | (fsr(W.plo, bp) & 0xFFFFu);
    asm volatile("prefetch.global.L2 [%0];" ::"l"(ix.table + 2ull * gf_home_bucket(key, ix.bucket_shift)));
}
/* visit every (contig, position) the k-mer at offset i maps to */
template <class EW, class F>
__device__ __forceinline__ void for_each_site(const GfDevIndex& ix, const EW& W, int i, F f) {
    const uint32_t bp = (uint32_t)i;
    if ((fsr(W.pv, bp) & 0xFFFFu) != 0xFFFFu) return;
    const uint32_t key = ((fsr(W.phi, bp) & 0xFFFFu) << 16) | (fsr(W.plo, bp) & 0xFFFFu);
    uint32_t val = gf_table_find(ix, key);
    if (val == GF_EMPTY_VAL) return;
    uint32_t kind = val >> 30;
    if (kind == GF_KIND_UNIQUE) {
        int32_t c, p;
        gf_site_decode(ix, val & 0x3FFFFFFFu, &c, &p);
        f(c, p);
    } else if (kind == GF_KIND_NORMAL) {
        uint32_t cnt = val & 7u, off = (val >> 3) & 0x07FFFFFFu;
        for (uint32_t j = 0; j < cnt; j++) {
            int32_t c, p;
            gf_site_decode(ix, __ldg(ix.dupes + off + j), &c, &p);
            f(c, p);
        }
    }
}

/* next set bit of plane `pl` (nw words) at position >= from, or `none` */
__device__ __forceinline__ int next_bit(const uint32_t* pl, int nw, int from, int none) {
    if (from < 0) from = 0;
    int w = from >> 5;
    if (w >= nw) return none;
    uint32_t x = pl[w] & (0xFFFFFFFFu << (from & 31));
    while (!x) {
        if (++w >= nw) return none;
        x = pl[w];
    }
    return 32 * w + __ffs(x) - 1;
}
__device__ __forceinline__ int next_zero(const uint32_t* pl, int nw, int from, int none) {
    int w = from >> 5;
    if (w >= nw) return none;
    uint32_t x = ~pl[w] & (0xFFFFFFFFu << (from & 31));
    while (!x) {
        if (++w >= nw) return none;
        x = ~pl[w];
    }
    return 32 * w + __ffs(x) - 1;
}

struct SegResult { int n; int s0, e0, s1, e1; long long gp0, gp1; }; /* entries in TOP, SECOND order */

/* Indexer::map_read (indexer.rs:252-538) on the ASCII sequence in W.seq.  All lanes return the same result. */
template <class EW>
__device__ SegResult exact_map_read(const GfDevIndex& ix, EW& W, int len, long long* gkeys, int* gcnt, bool prefetch) {
    const uint32_t lane = gf_lane();
    SegResult R;
    R.n = 0; R.s0 = R.e0 = R.s1 = R.e1 = 0; R.gp0 = R.gp1 = 0;
    if (len < 16) return R;
    exact_planes(W, len);
    const int nprobe = ((len - 16) >> 1) + 1;
    long long* tk = W.tkeys;
    int* tc = W.tcnt;
    uint32_t tsize = EW::TBL_SLOTS;
    /* first pass: every 2nd offset votes for pack(contig, position - i)  (:277-321); shared table first, the global
     * one when the read casts more distinct votes than 3/4 of the shared slots */
    if (prefetch)
        for (int j = (int)lane; j < nprobe; j += 32) prefetch_site_bucket(ix, W, 2 * j);
    for (int round = 0; round < 2; round++) {
        const uint32_t tmask = tsize - 1;
        for (uint32_t s = lane; s < tsize; s += 32) { tk[s] = EX_EMPTY_KEY; tc[s] = 0; }
        if (lane == 0) { W.distinct = 0; W.overflow = 0; }
        __syncwarp();
        const int limit = (int)(tsize - tsize / 4);
        for (int j = (int)lane; j < nprobe; j += 32) {
            int i = 2 * j;
            for_each_site(ix, W, i, [&](int32_t c, int32_t p) {
                vote_insert(tk, tc, tmask, gf_gp_pack(c, p - i), &W.distinct, limit, &W.overflow);
            });
        }
        __syncwarp();
        if (!W.overflow || round == 1) break;
        __syncwarp();
        tk = gkeys; tc = gcnt; tsize = EW::GLOBAL_SLOTS;
    }
    /* top-2 (:324-346) */
    long long k1 = 0, k2 = 0;
    int c1 = 0, c2 = 0;
    for (uint32_t s = lane; s < tsize; s += 32) {
        long long k = tk[s];
        if (k == EX_EMPTY_KEY) continue;
        int c = tc[s];
        if (vote_better(c, k, c1, k1)) { k2 = k1; c2 = c1; k1 = k; c1 = c; }
        else if (vote_better(c, k, c2, k2)) { k2 = k; c2 = c; }
    }
    long long bk = k1; int bc = c1;
    for (int o = 16; o > 0; o >>= 1) {
        long long ok_ = __shfl_xor_sync(FULL, bk, o);
        int oc = __shfl_xor_sync(FULL, bc, o);
        if (vote_better(oc, ok_, bc, bk)) { bk = ok_; bc = oc; }
    }
    long long sk = (k1 == bk && c1 == bc) ? k2 : k1;
    int sc = (k1 == bk && c1 == bc) ? c2 : c1;
    for (int o = 16; o > 0; o >>= 1) {
        long long ok_ = __shfl_xor_sync(FULL, sk, o);
        int oc = __shfl_xor_sync(FULL, sc, o);
        if (vote_better(oc, ok_, sc, sk)) { sk = ok_; sc = oc; }
    }
    const long long gp1 = bc > 0 ? bk : 0, gp2 = sc > 0 ? sk : 0;
    const int count1 = bc, count2 = sc;
    if (count1 * 2 < ix.major_req || count2 * 2 < ix.minor_req) return R; /* :353-360 */

    /* second pass: per-offset flag, then mask[p] = max over the 16 windows covering p  (:362-521, :716-732) */
    const int nwin = len - 15;
    if (prefetch)
        for (int i = (int)lane; i < nwin; i += 32)
            if (i & 1) prefetch_site_bucket(ix, W, i); /* (the even offsets were fetched by pass 1) */
    for (int i = (int)lane; i < nwin; i += 32) {
        int f = 0;
        for_each_site(ix, W, i, [&](int32_t c, int32_t p) {
            long long g = gf_gp_pack(c, p - i);
            long long d1 = g - gp1, d2 = g - gp2;
            if (d1 < 0) d1 = -d1;
            if (d2 < 0) d2 = -d2;
            int ff = d1 <= 1 ? 3 : (d2 <= 1 ? 2 : (g == 0 ? 1 : 0));
            f = max(f, ff);
        });
        W.flag[i] = (uint8_t)f;
    }
    __syncwarp();
    /* mask[p] = max flag of the (<= 16) windows covering p, kept as two planes: == MATCH_TOP (3), == MATCH_SECOND (2) */
    int mism = 0;
    const int nwm = (len + 31) >> 5;
    for (int w = 0; w < nwm; w++) {
        const int p = 32 * w + (int)lane;
        int m = 0;
        if (p < len) {
            const int lo = max(0, p - 15), hi = min(p, nwin - 1);
            for (int i = lo; i <= hi; i++) m = max(m, (int)W.flag[i]);
            if (m <= 1) mism++; /* MATCH_NONE or MATCH_UNKNOWN (:523-528) */
        }
        const uint32_t b3 = __ballot_sync(FULL, m == 3), b2 = __ballot_sync(FULL, m == 2);
        if (lane == 0) { W.m3[w] = b3; W.m2[w] = b2; }
    }
    mism = (int)__reduce_add_sync(FULL, (unsigned)mism);
    __syncwarp();
    if (mism > ix.mismatch_thr) return R; /* :530-535 */

    /* segment_mask (:616-679): every start s < len - 1 with mask[s] == target is tried, the walk tolerates gaps of up to 9
     * lower values and stops at any higher one; the longest run wins, the first one on ties (strict '>'), and only if
     * end - start > 20.  The walk is memoryless, so the starts fall into disjoint chains of target positions (linked when at
     * most 9 lower values and nothing higher lie between) and only a chain's first position can win: one pass over the
     * chains, jumping from gap to gap with bit scans. */
    for (int t = 0; t < 2; t++) {
        const uint32_t* T = t == 0 ? W.m3 : W.m2;
        const uint32_t* H = t == 0 ? nullptr : W.m3; /* values above the target */
        int best_len = 0, best_s = 0;
        int s0 = next_bit(T, nwm, 0, -1);
        while (s0 >= 0 && s0 < len - 1) {
            int pos = s0, last_t;
            for (;;) {
                const int run_end = min(next_zero(T, nwm, pos, len), len); /* pos .. run_end - 1 are target */
                last_t = run_end - 1;
                const int nt = next_bit(T, nwm, run_end, -1);
                if (nt < 0 || nt - run_end > 9) break;                       /* gap of >= 10 lower values: the walk gives up */
                if (H && next_bit(H, nwm, run_end, len) < nt) break;         /* a higher value first: break (:648-650) */
                pos = nt;
            }
            if (last_t - s0 > best_len) { best_len = last_t - s0; best_s = s0; }
            s0 = next_bit(T, nwm, last_t + 1, -1);
        }
        if (best_len > 20) {
            if (R.n == 0) { R.s0 = best_s; R.e0 = best_s + best_len; R.gp0 = t == 0 ? gp1 : gp2; }
            else { R.s1 = best_s; R.e1 = best_s + best_len; R.gp1 = t == 0 ? gp1 : gp2; }
            R.n++;
        }
    }
    return R;
}

/* i64_to_gp (indexer.rs:708-714) */
__device__ __forceinline__ void gp_unpack(long long v, int32_t* contig, int32_t* position) {
    *contig = (int32_t)(int16_t)(v >> 32);
    *position = (int32_t)(uint32_t)(v & 0xFFFFFFFFll);
}

/* Indexer::in_required_direction (indexer.rs:541-608), left/right already ordered by seq_start */
__device__ bool in_required_direction(const GfDevIndex& ix, int32_t lc, int32_t lp, int32_t rc, int32_t rp) {
    if (lp > 0 && rp > 0) return true;
    if (lp < 0 && rp < 0) return false;
    bool lrev = ix.gene_rev[lc] != 0, rrev = ix.gene_rev[rc] != 0;
    if (lrev && !rrev) return false;
    if (!lrev && rrev) return true;
    if (lc < rc) return true;
    return false; /* :597-599 compares left with left -> never true */
}

template <class EW>
__global__ void __launch_bounds__(EX_WARPS * 32) k_exact(ExactParams P) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    EW* Wall = reinterpret_cast<EW*>(smem_raw);
    const uint32_t lane = gf_lane();
    const uint32_t wib = threadIdx.x >> 5;
    EW& W = Wall[wib];
    const uint64_t gwarp = (uint64_t)blockIdx.x * EX_WARPS + wib;
    const uint64_t n_warps = (uint64_t)gridDim.x * EX_WARPS;
    long long* gkeys = P.gtbl_keys + gwarp * EW::GLOBAL_SLOTS;
    int* gcnt = P.gtbl_cnt + gwarp * EW::GLOBAL_SLOTS;
    const uint32_t n_surv = min(P.counters->n_survivors, P.survivors_cap);
    /* many survivors per resident warp (repeat-rich panels): the kernel's rate is lookups in flight, so every pass asks for all
     * its table buckets first (35 -> 26 ms for 2.5 M survivors); with a few waves of survivors the extra pass only delays each
     * warp's own chain (+15 % measured), so it is left out */
    const bool prefetch = (uint64_t)n_surv > 8 * n_warps;

    for (uint64_t sidx = gwarp; sidx < n_surv; sidx += n_warps) {
        const uint2 sv = P.survivors[sidx];
        const uint32_t pair = sv.x, source = sv.y & 3u;
        const int olen = (int)((sv.y >> 2) & 0xFFFu), diff = (int)((sv.y >> 14) & 3u);
        __syncwarp();
        const int len = load_sequence(P.b, pair, source, olen, W.seq, EW::SEQ_CAP - 16);
        if (len < 0) { if (lane == 0) atomicOr(&P.counters->error_flags, 1u); continue; }
        if (lane == 0) for (int k = 0; k < 16; k++) W.seq[len + k] = 0;
        __syncwarp();
        for (int attempt = 0; attempt < 2; attempt++) {
            SegResult R = exact_map_read(P.ix, W, len, gkeys, gcnt, prefetch);
            if (R.n < 2) break; /* mapable = false (fusion_mapper.rs:107-113): no retry */
            /* order by seq_start (fusion_mapper.rs:163-165 / indexer.rs:549-551) */
            int ls = R.s0, le = R.e0, rs = R.s1, re = R.e1;
            long long lg = R.gp0, rg = R.gp1;
            if (ls > rs) { int t; t = ls; ls = rs; rs = t; t = le; le = re; re = t; long long tg = lg; lg = rg; rg = tg; }
            int32_t lc, lp, rc, rp;
            gp_unpack(lg, &lc, &lp);
            gp_unpack(rg, &rc, &rp);
            (void)re; (void)ls;
            if (in_required_direction(P.ix, lc, lp, rc, rp)) {
                /* make_match (fusion_mapper.rs:154-194) */
                int read_break = (le + rs) / 2;
                if (lane == 0) {
                    unsigned long long slot = atomicAdd(P.n_out, 1ull);
                    if (slot < P.out_cap) {
                        gf_match m;
                        m.pair_idx = P.b.pair_base + pair;
                        m.read_break = read_break;
                        m.l_pos = lp + read_break;
                        m.r_pos = rp + read_break + 1;
                        m.gap = rs - le - 1;
                        m.l_dist = 0;
                        m.r_dist = 0;
                        m.seq_len = len;
                        m.l_contig = (int16_t)lc;
                        m.r_contig = (int16_t)rc;
                        m.merge_olen = source == 0 ? (int16_t)olen : (int16_t)-1;
                        m.merge_diff = source == 0 ? (int16_t)diff : (int16_t)0;
                        m.source = (uint8_t)source;
                        m.used_rc = (uint8_t)attempt;
                        /* set_reversed(true) only on the R1/R2 retries (pescanner.rs:483,506), never merged (:455-469) */
                        m.reversed = (uint8_t)(attempt == 1 && source != 0);
                        m.filter_flags = 0;
                        P.out[slot] = m;
                    }
                }
                break;
            }
            if (attempt == 0) {
                revcomp_inplace(W.seq, len); /* "else if mapable" retry on the reverse complement */
            }
        }
    }
}

/* ------------------------------------------------------------------------------------------------ */
/* k_verify: calc_distance / calc_ed / edit_distance                                                 */
constexpr int VF_WARPS = 4;

struct VerifyParams {
    GfDevIndex ix;
    GfDevBatch b;
    GfMapCounters* counters;
    gf_match* out;
    unsigned long long out_cap;
    const unsigned long long* n_out;
};

/* Levenshtein distance of pattern a[0..m) and text b[0..m) (equal lengths, m >= 1, m <= 2048), the
 * recurrences of edit_distance_bpv (edit_distance.rs:12-92) with block r in lane r.  `a_rc`: the pattern is
 * the reverse complement of part[0..m) (calc_ed start<0 branch, fusion_mapper.rs:237-246). */
__device__ int warp_edit_distance(const uint8_t* part, int m, bool a_rc, const uint8_t* __restrict__ text) {
    const uint32_t lane = gf_lane();
    const int nb = ((m - 1) >> 6) + 1, tmax = nb - 1, tlen = m - 64 * tmax;
    auto a_at = [&](int k) -> uint8_t { return a_rc ? gf_complement_ascii(part[m - 1 - k]) : part[k]; };
    unsigned long long pA = 0, pC = 0, pG = 0, pT = 0, pN = 0, pO = 0; /* match masks of this lane's block */
    if ((int)lane < nb) {
        for (int j = 0; j < 64; j++) {
            int k = 64 * (int)lane + j;
            if (k >= m) break;
            uint8_t ch = a_at(k);
            unsigned long long bit = 1ull << j;
            if (ch == 'A') pA |= bit; else if (ch == 'C') pC |= bit; else if (ch == 'G') pG |= bit;
            else if (ch == 'T') pT |= bit; else if (ch == 'N') pN |= bit; else pO |= bit;
        }
    }
    unsigned long long vp = 0, vn = 0;
    if ((int)lane < tmax) vp = ~0ull;
    else if ((int)lane == tmax) vp = tlen >= 64 ? ~0ull : ((1ull << tlen) - 1ull);
    const unsigned long long top = 1ull << (tlen - 1), lmb = 1ull << 63;
    int d = m;
    uint32_t hp_out = 0, hn_out = 0;
    const int steps = m + nb - 1;
    for (int t = 0; t < steps; t++) {
        uint32_t hp_in = __shfl_up_sync(FULL, hp_out, 1);
        uint32_t hn_in = __shfl_up_sync(FULL, hn_out, 1);
        int j = t - (int)lane;
        if ((int)lane < nb && j >= 0 && j < m) {
            uint8_t ch = __ldg(text + j);
            unsigned long long x;
            if (ch == 'A') x = pA; else if (ch == 'C') x = pC; else if (ch == 'G') x = pG;
            else if (ch == 'T') x = pT; else if (ch == 'N') x = pN;
            else {
                x = 0;
                if (pO) for (int q = 0; q < 64; q++) { int k = 64 * (int)lane + q; if (k < m && ((pO >> q) & 1ull) && a_at(k) == ch) x |= 1ull << q; }
            }
            if (lane > 0 && hn_in) x |= 1ull;
            unsigned long long d0 = (((x & vp) + vp) ^ vp) | x | vn;
            unsigned long long hp = vn | ~(d0 | vp);
            unsigned long long hn = d0 & vp;
            unsigned long long x2 = hp << 1;
            if (lane == 0 || hp_in) x2 |= 1ull;
            vp = (hn << 1) | ~(d0 | x2);
            if (lane > 0 && hn_in) vp |= 1ull;
            vn = d0 & x2;
            hp_out = (hp & lmb) ? 1u : 0u;
            hn_out = (hn & lmb) ? 1u : 0u;
            if ((int)lane == tmax) {
                if (hp & top) d++;
                else if (hn & top) d--;
            }
        }
    }
    return __shfl_sync(FULL, d, tmax);
}

/* 32 / G equal-length edit distances at once, one per group of G consecutive lanes: the same systolic recurrences as
 * warp_edit_distance with the block index = lane % G, so 32 / G jobs cost max(m) + blocks steps instead of their sum — and
 * 32 / G times fewer warp instructions per job than one job per warp (ncu, round 2: a candidate's two distances kept 7.5 of
 * 32 lanes busy and k_verify was issue bound at 13.8 k warp instructions per candidate).  Every lane of a group passes the
 * group's job; needs <= G blocks (m <= 64 G); m == 0 = no job (result 0). */
template <int G>
__device__ int group_edit_distance(const uint8_t* part, int m, bool a_rc, const uint8_t* __restrict__ text) {
    const uint32_t lane = gf_lane(), hl = lane % G;
    const int nb = m > 0 ? ((m - 1) >> 6) + 1 : 0, tmax = nb - 1, tlen = m - 64 * tmax;
    auto a_at = [&](int k) -> uint8_t { return a_rc ? gf_complement_ascii(part[m - 1 - k]) : part[k]; };
    unsigned long long pA = 0, pC = 0, pG = 0, pT = 0, pN = 0, pO = 0;
    if ((int)hl < nb) {
        for (int j = 0; j < 64; j++) {
            int k = 64 * (int)hl + j;
            if (k >= m) break;
            uint8_t ch = a_at(k);
            unsigned long long bit = 1ull << j;
            if (ch == 'A') pA |= bit; else if (ch == 'C') pC |= bit; else if (ch == 'G') pG |= bit;
            else if (ch == 'T') pT |= bit; else if (ch == 'N') pN |= bit; else pO |= bit;
        }
    }
    unsigned long long vp = 0, vn = 0;
    if ((int)hl < tmax) vp = ~0ull;
    else if ((int)hl == tmax) vp = tlen >= 64 ? ~0ull : ((1ull << tlen) - 1ull);
    const unsigned long long top = nb > 0 ? 1ull << (tlen - 1) : 0ull, lmb = 1ull << 63;
    int d = m;
    uint32_t hp_out = 0, hn_out = 0;
    const int my_steps = m > 0 ? m + nb - 1 : 0;
    const int steps = (int)__reduce_max_sync(FULL, (unsigned)my_steps);
    for (int t = 0; t < steps; t++) {
        uint32_t hp_in = __shfl_up_sync(FULL, hp_out, 1, G);
        uint32_t hn_in = __shfl_up_sync(FULL, hn_out, 1, G);
        int j = t - (int)hl;
        if ((int)hl < nb && j >= 0 && j < m) {
            uint8_t ch = __ldg(text + j);
            unsigned long long x;
            if (ch == 'A') x = pA; else if (ch == 'C') x = pC; else if (ch == 'G') x = pG;
            else if (ch == 'T') x = pT; else if (ch == 'N') x = pN;
            else {
                x = 0;
                if (pO) for (int q = 0; q < 64; q++) { int k = 64 * (int)hl + q; if (k < m && ((pO >> q) & 1ull) && a_at(k) == ch) x |= 1ull << q; }
            }
            if (hl > 0 && hn_in) x |= 1ull;
            unsigned long long dd0 = (((x & vp) + vp) ^ vp) | x | vn;
            unsigned long long hp = vn | ~(dd0 | vp);
            unsigned long long hn = dd0 & vp;
            unsigned long long x2 = hp << 1;
            if (hl == 0 || hp_in) x2 |= 1ull;
            vp = (hn << 1) | ~(dd0 | x2);
            if (hl > 0 && hn_in) vp |= 1ull;
            vn = dd0 & x2;
            hp_out = (hp & lmb) ? 1u : 0u;
            hn_out = (hn & lmb) ? 1u : 0u;
            if ((int)hl == tmax) {
                if (hp & top) d++;
                else if (hn & top) d--;
            }
        }
    }
    const int r = __shfl_sync(FULL, d, (int)(lane - hl) + (tmax > 0 ? tmax : 0));
    return m > 0 ? r : 0;
}

/* the checks of FusionMapper::calc_ed (fusion_mapper.rs:224-251) that come before the edit distance: returns true when
 * `*res` already is the answer (-1 / -2 sentinels, empty side), otherwise the equal-length job (text, rc) */
__device__ bool calc_ed_setup(const GfDevIndex& ix, int plen, int32_t contig, int32_t start, int32_t end, int* res,
                              const uint8_t** text, bool* rc, uint32_t* panic) {
    if ((start >= 0 && end <= 0) || (start <= 0 && end >= 0)) { *res = -1; return true; }
    const int32_t glen = (int32_t)ix.gene_len[contig];
    const int32_t as = start < 0 ? -start : start, ae = end < 0 ? -end : end;
    if (as >= glen || ae >= glen) { *res = -2; return true; }
    *rc = start < 0;
    if (*rc) { int32_t tmp = start; start = -end; end = -tmp; }
    const int reflen = end - start + 1;
    if (plen == 0) { *res = reflen; return true; }      /* edit_distance: asize == 0 -> bsize */
    if (reflen == 0) { *res = plen; return true; }
    if (((plen - 1) >> 6) + 1 > 10) *panic = 1; /* the reference falls into its panicking DP branch (>640) */
    *text = ix.gene_ascii + ix.gene_start[contig] + start;
    return false;
}

constexpr int VG_CAND = 4; /* candidates a warp verifies together */
template <int CAP>
struct VerifyGrpWarp {
    uint8_t seq[VG_CAND][CAP];
    const uint8_t* text[2 * VG_CAND]; /* per job (2 c = left, 2 c + 1 = right of candidate c): the gene bytes to compare with */
    int m[2 * VG_CAND];               /* job length, 0 = no distance to compute (sentinel, empty side, missing candidate) */
    int res[2 * VG_CAND];
    int off[2 * VG_CAND];             /* where the job's part starts in seq[c] */
    int rc[2 * VG_CAND];
    int len[VG_CAND];
};

template <int CAP>
__global__ void __launch_bounds__(VF_WARPS * 32) k_verify(VerifyParams P) {
    __shared__ VerifyGrpWarp<CAP> Wall[VF_WARPS];
    const uint32_t lane = gf_lane(), wib = threadIdx.x >> 5;
    VerifyGrpWarp<CAP>& W = Wall[wib];
    const uint64_t n_warps = (uint64_t)gridDim.x * VF_WARPS;
    unsigned long long n = *P.n_out;
    if (n > P.out_cap) n = P.out_cap;
    const unsigned long long from = P.counters->verify_from;
    for (uint64_t c0 = from + ((uint64_t)blockIdx.x * VF_WARPS + wib) * VG_CAND; c0 < n; c0 += n_warps * VG_CAND) {
        __syncwarp();
        const int cnt = (int)min((unsigned long long)VG_CAND, n - c0);
        for (int c = 0; c < VG_CAND; c++) { /* cooperative loads, one candidate after the other */
            int len = -1;
            if (c < cnt) {
                const gf_match m = P.out[c0 + c];
                len = load_sequence(P.b, (uint32_t)(m.pair_idx - P.b.pair_base), m.source, m.merge_olen, W.seq[c], CAP - 16);
                if (len >= 0 && m.used_rc) revcomp_inplace(W.seq[c], len);
                if (len < 0 && lane == 0) atomicOr(&P.counters->error_flags, 1u);
            }
            if (lane == 0) W.len[c] = len;
        }
        __syncwarp();
        /* the checks of calc_ed per job (lane j < 8 = job j) */
        uint32_t panic = 0;
        if (lane < 2 * VG_CAND) {
            const int c = (int)(lane >> 1);
            const bool right = (lane & 1u) != 0;
            int res = 0, m_job = 0, off = 0;
            const uint8_t* text = nullptr;
            bool rc = false;
            if (c < cnt && W.len[c] >= 0) {
                const gf_match m = P.out[c0 + c];
                const int rb = m.read_break, left_len = rb + 1, right_len = W.len[c] - (rb + 1);
                const int plen = right ? right_len : left_len;
                off = right ? rb + 1 : 0;
                const bool done = right ? calc_ed_setup(P.ix, right_len, m.r_contig, m.r_pos, m.r_pos + right_len - 1, &res, &text, &rc, &panic)
                                        : calc_ed_setup(P.ix, left_len, m.l_contig, m.l_pos - left_len + 1, m.l_pos, &res, &text, &rc, &panic);
                m_job = done ? 0 : plen;
            }
            W.res[lane] = res; W.m[lane] = m_job; W.off[lane] = off; W.text[lane] = text; W.rc[lane] = rc ? 1 : 0;
        }
        __syncwarp();
        int mx = 0;
        for (int j = 0; j < 2 * VG_CAND; j++) mx = max(mx, W.m[j]);
        /* all 8 jobs at once with 4 lanes each when every job fits 4 blocks (256 columns: every unmerged read), else 4 jobs
         * of 8 lanes twice, else 2 jobs of 16 lanes four times */
        if (mx > 0) {
            if (mx <= 256) {
                const int j = (int)(lane >> 2);
                const int d = group_edit_distance<4>(W.seq[j >> 1] + W.off[j], W.m[j], W.rc[j] != 0, W.text[j]);
                if ((lane & 3u) == 0 && W.m[j] > 0) W.res[j] = d;
            } else if (mx <= 512) {
                for (int r = 0; r < 2; r++) {
                    const int j = 4 * r + (int)(lane >> 3);
                    const int d = group_edit_distance<8>(W.seq[j >> 1] + W.off[j], W.m[j], W.rc[j] != 0, W.text[j]);
                    if ((lane & 7u) == 0 && W.m[j] > 0) W.res[j] = d;
                }
            } else if (mx <= 1024) {
                for (int r = 0; r < 4; r++) {
                    const int j = 2 * r + (int)(lane >> 4);
                    const int d = group_edit_distance<16>(W.seq[j >> 1] + W.off[j], W.m[j], W.rc[j] != 0, W.text[j]);
                    if ((lane & 15u) == 0 && W.m[j] > 0) W.res[j] = d;
                }
            } else {
                for (int j = 0; j < 2 * VG_CAND; j++) {
                    if (W.m[j] == 0) continue; /* warp-uniform */
                    const int d = warp_edit_distance(W.seq[j >> 1] + W.off[j], W.m[j], W.rc[j] != 0, W.text[j]);
                    if (lane == 0) W.res[j] = d;
                }
            }
        }
        __syncwarp();
        panic = __reduce_or_sync(FULL, panic);
        /* what filter_matches would decide (fusion_mapper.rs:298-377); the record is kept either way */
        for (int c = 0; c < cnt; c++) {
            const int len = W.len[c];
            if (len < 0) continue;
            const gf_match m = P.out[c0 + c];
            const int rb = m.read_break, left_len = rb + 1, right_len = len - (rb + 1);
            const uint8_t* sq = W.seq[c];
            int chg_l = 0, chg_r = 0; /* dis_connected_count (src/utils/mod.rs:48-56) of both sides of the break */
            for (int i = (int)lane; i + 1 < left_len; i += 32) chg_l += sq[i] != sq[i + 1];
            for (int i = (int)lane; i + 1 < right_len; i += 32) chg_r += sq[rb + 1 + i] != sq[rb + 2 + i];
            chg_l = (int)__reduce_add_sync(FULL, (unsigned)chg_l);
            chg_r = (int)__reduce_add_sync(FULL, (unsigned)chg_r);
            if (lane == 0) {
                const int ld = W.res[2 * c], rd = W.res[2 * c + 1];
                uint32_t ff = 0;
                if (left_len < 20 || chg_l < 7 || right_len < 20 || chg_r < 7) ff |= GF_FILTER_COMPLEXITY;
                if (ld + rd >= 5) ff |= GF_FILTER_DISTANCE;
                int dpos = m.l_pos - m.r_pos;
                if (dpos < 0) dpos = -dpos;
                if (m.l_contig == m.r_contig && dpos < P.ix.deletion_thr) ff |= GF_FILTER_INDEL;
                P.out[c0 + c].l_dist = ld;
                P.out[c0 + c].r_dist = rd;
                P.out[c0 + c].filter_flags = (uint8_t)ff;
            }
        }
        if (panic && lane == 0) atomicAdd(&P.counters->n_ref_panic, 1u);
    }
}

/* ------------------------------------------------------------------------------------------------ */
/* k_adjust_break: FusionResult::adjust_fusion_break / calc_ed (fusion_result.rs:299-397), warp per match */
struct AdjustParams {
    const uint8_t* bytes;
    const gf_break_ref* refs;
    const gf_break_job* jobs;
    unsigned long long n_jobs;
    gf_break_out* out;
    unsigned int* n_flagged;
};
__device__ __forceinline__ int ed_equal_len(const uint8_t* a, const uint8_t* b, int m) { /* both of length m */
    return m > 0 ? warp_edit_distance(a, m, false, b) : 0;
}
__global__ void __launch_bounds__(VF_WARPS * 32) k_adjust_break(AdjustParams P) {
    const uint32_t lane = gf_lane();
    const uint64_t n_warps = (uint64_t)gridDim.x * VF_WARPS;
    for (uint64_t j = (uint64_t)blockIdx.x * VF_WARPS + (threadIdx.x >> 5); j < P.n_jobs; j += n_warps) {
        const gf_break_job job = P.jobs[j];
        const gf_break_ref ref = P.refs[job.result];
        const uint8_t* seq = P.bytes + job.seq_off;
        const uint8_t* lref = P.bytes + ref.left_off;
        const uint8_t* rref = P.bytes + ref.right_off;
        const int len = (int)job.seq_len, nl = (int)ref.left_len, nr = (int)ref.right_len;
        int smallest = 0xFFFF, shift = 0, best_l = 0, best_r = 0;
        bool undefined = false, panic = false;
        for (int s = -3; s <= 3; s++) {
            const int left_len = job.read_break + s + 1, right_len = len - left_len;
            if (left_len < 0 || right_len < 0) { undefined = true; break; }
            const uint8_t* right_seq = seq + left_len;
            /* calc_ed computes both full-length distances of every shift, winning or not, and the reference's edit_distance
             * panics on more than 10 blocks (640 columns) on both sides; the two strings of each have equal length */
            const int lc2 = min(left_len, nl), rc2 = min(right_len, nr);
            if (lc2 > 640 || rc2 > 640) panic = true;
            /* the 20 bases on either side of the break decide (:340-372) */
            const int lc = min(lc2, 20), rc = min(rc2, 20);
            const int total = ed_equal_len(seq + left_len - lc, lref + nl - lc, lc) + ed_equal_len(right_seq, rref, rc);
            if (total < smallest) { /* strict: the first (most negative) best shift wins (:307-313) */
                best_l = ed_equal_len(seq + left_len - lc2, lref + nl - lc2, lc2);
                best_r = ed_equal_len(right_seq, rref, rc2);
                smallest = total;
                shift = s;
            }
        }
        if (lane == 0) {
            gf_break_out o;
            o.shift = undefined ? 0 : shift;
            o.left_distance = undefined ? 0 : best_l;
            o.right_distance = undefined ? 0 : best_r;
            o.status = undefined ? 1 : panic ? 2 : 0; /* status 2 keeps the computed shift and distances */
            P.out[j] = o;
            if (undefined || panic) atomicAdd(P.n_flagged, 1u);
        }
    }
}

/* ------------------------------------------------------------------------------------------------ */
/* k_finish: the per-record part of FusionMapper::filter_matches (fusion_mapper.rs:298-377: a record with any filter flag is
 * removed) and the key sort_matches orders by (add_match bucket :263, read_break descending, read length ascending,
 * read_match.rs:203-229; the name tie-break stays with the host, which owns the names).  Thread per record. */
__global__ void k_finish(const gf_match* __restrict__ in, const unsigned long long* __restrict__ n_in, unsigned long long in_cap,
                         gf_match* __restrict__ out, unsigned long long* __restrict__ keys, unsigned long long* __restrict__ n_out,
                         uint32_t n_genes, uint32_t mode) {
    unsigned long long n = *n_in;
    if (n > in_cap) n = in_cap;
    for (unsigned long long i = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x; i < n;
         i += (unsigned long long)gridDim.x * blockDim.x) {
        const gf_match m = in[i];
        if ((mode & GF_OUT_DROP_FILTERED) && m.filter_flags) continue;
        const unsigned long long slot = atomicAdd(n_out, 1ull);
        out[slot] = m;
        keys[slot] = gf_match_order_key(n_genes, &m);
    }
}

template <class K>
cudaError_t set_smem(K kernel, size_t bytes) {
    if (bytes <= 48 * 1024) return cudaSuccess;
    return cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes);
}

}  // namespace

/* blocks of `kernel` that are resident on one SM at once (registers / shared memory / threads) */
template <class K>
static unsigned resident_blocks(K kernel, int threads, size_t smem) {
    int nb = 0;
    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nb, kernel, threads, smem) != cudaSuccess || nb < 1) nb = 1;
    return (unsigned)nb;
}

/* ================================================================================================== */
/* later chunks of one call: the survivor list starts again at 0, its count so far moves to the running total */
__global__ void k_roll_counters(GfMapCounters* c, const unsigned long long* n_out, unsigned long long out_cap) {
    c->n_survivors_total += c->n_survivors;
    c->n_survivors = 0;
    c->verify_from = min(*n_out, out_cap); /* records before this index were verified with their own chunk */
}

int gf_map_device_batch(gf_index* idx, const GfDevBatch& b, gf_match* d_out, uint64_t out_cap,
                        unsigned long long* d_n_out, cudaStream_t st, GfChunkEvents* ev, bool first, gf_index* store_owner) {
    const bool record_events = ev != nullptr;
    if (ev)
        for (cudaEvent_t& e : ev->e)
            if (!e) GF_CUDA_TRY(cudaEventCreate(&e));
    const bool paired = b.seq2 != nullptr;
    if (b.n > 0xFFFFFFFFull) {
        gf_set_error("batch too large (n > 2^32-1 pairs): split it");
        return GF_E_LIMIT;
    }
    /* workspace */
    const uint64_t surv_cap64 = (paired ? 2 : 1) * b.n + 1;
    const uint32_t surv_cap = (uint32_t)(surv_cap64 > 0xFFFFFFFFull ? 0xFFFFFFFFull : surv_cap64);
    GF_CUDA_TRY(idx->ws_survivors.reserve(sizeof(uint2) * (size_t)surv_cap));
    GF_CUDA_TRY(idx->ws_counters.reserve(sizeof(GfMapCounters)));
    GfMapCounters* d_cnt = idx->ws_counters.as<GfMapCounters>();
    if (first) {
        GF_CUDA_TRY(cudaMemsetAsync(d_cnt, 0, sizeof(GfMapCounters), st));
        GF_CUDA_TRY(cudaMemsetAsync(d_n_out, 0, sizeof(unsigned long long), st));
    } else {
        k_roll_counters<<<1, 1, 0, st>>>(d_cnt, d_n_out, out_cap);
    }
    if (record_events) { GF_CUDA_TRY(cudaEventRecord(ev->e[0], st)); idx->split_events = false; }

    const int need_major = (idx->params.major_gene_key_requirement + 1) / 2;
    const int need_minor = (idx->params.minor_gene_key_requirement + 1) / 2;
    ScreenParams sp;
    sp.ix = idx->dev;
    sp.b = b;
    sp.survivors = idx->ws_survivors.as<uint2>();
    sp.survivors_cap = surv_cap;
    sp.counters = d_cnt;
    sp.need_total = need_major + need_minor;
    sp.need_minor = need_minor;

    if (b.n) {
        const int threads = 256, warps = threads / 32;
        const bool small = b.max_len != 0 && b.max_len <= 256;
        const size_t smem = (small ? sizeof(ScreenWarp<8>) : sizeof(ScreenWarp<32>)) * warps;
        const int blocks_per_sm = 3; /* 80 registers x 256 threads -> 3 resident blocks per SM */
        uint64_t want = (b.n + warps - 1) / warps;
        unsigned grid = (unsigned)std::min<uint64_t>(want, (uint64_t)idx->sm_count * blocks_per_sm);
        if (small) {
            /* split pipeline: prep -> seed -> diag / scan (gf_screen_split.cuh) */
            const bool w5 = b.max_len <= 160;
            const int NW3 = w5 ? split::SL<5>::NW3 : split::SL<8>::NW3;
            const uint32_t cap = surv_cap;
            const size_t groups = ((size_t)cap + 31) / 32;
            /* list mode (several indices, one batch): k_prep's output does not depend on the index, so only the first
             * handle of the list (`store_owner`) converts / merges / stores the sequences; the others read its store */
            gf_index* own = store_owner ? store_owner : idx;
            if (!store_owner) {
                GF_CUDA_TRY(idx->ws_seq_words.reserve(groups * NW3 * 32 * sizeof(uint32_t)));
                GF_CUDA_TRY(idx->ws_seq_meta.reserve((size_t)cap * sizeof(uint4)));
            }
            GF_CUDA_TRY(idx->ws_seq_seed.reserve((size_t)cap * sizeof(uint2)));
            GF_CUDA_TRY(idx->ws_seq_lists.reserve((size_t)cap * sizeof(uint32_t) + 64));
            split::SeqStore ss;
            ss.words = own->ws_seq_words.as<uint32_t>();
            ss.meta = own->ws_seq_meta.as<uint4>();
            ss.seed = idx->ws_seq_seed.as<uint2>();
            ss.counters = idx->ws_seq_lists.as<unsigned int>();
            ss.list = idx->ws_seq_lists.as<uint32_t>() + 16;
            ss.cap = cap;
            GF_CUDA_TRY(cudaMemsetAsync(ss.counters, 0, 64, st));
            if (store_owner) { /* the slot counts of the shared store */
                const unsigned int* oc = store_owner->ws_seq_lists.as<unsigned int>();
                GF_CUDA_TRY(cudaMemcpyAsync(ss.counters, oc, sizeof(unsigned int), cudaMemcpyDeviceToDevice, st));
                GF_CUDA_TRY(cudaMemcpyAsync(ss.counters + 5, oc + 5, sizeof(unsigned int), cudaMemcpyDeviceToDevice, st));
            }
            split::PrepParams pp;
            pp.b = b;
            pp.st = ss;
            pp.counters = d_cnt;
            const size_t psm = sizeof(uint32_t) * tpp::WARPS * (w5 ? tpp::Lay<5>::NWORDS : tpp::Lay<8>::NWORDS) * 32;
            const uint64_t want_b = (b.n + tpp::WARPS * 32 - 1) / (tpp::WARPS * 32);
            /* persistent grids: exactly as many blocks as are resident at once (a partial second wave would idle SMs) */
#define GF_LAUNCH_PREP2(WW, PE, PK)                                                        \
    do {                                                                                   \
        GF_CUDA_TRY(set_smem(split::k_prep<WW, PE, PK>, psm));                             \
        const unsigned pgrid = (unsigned)std::min<uint64_t>(                               \
            want_b, (uint64_t)idx->sm_count * resident_blocks(split::k_prep<WW, PE, PK>, tpp::WARPS * 32, psm)); \
        split::k_prep<WW, PE, PK><<<pgrid, tpp::WARPS * 32, psm, st>>>(pp);                \
    } while (0)
#define GF_LAUNCH_PREP(WW, PE) do { if (b.pk1) GF_LAUNCH_PREP2(WW, PE, true); else GF_LAUNCH_PREP2(WW, PE, false); } while (0)
            if (!store_owner) {
                if (w5) { if (paired) GF_LAUNCH_PREP(5, true); else GF_LAUNCH_PREP(5, false); }
                else { if (paired) GF_LAUNCH_PREP(8, true); else GF_LAUNCH_PREP(8, false); }
            }
#undef GF_LAUNCH_PREP2
#undef GF_LAUNCH_PREP
            if (record_events) GF_CUDA_TRY(cudaEventRecord(ev->e[1], st));
            split::SeedParams sdp;
            sdp.ix = idx->dev;
            sdp.st = ss;
            sdp.need_total = sp.need_total;
            sdp.need_minor = sp.need_minor;
            split::ClassParams cp;
            cp.ix = idx->dev;
            cp.st = ss;
            cp.survivors = sp.survivors;
            cp.survivors_cap = sp.survivors_cap;
            cp.counters = d_cnt;
            cp.need_total = sp.need_total;
            cp.need_minor = sp.need_minor;
            const unsigned smc = (unsigned)idx->sm_count;
#define GF_EV(k) do { if (record_events) GF_CUDA_TRY(cudaEventRecord(ev->e[k], st)); } while (0)
            /* k_diag and k_scan back to back: running them side by side on two streams with split grids measured the same
             * (2.8 vs 2.9 ms), so there is one path */
#define GF_LAUNCH_CLASSES(WW)                                                                                         \
    do {                                                                                                              \
        split::k_seed<WW><<<smc * resident_blocks(split::k_seed<WW>, 256, 0), 256, 0, st>>>(sdp);                     \
        GF_EV(2);                                                                                                     \
        split::k_diag<WW><<<smc * resident_blocks(split::k_diag<WW>, 256, 0), 256, 0, st>>>(cp);                      \
        GF_EV(3);                                                                                                     \
        split::k_scan<WW><<<smc * resident_blocks(split::k_scan<WW>, 256, 0), 256, 0, st>>>(cp);                      \
    } while (0)
            if (w5) GF_LAUNCH_CLASSES(5); else GF_LAUNCH_CLASSES(8);
#undef GF_LAUNCH_CLASSES
#undef GF_EV
            if (record_events) idx->split_events = true;
            idx->launches += 3;
        } else {
            /* reads longer than 256 bases: warp per pair, same filter + gene-plane structures */
            GF_CUDA_TRY(set_smem(k_screen<32, true>, smem));
            GF_CUDA_TRY(set_smem(k_screen<32, false>, smem));
            if (paired) k_screen<32, true><<<grid, threads, smem, st>>>(sp);
            else k_screen<32, false><<<grid, threads, smem, st>>>(sp);
        }
        GF_CUDA_TRY(cudaGetLastError());
        idx->launches++;
    }
    if (record_events) GF_CUDA_TRY(cudaEventRecord(ev->e[4], st));

    if (b.n) {
        /* exact path over the (device-side) survivor count: persistent grid of all resident warps, no host round trip */
        const bool ex_small = b.max_len != 0 && b.max_len <= 256;
        const size_t ex_smem = (ex_small ? sizeof(ExactWarpSmall) : sizeof(ExactWarpLarge)) * EX_WARPS;
        const int ex_gslots = ex_small ? ExactWarpSmall::GLOBAL_SLOTS : ExactWarpLarge::GLOBAL_SLOTS;
        if (ex_small) GF_CUDA_TRY(set_smem(k_exact<ExactWarpSmall>, ex_smem));
        else GF_CUDA_TRY(set_smem(k_exact<ExactWarpLarge>, ex_smem));
        const unsigned ex_res = ex_small ? resident_blocks(k_exact<ExactWarpSmall>, EX_WARPS * 32, ex_smem)
                                         : resident_blocks(k_exact<ExactWarpLarge>, EX_WARPS * 32, ex_smem);
        const unsigned ex_grid = (unsigned)idx->sm_count * std::min(ex_res, 10u);
        const size_t n_ex_warps = (size_t)ex_grid * EX_WARPS;
        static_assert(sizeof(long long) == 8, "");
        GfBuf& gt = idx->ws_gtbl; /* per-warp global vote tables (reads whose votes overflow the shared table) */
        GF_CUDA_TRY(gt.reserve(n_ex_warps * ex_gslots * (sizeof(long long) + sizeof(int))));
        ExactParams ep;
        ep.ix = idx->dev;
        ep.b = b;
        ep.survivors = idx->ws_survivors.as<uint2>();
        ep.survivors_cap = surv_cap;
        ep.counters = d_cnt;
        ep.out = d_out;
        ep.out_cap = out_cap;
        ep.n_out = d_n_out;
        ep.gtbl_keys = gt.as<long long>();
        ep.gtbl_cnt = (int*)(gt.as<long long>() + n_ex_warps * ex_gslots);
        if (ex_small) k_exact<ExactWarpSmall><<<ex_grid, EX_WARPS * 32, ex_smem, st>>>(ep);
        else k_exact<ExactWarpLarge><<<ex_grid, EX_WARPS * 32, ex_smem, st>>>(ep);
        GF_CUDA_TRY(cudaGetLastError());
        VerifyParams vp;
        vp.ix = idx->dev;
        vp.b = b;
        vp.counters = d_cnt;
        vp.out = d_out;
        vp.out_cap = out_cap;
        vp.n_out = d_n_out;
        if (ex_small)
            k_verify<544><<<(unsigned)idx->sm_count * std::min(resident_blocks(k_verify<544>, VF_WARPS * 32, 0), 8u), VF_WARPS * 32, 0, st>>>(vp);
        else
            k_verify<EX_SEQ_CAP><<<(unsigned)idx->sm_count * std::min(resident_blocks(k_verify<EX_SEQ_CAP>, VF_WARPS * 32, 0), 8u), VF_WARPS * 32, 0, st>>>(vp);
        GF_CUDA_TRY(cudaGetLastError());
        idx->launches += 2;
    }
    if (record_events) GF_CUDA_TRY(cudaEventRecord(ev->e[5], st));
    return GF_OK;
}

int gf_map_device_batches(gf_index* const* hs, uint32_t nh, const GfDevBatch& b, gf_match* const* d_outs, uint64_t out_cap,
                          unsigned long long* const* d_n_outs, cudaStream_t st) {
    /* workspace per pair of a chunk: two store slots (reads <= 256 bases) + list + survivor entries */
    const bool small = b.max_len != 0 && b.max_len <= 256;
    const uint64_t per_pair = (small ? 2ull * ((b.max_len <= 160 ? split::SL<5>::NW3 : split::SL<8>::NW3) * 4 + 16 + 8) : 0ull) + 8 + 16;
    uint64_t chunk = std::max<uint64_t>(1u << 20, (5ull << 30) / per_pair);
    if (const char* e = getenv("GF_DEVICE_CHUNK_PAIRS")) { long long v = atoll(e); if (v >= 1024) chunk = (uint64_t)v; }
    const uint64_t n_chunks = b.n ? (b.n + chunk - 1) / chunk : 1;
    const uint64_t per = b.n ? (b.n + n_chunks - 1) / n_chunks : 0;
    for (uint32_t h = 0; h < nh; h++) {
        if (hs[h]->chunk_events.size() < n_chunks) hs[h]->chunk_events.resize(n_chunks);
        hs[h]->n_chunks_timed = (uint32_t)n_chunks;
    }
    for (uint64_t c = 0; c < n_chunks; c++) {
        const uint64_t lo = c * per, hi = std::min(b.n, lo + per);
        GfDevBatch cb = b;
        cb.n = hi - lo;
        cb.s1 += lo; cb.e1 += lo; cb.qs1 += lo;
        if (cb.s2) { cb.s2 += lo; cb.e2 += lo; cb.qs2 += lo; }
        cb.pair_base = b.pair_base + lo;
        for (uint32_t h = 0; h < nh; h++) {
            int rc = gf_map_device_batch(hs[h], cb, d_outs[h], out_cap, d_n_outs[h], st, &hs[h]->chunk_events[c], c == 0,
                                         h ? hs[0] : nullptr);
            if (rc != GF_OK) return rc;
        }
    }
    return GF_OK;
}

int gf_finish_records_device(gf_index* idx, const gf_match* d_in, const unsigned long long* d_n_in, uint64_t in_cap,
                             gf_match* d_out2, unsigned long long* d_keys, unsigned long long* d_n_out2, uint32_t mode,
                             cudaStream_t st) {
    GF_CUDA_TRY(cudaMemsetAsync(d_n_out2, 0, sizeof(unsigned long long), st));
    k_finish<<<(unsigned)idx->sm_count, 256, 0, st>>>(d_in, d_n_in, in_cap, d_out2, d_keys, d_n_out2, idx->n_genes, mode);
    GF_CUDA_TRY(cudaGetLastError());
    idx->launches++;
    return GF_OK;
}

int gf_fast_merge_device(gf_index* idx, const GfDevBatch& b, gf_merge_info* d_out, cudaStream_t st) {
    if (!b.n) return GF_OK;
    GF_CUDA_TRY(idx->ws_counters.reserve(sizeof(GfMapCounters)));
    GF_CUDA_TRY(cudaMemsetAsync(idx->ws_counters.p, 0, sizeof(GfMapCounters), st));
    if (b.max_len != 0 && b.max_len <= 256) {
        const bool w5 = b.max_len <= 160;
        const size_t tsm = sizeof(uint32_t) * tpp::WARPS * (w5 ? tpp::Lay<5>::NWORDS : tpp::Lay<8>::NWORDS) * 32;
        unsigned tgrid = (unsigned)std::min<uint64_t>((b.n + tpp::WARPS * 32 - 1) / (tpp::WARPS * 32), (uint64_t)idx->sm_count * 3);
        if (w5) {
            GF_CUDA_TRY(set_smem(tpp::k_merge_only_tpp<5>, tsm));
            tpp::k_merge_only_tpp<5><<<tgrid, tpp::WARPS * 32, tsm, st>>>(b, d_out, idx->ws_counters.as<GfMapCounters>());
        } else {
            GF_CUDA_TRY(set_smem(tpp::k_merge_only_tpp<8>, tsm));
            tpp::k_merge_only_tpp<8><<<tgrid, tpp::WARPS * 32, tsm, st>>>(b, d_out, idx->ws_counters.as<GfMapCounters>());
        }
        GF_CUDA_TRY(cudaGetLastError());
        return GF_OK;
    }
    const int threads = 256, warps = 8;
    const size_t smem = sizeof(ScreenWarp<32>) * warps;
    GF_CUDA_TRY(set_smem(k_merge_only<32>, smem));
    unsigned grid = (unsigned)std::min<uint64_t>((b.n + warps - 1) / warps, (uint64_t)idx->sm_count * 4);
    k_merge_only<32><<<grid, threads, smem, st>>>(b, d_out, idx->ws_counters.as<GfMapCounters>());
    GF_CUDA_TRY(cudaGetLastError());
    return GF_OK;
}

/* report stage: adjust_fusion_break for n_jobs matches, everything already on the device; *d_n_flagged counts jobs on which
 * the reference would panic: a shifted break leaves the read (status 1) or a full-length distance needs more than 640
 * columns (status 2) */
int gf_adjust_break_device(gf_index* idx, const uint8_t* d_bytes, const gf_break_ref* d_refs, const gf_break_job* d_jobs,
                           uint64_t n_jobs, gf_break_out* d_out, unsigned int* d_n_flagged, cudaStream_t st) {
    if (!n_jobs) return GF_OK;
    AdjustParams ap;
    ap.bytes = d_bytes;
    ap.refs = d_refs;
    ap.jobs = d_jobs;
    ap.n_jobs = n_jobs;
    ap.out = d_out;
    ap.n_flagged = d_n_flagged;
    const uint64_t want = (n_jobs + VF_WARPS - 1) / VF_WARPS;
    const unsigned grid = (unsigned)std::min<uint64_t>(want, (uint64_t)idx->sm_count * resident_blocks(k_adjust_break, VF_WARPS * 32, 0));
    k_adjust_break<<<grid, VF_WARPS * 32, 0, st>>>(ap);
    GF_CUDA_TRY(cudaGetLastError());
    idx->launches++;
    return GF_OK;
}
