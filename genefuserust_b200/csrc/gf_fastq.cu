/*
 * gf_fastq.cu — FASTQ ingest on the device (SURVEY.md 8f rank 2): raw FASTQ text -> per-record tables, so the
 * mapping kernels read sequences and qualities straight out of the text buffer (no host-side parsing, no repacking).
 *
 * Mirrors FastqReader::read (/root/reference/src/core/fastq_reader.rs:75-147): a record is four lines (name,
 * sequence, strand, quality), each line loses ONE trailing '\n' and nothing else ('\r' is kept, nothing is validated);
 * reading stops at the first record that cannot be completed, so an incomplete trailing record is dropped.
 *
 *   k_nl_count   16 bytes per thread (128-bit loads), newlines per 4 KB tile
 *   exclusive scan of the tile counts (gf_exclusive_scan_u32)
 *   k_nl_write   positions of all newlines, in order
 *   k_records    record i: sequence = (NL[4i], NL[4i+1]), quality = (NL[4i+2], NL[4i+3]); max length; checks
 */
#include <algorithm>

#include "gf_internal.h"
#include "gf_inflate.cuh"

namespace {

constexpr int NL_THREADS = 256;
constexpr int NL_TILE = NL_THREADS * 16;

__device__ __forceinline__ uint32_t newline_mask16(const uint8_t* __restrict__ text, uint64_t bytes, uint64_t pos) {
    /* bit t set <=> text[pos + t] == '\n' */
    uint32_t m = 0;
    if (pos + 16 <= bytes && ((uintptr_t)(text + pos) & 15u) == 0) {
        uint4 v = __ldg(reinterpret_cast<const uint4*>(text + pos));
        uint32_t w[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
        for (int j = 0; j < 4; j++) {
            uint32_t y = w[j] ^ 0x0A0A0A0Au;
            uint32_t z = ~(((y & 0x7F7F7F7Fu) + 0x7F7F7F7Fu) | y) & 0x80808080u; /* bit 7 of every zero byte */
            m |= ((((z >> 7) * 0x01020408u) >> 24) & 0xFu) << (4 * j);
        }
    } else {
        for (int t = 0; t < 16; t++)
            if (pos + t < bytes && text[pos + t] == '\n') m |= 1u << t;
    }
    return m;
}
__global__ void k_nl_count(const uint8_t* __restrict__ text, uint64_t bytes, uint32_t* __restrict__ tile_counts,
                           unsigned long long* __restrict__ total) {
    __shared__ uint32_t ws[NL_THREADS / 32];
    uint64_t pos = (uint64_t)blockIdx.x * NL_TILE + (uint64_t)threadIdx.x * 16;
    uint32_t c = pos < bytes ? __popc(newline_mask16(text, bytes, pos)) : 0u;
    c = __reduce_add_sync(0xFFFFFFFFu, c);
    if ((threadIdx.x & 31) == 0) ws[threadIdx.x >> 5] = c;
    __syncthreads();
    if (threadIdx.x == 0) {
        uint32_t t = 0;
        for (int w = 0; w < NL_THREADS / 32; w++) t += ws[w];
        tile_counts[blockIdx.x] = t;
        if (t) atomicAdd(total, (unsigned long long)t); /* 64-bit: the u32 scan below must not wrap unnoticed */
    }
}
__global__ void k_nl_write(const uint8_t* __restrict__ text, uint64_t bytes, const uint32_t* __restrict__ tile_off,
                           unsigned long long* __restrict__ nl) {
    __shared__ uint32_t ws[NL_THREADS / 32];
    uint64_t pos = (uint64_t)blockIdx.x * NL_TILE + (uint64_t)threadIdx.x * 16;
    uint32_t m = pos < bytes ? newline_mask16(text, bytes, pos) : 0u;
    uint32_t c = __popc(m), incl = c;
    const uint32_t lane = threadIdx.x & 31;
    for (int o = 1; o < 32; o <<= 1) {
        uint32_t t = __shfl_up_sync(0xFFFFFFFFu, incl, o);
        if (lane >= (uint32_t)o) incl += t;
    }
    if (lane == 31) ws[threadIdx.x >> 5] = incl;
    __syncthreads();
    uint32_t woff = 0;
    for (int w = 0; w < (int)(threadIdx.x >> 5); w++) woff += ws[w];
    uint32_t dst = tile_off[blockIdx.x] + woff + incl - c;
    while (m) {
        int t = __ffs(m) - 1;
        m &= m - 1;
        nl[dst++] = pos + (uint64_t)t;
    }
}
/* err bits: 1 = quality and sequence lengths differ */
__global__ void k_records(const unsigned long long* __restrict__ nl, uint64_t n_records, unsigned long long* __restrict__ s,
                          unsigned long long* __restrict__ e, unsigned long long* __restrict__ qs,
                          unsigned int* __restrict__ max_len, unsigned int* __restrict__ err) {
    uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    uint32_t len = 0, bad = 0;
    if (i < n_records) {
        /* line j spans (nl[j], nl[j+1]) in the shifted table; record i = lines 4i (name), 4i+1 (sequence), 4i+2, 4i+3 (quality) */
        unsigned long long a = nl[4 * i + 1] + 1, b = nl[4 * i + 2], qa = nl[4 * i + 3] + 1, qb = nl[4 * i + 4];
        s[i] = a;
        e[i] = b;
        qs[i] = qa;
        len = (uint32_t)(b - a);
        bad = (qb - qa) != (b - a);
    }
    len = __reduce_max_sync(0xFFFFFFFFu, len);
    bad = __reduce_or_sync(0xFFFFFFFFu, bad);
    if ((threadIdx.x & 31) == 0) {
        if (len) atomicMax(max_len, len);
        if (bad) atomicOr(err, 1u);
    }
}

}  // namespace

int gf_fastq_parse_device(const uint8_t* d_text, uint64_t bytes, GfFastqTable* out, cudaStream_t st, bool final_chunk) {
    out->n_records = 0;
    out->max_len = 0;
    if (bytes == 0) return GF_OK;
    const uint64_t n_tiles = (bytes + NL_TILE - 1) / NL_TILE;
    if (n_tiles > 0x7FFFFFFFull) { gf_set_error("FASTQ buffer too large for one call (> 8 TiB)"); return GF_E_LIMIT; }
    GF_CUDA_TRY(out->cnt.reserve(sizeof(uint32_t) * (n_tiles + 2) + 16));
    GF_CUDA_TRY(out->off.reserve(sizeof(uint32_t) * (n_tiles + 1)));
    GF_CUDA_TRY(out->tmp.reserve(sizeof(uint32_t) * gf_scan_tmp_elems(n_tiles)));
    uint32_t *d_cnt = out->cnt.as<uint32_t>(), *d_off = out->off.as<uint32_t>(), *d_tmp = out->tmp.as<uint32_t>();
    /* 64-bit newline total behind the tile counts (8-byte aligned) */
    unsigned long long* d_total = reinterpret_cast<unsigned long long*>(d_cnt + ((n_tiles + 2 + 1) & ~1ull));
    GF_CUDA_TRY(cudaMemsetAsync(d_total, 0, sizeof(unsigned long long), st));
    k_nl_count<<<(unsigned)n_tiles, NL_THREADS, 0, st>>>(d_text, bytes, d_cnt, d_total);
    GF_CUDA_TRY(gf_exclusive_scan_u32(d_cnt, d_off, n_tiles, d_tmp, st));
    uint32_t n_nl = 0;
    unsigned long long n_nl64 = 0;
    uint8_t last = 0;
    GF_CUDA_TRY(cudaMemcpyAsync(&n_nl, d_off + n_tiles, sizeof(uint32_t), cudaMemcpyDeviceToHost, st));
    GF_CUDA_TRY(cudaMemcpyAsync(&n_nl64, d_total, sizeof(n_nl64), cudaMemcpyDeviceToHost, st));
    GF_CUDA_TRY(cudaMemcpyAsync(&last, d_text + bytes - 1, 1, cudaMemcpyDeviceToHost, st));
    GF_CUDA_TRY(cudaStreamSynchronize(st));
    if (n_nl64 != (unsigned long long)n_nl) {
        gf_set_error("FASTQ buffer holds 2^32 or more lines: pass it in pieces (gf_fastq_stream_*)");
        return GF_E_LIMIT;
    }
    /* a non-empty unterminated last line still counts as a line (read_line returns > 0): virtual newline at `bytes` — but
     * only at the end of the file: in a streamed chunk the rest of that line has not arrived yet */
    if (!final_chunk) last = '\n';
    const uint64_t n_lines = (uint64_t)n_nl + (last != '\n' ? 1 : 0);
    GF_CUDA_TRY(out->nl.reserve(sizeof(unsigned long long) * (n_lines + 2)));
    unsigned long long* nl = out->nl.as<unsigned long long>();
    /* nl[0] = -1 (virtual newline before the first byte), nl[1..] = real newlines */
    const unsigned long long minus1 = ~0ull;
    GF_CUDA_TRY(cudaMemcpyAsync(nl, &minus1, sizeof(minus1), cudaMemcpyHostToDevice, st));
    k_nl_write<<<(unsigned)n_tiles, NL_THREADS, 0, st>>>(d_text, bytes, d_off, nl + 1);
    if (last != '\n') {
        const unsigned long long endpos = bytes;
        GF_CUDA_TRY(cudaMemcpyAsync(nl + 1 + n_nl, &endpos, sizeof(endpos), cudaMemcpyHostToDevice, st));
    }
    const uint64_t n_records = n_lines / 4;
    out->n_records = n_records;
    if (n_records) {
        GF_CUDA_TRY(out->s.reserve(sizeof(unsigned long long) * n_records));
        GF_CUDA_TRY(out->e.reserve(sizeof(unsigned long long) * n_records));
        GF_CUDA_TRY(out->qs.reserve(sizeof(unsigned long long) * n_records));
        unsigned int* d_flags = reinterpret_cast<unsigned int*>(d_cnt); /* reuse: [0] max_len, [1] err */
        GF_CUDA_TRY(cudaMemsetAsync(d_flags, 0, 2 * sizeof(unsigned int), st));
        /* record i uses lines 4i..4i+3; line j spans (nl[j], nl[j+1]) in the shifted table */
        k_records<<<(unsigned)((n_records + 255) / 256), 256, 0, st>>>(nl, n_records, out->s.as<unsigned long long>(),
                                                                       out->e.as<unsigned long long>(),
                                                                       out->qs.as<unsigned long long>(), d_flags, d_flags + 1);
        unsigned int h[2] = {0, 0};
        GF_CUDA_TRY(cudaMemcpyAsync(h, d_flags, sizeof(h), cudaMemcpyDeviceToHost, st));
        GF_CUDA_TRY(cudaStreamSynchronize(st));
        out->max_len = h[0];
        if (h[1] & 1u) {
            gf_set_error("FASTQ: a quality line and its sequence line differ in length (the reference indexes qualities by "
                         "sequence position and panics when they are shorter, src/core/read.rs:349)");
            return GF_E_INVALID;
        }
    }
    GF_CUDA_TRY(cudaGetLastError());
    return GF_OK;
}

/* ---- the FASTQ lines of the pairs that have a record (gf_fastq_stream_keep_reads) ----
 * Runs after k_verify / gf_finish_records_device, while the chunk's text and newline tables are still resident:
 *   k_reads_mark     bit h of mask[local pair] for every record of index h of the list (the counts are read on the device)
 *   k_reads_size     per pair: a 0/1 "has a record" word and the bytes of its 4 or 8 lines (0 when unmarked); 64-bit total
 *   two exclusive scans: the 0/1 words -> slot in the ascending list of matched pairs, bytes -> offset in the text arena
 *   k_reads_compact  descriptor and mask of every matched pair at its slot
 *   k_reads_gather   one warp per matched pair copies its lines, without the newlines, into the arena
 * The arena holds the lines of the matched pairs only: it is not sized for the chunk's whole text (600 MB of device memory
 * with the default 256 MiB chunks, for the ~1 MB that a chunk's matched pairs usually take).  Their total is known on the
 * device only, so k_reads_gather is launched against the arena as it is and copies nothing when the total does not fit; the
 * host sees that after the call's end-of-call synchronisation, grows the arena to the total and launches the gather again
 * (gf_fastq_regather_reads): one extra launch and synchronisation each time the arena grows, which is rare — it is grow-only
 * and starts at RD_ARENA_MIN.  A list stream gathers the union of its indices' matched pairs once; the masks tell the host
 * which index each pair belongs to. */
namespace {

constexpr int RD_THREADS = 256;
constexpr size_t RD_ARENA_MIN = 256u << 10;

__device__ __forceinline__ void line_span(const unsigned long long* __restrict__ nl, uint64_t j, unsigned long long* a,
                                          uint32_t* len) {
    /* line j spans (nl[j], nl[j + 1]) in the shifted table (nl[0] = -1: the +1 wraps to 0) */
    *a = nl[j] + 1;
    *len = (uint32_t)(nl[j + 1] - *a);
}

/* blockIdx.y = index h of the list */
__global__ void k_reads_mark(GfRecordLists lists, unsigned long long* __restrict__ mask) {
    const uint32_t h = blockIdx.y;
    const gf_match* __restrict__ rec = lists.rec[h];
    const unsigned long long n = *lists.n[h];
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (uint64_t)gridDim.x * blockDim.x)
        atomicOr(&mask[rec[i].pair_idx], 1ull << h);
}

__global__ void k_reads_size(const unsigned long long* __restrict__ nl1, const unsigned long long* __restrict__ nl2, uint64_t n,
                             const unsigned long long* __restrict__ mask, uint32_t* __restrict__ has, uint32_t* __restrict__ bytes,
                             unsigned long long* __restrict__ total) {
    const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    unsigned long long b = 0;
    const bool marked = mask[i] != 0;
    has[i] = marked ? 1u : 0u; /* (the scan counts pairs, not mask bits) */
    if (marked) {
        /* record i = lines 4i .. 4i+3: its lines = from the name line's start to the quality line's end, less 3 newlines */
        b = nl1[4 * i + 4] - (nl1[4 * i] + 1) - 3;
        if (nl2) b += nl2[4 * i + 4] - (nl2[4 * i] + 1) - 3;
        atomicAdd(total, b); /* 64-bit: the u32 scan of `bytes` must not wrap unnoticed (few pairs are flagged) */
    }
    bytes[i] = (uint32_t)b;
}

__global__ void k_reads_compact(const unsigned long long* __restrict__ nl1, const unsigned long long* __restrict__ nl2, uint64_t n,
                                const unsigned long long* __restrict__ mask, const uint32_t* __restrict__ slot,
                                const uint32_t* __restrict__ off, gf_fastq_read_pair* __restrict__ out,
                                unsigned long long* __restrict__ out_mask) {
    const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const unsigned long long mk = mask[i];
    if (!mk) return;
    gf_fastq_read_pair p;
    p.pair_idx = i;
    p.text_off = off[i];
    unsigned long long a;
#pragma unroll
    for (int l = 0; l < 4; l++) line_span(nl1, 4 * i + l, &a, &p.len[0][l]);
#pragma unroll
    for (int l = 0; l < 4; l++) {
        p.len[1][l] = 0;
        if (nl2) line_span(nl2, 4 * i + l, &a, &p.len[1][l]);
    }
    out[slot[i]] = p;
    out_mask[slot[i]] = mk;
}

__global__ void k_reads_gather(const uint8_t* __restrict__ text1, const unsigned long long* __restrict__ nl1,
                               const uint8_t* __restrict__ text2, const unsigned long long* __restrict__ nl2,
                               const gf_fastq_read_pair* __restrict__ pairs, const uint32_t* __restrict__ n_pairs,
                               const unsigned long long* __restrict__ total, uint64_t arena_cap, uint8_t* __restrict__ arena) {
    const uint32_t lane = threadIdx.x & 31u;
    if (*total > arena_cap) return; /* the host grows the arena and launches again */
    const uint32_t n = *n_pairs;
    const uint64_t warps = (uint64_t)gridDim.x * (blockDim.x >> 5);
    for (uint64_t w = (uint64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5); w < n; w += warps) {
        const uint64_t i = pairs[w].pair_idx;
        uint8_t* dst = arena + pairs[w].text_off;
        for (int m = 0; m < (nl2 ? 2 : 1); m++) {
            const uint8_t* src = m ? text2 : text1;
            const unsigned long long* nl = m ? nl2 : nl1;
            for (int l = 0; l < 4; l++) {
                unsigned long long a;
                uint32_t len;
                line_span(nl, 4 * i + l, &a, &len);
                for (uint32_t b = lane; b < len; b += 32) dst[b] = __ldg(src + a + b);
                dst += len;
            }
        }
    }
}

}  // namespace

int gf_fastq_gather_reads(gf_index* idx, const uint8_t* const text[2], uint64_t n, const GfRecordLists& lists, uint32_t nh,
                          GfHostSlot* h, cudaStream_t st) {
    GfFastqReadsWork& w = idx->fq_reads;
    const bool pe = text[1] != nullptr;
    const unsigned long long* nl1 = idx->fq[0].nl.as<unsigned long long>();
    const unsigned long long* nl2 = pe ? idx->fq[1].nl.as<unsigned long long>() : nullptr;
    w.text1 = text[0];
    w.text2 = text[1];
    w.n = n;
    w.arena_used = 0;
    if (n == 0) return GF_OK;
    if (n >= 0xFFFFFFFFull) { gf_set_error("FASTQ chunk holds 2^32 or more records"); return GF_E_LIMIT; }
    GF_CUDA_TRY(w.mask.reserve(sizeof(unsigned long long) * n));
    GF_CUDA_TRY(w.has.reserve(sizeof(uint32_t) * (n + 1)));
    GF_CUDA_TRY(w.slot.reserve(sizeof(uint32_t) * (n + 1)));
    GF_CUDA_TRY(w.bytes.reserve(sizeof(uint32_t) * (n + 1)));
    GF_CUDA_TRY(w.off.reserve(sizeof(uint32_t) * (n + 1)));
    GF_CUDA_TRY(w.tmp.reserve(sizeof(uint32_t) * gf_scan_tmp_elems(n)));
    GF_CUDA_TRY(w.total.reserve(sizeof(unsigned long long)));
    GF_CUDA_TRY(w.pairs.reserve(sizeof(gf_fastq_read_pair) * n));
    GF_CUDA_TRY(w.pair_mask.reserve(sizeof(unsigned long long) * n));
    unsigned long long* mask = w.mask.as<unsigned long long>();
    uint32_t *has = w.has.as<uint32_t>(), *slot = w.slot.as<uint32_t>(), *bytes = w.bytes.as<uint32_t>(), *off = w.off.as<uint32_t>();
    unsigned long long* total = w.total.as<unsigned long long>();
    GF_CUDA_TRY(cudaMemsetAsync(mask, 0, sizeof(unsigned long long) * n, st));
    GF_CUDA_TRY(cudaMemsetAsync(total, 0, sizeof(unsigned long long), st));
    const unsigned grid = (unsigned)std::max<uint64_t>(1, std::min<uint64_t>((n + RD_THREADS - 1) / RD_THREADS, 4ull * idx->sm_count));
    const unsigned per_pair = (unsigned)((n + RD_THREADS - 1) / RD_THREADS);
    k_reads_mark<<<dim3(grid, nh), RD_THREADS, 0, st>>>(lists, mask);
    k_reads_size<<<per_pair, RD_THREADS, 0, st>>>(nl1, nl2, n, mask, has, bytes, total);
    GF_CUDA_TRY(gf_exclusive_scan_u32(has, slot, n, w.tmp.as<uint32_t>(), st));
    GF_CUDA_TRY(gf_exclusive_scan_u32(bytes, off, n, w.tmp.as<uint32_t>(), st));
    k_reads_compact<<<per_pair, RD_THREADS, 0, st>>>(nl1, nl2, n, mask, slot, off, w.pairs.as<gf_fastq_read_pair>(),
                                                      w.pair_mask.as<unsigned long long>());
    GF_CUDA_TRY(w.text.reserve(RD_ARENA_MIN));
    w.arena_used = w.text.cap;
    k_reads_gather<<<grid, RD_THREADS, 0, st>>>(text[0], nl1, text[1], nl2, w.pairs.as<gf_fastq_read_pair>(), slot + n, total,
                                                 w.arena_used, w.text.as<uint8_t>());
    idx->launches += 4 + 2 * gf_scan_launches(n);
    /* the totals travel with the call's other end-of-call copies into the pinned slot */
    GF_CUDA_TRY(cudaMemcpyAsync(&h->n_read_pairs, slot + n, sizeof(uint32_t), cudaMemcpyDeviceToHost, st));
    GF_CUDA_TRY(cudaMemcpyAsync(&h->read_bytes, off + n, sizeof(uint32_t), cudaMemcpyDeviceToHost, st));
    GF_CUDA_TRY(cudaMemcpyAsync(&h->read_bytes64, total, sizeof(unsigned long long), cudaMemcpyDeviceToHost, st));
    GF_CUDA_TRY(cudaGetLastError());
    return GF_OK;
}

/* ---- BGZF members -> text, one WARP per member (csrc/gf_inflate.cuh holds the tables, the symbol decoder and a single-thread
 * reference version that the CPU tests check against zlib).  Decoding a DEFLATE stream is a chain of dependent steps, so lane 0
 * walks it alone — header, tables, symbol after symbol, literals stored as they come — and the other 31 lanes join for what is
 * parallel: every match is copied by the whole warp (byte i of it is byte i mod dist of the `dist` bytes before it, so an
 * overlapping match is no special case).  A thread per member was measured first: the 32 streams of a warp are never at the same
 * instruction, the warp runs them one after the other and every copied byte costs an L2 round trip (1.1 GB/s of text per GPU);
 * a warp per member keeps ~26 members in flight per SM.  With one useful lane per warp the kernel is bound by instruction issue
 * (ncu: 65 % issue utilisation, 7.0 G warp instructions per 3831 members = 10.3 ms), so what counts is instructions per symbol.
 * Measured and rejected: lane 0 noting up to 64 matches per round in a shared-memory list that the warp then copies in order — no
 * fewer instructions (7.5 G) and the L2 round trips no longer overlap with the decoding: 16.9 ms.  Blocks of 4 warps at 72 registers (no spills), 7 per SM: 8.9 ms (8-warp blocks capped at 64 registers with
 * spills: 10.3 ms).  The decoding tables of a block's warps live in shared memory (2.5 KB each) next to the four CRC-32 tables.  Every member's sizes and CRC-32 are known from its header
 * and trailer: a member that does not come out exactly is reported through `status`, never used. ---- */
namespace {
constexpr int INF_WARPS = 4;
constexpr size_t INF_TABLES = (sizeof(gfinf::Tables) + 15) / 16 * 16;
constexpr size_t INF_SMEM = INF_WARPS * INF_TABLES + (4 * 256 + 32) * sizeof(uint32_t);

struct Bits32 { /* gfinf::Bits with 32-bit loads (lane 0 only) */
    const uint8_t* in;
    uint32_t n, pos;
    uint64_t buf;
    uint32_t cnt;
    __device__ __forceinline__ bool word_ok() const { return (((uintptr_t)(in + pos)) & 3u) == 0 && pos + 4 <= n; }
    __device__ __forceinline__ void refill() { /* >= 32 valid bits afterwards (zeros behind the input: `over` tells) */
        if (cnt > 32) return;
        while (cnt <= 56 && !word_ok()) { /* up to the next aligned word, or the last bytes of the input */
            const uint64_t b = pos < n ? __ldg(in + pos) : 0u;
            pos++;
            buf |= b << cnt;
            cnt += 8;
        }
        if (cnt <= 32) { /* (then word_ok() holds) */
            buf |= (uint64_t)__ldg(reinterpret_cast<const uint32_t*>(in + pos)) << cnt;
            pos += 4;
            cnt += 32;
        }
    }
    __device__ __forceinline__ uint32_t peek(uint32_t k) const { return (uint32_t)(buf & ((1ull << k) - 1ull)); }
    __device__ __forceinline__ void drop(uint32_t k) { buf >>= k; cnt -= k; }
    __device__ __forceinline__ uint32_t take(uint32_t k) { const uint32_t v = peek(k); drop(k); return v; }
    __device__ __forceinline__ uint32_t used_bytes() const { return pos - (cnt >> 3); }
    __device__ __forceinline__ bool over() const { return used_bytes() > n; }
};

__constant__ uint16_t c_lbase[29] = {3, 4, 5, 6, 7, 8, 9, 10, 11, 13, 15, 17, 19, 23, 27, 31, 35, 43, 51, 59, 67, 83, 99, 115, 131, 163, 195, 227, 258};
__constant__ uint8_t c_lext[29] = {0, 0, 0, 0, 0, 0, 0, 0, 1, 1, 1, 1, 2, 2, 2, 2, 3, 3, 3, 3, 4, 4, 4, 4, 5, 5, 5, 5, 0};
__constant__ uint16_t c_dbase[30] = {1, 2, 3, 4, 5, 7, 9, 13, 17, 25, 33, 49, 65, 97, 129, 193, 257, 385, 513, 769, 1025, 1537, 2049, 3073, 4097, 6145, 8193, 12289, 16385, 24577};
__constant__ uint8_t c_dext[30] = {0, 0, 0, 0, 1, 1, 2, 2, 3, 3, 4, 4, 5, 5, 6, 6, 7, 7, 8, 8, 9, 9, 10, 10, 11, 11, 12, 12, 13, 13};
__constant__ uint8_t c_order[19] = {16, 17, 18, 0, 8, 7, 9, 6, 10, 5, 11, 4, 12, 3, 13, 2, 14, 1, 15};

/* lane 0: the header of the next block; returns an error code, sets *stored (a stored block was copied, no symbols follow) */
__device__ int block_header(Bits32& b, gfinf::Tables& T, uint8_t* out, uint32_t out_len, uint32_t* op, uint32_t* last, bool* stored) {
    using namespace gfinf;
    b.refill();
    *last = b.take(1);
    const uint32_t type = b.take(2);
    *stored = false;
    if (type == 3) return E_BTYPE;
    if (type == 0) {
        b.drop(b.cnt & 7u);
        while (b.cnt < 32) { const uint64_t x = b.pos < b.n ? __ldg(b.in + b.pos) : 0u; b.pos++; b.buf |= x << b.cnt; b.cnt += 8; }
        const uint32_t len = b.take(16), nlen = b.take(16);
        if ((len ^ 0xFFFFu) != nlen) return E_STORED;
        uint32_t ip = b.used_bytes();
        if (ip + len > b.n) return E_INPUT;
        if (*op + len > out_len) return E_OUTPUT;
        for (uint32_t i = 0; i < len; i++) out[*op + i] = __ldg(b.in + ip + i);
        *op += len;
        b.pos = ip + len; b.buf = 0; b.cnt = 0;
        *stored = true;
        return OK;
    }
    if (type == 1) {
        fixed_lengths(T.lens);
        build(T.lens, 288, T.lcount, T.lsym, T.lit, LBITS);
        build(T.lens + 288, 30, T.dcount, T.dsym, T.dist, DBITS);
        return OK;
    }
    const uint32_t nlen = b.take(5) + 257, ndist = b.take(5) + 1, ncode = b.take(4) + 4;
    if (nlen > 286 || ndist > 30) return E_CODELEN;
    uint8_t cl[19];
    for (int i = 0; i < 19; i++) cl[i] = 0;
    for (uint32_t i = 0; i < ncode; i++) { b.refill(); cl[c_order[i]] = (uint8_t)b.take(3); }
    if (build(cl, 19, T.dcount, T.dsym, T.dist, 7) != 0) return E_CODELEN;
    uint32_t i = 0;
    while (i < nlen + ndist) {
        b.refill();
        const int s = decode_sym(b, T.dist, 7, T.dcount, T.dsym);
        if (s < 0) return E_CODELEN;
        if (s < 16) { T.lens[i++] = (uint8_t)s; continue; }
        uint32_t rep, val = 0;
        if (s == 16) { if (i == 0) return E_CODELEN; val = T.lens[i - 1]; rep = 3 + b.take(2); }
        else if (s == 17) rep = 3 + b.take(3);
        else rep = 11 + b.take(7);
        if (i + rep > nlen + ndist) return E_CODELEN;
        while (rep--) T.lens[i++] = (uint8_t)val;
    }
    if (T.lens[256] == 0) return E_CODELEN;
    uint8_t dl[30];
    for (uint32_t d = 0; d < 30; d++) dl[d] = d < ndist ? T.lens[nlen + d] : 0;
    for (uint32_t s = nlen; s < 288; s++) T.lens[s] = 0;
    const int rl = build(T.lens, 288, T.lcount, T.lsym, T.lit, LBITS);
    if (rl < 0 || (rl > 0 && !(T.lcount[1] == 1 && T.lcount[0] == 287))) return E_CODELEN;
    const int rd = build(dl, 30, T.dcount, T.dsym, T.dist, DBITS);
    if (rd < 0 || (rd > 0 && !(T.dcount[1] == 1 && T.dcount[0] == 29))) return E_CODELEN;
    return OK;
}

__global__ void __launch_bounds__(INF_WARPS * 32, 7) k_bgzf_inflate(const uint8_t* __restrict__ comp, const GfBgzfMember* __restrict__ members,
                                                                uint32_t n, uint8_t* text, unsigned int* __restrict__ status) {
    using namespace gfinf;
    extern __shared__ __align__(16) unsigned char inf_smem[];
    uint32_t* crc_t = reinterpret_cast<uint32_t*>(inf_smem + INF_WARPS * INF_TABLES);
    uint32_t* x2n = crc_t + 4 * 256;
    crc_tables(crc_t, (int)threadIdx.x, INF_WARPS * 32);
    if (threadIdx.x == INF_WARPS * 32 - 1) crc_x2n_table(x2n);
    __syncthreads();
    crc_tables_rest(crc_t, (int)threadIdx.x, INF_WARPS * 32);
    __syncthreads();
    const uint32_t lane = threadIdx.x & 31u, wib = threadIdx.x >> 5;
    const uint32_t i = blockIdx.x * INF_WARPS + wib;
    if (i >= n) return;
    Tables& T = *reinterpret_cast<Tables*>(inf_smem + wib * INF_TABLES);
    const GfBgzfMember m = members[i];
    uint8_t* out = text + m.out_off;
    const uint32_t out_len = m.isize;
    Bits32 b{comp + m.in_off, m.clen, 0, 0, 0};
    uint32_t op = 0, last = 0; /* lane 0's: where the next decoded byte goes (the match being copied is counted already) */
    bool in_block = false;
    int err = OK;
    /* The copy of a match overlaps with the decoding of what follows it: every lane asks for its source byte (an L2 round
     * trip), lane 0 decodes on to the next match while the bytes are on their way, then they are stored. */
    uint32_t c_len = 0, c_dist = 0, c_op = 0; /* the match being copied (c_len == 0: none) */
    for (;;) {
        const bool mine = lane < c_len;
        const uint8_t* src = out + c_op - c_dist;
        const bool apart = c_dist >= c_len; /* else byte k of the match is byte k mod dist of the `dist` bytes before it */
        uint8_t v = 0;
        uint32_t si = lane;
        if (!apart) si = lane % c_dist; /* (warp-uniform branch: the division is only paid by overlapping matches) */
        if (mine) v = __ldcg(src + si);
        /* lane 0 decodes up to the next match (state 0), the end of the member (1) or an error (2) */
        uint32_t state = 0, len = 0, dist = 0;
        if (lane == 0) {
            for (;;) {
                if (!in_block) {
                    if (last) { state = 1; break; }
                    bool stored = false;
                    err = block_header(b, T, out, out_len, &op, &last, &stored);
                    if (err == OK && b.over()) err = E_INPUT;
                    if (err != OK) { state = 2; break; }
                    in_block = !stored;
                    continue;
                }
                b.refill();
                int s = decode_sym(b, T.lit, LBITS, T.lcount, T.lsym);
                if (s < 0) { err = E_SYMBOL; state = 2; break; }
                if (s < 256) {
                    if (op >= out_len) { err = E_OUTPUT; state = 2; break; }
                    out[op++] = (uint8_t)s;
                    continue;
                }
                if (s == 256) {
                    in_block = false;
                    if (b.over()) { err = E_INPUT; state = 2; break; }
                    continue;
                }
                s -= 257;
                if (s >= 29) { err = E_SYMBOL; state = 2; break; }
                len = c_lbase[s] + b.take(c_lext[s]);
                b.refill();
                const int d = decode_sym(b, T.dist, DBITS, T.dcount, T.dsym);
                if (d < 0 || d >= 30) { err = E_SYMBOL; state = 2; break; }
                dist = c_dbase[d] + b.take(c_dext[d]);
                if (dist > op) { err = E_DIST; state = 2; break; }
                if (op + len > out_len) { err = E_OUTPUT; state = 2; break; }
                break; /* state 0: a match for the whole warp */
            }
        }
        if (mine) out[c_op + lane] = v;
        if (c_len > 32)
            for (uint32_t k = lane + 32; k < c_len; k += 32) out[c_op + k] = __ldcg(src + (apart ? k : k % c_dist));
        const uint32_t packed = __shfl_sync(0xFFFFFFFFu, state | (len << 2) | (dist << 11), 0); /* len <= 258, dist <= 32768 */
        const uint32_t op0 = __shfl_sync(0xFFFFFFFFu, op, 0);
        if ((packed & 3u) != 0) break;
        c_len = (packed >> 2) & 0x1FFu;
        c_dist = packed >> 11;
        c_op = op0;
        if (lane == 0) op += c_len;
        __syncwarp(); /* what lane 0 and the copy stored is visible to the lanes that read it next */
    }
    if (lane == 0) {
        if (err == OK && op != out_len) err = E_OUTPUT;
        if (err == OK && b.used_bytes() != m.clen) err = E_TRAILING;
    }
    err = __shfl_sync(0xFFFFFFFFu, err, 0);
    __syncwarp();
    if (err == OK) {
        /* CRC-32 of the trailer: every lane takes one slice (the bytes were written by all lanes: read around L1), the partial
         * values are combined as zlib's crc32_combine does: crc(A B) = crc(A) x^(8 |B|) mod P ^ crc(B) */
        const uint32_t per = ((out_len + 31) / 32 + 3) & ~3u;
        const uint32_t a0 = min(lane * per, out_len), b0 = min((lane + 1) * per, out_len);
        uint32_t c = 0xFFFFFFFFu, k = a0;
        for (; k < b0 && (((uintptr_t)(out + k)) & 3u); k++) c = crc_t[(c ^ __ldcg(out + k)) & 0xFFu] ^ (c >> 8);
        for (; k + 4 <= b0; k += 4) {
            c ^= __ldcg(reinterpret_cast<const uint32_t*>(out + k));
            c = crc_t[3 * 256 + (c & 0xFFu)] ^ crc_t[2 * 256 + ((c >> 8) & 0xFFu)] ^ crc_t[256 + ((c >> 16) & 0xFFu)] ^ crc_t[c >> 24];
        }
        for (; k < b0; k++) c = crc_t[(c ^ __ldcg(out + k)) & 0xFFu] ^ (c >> 8);
        const uint32_t part = b0 > a0 ? crc_multmodp(crc_x8n(out_len - b0, x2n), ~c) : 0u;
        const uint32_t total = __reduce_xor_sync(0xFFFFFFFFu, part);
        if (total != m.crc) err = 9;
    }
    if (lane == 0 && err != OK) {
        atomicOr(&status[0], 1u << err);
        atomicMax(&status[1], i + 1u);
    }
}
}  // namespace

int gf_bgzf_inflate_device(const uint8_t* d_comp, const GfBgzfMember* d_members, uint32_t n, uint8_t* d_text, unsigned int* d_status,
                           cudaStream_t st) {
    GF_CUDA_TRY(cudaFuncSetAttribute(k_bgzf_inflate, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)INF_SMEM));
    GF_CUDA_TRY(cudaMemsetAsync(d_status, 0, 2 * sizeof(unsigned int), st));
    if (n == 0) return GF_OK;
    k_bgzf_inflate<<<(n + INF_WARPS - 1) / INF_WARPS, INF_WARPS * 32, INF_SMEM, st>>>(d_comp, d_members, n, d_text, d_status);
    GF_CUDA_TRY(cudaGetLastError());
    return GF_OK;
}

int gf_fastq_regather_reads(gf_index* idx, uint64_t bytes, cudaStream_t st) {
    GfFastqReadsWork& w = idx->fq_reads;
    if (w.n == 0 || bytes <= w.arena_used) return GF_OK;
    GF_CUDA_TRY(w.text.reserve(bytes));
    w.arena_used = w.text.cap;
    const unsigned grid = (unsigned)std::max<uint64_t>(1, std::min<uint64_t>((w.n + RD_THREADS - 1) / RD_THREADS, 4ull * idx->sm_count));
    const unsigned long long* nl2 = w.text2 ? idx->fq[1].nl.as<unsigned long long>() : nullptr;
    k_reads_gather<<<grid, RD_THREADS, 0, st>>>(w.text1, idx->fq[0].nl.as<unsigned long long>(), w.text2, nl2,
                                                 w.pairs.as<gf_fastq_read_pair>(), w.slot.as<uint32_t>() + w.n,
                                                 w.total.as<unsigned long long>(), w.arena_used, w.text.as<uint8_t>());
    idx->launches++;
    GF_CUDA_TRY(cudaGetLastError());
    GF_CUDA_TRY(cudaStreamSynchronize(st));
    return GF_OK;
}
