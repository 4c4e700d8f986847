/*
 * gf_index.cu — GPU build of the fusion-gene 16-mer index.
 *
 * Replaces Indexer::make_index / index_contig / fill_bloom_filter
 * (/root/reference/src/core/indexer.rs:122-250):
 *
 *   k_extract_flags / k_extract_items   every window of every gene, both strands, last forward window and
 *                                       first reverse window excluded (index_contig iterates 0..len-16
 *                                       EXCLUSIVE, :188; reverse strand start = 1-len, :168)
 *   k_radix_hist / k_radix_scatter      hand-written stable LSD radix sort of (key, site) by key, 4 x 8 bits
 *   k_classify                          run-length classification 1 / 2..T / >T occurrences
 *                                       (= the dedup state machine of :202-239, T = skip_key_dup_threshold)
 *   k_build_table                       dupe lists + open-addressed table (layout: gf_device.cuh)
 *
 * The 512 MiB bitmap (:243-250) is not materialised: it is an exact membership set of the table's keys,
 * so "bitmap hit" == "key present in the table".
 */
#include <algorithm>
#include <chrono>
#include <cstdio>
#include <cstdlib>
#include <cstring>

#include "gf_internal.h"

namespace {

constexpr int SCAN_THREADS = 256;
constexpr int SCAN_ITEMS = 8;
constexpr int SCAN_TILE = SCAN_THREADS * SCAN_ITEMS; /* 2048 */

/* ---- exclusive scan (u32), writes n+1 outputs (out[n] = total) -------------------------------- */
__global__ void k_scan_reduce(const uint32_t* __restrict__ in, uint64_t n, uint32_t* __restrict__ block_sums) {
    __shared__ uint32_t warp_sums[SCAN_THREADS / 32];
    uint64_t base = (uint64_t)blockIdx.x * SCAN_TILE;
    uint32_t s = 0;
    for (int k = 0; k < SCAN_ITEMS; k++) {
        uint64_t i = base + (uint64_t)k * SCAN_THREADS + threadIdx.x;
        if (i < n) s += in[i];
    }
    for (int o = 16; o > 0; o >>= 1) s += __shfl_down_sync(0xFFFFFFFFu, s, o);
    if ((threadIdx.x & 31) == 0) warp_sums[threadIdx.x >> 5] = s;
    __syncthreads();
    if (threadIdx.x == 0) {
        uint32_t t = 0;
        for (int w = 0; w < SCAN_THREADS / 32; w++) t += warp_sums[w];
        block_sums[blockIdx.x] = t;
    }
}

/* each thread owns SCAN_ITEMS consecutive elements -> in-order scan */
__global__ void k_scan_apply(const uint32_t* __restrict__ in, uint64_t n, const uint32_t* __restrict__ block_offs,
                             uint32_t* __restrict__ out) {
    __shared__ uint32_t warp_sums[SCAN_THREADS / 32];
    uint64_t base = (uint64_t)blockIdx.x * SCAN_TILE + (uint64_t)threadIdx.x * SCAN_ITEMS;
    uint32_t v[SCAN_ITEMS];
    uint32_t s = 0;
    for (int k = 0; k < SCAN_ITEMS; k++) {
        uint64_t i = base + k;
        v[k] = i < n ? in[i] : 0;
        s += v[k];
    }
    uint32_t incl = s;
    uint32_t lane = threadIdx.x & 31;
    for (int o = 1; o < 32; o <<= 1) {
        uint32_t t = __shfl_up_sync(0xFFFFFFFFu, incl, o);
        if (lane >= (uint32_t)o) incl += t;
    }
    if (lane == 31) warp_sums[threadIdx.x >> 5] = incl;
    __syncthreads();
    uint32_t woff = 0;
    for (int w = 0; w < (int)(threadIdx.x >> 5); w++) woff += warp_sums[w];
    uint32_t run = block_offs[blockIdx.x] + woff + incl - s;
    for (int k = 0; k < SCAN_ITEMS; k++) {
        uint64_t i = base + k;
        if (i < n) out[i] = run;
        run += v[k];
    }
    if (blockIdx.x == gridDim.x - 1 && threadIdx.x == SCAN_THREADS - 1) out[n] = block_offs[gridDim.x];
}

/* single-block scan for the top level (n <= a few thousand) */
__global__ void k_scan_small(uint32_t* data, uint32_t n) {
    /* data[0..n) -> exclusive scan in place, data[n] = total; one thread: top levels are tiny */
    if (threadIdx.x == 0 && blockIdx.x == 0) {
        uint32_t run = 0;
        for (uint32_t i = 0; i < n; i++) {
            uint32_t v = data[i];
            data[i] = run;
            run += v;
        }
        data[n] = run;
    }
}

/* recursive host driver; `tmp` must hold the block-sum pyramid (see scan_tmp_elems) */
size_t scan_tmp_elems(uint64_t n) {
    size_t total = 0;
    while (n > 1024) {
        uint64_t nb = (n + SCAN_TILE - 1) / SCAN_TILE;
        total += nb + 1;
        n = nb;
    }
    return total + 2048;
}
cudaError_t exclusive_scan(const uint32_t* in, uint32_t* out, uint64_t n, uint32_t* tmp, cudaStream_t st) {
    if (n == 0) return cudaMemsetAsync(out, 0, sizeof(uint32_t), st);
    uint64_t nb = (n + SCAN_TILE - 1) / SCAN_TILE;
    uint32_t* sums = tmp; /* nb + 1 */
    k_scan_reduce<<<(unsigned)nb, SCAN_THREADS, 0, st>>>(in, n, sums);
    if (nb <= 1024) {
        k_scan_small<<<1, 32, 0, st>>>(sums, (uint32_t)nb);
    } else {
        /* scan the block sums in place through a scratch copy one level up */
        uint32_t* next = tmp + nb + 1;
        cudaError_t e = exclusive_scan(sums, sums, nb, next, st);
        if (e != cudaSuccess) return e;
    }
    k_scan_apply<<<(unsigned)nb, SCAN_THREADS, 0, st>>>(in, n, sums, out);
    return cudaGetLastError();
}

/* ---- k-mer extraction ---------------------------------------------------------------------------- */
/* One thread per arena position g (a candidate window start).  Gene bytes are upper-case ASCII, padding is
 * 0 -> a window that touches padding is invalid by itself.
 *   forward item : valid window and byte g+16 still inside the gene  (excludes the window at len-16)
 *   reverse item : valid window and byte g-1 still inside the gene   (excludes the window at 0)        */
constexpr int EX_THREADS = 256;
__device__ __forceinline__ void extract_window(const uint8_t* tile, int t, uint32_t* key, bool* fwd, bool* rev) {
    /* tile[0] = byte g-1 of thread 0 */
    bool ok = gf_kmer_from_ascii(tile + t + 1, key);
    *fwd = ok && tile[t + 17] != 0;
    *rev = ok && tile[t] != 0;
}
__device__ __forceinline__ void load_tile(const uint8_t* __restrict__ arena, uint64_t arena_len, uint64_t g0, uint8_t* tile) {
    for (int k = threadIdx.x; k < EX_THREADS + 17; k += EX_THREADS) {
        int64_t g = (int64_t)g0 + k - 1;
        tile[k] = (g >= 0 && (uint64_t)g < arena_len) ? arena[g] : 0;
    }
    __syncthreads();
}
__global__ void k_extract_flags(const uint8_t* __restrict__ arena, uint64_t arena_len, uint32_t* __restrict__ flags) {
    __shared__ uint8_t tile[EX_THREADS + 32];
    uint64_t g0 = (uint64_t)blockIdx.x * EX_THREADS;
    load_tile(arena, arena_len, g0, tile);
    uint64_t g = g0 + threadIdx.x;
    if (g >= arena_len) return;
    uint32_t key;
    bool f, r;
    extract_window(tile, threadIdx.x, &key, &f, &r);
    flags[2 * g] = f;
    flags[2 * g + 1] = r;
}
__global__ void k_extract_items(const uint8_t* __restrict__ arena, uint64_t arena_len,
                                const uint32_t* __restrict__ pos, unsigned long long* __restrict__ items) {
    __shared__ uint8_t tile[EX_THREADS + 32];
    uint64_t g0 = (uint64_t)blockIdx.x * EX_THREADS;
    load_tile(arena, arena_len, g0, tile);
    uint64_t g = g0 + threadIdx.x;
    if (g >= arena_len) return;
    uint32_t key;
    bool f, r;
    extract_window(tile, threadIdx.x, &key, &f, &r);
    if (f) items[pos[2 * g]] = ((unsigned long long)key << 32) | (uint32_t)g;
    if (r) items[pos[2 * g + 1]] = ((unsigned long long)gf_key_revcomp(key) << 32) | (GF_SITE_STRAND | (uint32_t)(g + 15));
}

/* ---- stable LSD radix sort on the key half (bits 32..63), 8 bits per pass ---------------------------- */
constexpr int RS_WARPS = 8;
constexpr int RS_TILE = 2048; /* items per warp */

__global__ void k_radix_hist(const unsigned long long* __restrict__ items, uint64_t n, int shift,
                             uint32_t* __restrict__ hist, uint32_t n_tiles) {
    __shared__ uint32_t sh[RS_WARPS][256];
    uint32_t warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    uint32_t tile = blockIdx.x * RS_WARPS + warp;
    for (int d = lane; d < 256; d += 32) sh[warp][d] = 0;
    __syncwarp();
    if (tile < n_tiles) {
        uint64_t base = (uint64_t)tile * RS_TILE;
        for (int c = 0; c < RS_TILE; c += 32) {
            uint64_t i = base + c + lane;
            uint32_t d = i < n ? (uint32_t)((items[i] >> shift) & 0xFF) : 256u + lane;
            uint32_t peers = __match_any_sync(0xFFFFFFFFu, d);
            if (i < n && (peers & gf_lanemask_lt()) == 0) sh[warp][d] += __popc(peers);
            __syncwarp();
        }
        for (int d = lane; d < 256; d += 32) hist[(uint64_t)d * n_tiles + tile] = sh[warp][d];
    }
}
__global__ void k_radix_scatter(const unsigned long long* __restrict__ items, uint64_t n, int shift,
                                const uint32_t* __restrict__ offs, uint32_t n_tiles,
                                unsigned long long* __restrict__ out) {
    __shared__ uint32_t sh[RS_WARPS][256];
    uint32_t warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    uint32_t tile = blockIdx.x * RS_WARPS + warp;
    if (tile >= n_tiles) return;
    for (int d = lane; d < 256; d += 32) sh[warp][d] = offs[(uint64_t)d * n_tiles + tile];
    __syncwarp();
    uint64_t base = (uint64_t)tile * RS_TILE;
    for (int c = 0; c < RS_TILE; c += 32) {
        uint64_t i = base + c + lane;
        unsigned long long it = i < n ? items[i] : 0ull;
        uint32_t d = i < n ? (uint32_t)((it >> shift) & 0xFF) : 256u + lane;
        uint32_t peers = __match_any_sync(0xFFFFFFFFu, d);
        uint32_t rank = __popc(peers & gf_lanemask_lt());
        uint32_t dst = 0;
        if (i < n) dst = sh[warp][d] + rank;
        __syncwarp();
        if (i < n && rank == 0) sh[warp][d] += __popc(peers);
        __syncwarp();
        if (i < n) out[dst] = it;
    }
}

/* ---- run-length classification --------------------------------------------------------------------- */
__device__ __forceinline__ uint32_t run_len_capped(const unsigned long long* items, uint64_t n, uint64_t i, uint32_t cap) {
    uint32_t key = (uint32_t)(items[i] >> 32);
    uint32_t cnt = 1;
    while (cnt < cap && i + cnt < n && (uint32_t)(items[i + cnt] >> 32) == key) cnt++;
    return cnt;
}
/* stats: [0] keys [1] unique [2] normal [3] high */
__global__ void k_classify(const unsigned long long* __restrict__ items, uint64_t n, uint32_t thr,
                           uint32_t* __restrict__ ncnt, unsigned long long* __restrict__ stats) {
    uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    bool head = i == 0 || (uint32_t)(items[i] >> 32) != (uint32_t)(items[i - 1] >> 32);
    uint32_t c = 0;
    if (head) {
        uint32_t len = run_len_capped(items, n, i, thr + 1);
        atomicAdd(&stats[0], 1ull);
        if (len == 1) atomicAdd(&stats[1], 1ull);
        else if (len <= thr) { atomicAdd(&stats[2], 1ull); c = len; }
        else atomicAdd(&stats[3], 1ull);
    }
    ncnt[i] = c;
}
__global__ void k_build_table(const unsigned long long* __restrict__ items, uint64_t n, uint32_t thr,
                              const uint32_t* __restrict__ dupe_off, uint32_t* __restrict__ dupes,
                              unsigned long long* __restrict__ table, uint32_t bucket_shift, uint32_t bucket_mask,
                              unsigned int* __restrict__ max_disp, unsigned long long* __restrict__ filter,
                              uint32_t filter_words, unsigned long long* __restrict__ filter_multi,
                              uint32_t filter_multi_words) {
    uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    uint32_t key = (uint32_t)(items[i] >> 32);
    bool head = i == 0 || key != (uint32_t)(items[i - 1] >> 32);
    if (!head) return;
    uint32_t len = run_len_capped(items, n, i, thr + 1);
    uint32_t val;
    if (len == 1) {
        val = (GF_KIND_UNIQUE << 30) | (uint32_t)(items[i] & 0x3FFFFFFFull);
    } else if (len <= thr) {
        uint32_t off = dupe_off[i];
        for (uint32_t j = 0; j < len; j++) dupes[off + j] = (uint32_t)(items[i + j] & 0x3FFFFFFFull);
        val = (GF_KIND_NORMAL << 30) | (off << 3) | len;
    } else {
        val = (GF_KIND_HIGH << 30);
    }
    if (len <= thr) { /* unique and NORMAL keys vote; HIGH keys never do and stay out of the filter */
        uint32_t al, ah;
        gf_filter_masks(key, &al, &ah);
        atomicOr(filter + gf_filter_word(key, filter_words), ((unsigned long long)ah << 32) | al);
        if (len > 1) atomicOr(filter_multi + gf_multi_word(key, filter_multi_words), gf_multi_mask(key));
    }
    unsigned long long entry = ((unsigned long long)val << 32) | key;
    uint32_t b = gf_home_bucket(key, bucket_shift);
    uint32_t disp = 0;
    for (;;) {
        unsigned long long* slot = table + 4ull * b;
        bool done = false;
        for (int s = 0; s < 4 && !done; s++) {
            if (slot[s] == ~0ull) done = atomicCAS(slot + s, ~0ull, entry) == ~0ull;
        }
        if (done) break;
        b = (b + 1) & bucket_mask;
        disp++;
    }
    if (disp) atomicMax(max_disp, disp);
}

/* ---- L2-resident screen structures ------------------------------------------------------------------ */
/* gene arena -> bit-planes (thread per 32-base word) */
__global__ void k_gene_planes(const uint8_t* __restrict__ arena, uint64_t arena_len, uint32_t n_words,
                              uint32_t* __restrict__ lo, uint32_t* __restrict__ hi, uint32_t* __restrict__ v) {
    uint32_t w = blockIdx.x * blockDim.x + threadIdx.x;
    if (w >= n_words) return;
    uint32_t blo = 0, bhi = 0, bv = 0;
    for (int j = 0; j < 32; j++) {
        uint64_t g = 32ull * w + j;
        uint32_t c = g < arena_len ? arena[g] : 0u;
        if (gf_is_acgt_upper(c)) {
            bv |= 1u << j;
            blo |= gf_code_lo(c) << j;
            bhi |= gf_code_hi(c) << j;
        }
    }
    lo[w] = blo; hi[w] = bhi; v[w] = bv;
}
/* per window and strand: number of sites its k-mer votes for if the window is an indexed site (0 otherwise / HIGH) */
__device__ __forceinline__ uint32_t window_sites(const GfDevIndex& ix, uint32_t key) {
    uint32_t val = gf_table_find(ix, key);
    if (val == GF_EMPTY_VAL) return 0u;
    uint32_t kind = val >> 30;
    return kind == GF_KIND_UNIQUE ? 1u : (kind == GF_KIND_NORMAL ? (val & 7u) : 0u);
}
__global__ void k_window_class(GfDevIndex ix, const uint8_t* __restrict__ arena, uint64_t arena_len,
                               uint32_t* __restrict__ cf, uint32_t* __restrict__ cr, uint32_t stride) {
    __shared__ uint8_t tile[EX_THREADS + 32];
    uint64_t g0 = (uint64_t)blockIdx.x * EX_THREADS;
    load_tile(arena, arena_len, g0, tile);
    uint64_t g = g0 + threadIdx.x;
    uint32_t key = 0;
    bool f = false, r = false;
    if (g < arena_len) extract_window(tile, threadIdx.x, &key, &f, &r);
    uint32_t nf = f ? window_sites(ix, key) : 0u;
    uint32_t nr = r ? window_sites(ix, gf_key_revcomp(key)) : 0u;
    for (int b = 0; b < 3; b++) {
        uint32_t mf = __ballot_sync(0xFFFFFFFFu, (nf >> b) & 1u), mr = __ballot_sync(0xFFFFFFFFu, (nr >> b) & 1u);
        if ((threadIdx.x & 31) == 0) { cf[(size_t)b * stride + (g >> 5)] = mf; cr[(size_t)b * stride + (g >> 5)] = mr; }
    }
}

/* ---- parity hook: lookups ---------------------------------------------------------------------------- */
__global__ void k_lookup(GfDevIndex ix, const uint32_t* __restrict__ kmers, uint64_t n, gf_lookup* __restrict__ out) {
    uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    gf_lookup o;
    memset(&o, 0, sizeof(o));
    uint32_t v = gf_table_find(ix, gf_key_from_refcode(kmers[i]));
    if (v != GF_EMPTY_VAL) {
        uint32_t kind = v >> 30;
        if (kind == GF_KIND_UNIQUE) {
            int32_t c, p;
            gf_site_decode(ix, v & 0x3FFFFFFFu, &c, &p);
            o.kind = 1;
            o.n_sites = 1;
            o.contig[0] = (int16_t)c;
            o.position[0] = p;
        } else if (kind == GF_KIND_NORMAL) {
            uint32_t cnt = v & 7u, off = (v >> 3) & 0x07FFFFFFu;
            o.kind = 2;
            o.n_sites = (int32_t)cnt;
            for (uint32_t j = 0; j < cnt; j++) {
                int32_t c, p;
                gf_site_decode(ix, ix.dupes[off + j], &c, &p);
                /* insertion sort by (contig, position): the order inside a dupe list is unobservable */
                int k = (int)j;
                while (k > 0 && (o.contig[k - 1] > c || (o.contig[k - 1] == c && o.position[k - 1] > p))) {
                    o.contig[k] = o.contig[k - 1];
                    o.position[k] = o.position[k - 1];
                    k--;
                }
                o.contig[k] = (int16_t)c;
                o.position[k] = p;
            }
        } else {
            o.kind = 3;
        }
    }
    out[i] = o;
}

}  // namespace

/* exported to the other translation units (gf_fastq.cu) */
size_t gf_scan_tmp_elems(uint64_t n) { return scan_tmp_elems(n); }
cudaError_t gf_exclusive_scan_u32(const uint32_t* in, uint32_t* out, uint64_t n, uint32_t* tmp, cudaStream_t st) {
    return exclusive_scan(in, out, n, tmp, st);
}
uint32_t gf_scan_launches(uint64_t n) {
    if (n == 0) return 0;
    const uint64_t nb = (n + SCAN_TILE - 1) / SCAN_TILE;
    return 2 + (nb <= 1024 ? 1 : gf_scan_launches(nb));
}

/* ======================================================================================================= */
namespace {
struct PhaseTimer { /* GF_DEBUG_TIMING=1: host wall clock per build phase on stderr */
    bool on;
    std::chrono::steady_clock::time_point t0;
    PhaseTimer() : on(getenv("GF_DEBUG_TIMING") != nullptr), t0(std::chrono::steady_clock::now()) {}
    void mark(const char* what) {
        if (!on) return;
        cudaDeviceSynchronize();
        auto t1 = std::chrono::steady_clock::now();
        fprintf(stderr, "[gf build] %-28s %8.2f ms\n", what, std::chrono::duration<double, std::milli>(t1 - t0).count());
        t0 = t1;
    }
};
}  // namespace

namespace {
/* error paths return through GF_CUDA_TRY: temporaries and events are released by these guards */
struct DevTmp {
    void* p = nullptr;
    ~DevTmp() { if (p) cudaFree(p); }
};
struct EventGuard {
    cudaEvent_t e = nullptr;
    ~EventGuard() { if (e) cudaEventDestroy(e); }
};
/* one device allocation for every temporary of the build (cudaMalloc/cudaFree are slow, synchronising calls) */
struct BuildWorkspace {
    char* base = nullptr;
    size_t cap = 0, used = 0;
    ~BuildWorkspace() { if (base) cudaFree(base); }
    cudaError_t init(size_t bytes) { cap = bytes; return cudaMalloc((void**)&base, bytes); }
    template <class T>
    T* take(size_t n) {
        size_t bytes = (n * sizeof(T) + 255) & ~(size_t)255;
        if (used + bytes > cap) return nullptr;
        T* p = reinterpret_cast<T*>(base + used);
        used += bytes;
        return p;
    }
};
/* planes lo, hi, valid, cf[3], cr[3] (each `stride` words) -> two interleaved arrays of 8 words per arena word */
__global__ void k_interleave_planes(const uint32_t* __restrict__ pl, uint32_t stride, uint32_t* __restrict__ g_if,
                                    uint32_t* __restrict__ g_ir) {
    const uint32_t w = blockIdx.x * blockDim.x + threadIdx.x;
    if (w >= stride) return;
    const uint32_t lo = pl[w], hi = pl[(size_t)stride + w], v = pl[2ull * stride + w];
    uint4* f = reinterpret_cast<uint4*>(g_if + 8ull * w);
    uint4* r = reinterpret_cast<uint4*>(g_ir + 8ull * w);
    f[0] = make_uint4(lo, hi, v, pl[3ull * stride + w]);
    f[1] = make_uint4(pl[4ull * stride + w], pl[5ull * stride + w], 0u, 0u);
    r[0] = make_uint4(lo, hi, v, pl[6ull * stride + w]);
    r[1] = make_uint4(pl[7ull * stride + w], pl[8ull * stride + w], 0u, 0u);
}

}  // namespace

int gf_build_index_device(gf_index* idx, const gf_gene_span* genes, uint32_t n_genes) {
    PhaseTimer pt;
    /* index_contig (:202-239): the 2nd occurrence always opens a dupe list of 2; occurrence n >= 3 is pushed
     * while the list holds < threshold sites  =>  NORMAL iff 2 <= n <= max(threshold, 2), HIGH beyond */
    const uint32_t thr = (uint32_t)std::max(idx->params.skip_key_dup_threshold, 2);
    cudaStream_t st = idx->stream;

    /* host: padded upper-case arena */
    idx->n_genes = n_genes;
    idx->gene_start.resize(n_genes);
    idx->gene_len.resize(n_genes);
    std::vector<uint8_t> rev(n_genes ? n_genes : 1, 0);
    uint64_t cur = GF_GENE_PAD, gene_bytes = 0;
    for (uint32_t g = 0; g < n_genes; g++) {
        idx->gene_start[g] = (uint32_t)cur;
        idx->gene_len[g] = genes[g].len;
        rev[g] = genes[g].reversed ? 1 : 0;
        gene_bytes += genes[g].len;
        cur += genes[g].len + GF_GENE_PAD;
        cur = (cur + 15) & ~15ull;
        if (cur >= GF_MAX_GOFF) {
            gf_set_error("gene panel too large for the 29-bit site encoding (sum of gene lengths + padding >= 2^29)");
            return GF_E_LIMIT;
        }
    }
    const uint64_t arena_len = cur;
    std::vector<uint8_t> arena(arena_len, 0);
    for (uint32_t g = 0; g < n_genes; g++) {
        uint8_t* dst = arena.data() + idx->gene_start[g];
        const uint8_t* src = genes[g].seq;
        for (uint32_t k = 0; k < genes[g].len; k++) {
            uint8_t c = src[k];
            if (c >= 'a' && c <= 'z') c = (uint8_t)(c - 32); /* to_uppercase, indexer.rs:159 */
            if (c == 0) c = 1;                                /* 0 is the padding marker; both are non-ACGT */
            dst[k] = c;
        }
    }

    pt.mark("host arena");
    /* granule -> contig table (site decoding) */
    std::vector<uint16_t> granule((arena_len >> 11) + 2, 0);
    for (uint32_t g = 0; g < n_genes; g++)
        if (genes[g].len)
            for (uint64_t q = idx->gene_start[g] >> 11; q <= ((uint64_t)idx->gene_start[g] + genes[g].len - 1) >> 11; q++)
                granule[q] = (uint16_t)g;
    EventGuard g0, g1;
    GF_CUDA_TRY(cudaEventCreate(&g0.e));
    GF_CUDA_TRY(cudaEventCreate(&g1.e));
    const cudaEvent_t e0 = g0.e, e1 = g1.e;
    GF_CUDA_TRY(cudaMalloc(&idx->d_gene_ascii, arena_len));
    GF_CUDA_TRY(cudaMalloc(&idx->d_gene_start, sizeof(uint32_t) * (n_genes + 1)));
    GF_CUDA_TRY(cudaMalloc(&idx->d_gene_len, sizeof(uint32_t) * (n_genes + 1)));
    GF_CUDA_TRY(cudaMalloc(&idx->d_gene_rev, n_genes + 1));
    GF_CUDA_TRY(cudaMalloc(&idx->d_granule, sizeof(uint16_t) * granule.size()));
    GF_CUDA_TRY(cudaMemcpyAsync(idx->d_granule, granule.data(), sizeof(uint16_t) * granule.size(), cudaMemcpyHostToDevice, st));
    idx->dev.granule_contig = (const uint16_t*)idx->d_granule;
    GF_CUDA_TRY(cudaMemcpyAsync(idx->d_gene_ascii, arena.data(), arena_len, cudaMemcpyHostToDevice, st));
    if (n_genes) {
        GF_CUDA_TRY(cudaMemcpyAsync(idx->d_gene_start, idx->gene_start.data(), sizeof(uint32_t) * n_genes,
                                    cudaMemcpyHostToDevice, st));
        GF_CUDA_TRY(cudaMemcpyAsync(idx->d_gene_len, idx->gene_len.data(), sizeof(uint32_t) * n_genes,
                                    cudaMemcpyHostToDevice, st));
        GF_CUDA_TRY(cudaMemcpyAsync(idx->d_gene_rev, rev.data(), n_genes, cudaMemcpyHostToDevice, st));
    }
    GF_CUDA_TRY(cudaEventRecord(e0, st));

    pt.mark("upload genes");
    /* 1. flags -> positions -> compacted (key, site) items */
    const uint64_t n_flags = 2 * arena_len;
    const uint64_t max_tiles = (n_flags + RS_TILE - 1) / RS_TILE, max_hist = 256ull * max_tiles;
    BuildWorkspace ws;
    {
        size_t need = 4 * (n_flags + 64) * 4 /* flags, pos, ncnt, doff */ + 8 * (n_flags + 64) * 2 /* items x2 */ +
                      4 * (max_hist + 64) * 2 + 4 * (scan_tmp_elems(n_flags + 1) * 2 + scan_tmp_elems(max_hist)) + 4096 +
                      256 * 16;
        GF_CUDA_TRY(ws.init(need));
    }
    uint32_t* d_flags = ws.take<uint32_t>(n_flags);
    uint32_t* d_pos = ws.take<uint32_t>(n_flags + 1);
    uint32_t* d_tmp = ws.take<uint32_t>(scan_tmp_elems(n_flags));
    const unsigned ex_blocks = (unsigned)((arena_len + EX_THREADS - 1) / EX_THREADS);
    k_extract_flags<<<ex_blocks, EX_THREADS, 0, st>>>((const uint8_t*)idx->d_gene_ascii, arena_len, d_flags);
    GF_CUDA_TRY(exclusive_scan(d_flags, d_pos, n_flags, d_tmp, st));
    uint32_t n_items32 = 0;
    GF_CUDA_TRY(cudaMemcpyAsync(&n_items32, d_pos + n_flags, sizeof(uint32_t), cudaMemcpyDeviceToHost, st));
    GF_CUDA_TRY(cudaStreamSynchronize(st));
    const uint64_t n_items = n_items32;
    unsigned long long* d_items = ws.take<unsigned long long>(n_items + 1);
    unsigned long long* d_items2 = ws.take<unsigned long long>(n_items + 1);
    k_extract_items<<<ex_blocks, EX_THREADS, 0, st>>>((const uint8_t*)idx->d_gene_ascii, arena_len, d_pos, d_items);
    GF_CUDA_TRY(cudaGetLastError());

    pt.mark("extract k-mers");
    /* 2. radix sort by key */
    if (n_items > 1) {
        const uint32_t n_tiles = (uint32_t)((n_items + RS_TILE - 1) / RS_TILE);
        const uint64_t n_hist = 256ull * n_tiles;
        uint32_t* d_hist = ws.take<uint32_t>(n_hist);
        uint32_t* d_offs = ws.take<uint32_t>(n_hist + 1);
        uint32_t* d_stmp = ws.take<uint32_t>(scan_tmp_elems(n_hist));
        if (!d_hist || !d_offs || !d_stmp) { gf_set_error("internal: build workspace too small"); return GF_E_CUDA; }
        const unsigned rs_blocks = (n_tiles + RS_WARPS - 1) / RS_WARPS;
        for (int pass = 0; pass < 4; pass++) {
            int shift = 32 + 8 * pass;
            k_radix_hist<<<rs_blocks, RS_WARPS * 32, 0, st>>>(d_items, n_items, shift, d_hist, n_tiles);
            GF_CUDA_TRY(exclusive_scan(d_hist, d_offs, n_hist, d_stmp, st));
            k_radix_scatter<<<rs_blocks, RS_WARPS * 32, 0, st>>>(d_items, n_items, shift, d_offs, n_tiles, d_items2);
            std::swap(d_items, d_items2);
        }
        GF_CUDA_TRY(cudaGetLastError());
        GF_CUDA_TRY(cudaStreamSynchronize(st));
    }

    pt.mark("radix sort");
    /* 3. classify runs */
    uint32_t* d_ncnt = ws.take<uint32_t>(n_items + 1);
    uint32_t* d_doff = ws.take<uint32_t>(n_items + 2);
    uint32_t* d_tmp2 = ws.take<uint32_t>(scan_tmp_elems(n_items + 1));
    unsigned long long* d_stats = ws.take<unsigned long long>(8);
    if (!d_flags || !d_pos || !d_tmp || !d_items || !d_items2 || !d_ncnt || !d_doff || !d_tmp2 || !d_stats) {
        gf_set_error("internal: build workspace too small");
        return GF_E_CUDA;
    }
    GF_CUDA_TRY(cudaMemsetAsync(d_stats, 0, sizeof(unsigned long long) * 8, st));
    unsigned long long h_stats[8] = {0, 0, 0, 0, 0, 0, 0, 0};
    uint32_t n_dupes = 0;
    if (n_items) {
        const unsigned cb = (unsigned)((n_items + 255) / 256);
        k_classify<<<cb, 256, 0, st>>>(d_items, n_items, thr, d_ncnt, d_stats);
        GF_CUDA_TRY(exclusive_scan(d_ncnt, d_doff, n_items, d_tmp2, st));
        GF_CUDA_TRY(cudaMemcpyAsync(&n_dupes, d_doff + n_items, sizeof(uint32_t), cudaMemcpyDeviceToHost, st));
        GF_CUDA_TRY(cudaMemcpyAsync(h_stats, d_stats, sizeof(h_stats), cudaMemcpyDeviceToHost, st));
        GF_CUDA_TRY(cudaStreamSynchronize(st));
    }
    if (n_dupes >= (1u << 27)) {
        gf_set_error("too many NORMAL dupe sites for the 27-bit dupe offset");
        return GF_E_LIMIT;
    }

    pt.mark("classify");
    /* 4. table */
    const uint64_t n_keys = h_stats[0];
    uint32_t bucket_bits = 6;
    while ((1ull << bucket_bits) * 2 < n_keys) bucket_bits++; /* <= 2 keys per 4-slot bucket on average */
    const uint64_t n_buckets = 1ull << bucket_bits;
    GF_CUDA_TRY(cudaMalloc(&idx->d_table, n_buckets * 32));
    GF_CUDA_TRY(cudaMemsetAsync(idx->d_table, 0xFF, n_buckets * 32, st));
    GF_CUDA_TRY(cudaMalloc(&idx->d_dupes, sizeof(uint32_t) * ((size_t)n_dupes + 8)));
    unsigned int* d_maxdisp = (unsigned int*)(d_stats + 6);
    /* blocked Bloom filter, 8 bits per key (the filter must stay L2-resident next to the gene planes), whole 64-bit words,
     * at least 1024 words */
    const int filter_bits = 8;
    const uint32_t filter_words = (uint32_t)std::max<uint64_t>(1024, (n_keys * (uint64_t)filter_bits + 63) / 64);
    /* + the multi filter behind it: 16 bits per NORMAL key */
    const uint32_t filter_multi_words = (uint32_t)std::max<uint64_t>(1024, (h_stats[2] * 16 + 63) / 64);
    GF_CUDA_TRY(cudaMalloc(&idx->d_filter, sizeof(unsigned long long) * ((size_t)filter_words + filter_multi_words)));
    GF_CUDA_TRY(cudaMemsetAsync(idx->d_filter, 0, sizeof(unsigned long long) * ((size_t)filter_words + filter_multi_words), st));
    unsigned long long* d_filter_multi = (unsigned long long*)idx->d_filter + filter_words;
    if (n_items) {
        const unsigned cb = (unsigned)((n_items + 255) / 256);
        k_build_table<<<cb, 256, 0, st>>>(d_items, n_items, thr, d_doff, (uint32_t*)idx->d_dupes,
                                          (unsigned long long*)idx->d_table, 32 - bucket_bits,
                                          (uint32_t)(n_buckets - 1), d_maxdisp, (unsigned long long*)idx->d_filter,
                                          filter_words, d_filter_multi, filter_multi_words);
        GF_CUDA_TRY(cudaGetLastError());
    }
    unsigned int h_maxdisp = 0;
    GF_CUDA_TRY(cudaMemcpyAsync(&h_maxdisp, d_maxdisp, sizeof(unsigned int), cudaMemcpyDeviceToHost, st));
    GF_CUDA_TRY(cudaStreamSynchronize(st));

    pt.mark("table + filter");
    idx->dev.table = (const uint4*)idx->d_table;
    idx->dev.dupes = (const uint32_t*)idx->d_dupes;
    idx->dev.gene_ascii = (const uint8_t*)idx->d_gene_ascii;
    idx->dev.gene_start = (const uint32_t*)idx->d_gene_start;
    idx->dev.gene_len = (const uint32_t*)idx->d_gene_len;
    idx->dev.gene_rev = (const uint8_t*)idx->d_gene_rev;
    idx->dev.n_genes = n_genes;
    idx->dev.max_sites = thr;
    idx->dev.bucket_shift = 32 - bucket_bits;
    idx->dev.bucket_mask = (uint32_t)(n_buckets - 1);
    idx->dev.major_req = idx->params.major_gene_key_requirement;
    idx->dev.minor_req = idx->params.minor_gene_key_requirement;
    idx->dev.mismatch_thr = idx->params.mismatch_threshold;
    idx->dev.deletion_thr = idx->params.deletion_threshold;
    idx->dev.filter = (const unsigned long long*)idx->d_filter;
    idx->dev.filter_words = filter_words;
    idx->dev.filter_multi = d_filter_multi;
    idx->dev.filter_multi_words = filter_multi_words;

    /* gene bit-planes (lo, hi, valid) + per-window site-count planes (3 bits x 2 strands), built as 9 separate planes in a
     * temporary and interleaved into the two resident arrays g_if / g_ir (one 32-byte entry per arena word and strand; the
     * allocation is 256-byte aligned, so every entry is sector aligned).  72 pad words: the longest diagonal walk reads
     * (2048 + 64) / 32 + 2 words beyond its start. */
    const uint32_t n_pw = (uint32_t)((arena_len + 31) / 32);
    const size_t plane_stride = ((size_t)n_pw + 72 + 7) & ~(size_t)7;
    DevTmp tmp_planes;
    GF_CUDA_TRY(cudaMalloc(&tmp_planes.p, sizeof(uint32_t) * plane_stride * 9));
    GF_CUDA_TRY(cudaMemsetAsync(tmp_planes.p, 0, sizeof(uint32_t) * plane_stride * 9, st));
    GF_CUDA_TRY(cudaMalloc(&idx->d_planes, sizeof(uint32_t) * plane_stride * 16));
    uint32_t* pl = (uint32_t*)tmp_planes.p;
    uint32_t* gi = (uint32_t*)idx->d_planes;
    k_gene_planes<<<(n_pw + 255) / 256, 256, 0, st>>>((const uint8_t*)idx->d_gene_ascii, arena_len, n_pw, pl,
                                                      pl + plane_stride, pl + 2 * plane_stride);
    k_window_class<<<ex_blocks, EX_THREADS, 0, st>>>(idx->dev, (const uint8_t*)idx->d_gene_ascii, arena_len,
                                                     pl + 3 * plane_stride, pl + 6 * plane_stride,
                                                     (uint32_t)plane_stride);
    idx->dev.g_if = gi;
    idx->dev.g_ir = gi + 8 * plane_stride;
    k_interleave_planes<<<(unsigned)((plane_stride + 255) / 256), 256, 0, st>>>(pl, (uint32_t)plane_stride, gi, gi + 8 * plane_stride);
    GF_CUDA_TRY(cudaGetLastError());
    GF_CUDA_TRY(cudaEventRecord(e1, st));
    GF_CUDA_TRY(cudaStreamSynchronize(st));
    float ms = 0;
    GF_CUDA_TRY(cudaEventElapsedTime(&ms, e0, e1));

    pt.mark("gene planes + window class");
    gf_index_info& inf = idx->info;
    inf.n_sites = n_items;
    inf.n_keys = n_keys;
    inf.n_unique = h_stats[1];
    inf.n_normal = h_stats[2];
    inf.n_high = h_stats[3];
    inf.table_slots = n_buckets * 4;
    inf.table_bytes = n_buckets * 32;
    inf.max_displacement = h_maxdisp;
    inf.gene_bytes = gene_bytes;
    inf.device_bytes = n_buckets * 32 + sizeof(uint32_t) * ((size_t)n_dupes + 8) + arena_len + 9ull * (n_genes + 1) +
                       sizeof(uint32_t) * plane_stride * 16 + sizeof(unsigned long long) * ((size_t)filter_words + filter_multi_words);
    inf.build_ms = ms;
    return GF_OK;
}

int gf_lookup_device(gf_index* idx, const uint32_t* kmers, uint64_t n, gf_lookup* out) {
    if (n == 0) return GF_OK;
    DevTmp k, o;
    GF_CUDA_TRY(cudaMalloc(&k.p, sizeof(uint32_t) * n));
    GF_CUDA_TRY(cudaMalloc(&o.p, sizeof(gf_lookup) * n));
    GF_CUDA_TRY(cudaMemcpyAsync(k.p, kmers, sizeof(uint32_t) * n, cudaMemcpyHostToDevice, idx->stream));
    k_lookup<<<(unsigned)((n + 127) / 128), 128, 0, idx->stream>>>(idx->dev, (const uint32_t*)k.p, n, (gf_lookup*)o.p);
    GF_CUDA_TRY(cudaGetLastError());
    GF_CUDA_TRY(cudaMemcpyAsync(out, o.p, sizeof(gf_lookup) * n, cudaMemcpyDeviceToHost, idx->stream));
    GF_CUDA_TRY(cudaStreamSynchronize(idx->stream));
    return GF_OK;
}
