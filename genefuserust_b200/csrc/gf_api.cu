/*
 * gf_api.cu — the C ABI (include/genefuse_gpu.h): handles, host<->device staging, stream pipeline.
 * No CPU fallback: every compute entry point needs a CUDA device and fails with GF_E_CUDA otherwise.
 */
#include <algorithm>
#include <chrono>
#include <cstdlib>
#include <condition_variable>
#include <cstring>
#include <mutex>
#include <thread>

#include "gf_internal.h"

static thread_local std::string g_last_error;
void gf_set_error(const std::string& msg) { g_last_error = msg; }

/* packed upload, a chunk whose reads all have one length: off[i] = base + i * len (n + 1 entries), and where read i's plane
 * words start: pko[i] = i * 2 * ceil(len / 32) — nothing the host would have to send */
__global__ void k_fill_uniform(uint64_t* off, uint32_t* pko, uint64_t base, uint32_t len, uint64_t n) {
    const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i <= n) off[i] = base + i * len;
    if (i < n) pko[i] = (uint32_t)(i * 2u * ((len + 31u) >> 5));
}

namespace {

constexpr uint64_t CHUNK_TARGET_BYTES = 192ull << 20; /* sequence+quality bytes per pipeline chunk */

int fail(int code, const std::string& msg) {
    gf_set_error(msg);
    return code;
}

void accumulate(gf_map_stats& st, const GfHostSlot& h) {
    st.n_sequences += h.counters.n_sequences;
    st.n_probes_pass1 += h.counters.n_probes;
    st.n_survivors += h.counters.n_survivors + h.counters.n_survivors_total;
    st.n_matches += h.n_out;
    st.seq_bytes += h.counters.seq_bytes;
}

int check_flags(const GfHostSlot& h) {
    if (h.counters.error_flags & 1u)
        return fail(GF_E_INVALID, "a read is longer than the kernel capacity (max_len hint too small, or > 1024 bases)");
    if (h.counters.error_flags & 2u) return fail(GF_E_CUDA, "internal: survivor list overflow");
    return GF_OK;
}

/* gf_map_pairs_device* return with work in flight on the caller's stream; that work uses the handle's workspace
 * (counters, survivor list, sequence store, vote tables, the pinned result slot).  Every entry point that touches the
 * workspace first makes its own stream wait for it. */
int wait_prior_device_work(gf_index* idx, cudaStream_t st) {
    if (idx->busy) GF_CUDA_TRY(cudaStreamWaitEvent(st, idx->ev_busy, 0));
    return GF_OK;
}
int mark_device_work(gf_index* idx, cudaStream_t st) {
    GF_CUDA_TRY(cudaEventRecord(idx->ev_busy, st));
    idx->busy = true;
    return GF_OK;
}

/* Host offsets of one mate: ascending, every record at most `limit` long.  Returns the longest record in *max_len.
 * (Several threads: ~1 ms per 10 M reads.) */
int scan_offsets(const uint64_t* off1, const uint64_t* off2, uint64_t n, uint64_t limit, uint64_t* max_len, unsigned max_threads = 16) {
    const unsigned nt = n < (1u << 16) ? 1u : std::max(1u, std::min(max_threads, std::thread::hardware_concurrency()));
    std::vector<uint64_t> part(nt, 0);
    std::vector<char> bad(nt, 0);
    auto work = [&](unsigned t) {
        uint64_t mx = 0;
        bool b = false;
        for (uint64_t i = n * t / nt; i < n * (t + 1) / nt; i++) {
            const uint64_t a = off1[i], e = off1[i + 1];
            b |= e < a;
            mx = std::max(mx, e - a);
            if (off2) {
                const uint64_t a2 = off2[i], e2 = off2[i + 1];
                b |= e2 < a2;
                mx = std::max(mx, e2 - a2);
            }
        }
        part[t] = mx;
        bad[t] = b;
    };
    if (nt == 1) work(0);
    else {
        std::vector<std::thread> th;
        for (unsigned t = 0; t < nt; t++) th.emplace_back(work, t);
        for (auto& x : th) x.join();
    }
    uint64_t mx = 0;
    for (unsigned t = 0; t < nt; t++) {
        if (bad[t]) return fail(GF_E_INVALID, "offsets are not ascending");
        mx = std::max(mx, part[t]);
    }
    if (mx > limit) return fail(GF_E_INVALID, "a read is longer than the kernel capacity (max_len hint too small, or > 1024 bases)");
    *max_len = mx;
    return GF_OK;
}

void destroy_handle(gf_index* idx) {
    if (!idx) return;
    cudaSetDevice(idx->device);
    if (idx->busy && idx->ev_busy) cudaEventSynchronize(idx->ev_busy); /* device-batch work still in flight on a caller's stream */
    if (idx->stream) cudaStreamSynchronize(idx->stream);
    if (idx->copy_stream) cudaStreamSynchronize(idx->copy_stream);
    cudaFree(idx->d_table);
    cudaFree(idx->d_dupes);
    cudaFree(idx->d_gene_ascii);
    cudaFree(idx->d_gene_start);
    cudaFree(idx->d_gene_len);
    cudaFree(idx->d_gene_rev);
    cudaFree(idx->d_planes);
    cudaFree(idx->d_filter);
    cudaFree(idx->d_granule);
    idx->ws_survivors.release();
    idx->ws_counters.release();
    idx->ws_gtbl.release();
    idx->ws_seq_words.release();
    idx->ws_seq_meta.release();
    idx->ws_seq_seed.release();
    idx->ws_seq_lists.release();
    idx->fq[0].release();
    idx->fq[1].release();
    idx->fq_reads.release();
    idx->bgzf_comp[0].release(); idx->bgzf_comp[1].release();
    idx->bgzf_members[0].release(); idx->bgzf_members[1].release();
    idx->bgzf_status.release();
    for (auto& s : idx->stage) {
        s.seq1.release(); s.qual1.release(); s.off1.release();
        s.seq2.release(); s.qual2.release(); s.off2.release();
        s.out.release(); s.nout.release(); s.out2.release(); s.keys.release();
        for (int m = 0; m < 2; m++) {
            s.pk[m].release(); s.pko[m].release(); s.pkx[m].release(); s.pxo[m].release();
        }
        if (s.copied) cudaEventDestroy(s.copied);
        if (s.done) cudaEventDestroy(s.done);
    }
    for (auto& ps : idx->pack_set) {
        for (int m = 0; m < 2; m++) { ps.h_pk[m].release(); ps.h_pko[m].release(); ps.h_pkx[m].release(); ps.h_pxo[m].release(); }
        if (ps.copied) cudaEventDestroy(ps.copied);
    }
    if (idx->h_slots) cudaFreeHost(idx->h_slots);
    for (cudaEvent_t e : {idx->ev_start, idx->ev_end, idx->ev_ingest})
        if (e) cudaEventDestroy(e);
    for (GfChunkEvents& ce : idx->chunk_events)
        for (cudaEvent_t e : ce.e)
            if (e) cudaEventDestroy(e);
    if (idx->stream) cudaStreamDestroy(idx->stream);
    if (idx->copy_stream) cudaStreamDestroy(idx->copy_stream);
    if (idx->ev_busy) cudaEventDestroy(idx->ev_busy);
    delete idx;
}

}  // namespace

/* list mode: all handles are locked in address order (two list calls sharing handles cannot deadlock) */
struct ListLock {
    std::vector<gf_index*> order;
    explicit ListLock(gf_index* const* hs, uint32_t nh) : order(hs, hs + nh) {
        std::sort(order.begin(), order.end());
        for (gf_index* h : order) h->mu.lock();
    }
    ~ListLock() { for (auto it = order.rbegin(); it != order.rend(); ++it) (*it)->mu.unlock(); }
};
int gf_validate_list(gf_index* const* hs, uint32_t nh) {
    if (!hs || nh == 0) return fail(GF_E_INVALID, "empty index list");
    for (uint32_t h = 0; h < nh; h++) {
        if (!hs[h]) return fail(GF_E_INVALID, "NULL index in the list");
        if (hs[h]->device != hs[0]->device) return fail(GF_E_INVALID, "all indices of a list must live on one device");
        for (uint32_t g = 0; g < h; g++)
            if (hs[g] == hs[h]) return fail(GF_E_INVALID, "the same index is listed twice");
    }
    return GF_OK;
}

extern "C" {

const char* gf_last_error(void) { return g_last_error.c_str(); }
int gf_abi_version(void) { return GF_ABI_VERSION; }

int gf_device_count(void) {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) {
        cudaGetLastError();
        return 0;
    }
    return n;
}

void gf_default_params(gf_params* p) {
    /* src/aux/global_settings.rs:15-29 */
    p->skip_key_dup_threshold = 5;
    p->major_gene_key_requirement = 40;
    p->minor_gene_key_requirement = 20;
    p->mismatch_threshold = 10;
    p->deletion_threshold = 50;
}

int gf_index_create(const gf_gene_span* genes, uint32_t n_genes, const gf_params* params, int device,
                    gf_index** out) {
    if (!out) return fail(GF_E_INVALID, "out is NULL");
    *out = nullptr;
    if (n_genes && !genes) return fail(GF_E_INVALID, "genes is NULL");
    if (n_genes > 32767) return fail(GF_E_LIMIT, "more than 32767 genes: contig ids are i16 (src/core/common.rs:5)");
    gf_params p;
    if (params) p = *params; else gf_default_params(&p);
    if (p.skip_key_dup_threshold < 0 || p.skip_key_dup_threshold > GF_MAX_DUPES)
        return fail(GF_E_LIMIT, "skip_key_dup_threshold must be in [0, 7] (3-bit site count)");
    for (uint32_t g = 0; g < n_genes; g++)
        if (genes[g].len && !genes[g].seq) return fail(GF_E_INVALID, "gene with len > 0 and seq == NULL");
    int ndev = gf_device_count();
    if (ndev <= 0) return fail(GF_E_CUDA, "no CUDA device available (this library has no CPU fallback)");
    if (device < 0 || device >= ndev) return fail(GF_E_INVALID, "device index out of range");
    GF_CUDA_TRY(cudaSetDevice(device));

    /* GF_L2_FETCH_GRANULARITY=32|64|128 (opt-in, experiments only): sets cudaLimitMaxL2FetchGranularity for the whole
     * primary context.  Measured: it does not change the DRAM sectors fetched per random bucket probe
     * (profiles/r01_screen_v1_summary.md), so the library leaves the context's limit alone by default. */
    if (const char* e = getenv("GF_L2_FETCH_GRANULARITY")) {
        const size_t gran = (size_t)atoi(e);
        if (gran == 32 || gran == 64 || gran == 128)
            if (cudaDeviceSetLimit(cudaLimitMaxL2FetchGranularity, gran) != cudaSuccess) cudaGetLastError();
    }

    gf_index* idx = new gf_index();
    idx->device = device;
    idx->params = p;
    int rc = GF_OK;
    do {
        cudaDeviceProp prop;
        if (cudaGetDeviceProperties(&prop, device) != cudaSuccess) { rc = fail(GF_E_CUDA, "cudaGetDeviceProperties failed"); break; }
        idx->sm_count = prop.multiProcessorCount;
        if (cudaStreamCreateWithFlags(&idx->stream, cudaStreamNonBlocking) != cudaSuccess ||
            cudaStreamCreateWithFlags(&idx->copy_stream, cudaStreamNonBlocking) != cudaSuccess) {
            rc = fail(GF_E_CUDA, "cudaStreamCreate failed");
            break;
        }
        bool ok = cudaEventCreate(&idx->ev_start) == cudaSuccess && cudaEventCreate(&idx->ev_end) == cudaSuccess &&
                  cudaEventCreate(&idx->ev_ingest) == cudaSuccess &&
                  cudaEventCreateWithFlags(&idx->ev_busy, cudaEventDisableTiming) == cudaSuccess;
        for (auto& s : idx->stage)
            ok = ok && cudaEventCreateWithFlags(&s.copied, cudaEventDisableTiming) == cudaSuccess &&
                 cudaEventCreateWithFlags(&s.done, cudaEventDisableTiming) == cudaSuccess;
        for (auto& ps : idx->pack_set) ok = ok && cudaEventCreateWithFlags(&ps.copied, cudaEventDisableTiming) == cudaSuccess;
        ok = ok && cudaMallocHost((void**)&idx->h_slots, sizeof(GfHostSlot) * (GF_STAGES + 1)) == cudaSuccess;
        if (!ok) { rc = fail(GF_E_CUDA, "event / pinned allocation failed"); break; }
        memset(idx->h_slots, 0, sizeof(GfHostSlot) * (GF_STAGES + 1));
        rc = gf_build_index_device(idx, genes, n_genes);
    } while (0);
    if (rc != GF_OK) {
        std::string keep = g_last_error;
        destroy_handle(idx);
        cudaGetLastError();
        g_last_error = keep;
        return rc;
    }
    *out = idx;
    return GF_OK;
}

void gf_index_destroy(gf_index* idx) { destroy_handle(idx); }

int gf_index_get_info(const gf_index* idx, gf_index_info* out) {
    if (!idx || !out) return fail(GF_E_INVALID, "NULL argument");
    *out = idx->info;
    return GF_OK;
}

int gf_index_lookup(gf_index* idx, const uint32_t* kmers, uint64_t n, gf_lookup* out) {
    if (!idx || (n && (!kmers || !out))) return fail(GF_E_INVALID, "NULL argument");
    std::lock_guard<std::mutex> lk(idx->mu);
    GF_CUDA_TRY(cudaSetDevice(idx->device));
    return gf_lookup_device(idx, kmers, n, out);
}

void gf_sort_matches(gf_match* m, uint64_t n) {
    std::sort(m, m + n, [](const gf_match& a, const gf_match& b) {
        if (a.pair_idx != b.pair_idx) return a.pair_idx < b.pair_idx;
        return a.source < b.source;
    });
}

/* GF_OUT_BUCKET_ORDER: records by (device-computed key, pair_idx, source) */
static void order_by_keys(gf_match* m, const std::vector<unsigned long long>& keys, uint64_t n) {
    std::vector<uint64_t> perm(n);
    for (uint64_t i = 0; i < n; i++) perm[i] = i;
    std::sort(perm.begin(), perm.end(), [&](uint64_t a, uint64_t b) {
        if (keys[a] != keys[b]) return keys[a] < keys[b];
        if (m[a].pair_idx != m[b].pair_idx) return m[a].pair_idx < m[b].pair_idx;
        return m[a].source < m[b].source;
    });
    std::vector<gf_match> tmp(m, m + n);
    for (uint64_t i = 0; i < n; i++) m[i] = tmp[perm[i]];
}

int gf_index_set_output_mode(gf_index* idx, uint32_t mode) {
    if (!idx) return fail(GF_E_INVALID, "NULL argument");
    if (mode & ~(GF_OUT_DROP_FILTERED | GF_OUT_BUCKET_ORDER)) return fail(GF_E_INVALID, "unknown output mode bits");
    std::lock_guard<std::mutex> lk(idx->mu);
    idx->out_mode = mode;
    return GF_OK;
}

static int validate_batch(const gf_batch* in) {
    if (!in) return fail(GF_E_INVALID, "batch is NULL");
    if (in->n == 0) return GF_OK;
    if (!in->seq1 || !in->qual1 || !in->off1) return fail(GF_E_INVALID, "seq1/qual1/off1 must be set");
    bool pe = in->seq2 != nullptr;
    if (pe && (!in->qual2 || !in->off2)) return fail(GF_E_INVALID, "paired batch needs qual2 and off2");
    return GF_OK;
}

/* Host batch: chunked pipeline, up to GF_STAGES chunks in flight (the upload of a chunk overlaps the kernels of the chunks before;
 * with the arenas in pinned memory the chunks are taken from both ends of the batch: packed by the host threads from the back,
 * copied as ASCII from the front — see below).
 * nh > 1 = list mode: the same reads against several indices.  hs[0] owns the staging buffers, the streams and the
 * sequence store; every chunk is copied ONCE, converted / merged ONCE (k_prep) and then seeded, screened and verified
 * against each index in turn, on hs[0]'s stream. */
static int map_host_batch(gf_index* const* hs, uint32_t nh, const gf_batch* in, gf_match* const* outs, const uint64_t* caps,
                          uint64_t* n_outs) {
    gf_index* idx = hs[0];
    GF_CUDA_TRY(cudaSetDevice(idx->device));
    for (uint32_t h = 0; h < nh; h++) {
        hs[h]->stats = gf_map_stats{};
        hs[h]->stats.n_pairs = in->n;
        hs[h]->stats_pending = false;
        n_outs[h] = 0;
    }
    if (in->n == 0) return GF_OK;
    const bool pe = in->seq2 != nullptr;
    const uint64_t n = in->n;
    const uint64_t* off1 = in->off1;
    const uint64_t* off2 = in->off2;
    if (off1[n] < off1[0] || (pe && off2[n] < off2[0])) return fail(GF_E_INVALID, "offsets are not ascending");
    const uint64_t total_bytes = (off1[n] - off1[0]) + (pe ? off2[n] - off2[0] : 0);
    /* The host offsets are at hand: they must ascend, and no read may be longer than the caller's hint (or than 1024 bases);
     * the longest read selects the kernel capacity.  Without a hint the whole table is scanned here, before anything is
     * launched (several threads).  With a hint every pipeline chunk is checked against it just before it is issued (below),
     * while the device works on the chunk before: a violation fails the call before that chunk's kernels read anything. */
    uint32_t max_len;
    const bool check_per_chunk = in->max_len != 0;
    if (check_per_chunk) {
        if (in->max_len > 1024) return fail(GF_E_INVALID, "max_len hint above the kernel capacity of 1024 bases");
        max_len = in->max_len;
    } else {
        uint64_t mx = 0;
        int r = scan_offsets(off1, pe ? off2 : nullptr, n, 1024, &mx);
        if (r != GF_OK) return r;
        max_len = (uint32_t)std::max<uint64_t>(mx, 1);
    }
    for (uint32_t h = 0; h < nh; h++) {
        int r = wait_prior_device_work(hs[h], idx->stream);
        if (r != GF_OK) return r;
    }

    std::vector<unsigned long long> launches0(nh);
    for (uint32_t h = 0; h < nh; h++) launches0[h] = hs[h]->launches;
    std::vector<uint64_t> total_out(nh, 0), d2h(nh, 0);
    std::vector<std::vector<unsigned long long>> keys(nh); /* GF_OUT_BUCKET_ORDER: device-computed order keys */
    uint64_t h2d = 0;
    std::vector<char> panic(nh, 0);
    GF_CUDA_TRY(cudaEventRecord(idx->ev_start, idx->stream));

    /* qualities: zero-copy when they live in pinned host memory and the on-demand kernel (thread per pair) runs */
    const uint8_t *zq1 = nullptr, *zq2 = nullptr;
    {
        const char* e = getenv("GF_ZEROCOPY_QUAL");
        bool want = !(e && atoi(e) == 0) && max_len != 0 && max_len <= 256;
        auto mapped = [](const void* p) -> const uint8_t* {
            cudaPointerAttributes at;
            if (cudaPointerGetAttributes(&at, p) != cudaSuccess) { cudaGetLastError(); return nullptr; }
            return at.type == cudaMemoryTypeHost ? (const uint8_t*)at.devicePointer : nullptr;
        };
        if (want) {
            zq1 = mapped(in->qual1);
            zq2 = pe ? mapped(in->qual2) : nullptr;
            if (!zq1 || (pe && !zq2)) zq1 = zq2 = nullptr;
        }
    }
    const bool zc = zq1 != nullptr;
    /* packed upload: with the sequence arenas in pinned memory too, the host threads build the plane words and only they are
     * copied (gf_pack.cpp); k_exact / k_verify read the survivors' bases from the mapped arenas */
    const uint8_t *zs1 = nullptr, *zs2 = nullptr;
    if (zc && gf_pack_available()) {
        auto mapped = [](const void* p) -> const uint8_t* {
            cudaPointerAttributes at;
            if (cudaPointerGetAttributes(&at, p) != cudaSuccess) { cudaGetLastError(); return nullptr; }
            return at.type == cudaMemoryTypeHost ? (const uint8_t*)at.devicePointer : nullptr;
        };
        zs1 = mapped(in->seq1);
        zs2 = pe ? mapped(in->seq2) : nullptr;
        if (!zs1 || (pe && !zs2)) zs1 = zs2 = nullptr;
    }
    const bool can_pack = zs1 != nullptr;
    const bool pack_all = can_pack && gf_pack_forced();
    float ms_pack = 0;
    uint64_t n_packed_chunks = 0;
    /* pipeline chunks.  List mode: a chunk costs nh rounds of launches, so chunks are larger (the upload is a smaller share of a
     * chunk anyway). */
    uint64_t chunk_bytes = CHUNK_TARGET_BYTES * std::min<uint32_t>(nh, 4u);
    if (const char* e = getenv("GF_CHUNK_MB")) { long v = atol(e); if (v >= 1 && v <= 65536) chunk_bytes = (uint64_t)v << 20; }
    uint64_t n_chunks = std::max<uint64_t>(1, (2 * total_bytes + chunk_bytes - 1) / chunk_bytes);
    n_chunks = std::min<uint64_t>(n_chunks, n);
    const uint64_t per = (n + n_chunks - 1) / n_chunks;
    n_chunks = (n + per - 1) / per;

    for (uint32_t h = 0; h < nh; h++) hs[h]->stats.zero_copy_qual = zc ? 1u : 0u;

    /* Which chunks are packed?  The packers (host cores, memory-bound) and the copy engine (PCIe) are two resources that work
     * side by side: a packed chunk costs host time and a third of the copy time, an ASCII chunk no host time.  So the batch is
     * eaten from both ends: a driver thread keeps the packing threads busy with chunks taken from the BACK of the batch, one
     * after the other without a pause, into GF_PACK_SETS pinned buffer sets; the issuing thread uploads every packed chunk as
     * soon as it is ready and, whenever the copy engine is about to run dry, takes the next chunk from the FRONT and copies its
     * ASCII.  The two meet somewhere in the middle — where depends on how many cores there are and how fast the copies go, and
     * nothing has to be estimated beyond "how much copying is still queued" (cudaEventQuery).  Few cores => mostly ASCII chunks,
     * many cores => mostly packed ones; the issuing thread's thirty driver calls per chunk overlap with the packing.
     * The records of a call are sorted at the end, so the order in which chunks are issued does not matter. */
    struct InFlight { cudaEvent_t copied; double copy_ms; };
    std::vector<InFlight> in_flight;
    constexpr double COPY_BYTES_PER_MS = 45.0e6;
    auto queued_copy_ms = [&]() {
        double t = 0;
        for (size_t i = 0; i < in_flight.size();) {
            if (cudaEventQuery(in_flight[i].copied) == cudaSuccess) { in_flight[i] = in_flight.back(); in_flight.pop_back(); }
            else { t += in_flight[i].copy_ms; i++; }
        }
        cudaGetLastError(); /* cudaErrorNotReady is not an error here */
        return t;
    };
    const int nm = pe ? 2 : 1;
    uint64_t max_chunk_bytes[2] = {0, 0};
    for (uint64_t k = 0; k < n_chunks; k++) {
        const uint64_t lo = k * per, hi = std::min(n, lo + per);
        max_chunk_bytes[0] = std::max(max_chunk_bytes[0], off1[hi] - off1[lo]);
        if (pe) max_chunk_bytes[1] = std::max(max_chunk_bytes[1], off2[hi] - off2[lo]);
    }
    const bool use_packers = can_pack && (pack_all || n_chunks >= 2);
    /* state shared with the driver thread */
    enum { SET_FREE = 0, SET_PACKING, SET_READY, SET_COPYING };
    struct SetState { int state = SET_FREE; uint64_t chunk = 0; float ms = 0; GfPackMate pm[2]; };
    struct Shared {
        std::mutex mu;
        std::condition_variable cv_driver, cv_issuer;
        uint64_t front = 0, back = 0;
        bool stop = false, driver_done = true;
        SetState set[GF_PACK_SETS];
        std::vector<int> ready;
    } sh;
    sh.back = n_chunks;
    auto fill_mates = [&](GfPackMate* pmv, uint64_t k) {
        const uint64_t lo = k * per, hi = std::min(n, lo + per);
        for (int m = 0; m < nm; m++) {
            const uint64_t* off = m ? off2 : off1;
            pmv[m] = GfPackMate{};
            pmv[m].seq = (m ? in->seq2 : in->seq1) + off[lo];
            pmv[m].off = off + lo;
            pmv[m].off_base = off[lo];
            pmv[m].n = hi - lo;
            pmv[m].mate2 = m == 1;
            pmv[m].max_len = max_len;
        }
    };
    if (use_packers) {
        for (GfPackSet& ps : idx->pack_set)
            for (int m = 0; m < nm; m++) {
                const size_t wcap = sizeof(uint32_t) * 2 * (size_t)(max_chunk_bytes[m] / 32 + per + 1); /* >= 2 * sum ceil(len / 32) */
                GF_CUDA_TRY(ps.h_pk[m].reserve(wcap));
                GF_CUDA_TRY(ps.h_pkx[m].reserve(wcap));
                GF_CUDA_TRY(ps.h_pko[m].reserve(sizeof(uint32_t) * per));
                GF_CUDA_TRY(ps.h_pxo[m].reserve(sizeof(uint32_t) * per));
            }
    }
    auto driver = [&]() {
        cudaSetDevice(idx->device);
        for (;;) {
            int j = -1;
            uint64_t k = 0;
            {
                std::unique_lock<std::mutex> lk(sh.mu);
                for (;;) {
                    if (sh.stop || sh.front >= sh.back) break;
                    for (int u = 0; u < GF_PACK_SETS && j < 0; u++)
                        if (sh.set[u].state == SET_FREE) j = u;
                    if (j >= 0) break;
                    /* no free set: those being copied come back when their copy is through */
                    for (int u = 0; u < GF_PACK_SETS; u++)
                        if (sh.set[u].state == SET_COPYING && cudaEventQuery(idx->pack_set[u].copied) == cudaSuccess) sh.set[u].state = SET_FREE;
                    cudaGetLastError();
                    for (int u = 0; u < GF_PACK_SETS && j < 0; u++)
                        if (sh.set[u].state == SET_FREE) j = u;
                    if (j >= 0) break;
                    sh.cv_driver.wait_for(lk, std::chrono::microseconds(100));
                }
                if (j < 0) break;
                k = --sh.back;
                sh.set[j].state = SET_PACKING;
                sh.set[j].chunk = k;
            }
            SetState& st = sh.set[j];
            GfPackSet& ps = idx->pack_set[j];
            fill_mates(st.pm, k);
            for (int m = 0; m < nm; m++) {
                st.pm[m].compact = true;
                st.pm[m].words = ps.h_pk[m].as<uint32_t>();
                st.pm[m].woff = ps.h_pko[m].as<uint32_t>();
                st.pm[m].xwords = ps.h_pkx[m].as<uint32_t>();
                st.pm[m].xoff = ps.h_pxo[m].as<uint32_t>();
            }
            gf_pack_start(st.pm, nm, false, true); /* waits while the packing threads work for another handle */
            st.ms = gf_pack_wait();
            {
                std::lock_guard<std::mutex> lk(sh.mu);
                st.state = SET_READY;
                sh.ready.push_back(j);
            }
            sh.cv_issuer.notify_one();
        }
        {
            std::lock_guard<std::mutex> lk(sh.mu);
            sh.driver_done = true;
        }
        sh.cv_issuer.notify_one();
    };
    std::thread driver_thread;
    if (use_packers) {
        sh.driver_done = false;
        driver_thread = std::thread(driver);
    }
    auto stop_driver = [&]() {
        if (!driver_thread.joinable()) return;
        {
            std::lock_guard<std::mutex> lk(sh.mu);
            sh.stop = true;
        }
        sh.cv_driver.notify_one();
        driver_thread.join();
    };

    /* issue chunk k as issue number q (stage q % GF_STAGES): its copies (plane words of pack set `set`, or the ASCII) and launches */
    auto enqueue_chunk = [&](uint64_t q, uint64_t k, int set) -> int {
        GfStage& s = idx->stage[q % GF_STAGES];
        const bool packed = set >= 0;
        const GfPackMate* pm = packed ? sh.set[set].pm : nullptr;
        const uint64_t lo = k * per, hi = std::min(n, lo + per), cn = hi - lo;
        const uint64_t b1 = off1[lo], e1 = off1[hi];
        const uint64_t h2d_before = h2d;
        cudaStream_t cs = idx->copy_stream;
        if (packed) {
            const GfPackSet& ps = idx->pack_set[set];
            for (int m = 0; m < nm; m++) {
                const size_t wcap = sizeof(uint32_t) * 2 * (size_t)(max_chunk_bytes[m] / 32 + per + 1);
                GF_CUDA_TRY(s.pk[m].reserve(wcap));
                GF_CUDA_TRY(s.pkx[m].reserve(wcap));
                GF_CUDA_TRY(s.pko[m].reserve(sizeof(uint32_t) * per));
                GF_CUDA_TRY(s.pxo[m].reserve(sizeof(uint32_t) * per));
                GF_CUDA_TRY(cudaMemcpyAsync(s.pk[m].p, ps.h_pk[m].p, sizeof(uint32_t) * pm[m].n_words, cudaMemcpyHostToDevice, cs));
                h2d += sizeof(uint32_t) * pm[m].n_words;
                if (!pm[m].uniform_len) { /* (reads of one length: the device fills the table itself, below) */
                    GF_CUDA_TRY(cudaMemcpyAsync(s.pko[m].p, ps.h_pko[m].p, sizeof(uint32_t) * cn, cudaMemcpyHostToDevice, cs));
                    h2d += sizeof(uint32_t) * cn;
                }
                bool any_x = false;
                for (int t = 0; t < pm[m].n_threads; t++) any_x = any_x || pm[m].xregion_used[t] != 0;
                if (any_x) {
                    for (int t = 0; t < pm[m].n_threads; t++) { /* threads without a flagged read left their part of xoff alone */
                        const uint64_t a = cn * (uint64_t)t / pm[m].n_threads, b = cn * (uint64_t)(t + 1) / pm[m].n_threads;
                        if (!pm[m].xoff_written[t]) memset(ps.h_pxo[m].as<uint32_t>() + a, 0, sizeof(uint32_t) * (b - a));
                    }
                    GF_CUDA_TRY(cudaMemcpyAsync(s.pxo[m].p, ps.h_pxo[m].p, sizeof(uint32_t) * cn, cudaMemcpyHostToDevice, cs));
                    h2d += sizeof(uint32_t) * cn;
                } else {
                    GF_CUDA_TRY(cudaMemsetAsync(s.pxo[m].p, 0, sizeof(uint32_t) * cn, idx->stream));
                }
                for (int t = 0; t < pm[m].n_threads; t++) {
                    if (!pm[m].xregion_used[t]) continue;
                    GF_CUDA_TRY(cudaMemcpyAsync(s.pkx[m].as<uint32_t>() + pm[m].xregion_start[t],
                                                ps.h_pkx[m].as<uint32_t>() + pm[m].xregion_start[t],
                                                sizeof(uint32_t) * pm[m].xregion_used[t], cudaMemcpyHostToDevice, cs));
                    h2d += sizeof(uint32_t) * pm[m].xregion_used[t];
                }
            }
            GF_CUDA_TRY(cudaEventRecord(ps.copied, cs)); /* the set is free again from here on */
        } else {
            GF_CUDA_TRY(s.seq1.reserve(max_chunk_bytes[0] + 16));
            GF_CUDA_TRY(cudaMemcpyAsync(s.seq1.p, in->seq1 + b1, e1 - b1, cudaMemcpyHostToDevice, cs));
            h2d += e1 - b1;
        }
        GF_CUDA_TRY(s.off1.reserve(sizeof(uint64_t) * (per + 1)));
        if (!zc) {
            GF_CUDA_TRY(s.qual1.reserve(max_chunk_bytes[0] + 16));
            GF_CUDA_TRY(cudaMemcpyAsync(s.qual1.p, in->qual1 + b1, e1 - b1, cudaMemcpyHostToDevice, cs));
            h2d += e1 - b1;
        }
        if (packed && pm[0].uniform_len) { /* reads of one length: offsets and word offsets are made on the device */
            k_fill_uniform<<<(unsigned)((cn + 256) / 256), 256, 0, idx->stream>>>(s.off1.as<uint64_t>(), s.pko[0].as<uint32_t>(), b1,
                                                                                 pm[0].uniform_len, cn);
            idx->launches++;
        } else {
            GF_CUDA_TRY(cudaMemcpyAsync(s.off1.p, off1 + lo, sizeof(uint64_t) * (cn + 1), cudaMemcpyHostToDevice, cs));
            h2d += sizeof(uint64_t) * (cn + 1);
        }
        GfDevBatch db{};
        db.n = cn;
        db.seq1 = packed ? zs1 + b1 : s.seq1.as<uint8_t>();
        if (packed) {
            db.pk1 = s.pk[0].as<uint32_t>(); db.pko1 = s.pko[0].as<uint32_t>();
            db.pkx1 = s.pkx[0].as<uint32_t>(); db.pxo1 = s.pxo[0].as<uint32_t>();
        }
        db.qual1 = zc ? zq1 + b1 : s.qual1.as<uint8_t>(); /* kernels address it as qual1 + (off - base1) */
        db.s1 = s.off1.as<uint64_t>(); db.e1 = db.s1 + 1; db.qs1 = db.s1;
        db.base1 = b1;
        db.bytes1 = e1 - b1;
        db.pair_base = lo;
        db.max_len = max_len;
        if (pe) {
            const uint64_t b2 = off2[lo], e2 = off2[hi];
            GF_CUDA_TRY(s.off2.reserve(sizeof(uint64_t) * (per + 1)));
            if (!packed) {
                GF_CUDA_TRY(s.seq2.reserve(max_chunk_bytes[1] + 16));
                GF_CUDA_TRY(cudaMemcpyAsync(s.seq2.p, in->seq2 + b2, e2 - b2, cudaMemcpyHostToDevice, cs));
                h2d += e2 - b2;
            }
            if (!zc) {
                GF_CUDA_TRY(s.qual2.reserve(max_chunk_bytes[1] + 16));
                GF_CUDA_TRY(cudaMemcpyAsync(s.qual2.p, in->qual2 + b2, e2 - b2, cudaMemcpyHostToDevice, cs));
                h2d += e2 - b2;
            }
            if (packed && pm[1].uniform_len) {
                k_fill_uniform<<<(unsigned)((cn + 256) / 256), 256, 0, idx->stream>>>(s.off2.as<uint64_t>(), s.pko[1].as<uint32_t>(), b2,
                                                                                     pm[1].uniform_len, cn);
                idx->launches++;
            } else {
                GF_CUDA_TRY(cudaMemcpyAsync(s.off2.p, off2 + lo, sizeof(uint64_t) * (cn + 1), cudaMemcpyHostToDevice, cs));
                h2d += sizeof(uint64_t) * (cn + 1);
            }
            db.seq2 = packed ? zs2 + b2 : s.seq2.as<uint8_t>();
            if (packed) {
                db.pk2 = s.pk[1].as<uint32_t>(); db.pko2 = s.pko[1].as<uint32_t>();
                db.pkx2 = s.pkx[1].as<uint32_t>(); db.pxo2 = s.pxo[1].as<uint32_t>();
            }
            db.qual2 = zc ? zq2 + b2 : s.qual2.as<uint8_t>();
            db.s2 = s.off2.as<uint64_t>(); db.e2 = db.s2 ? db.s2 + 1 : nullptr; db.qs2 = db.s2;
            db.base2 = b2;
            db.bytes2 = e2 - b2;
        }
        GF_CUDA_TRY(cudaEventRecord(s.copied, cs));
        in_flight.push_back(InFlight{s.copied, (double)(h2d - h2d_before) / COPY_BYTES_PER_MS});
        s.n = cn;
        s.pair_base = lo;
        GF_CUDA_TRY(cudaStreamWaitEvent(idx->stream, s.copied, 0));
        for (uint32_t h = 0; h < nh; h++) {
            GfStage& sh_ = hs[h]->stage[q % GF_STAGES];
            sh_.out_cap = (pe ? 2 : 1) * cn;
            GF_CUDA_TRY(sh_.out.reserve(sizeof(gf_match) * (pe ? 2 : 1) * per));
            GF_CUDA_TRY(sh_.nout.reserve(2 * sizeof(unsigned long long)));
            int r = gf_map_device_batch(hs[h], db, sh_.out.as<gf_match>(), sh_.out_cap, sh_.nout.as<unsigned long long>(),
                                        idx->stream, nullptr, true, h ? idx : nullptr);
            if (r != GF_OK) return r;
            GfHostSlot* hsl = &hs[h]->h_slots[q % GF_STAGES];
            if (hs[h]->out_mode) { /* per-record filters + order keys on the device, before the records leave it */
                GF_CUDA_TRY(sh_.out2.reserve(sizeof(gf_match) * (pe ? 2 : 1) * per));
                GF_CUDA_TRY(sh_.keys.reserve(sizeof(unsigned long long) * (pe ? 2 : 1) * per));
                r = gf_finish_records_device(hs[h], sh_.out.as<gf_match>(), sh_.nout.as<unsigned long long>(), sh_.out_cap,
                                             sh_.out2.as<gf_match>(), sh_.keys.as<unsigned long long>(),
                                             sh_.nout.as<unsigned long long>() + 1, hs[h]->out_mode, idx->stream);
                if (r != GF_OK) return r;
                GF_CUDA_TRY(cudaMemcpyAsync(&hsl->n_out2, sh_.nout.as<unsigned long long>() + 1, sizeof(unsigned long long),
                                            cudaMemcpyDeviceToHost, idx->stream));
            }
            GF_CUDA_TRY(cudaMemcpyAsync(&hsl->counters, hs[h]->ws_counters.p, sizeof(GfMapCounters), cudaMemcpyDeviceToHost,
                                        idx->stream));
            GF_CUDA_TRY(cudaMemcpyAsync(&hsl->n_out, sh_.nout.p, sizeof(unsigned long long), cudaMemcpyDeviceToHost,
                                        idx->stream));
        }
        GF_CUDA_TRY(cudaEventRecord(s.done, idx->stream));
        return GF_OK;
    };
    auto collect = [&](uint64_t q) -> int {
        GF_CUDA_TRY(cudaEventSynchronize(idx->stage[q % GF_STAGES].done));
        for (uint32_t h = 0; h < nh; h++) {
            GfStage& sh_ = hs[h]->stage[q % GF_STAGES];
            GfHostSlot* hsl = &hs[h]->h_slots[q % GF_STAGES];
            int r = check_flags(*hsl);
            if (r != GF_OK) return r;
            accumulate(hs[h]->stats, *hsl);
            if (hsl->counters.n_ref_panic) panic[h] = 1;
            const uint32_t mode = hs[h]->out_mode;
            const uint64_t cnt = mode ? hsl->n_out2 : hsl->n_out; /* <= sh_.out_cap by construction */
            if (cnt && total_out[h] + cnt <= caps[h]) {
                GF_CUDA_TRY(cudaMemcpy(outs[h] + total_out[h], mode ? sh_.out2.p : sh_.out.p, sizeof(gf_match) * cnt,
                                       cudaMemcpyDeviceToHost));
                d2h[h] += sizeof(gf_match) * cnt;
                if (mode & GF_OUT_BUCKET_ORDER) {
                    keys[h].resize(total_out[h] + cnt);
                    GF_CUDA_TRY(cudaMemcpy(keys[h].data() + total_out[h], sh_.keys.p, sizeof(unsigned long long) * cnt,
                                           cudaMemcpyDeviceToHost));
                    d2h[h] += sizeof(unsigned long long) * cnt;
                }
            }
            d2h[h] += sizeof(GfMapCounters) + sizeof(unsigned long long);
            total_out[h] += cnt;
        }
        return GF_OK;
    };

    /* The issuing thread.  An ASCII chunk is taken from the front only when less than GF_ASCII_AHEAD_MS of copying is still
     * queued (default: half an ASCII chunk; measured 0 / 2 / 4 / 8 ms with 4 ms chunks: 39.3 / 35.8 / 36.5 / 40.9 ms per 10 M pairs), so the copy engine stays busy and nothing is committed to the slow way that the
     * packers could still have taken.  Up to GF_STAGES chunks are in flight; a chunk's results are collected when its stage is
     * needed again (or at the end). */
    double ascii_ahead_ms = 0.5 * (double)(max_chunk_bytes[0] + max_chunk_bytes[1]) / COPY_BYTES_PER_MS;
    if (const char* e = getenv("GF_ASCII_AHEAD_MS")) { const double v = atof(e); if (v >= 0) ascii_ahead_ms = v; }
    uint64_t issued = 0, collected = 0;
    int rc = GF_OK;
    while (rc == GF_OK && issued < n_chunks) {
        const bool ascii_ok = !use_packers || (!pack_all && queued_copy_ms() < ascii_ahead_ms);
        int set = -1;
        uint64_t k = 0;
        bool have = false;
        {
            std::unique_lock<std::mutex> lk(sh.mu);
            if (!sh.ready.empty()) {
                set = sh.ready.front();
                sh.ready.erase(sh.ready.begin());
                k = sh.set[set].chunk;
                have = true;
            } else if (sh.front < sh.back && ascii_ok) {
                k = sh.front++;
                have = true;
            } else {
                sh.cv_issuer.wait_for(lk, std::chrono::microseconds(50));
            }
        }
        if (!have) continue;
        if (set >= 0) {
            const SetState& st = sh.set[set];
            ms_pack += st.ms;
            n_packed_chunks++;
            if (st.pm[0].bad_offsets || (pe && st.pm[1].bad_offsets)) {
                rc = fail(GF_E_INVALID, "offsets are not ascending, or a read is longer than max_len / the kernel capacity");
                break;
            }
        } else if (check_per_chunk) {
            const uint64_t lo = k * per, cn = std::min(n, lo + per) - lo;
            uint64_t mx = 0;
            rc = scan_offsets(off1 + lo, pe ? off2 + lo : nullptr, cn, max_len, &mx, 1); /* inline: ~0.3 ms per chunk */
            if (rc != GF_OK) break;
        }
        while (rc == GF_OK && issued - collected >= (uint64_t)GF_STAGES) rc = collect(collected++); /* this issue reuses that stage */
        queued_copy_ms(); /* (forget the finished copies before that stage's event is recorded again) */
        if (rc == GF_OK) rc = enqueue_chunk(issued, k, set);
        if (set >= 0) {
            std::lock_guard<std::mutex> lk(sh.mu);
            sh.set[set].state = rc == GF_OK ? SET_COPYING : SET_FREE;
        }
        issued++;
    }
    stop_driver();
    while (rc == GF_OK && collected < issued) rc = collect(collected++);
    if (rc != GF_OK) {
        cudaStreamSynchronize(idx->stream);
        cudaStreamSynchronize(idx->copy_stream);
        return rc;
    }
    GF_CUDA_TRY(cudaEventRecord(idx->ev_end, idx->stream));
    GF_CUDA_TRY(cudaEventSynchronize(idx->ev_end));
    float ms = 0;
    GF_CUDA_TRY(cudaEventElapsedTime(&ms, idx->ev_start, idx->ev_end));
    rc = GF_OK;
    for (uint32_t h = 0; h < nh; h++) hs[h]->busy = false; /* the stream waited for it and has drained */
    for (uint32_t h = 0; h < nh; h++) {
        gf_map_stats& st = hs[h]->stats;
        st.ms_total = ms; /* of the whole call (all indices) */
        st.kernel_launches = hs[h]->launches - launches0[h];
        st.h2d_bytes = h ? 0 : h2d;
        st.ms_host_pack = h ? 0.f : ms_pack;
        st.packed_upload = n_packed_chunks == 0 ? 0u : (n_packed_chunks == n_chunks ? 1u : 2u);
        st.d2h_bytes = d2h[h];
        if (h) { /* k_prep ran once, on hs[0] */
            st.n_sequences = hs[0]->stats.n_sequences;
            st.n_probes_pass1 = hs[0]->stats.n_probes_pass1;
            st.seq_bytes = hs[0]->stats.seq_bytes;
        }
        n_outs[h] = total_out[h];
        if (total_out[h] > caps[h]) { rc = fail(GF_E_CAPACITY, "out_cap too small; *n_out holds the required count"); continue; }
        if (hs[h]->out_mode & GF_OUT_BUCKET_ORDER) order_by_keys(outs[h], keys[h], total_out[h]);
        else gf_sort_matches(outs[h], total_out[h]);
        if (panic[h] && rc == GF_OK)
            rc = fail(GF_E_REF_PANIC,
                      "a candidate needs an edit distance over more than 640 columns: the reference panics here "
                      "(src/core/edit_distance.rs:94-100,177-196); records were still written with exact distances");
    }
    return rc;
}

int gf_map_pairs(gf_index* idx, const gf_batch* in, gf_match* out, uint64_t out_cap, uint64_t* n_out) {
    if (!idx || !n_out) return fail(GF_E_INVALID, "NULL argument");
    *n_out = 0;
    int rc = validate_batch(in);
    if (rc != GF_OK) return rc;
    if (out_cap && !out) return fail(GF_E_INVALID, "out is NULL");
    std::lock_guard<std::mutex> lk(idx->mu);
    return map_host_batch(&idx, 1, in, &out, &out_cap, n_out);
}

int gf_list_map_pairs(gf_index* const* idx, uint32_t n_idx, const gf_batch* in, gf_match* const* out, const uint64_t* out_cap,
                      uint64_t* n_out) {
    if (!n_out || !out_cap || !out) return fail(GF_E_INVALID, "NULL argument");
    int rc = gf_validate_list(idx, n_idx);
    if (rc != GF_OK) return rc;
    rc = validate_batch(in);
    if (rc != GF_OK) return rc;
    for (uint32_t h = 0; h < n_idx; h++)
        if (out_cap[h] && !out[h]) return fail(GF_E_INVALID, "out is NULL");
    ListLock lk(idx, n_idx);
    return map_host_batch(idx, n_idx, in, out, out_cap, n_out);
}

int gf_map_pairs_device_list(gf_index* const* idx, uint32_t n_idx, const gf_batch* in_dev, gf_match* const* d_out,
                             uint64_t out_cap, uint64_t* const* d_n_out, void* cuda_stream) {
    if (!d_out || !d_n_out) return fail(GF_E_INVALID, "NULL argument");
    int rc = gf_validate_list(idx, n_idx);
    if (rc != GF_OK) return rc;
    rc = validate_batch(in_dev);
    if (rc != GF_OK) return rc;
    ListLock lk(idx, n_idx);
    GF_CUDA_TRY(cudaSetDevice(idx[0]->device));
    cudaStream_t st = (cudaStream_t)cuda_stream;
    GfDevBatch db{};
    db.n = in_dev->n;
    db.seq1 = in_dev->seq1;
    db.qual1 = in_dev->qual1;
    db.s1 = in_dev->off1; db.e1 = db.s1 + 1; db.qs1 = db.s1;
    db.seq2 = in_dev->seq2;
    db.qual2 = in_dev->qual2;
    db.s2 = in_dev->off2; db.e2 = db.s2 ? db.s2 + 1 : nullptr; db.qs2 = db.s2;
    db.bytes1 = in_dev->bytes1;
    db.bytes2 = in_dev->bytes2;
    db.max_len = in_dev->max_len;
    for (uint32_t h = 0; h < n_idx; h++) {
        if (!d_n_out[h]) return fail(GF_E_INVALID, "NULL argument");
        rc = wait_prior_device_work(idx[h], st);
        if (rc != GF_OK) return rc;
    }
    std::vector<unsigned long long> launches0(n_idx);
    std::vector<gf_match*> outs(d_out, d_out + n_idx);
    std::vector<unsigned long long*> nouts(n_idx);
    for (uint32_t h = 0; h < n_idx; h++) { launches0[h] = idx[h]->launches; nouts[h] = (unsigned long long*)d_n_out[h]; }
    for (uint32_t h = 0; h < n_idx; h++) GF_CUDA_TRY(cudaEventRecord(idx[h]->ev_start, st));
    rc = gf_map_device_batches(idx, n_idx, db, outs.data(), out_cap, nouts.data(), st);
    if (rc != GF_OK) return rc;
    for (uint32_t h = 0; h < n_idx; h++) {
        gf_index* x = idx[h];
        GfHostSlot* hsl = &x->h_slots[GF_SLOT_DEVICE];
        GF_CUDA_TRY(cudaMemcpyAsync(&hsl->counters, x->ws_counters.p, sizeof(GfMapCounters), cudaMemcpyDeviceToHost, st));
        GF_CUDA_TRY(cudaMemcpyAsync(&hsl->n_out, d_n_out[h], sizeof(unsigned long long), cudaMemcpyDeviceToHost, st));
        GF_CUDA_TRY(cudaEventRecord(x->ev_end, st));
        x->stats = gf_map_stats{};
        x->stats.n_pairs = in_dev->n;
        x->stats.kernel_launches = x->launches - launches0[h];
        x->stats_pending = true;
    }
    for (uint32_t h = 0; h < n_idx; h++) { /* after the LAST handle's work: the shared sequence store is read by all of them */
        rc = mark_device_work(idx[h], st);
        if (rc != GF_OK) return rc;
    }
    return GF_OK;
}

int gf_map_pairs_device(gf_index* idx, const gf_batch* in_dev, gf_match* d_out, uint64_t out_cap, uint64_t* d_n_out,
                        void* cuda_stream) {
    if (!idx || !d_n_out) return fail(GF_E_INVALID, "NULL argument");
    int rc = validate_batch(in_dev);
    if (rc != GF_OK) return rc;
    std::lock_guard<std::mutex> lk(idx->mu);
    GF_CUDA_TRY(cudaSetDevice(idx->device));
    cudaStream_t st = (cudaStream_t)cuda_stream;
    GfDevBatch db{};
    db.n = in_dev->n;
    db.seq1 = in_dev->seq1;
    db.qual1 = in_dev->qual1;
    db.s1 = in_dev->off1; db.e1 = db.s1 + 1; db.qs1 = db.s1;
    db.seq2 = in_dev->seq2;
    db.qual2 = in_dev->qual2;
    db.s2 = in_dev->off2; db.e2 = db.s2 ? db.s2 + 1 : nullptr; db.qs2 = db.s2;
    db.base1 = db.base2 = 0;
    db.bytes1 = in_dev->bytes1;
    db.bytes2 = in_dev->bytes2;
    db.pair_base = 0;
    db.max_len = in_dev->max_len;
    const unsigned long long launches0 = idx->launches;
    rc = wait_prior_device_work(idx, st);
    if (rc != GF_OK) return rc;
    GF_CUDA_TRY(cudaEventRecord(idx->ev_start, st));
    unsigned long long* nout1 = (unsigned long long*)d_n_out;
    rc = gf_map_device_batches(&idx, 1, db, &d_out, out_cap, &nout1, st);
    if (rc != GF_OK) return rc;
    GfHostSlot* h = &idx->h_slots[GF_SLOT_DEVICE];
    GF_CUDA_TRY(cudaMemcpyAsync(&h->counters, idx->ws_counters.p, sizeof(GfMapCounters), cudaMemcpyDeviceToHost, st));
    GF_CUDA_TRY(cudaMemcpyAsync(&h->n_out, d_n_out, sizeof(unsigned long long), cudaMemcpyDeviceToHost, st));
    GF_CUDA_TRY(cudaEventRecord(idx->ev_end, st));
    idx->stats = gf_map_stats{};
    idx->stats.n_pairs = in_dev->n;
    idx->stats.kernel_launches = idx->launches - launches0;
    idx->stats_pending = true;
    return mark_device_work(idx, st);
}

int gf_map_fastq(gf_index* idx, const uint8_t* fq1, uint64_t bytes1, const uint8_t* fq2, uint64_t bytes2, gf_match* out,
                 uint64_t out_cap, uint64_t* n_out, uint64_t* n_records) {
    if (!idx) return fail(GF_E_INVALID, "NULL argument");
    uint64_t consumed[2];
    return gf_map_fastq_text(&idx, 1, fq1, bytes1, fq2, bytes2, true, &out, &out_cap, n_out, n_records, consumed);
}

} /* extern "C" */

int gf_map_fastq_text(gf_index* const* hs, uint32_t nh, const uint8_t* fq1, uint64_t host1, const uint8_t* fq2, uint64_t host2,
                      bool final_chunk, gf_match* const* out, const uint64_t* out_cap, uint64_t* n_out, uint64_t* n_records,
                      uint64_t consumed[2], const GfFastqMembers* members, GfFastqReads* reads, bool* panic,
                      std::vector<uint8_t>* tail) {
    /* the text of a mate: host bytes, then (gf_fastq_stream, blocked gzip) the text of BGZF members that are still compressed */
    const uint64_t bytes1 = host1 + (members ? members[0].text_bytes : 0), bytes2 = host2 + (members && fq2 ? members[1].text_bytes : 0);
    if (!hs || !nh || !hs[0] || !n_out || !n_records) return fail(GF_E_INVALID, "NULL argument");
    *n_records = 0;
    consumed[0] = consumed[1] = 0;
    for (uint32_t h = 0; h < nh; h++) {
        n_out[h] = 0;
        if (panic) panic[h] = false;
        if (reads) { reads[h].pairs.clear(); reads[h].text.clear(); }
    }
    if ((host1 && !fq1) || (host2 && !fq2)) return fail(GF_E_INVALID, "NULL FASTQ buffer");
    for (uint32_t h = 0; h < nh; h++)
        if (out_cap[h] && !out[h]) return fail(GF_E_INVALID, "out is NULL");
    ListLock lk(hs, nh);
    gf_index* idx = hs[0]; /* the text, its newline tables, the sequence store and the gathered lines live in idx's workspace */
    GF_CUDA_TRY(cudaSetDevice(idx->device));
    const bool pe = fq2 != nullptr;
    cudaStream_t st = idx->stream;
    GfStage& sg = idx->stage[0];
    for (uint32_t h = 0; h < nh; h++) {
        hs[h]->stats = gf_map_stats{};
        hs[h]->stats_pending = false;
        int r = wait_prior_device_work(hs[h], st);
        if (r != GF_OK) return r;
        GF_CUDA_TRY(cudaEventRecord(hs[h]->ev_start, st));
    }
    /* raw text -> device (the sequence and quality "arenas" are the text itself) */
    GF_CUDA_TRY(sg.seq1.reserve(bytes1 + 32));
    if (host1) GF_CUDA_TRY(cudaMemcpyAsync(sg.seq1.p, fq1, host1, cudaMemcpyHostToDevice, st));
    if (pe) {
        GF_CUDA_TRY(sg.seq2.reserve(bytes2 + 32));
        if (host2) GF_CUDA_TRY(cudaMemcpyAsync(sg.seq2.p, fq2, host2, cudaMemcpyHostToDevice, st));
    }
    uint64_t h2d_members = 0;
    bool inflated = false;
    if (members) { /* compressed bytes cross PCIe, the members are inflated here (gf_fastq.cu: k_bgzf_inflate) */
        GF_CUDA_TRY(idx->bgzf_status.reserve(4 * sizeof(unsigned int)));
        if (pe && members[1].n_members) { /* (mate 2's buffers may still be in use by work queued on `st` before this call) */
            GF_CUDA_TRY(cudaEventRecord(sg.done, st));
            GF_CUDA_TRY(cudaStreamWaitEvent(idx->copy_stream, sg.done, 0));
        }
        for (int k = 0; k < (pe ? 2 : 1); k++) {
            const GfFastqMembers& mk = members[k];
            if (!mk.n_members) continue;
            /* the two mates side by side: mate 2's members go through the copy stream (a warp per member: one mate's members
             * alone leave half of the SMs' warp slots empty) */
            cudaStream_t ks = k ? idx->copy_stream : st;
            GF_CUDA_TRY(idx->bgzf_comp[k].reserve(mk.comp_bytes + 16));
            GF_CUDA_TRY(idx->bgzf_members[k].reserve(sizeof(GfBgzfMember) * mk.n_members));
            GF_CUDA_TRY(cudaMemcpyAsync(idx->bgzf_comp[k].p, mk.comp, mk.comp_bytes, cudaMemcpyHostToDevice, ks));
            GF_CUDA_TRY(cudaMemcpyAsync(idx->bgzf_members[k].p, mk.members, sizeof(GfBgzfMember) * mk.n_members, cudaMemcpyHostToDevice, ks));
            int r = gf_bgzf_inflate_device(idx->bgzf_comp[k].as<uint8_t>(), idx->bgzf_members[k].as<GfBgzfMember>(), mk.n_members,
                                           (k ? sg.seq2 : sg.seq1).as<uint8_t>() + (k ? host2 : host1),
                                           idx->bgzf_status.as<unsigned int>() + 2 * k, ks);
            if (r != GF_OK) return r;
            if (k) {
                GF_CUDA_TRY(cudaEventRecord(sg.copied, ks));
                GF_CUDA_TRY(cudaStreamWaitEvent(st, sg.copied, 0));
            }
            idx->launches++;
            h2d_members += mk.comp_bytes + sizeof(GfBgzfMember) * mk.n_members;
            inflated = true;
        }
        if (inflated) { /* nothing of a chunk with a corrupt member is used */
            unsigned int stt[4] = {0, 0, 0, 0};
            GF_CUDA_TRY(cudaMemcpyAsync(stt, idx->bgzf_status.p, sizeof(stt), cudaMemcpyDeviceToHost, st));
            GF_CUDA_TRY(cudaStreamSynchronize(st));
            for (int k = 0; k < (pe ? 2 : 1); k++)
                if (members[k].n_members && stt[2 * k])
                    return fail(GF_E_INVALID, std::string("gzip stream of mate ") + (k ? "2" : "1") + " is corrupt (BGZF block " +
                                                  std::to_string(stt[2 * k + 1] - 1) + " of the chunk, error bits " + std::to_string(stt[2 * k]) + ")");
        }
    }
    int rc = gf_fastq_parse_device(sg.seq1.as<uint8_t>(), bytes1, &idx->fq[0], st, final_chunk);
    if (rc == GF_OK && pe) rc = gf_fastq_parse_device(sg.seq2.as<uint8_t>(), bytes2, &idx->fq[1], st, final_chunk);
    if (rc != GF_OK) return rc;
    for (uint32_t h = 0; h < nh; h++) /* end of the ingest (the parse synchronises on its record count) */
        GF_CUDA_TRY(cudaEventRecord(hs[h]->ev_ingest, st));
    const uint64_t n = pe ? std::min(idx->fq[0].n_records, idx->fq[1].n_records) : idx->fq[0].n_records;
    *n_records = n;
    for (uint32_t h = 0; h < nh; h++) hs[h]->stats.n_pairs = n;
    idx->stats.h2d_bytes = host1 + (pe ? host2 : 0) + h2d_members;
    /* bytes the n whole records cover = one past the newline that ends record n - 1's quality line (shifted table: nl[4 n]) */
    for (int k = 0; k < (pe ? 2 : 1) && n; k++) {
        unsigned long long end = 0;
        GF_CUDA_TRY(cudaMemcpyAsync(&end, idx->fq[k].nl.as<unsigned long long>() + 4 * n, sizeof(end), cudaMemcpyDeviceToHost, st));
        GF_CUDA_TRY(cudaStreamSynchronize(st));
        consumed[k] = std::min<uint64_t>(end + 1, k ? bytes2 : bytes1);
    }
    /* the unconsumed text of a mate whose members were inflated here exists on the device only: it goes back now, before any
     * other call on idx can reuse the staging buffer */
    for (int k = 0; k < (pe ? 2 : 1) && tail && members && !final_chunk; k++) {
        tail[k].clear();
        if (!members[k].n_members) continue;
        const uint64_t from = consumed[k], len = (k ? bytes2 : bytes1) - from;
        tail[k].resize(len);
        if (len) GF_CUDA_TRY(cudaMemcpyAsync(tail[k].data(), (k ? sg.seq2 : sg.seq1).as<uint8_t>() + from, len, cudaMemcpyDeviceToHost, st));
        GF_CUDA_TRY(cudaStreamSynchronize(st));
    }
    if (n == 0) return GF_OK;
    GfDevBatch db{};
    db.n = n;
    db.seq1 = db.qual1 = sg.seq1.as<uint8_t>();
    db.s1 = idx->fq[0].s.as<uint64_t>();
    db.e1 = idx->fq[0].e.as<uint64_t>();
    db.qs1 = idx->fq[0].qs.as<uint64_t>();
    db.bytes1 = bytes1;
    db.max_len = idx->fq[0].max_len;
    if (pe) {
        db.seq2 = db.qual2 = sg.seq2.as<uint8_t>();
        db.s2 = idx->fq[1].s.as<uint64_t>();
        db.e2 = idx->fq[1].e.as<uint64_t>();
        db.qs2 = idx->fq[1].qs.as<uint64_t>();
        db.bytes2 = bytes2;
        db.max_len = std::max(db.max_len, idx->fq[1].max_len);
    }
    if (db.max_len == 0) db.max_len = 1;
    const uint64_t cap = (pe ? 2 : 1) * n;
    std::vector<unsigned long long> launches0(nh);
    for (uint32_t h = 0; h < nh; h++) launches0[h] = hs[h]->launches;
    GfRecordLists lists{};
    for (uint32_t h = 0; h < nh; h++) { /* every index into its own record buffers; k_prep ran once, for hs[0] */
        gf_index* x = hs[h];
        GfStage& xs = x->stage[0];
        GF_CUDA_TRY(xs.out.reserve(sizeof(gf_match) * cap));
        GF_CUDA_TRY(xs.nout.reserve(2 * sizeof(unsigned long long)));
        rc = gf_map_device_batch(x, db, xs.out.as<gf_match>(), cap, xs.nout.as<unsigned long long>(), st, nullptr, true,
                                 h ? idx : nullptr);
        if (rc != GF_OK) return rc;
        const uint32_t mode = x->out_mode;
        if (mode) {
            GF_CUDA_TRY(xs.out2.reserve(sizeof(gf_match) * cap));
            GF_CUDA_TRY(xs.keys.reserve(sizeof(unsigned long long) * cap));
            rc = gf_finish_records_device(x, xs.out.as<gf_match>(), xs.nout.as<unsigned long long>(), cap, xs.out2.as<gf_match>(),
                                          xs.keys.as<unsigned long long>(), xs.nout.as<unsigned long long>() + 1, mode, st);
            if (rc != GF_OK) return rc;
            GF_CUDA_TRY(cudaMemcpyAsync(&x->h_slots[0].n_out2, xs.nout.as<unsigned long long>() + 1, sizeof(unsigned long long),
                                        cudaMemcpyDeviceToHost, st));
        }
        if (h < GF_FASTQ_LIST_MAX) {
            lists.rec[h] = mode ? xs.out2.as<gf_match>() : xs.out.as<gf_match>();
            lists.n[h] = xs.nout.as<unsigned long long>() + (mode ? 1 : 0);
        }
    }
    GfHostSlot* h0 = &idx->h_slots[0];
    if (reads) { /* the lines of the pairs behind the final records, while the text and its newline tables are resident */
        if (nh > GF_FASTQ_LIST_MAX) return fail(GF_E_LIMIT, "more than 64 indices keep reads in one mapping call");
        const uint8_t* text[2] = {sg.seq1.as<uint8_t>(), pe ? sg.seq2.as<uint8_t>() : nullptr};
        rc = gf_fastq_gather_reads(idx, text, n, lists, nh, h0, st);
        if (rc != GF_OK) return rc;
    }
    for (uint32_t h = 0; h < nh; h++) {
        gf_index* x = hs[h];
        GF_CUDA_TRY(cudaMemcpyAsync(&x->h_slots[0].counters, x->ws_counters.p, sizeof(GfMapCounters), cudaMemcpyDeviceToHost, st));
        GF_CUDA_TRY(cudaMemcpyAsync(&x->h_slots[0].n_out, x->stage[0].nout.p, sizeof(unsigned long long), cudaMemcpyDeviceToHost, st));
        GF_CUDA_TRY(cudaEventRecord(x->ev_end, st));
    }
    GF_CUDA_TRY(cudaEventSynchronize(hs[nh - 1]->ev_end));
    bool too_small = false;
    for (uint32_t h = 0; h < nh; h++) {
        gf_index* x = hs[h];
        const GfHostSlot& hx = x->h_slots[0];
        x->busy = false;
        rc = check_flags(hx);
        if (rc != GF_OK) return rc;
        accumulate(x->stats, hx);
        float ms = 0;
        GF_CUDA_TRY(cudaEventElapsedTime(&ms, x->ev_start, x->ev_end));
        x->stats.ms_total = ms;
        GF_CUDA_TRY(cudaEventElapsedTime(&x->stats.ms_ingest, x->ev_start, x->ev_ingest));
        x->stats.kernel_launches = x->launches - launches0[h] + (h ? 0 : 3);
        n_out[h] = x->out_mode ? hx.n_out2 : hx.n_out;
        too_small |= n_out[h] > out_cap[h];
    }
    if (too_small) return fail(GF_E_CAPACITY, "out_cap too small; *n_out holds the required count");
    bool any_panic = false, any_rec = false;
    for (uint32_t h = 0; h < nh; h++) {
        gf_index* x = hs[h];
        const uint32_t mode = x->out_mode;
        const uint64_t n_rec = n_out[h];
        gf_match* o = out[h];
        if (n_rec) GF_CUDA_TRY(cudaMemcpy(o, mode ? x->stage[0].out2.p : x->stage[0].out.p, sizeof(gf_match) * n_rec, cudaMemcpyDeviceToHost));
        x->stats.d2h_bytes = sizeof(gf_match) * n_rec + sizeof(GfMapCounters) + 8;
        if (mode & GF_OUT_BUCKET_ORDER) {
            std::vector<unsigned long long> keys(n_rec);
            if (n_rec) GF_CUDA_TRY(cudaMemcpy(keys.data(), x->stage[0].keys.p, sizeof(unsigned long long) * n_rec, cudaMemcpyDeviceToHost));
            x->stats.d2h_bytes += sizeof(unsigned long long) * n_rec;
            order_by_keys(o, keys, n_rec);
        } else {
            gf_sort_matches(o, n_rec);
        }
        any_rec |= n_rec != 0;
        const bool p = x->h_slots[0].counters.n_ref_panic != 0;
        any_panic |= p;
        if (panic) panic[h] = p;
    }
    if (reads && any_rec) {
        if ((unsigned long long)h0->read_bytes != h0->read_bytes64)
            return fail(GF_E_LIMIT, "the lines of one chunk's matched pairs reach 2^32 bytes: feed smaller chunks");
        rc = gf_fastq_regather_reads(idx, h0->read_bytes64, st); /* (the arena was too small: grown, lines copied now) */
        if (rc != GF_OK) return rc;
        idx->stats.kernel_launches = idx->launches - launches0[0] + 3;
        /* the union of the indices' pairs; one index: it is that index's list as it is (every mask is 1) */
        GfFastqReads uni;
        GfFastqReads& u = nh == 1 ? reads[0] : uni;
        u.pairs.resize(h0->n_read_pairs);
        u.text.resize(h0->read_bytes);
        GF_CUDA_TRY(cudaMemcpy(u.pairs.data(), idx->fq_reads.pairs.p, sizeof(gf_fastq_read_pair) * h0->n_read_pairs,
                               cudaMemcpyDeviceToHost));
        if (h0->read_bytes) GF_CUDA_TRY(cudaMemcpy(u.text.data(), idx->fq_reads.text.p, h0->read_bytes, cudaMemcpyDeviceToHost));
        idx->stats.d2h_bytes += sizeof(gf_fastq_read_pair) * h0->n_read_pairs + h0->read_bytes + 2 * sizeof(uint32_t) + 8;
        if (nh > 1) { /* each index gets its own pairs, its text laid out as a stream over that index alone lays it out */
            std::vector<unsigned long long> masks(h0->n_read_pairs);
            GF_CUDA_TRY(cudaMemcpy(masks.data(), idx->fq_reads.pair_mask.p, sizeof(unsigned long long) * masks.size(),
                                   cudaMemcpyDeviceToHost));
            idx->stats.d2h_bytes += sizeof(unsigned long long) * masks.size();
            for (size_t j = 0; j < masks.size(); j++) {
                const gf_fastq_read_pair& p = u.pairs[j];
                uint64_t len = 0;
                for (int m = 0; m < 2; m++)
                    for (int l = 0; l < 4; l++) len += p.len[m][l];
                for (uint32_t h = 0; h < nh; h++) {
                    if (!((masks[j] >> h) & 1ull)) continue;
                    gf_fastq_read_pair q = p;
                    q.text_off = reads[h].text.size();
                    reads[h].pairs.push_back(q);
                    reads[h].text.insert(reads[h].text.end(), u.text.begin() + p.text_off, u.text.begin() + p.text_off + len);
                }
            }
        }
    }
    if (any_panic)
        return fail(GF_E_REF_PANIC, "a candidate needs an edit distance over more than 640 columns (reference panics)");
    return GF_OK;
}

extern "C" {

static_assert(sizeof(gf_map_stats) == 120 && sizeof(gf_match) == 48 && sizeof(gf_fastq_read_pair) == 48,
              "ABI layout (include/genefuse_gpu.h, _abi.py)");
int gf_get_map_stats(const gf_index* cidx, gf_map_stats* out) {
    gf_index* idx = const_cast<gf_index*>(cidx);
    if (!idx || !out) return fail(GF_E_INVALID, "NULL argument");
    std::lock_guard<std::mutex> lk(idx->mu);
    int rc = GF_OK;
    if (idx->stats_pending) {
        GF_CUDA_TRY(cudaSetDevice(idx->device));
        GF_CUDA_TRY(cudaEventSynchronize(idx->ev_end));
        const GfHostSlot& h = idx->h_slots[GF_SLOT_DEVICE];
        accumulate(idx->stats, h);
        /* per-stage device time: the sum over the chunks of the call, from the events between the launches */
        gf_map_stats& S = idx->stats;
        S.ms_screen = S.ms_exact = S.ms_merge = S.ms_prep = S.ms_seed = S.ms_diag = S.ms_scan = 0; /* fast_merge is fused into k_prep */
        for (uint32_t c = 0; c < idx->n_chunks_timed && c < idx->chunk_events.size(); c++) {
            const GfChunkEvents& ce = idx->chunk_events[c];
            float t = 0;
            GF_CUDA_TRY(cudaEventElapsedTime(&t, ce.e[0], ce.e[4])); S.ms_screen += t;
            GF_CUDA_TRY(cudaEventElapsedTime(&t, ce.e[4], ce.e[5])); S.ms_exact += t;
            if (idx->split_events) {
                GF_CUDA_TRY(cudaEventElapsedTime(&t, ce.e[0], ce.e[1])); S.ms_prep += t;
                GF_CUDA_TRY(cudaEventElapsedTime(&t, ce.e[1], ce.e[2])); S.ms_seed += t;
                GF_CUDA_TRY(cudaEventElapsedTime(&t, ce.e[2], ce.e[3])); S.ms_diag += t;
                GF_CUDA_TRY(cudaEventElapsedTime(&t, ce.e[3], ce.e[4])); S.ms_scan += t;
            }
        }
        GF_CUDA_TRY(cudaEventElapsedTime(&S.ms_total, idx->ev_start, idx->ev_end));
        idx->stats_pending = false;
        idx->busy = false; /* ev_end was recorded after the work ev_busy stands for */
        rc = check_flags(h);
        if (rc == GF_OK && h.counters.n_ref_panic)
            rc = fail(GF_E_REF_PANIC, "a candidate needs an edit distance over more than 640 columns (reference panics)");
    }
    *out = idx->stats;
    return rc;
}

/* FusionResult::adjust_fusion_break for a set of clustered matches (src/core/fusion_result.rs:299-397) */
int gf_adjust_fusion_break(gf_index* idx, const uint8_t* bytes, uint64_t n_bytes, const gf_break_ref* refs, uint32_t n_refs,
                           const gf_break_job* jobs, uint64_t n_jobs, gf_break_out* out) {
    if (!idx || (n_jobs && (!jobs || !out || !refs)) || (n_bytes && !bytes)) return fail(GF_E_INVALID, "NULL argument");
    if (n_jobs == 0) return GF_OK;
    for (uint64_t j = 0; j < n_jobs; j++) {
        const gf_break_job& b = jobs[j];
        if (b.result >= n_refs) return fail(GF_E_INVALID, "gf_break_job.result out of range");
        if (b.seq_off > n_bytes || b.seq_len > n_bytes - b.seq_off) return fail(GF_E_INVALID, "gf_break_job sequence outside the arena");
        if (b.seq_len > GF_MAX_SEQ_LEN) return fail(GF_E_LIMIT, "gf_break_job sequence longer than GF_MAX_SEQ_LEN");
    }
    for (uint32_t r = 0; r < n_refs; r++) {
        const gf_break_ref& f = refs[r];
        if (f.left_off > n_bytes || f.left_len > n_bytes - f.left_off || f.right_off > n_bytes || f.right_len > n_bytes - f.right_off)
            return fail(GF_E_INVALID, "gf_break_ref string outside the arena");
    }
    std::lock_guard<std::mutex> lk(idx->mu);
    GF_CUDA_TRY(cudaSetDevice(idx->device));
    GfStage& s = idx->stage[0];
    GF_CUDA_TRY(s.seq1.reserve(n_bytes + 16));
    GF_CUDA_TRY(s.off1.reserve(sizeof(gf_break_ref) * (size_t)n_refs));
    GF_CUDA_TRY(s.off2.reserve(sizeof(gf_break_job) * n_jobs));
    GF_CUDA_TRY(s.out.reserve(sizeof(gf_break_out) * n_jobs + 16));
    GF_CUDA_TRY(idx->ws_counters.reserve(sizeof(GfMapCounters)));
    cudaStream_t st = idx->stream;
    { int r = wait_prior_device_work(idx, st); if (r != GF_OK) return r; }
    unsigned int* d_flagged = &idx->ws_counters.as<GfMapCounters>()->n_ref_panic;
    GF_CUDA_TRY(cudaMemsetAsync(idx->ws_counters.p, 0, sizeof(GfMapCounters), st));
    if (n_bytes) GF_CUDA_TRY(cudaMemcpyAsync(s.seq1.p, bytes, n_bytes, cudaMemcpyHostToDevice, st));
    GF_CUDA_TRY(cudaMemcpyAsync(s.off1.p, refs, sizeof(gf_break_ref) * (size_t)n_refs, cudaMemcpyHostToDevice, st));
    GF_CUDA_TRY(cudaMemcpyAsync(s.off2.p, jobs, sizeof(gf_break_job) * n_jobs, cudaMemcpyHostToDevice, st));
    int rc = gf_adjust_break_device(idx, s.seq1.as<uint8_t>(), s.off1.as<gf_break_ref>(), s.off2.as<gf_break_job>(), n_jobs,
                                    s.out.as<gf_break_out>(), d_flagged, st);
    if (rc != GF_OK) return rc;
    GF_CUDA_TRY(cudaMemcpyAsync(out, s.out.p, sizeof(gf_break_out) * n_jobs, cudaMemcpyDeviceToHost, st));
    unsigned int n_flagged = 0;
    GF_CUDA_TRY(cudaMemcpyAsync(&n_flagged, d_flagged, sizeof(unsigned int), cudaMemcpyDeviceToHost, st));
    GF_CUDA_TRY(cudaStreamSynchronize(st));
    if (n_flagged)
        return fail(GF_E_REF_PANIC, "a shifted break point lies outside its read or a distance needs more than 640 columns "
                                    "(gf_break_out.status)");
    return GF_OK;
}

int gf_fast_merge(gf_index* idx, const gf_batch* in, gf_merge_info* out) {
    if (!idx || !out) return fail(GF_E_INVALID, "NULL argument");
    int rc = validate_batch(in);
    if (rc != GF_OK) return rc;
    if (in->n == 0) return GF_OK;
    if (!in->seq2) return fail(GF_E_INVALID, "gf_fast_merge needs a paired batch");
    std::lock_guard<std::mutex> lk(idx->mu);
    GF_CUDA_TRY(cudaSetDevice(idx->device));
    const uint64_t n = in->n;
    const uint64_t b1 = in->off1[0], e1 = in->off1[n], b2 = in->off2[0], e2 = in->off2[n];
    uint64_t mx = 0;
    rc = scan_offsets(in->off1, in->off2, n, in->max_len ? std::min<uint64_t>(in->max_len, 1024) : 1024, &mx);
    if (rc != GF_OK) return rc;
    rc = wait_prior_device_work(idx, idx->stream);
    if (rc != GF_OK) return rc;
    GfStage& s = idx->stage[0];
    GF_CUDA_TRY(s.seq1.reserve(e1 - b1 + 16));
    GF_CUDA_TRY(s.qual1.reserve(e1 - b1 + 16));
    GF_CUDA_TRY(s.off1.reserve(sizeof(uint64_t) * (n + 1)));
    GF_CUDA_TRY(s.seq2.reserve(e2 - b2 + 16));
    GF_CUDA_TRY(s.qual2.reserve(e2 - b2 + 16));
    GF_CUDA_TRY(s.off2.reserve(sizeof(uint64_t) * (n + 1)));
    GF_CUDA_TRY(s.out.reserve(sizeof(gf_merge_info) * n));
    cudaStream_t st = idx->stream;
    GF_CUDA_TRY(cudaMemcpyAsync(s.seq1.p, in->seq1 + b1, e1 - b1, cudaMemcpyHostToDevice, st));
    GF_CUDA_TRY(cudaMemcpyAsync(s.qual1.p, in->qual1 + b1, e1 - b1, cudaMemcpyHostToDevice, st));
    GF_CUDA_TRY(cudaMemcpyAsync(s.off1.p, in->off1, sizeof(uint64_t) * (n + 1), cudaMemcpyHostToDevice, st));
    GF_CUDA_TRY(cudaMemcpyAsync(s.seq2.p, in->seq2 + b2, e2 - b2, cudaMemcpyHostToDevice, st));
    GF_CUDA_TRY(cudaMemcpyAsync(s.qual2.p, in->qual2 + b2, e2 - b2, cudaMemcpyHostToDevice, st));
    GF_CUDA_TRY(cudaMemcpyAsync(s.off2.p, in->off2, sizeof(uint64_t) * (n + 1), cudaMemcpyHostToDevice, st));
    GfDevBatch db{};
    db.n = n;
    db.seq1 = s.seq1.as<uint8_t>();
    db.qual1 = s.qual1.as<uint8_t>();
    db.s1 = s.off1.as<uint64_t>(); db.e1 = db.s1 + 1; db.qs1 = db.s1;
    db.seq2 = s.seq2.as<uint8_t>();
    db.qual2 = s.qual2.as<uint8_t>();
    db.s2 = s.off2.as<uint64_t>(); db.e2 = db.s2 ? db.s2 + 1 : nullptr; db.qs2 = db.s2;
    db.base1 = b1;
    db.base2 = b2;
    db.bytes1 = e1 - b1;
    db.bytes2 = e2 - b2;
    db.max_len = (uint32_t)std::max<uint64_t>(mx, 1);
    rc = gf_fast_merge_device(idx, db, s.out.as<gf_merge_info>(), st);
    if (rc != GF_OK) return rc;
    GF_CUDA_TRY(cudaMemcpyAsync(out, s.out.p, sizeof(gf_merge_info) * n, cudaMemcpyDeviceToHost, st));
    GfHostSlot* h = &idx->h_slots[0];
    GF_CUDA_TRY(cudaMemcpyAsync(&h->counters, idx->ws_counters.p, sizeof(GfMapCounters), cudaMemcpyDeviceToHost, st));
    GF_CUDA_TRY(cudaStreamSynchronize(st));
    return check_flags(*h);
}

} /* extern "C" */

/* ---- multi-device handle ------------------------------------------------------------------------------ */
struct gf_multi {
    std::vector<gf_index*> idx;
};

extern "C" int gf_multi_create(const gf_gene_span* genes, uint32_t n_genes, const gf_params* params, const int* devices,
                               int n_devices, gf_multi** out) {
    if (!out) return fail(GF_E_INVALID, "out is NULL");
    *out = nullptr;
    if (n_devices <= 0 || !devices) return fail(GF_E_INVALID, "no devices given");
    gf_multi* m = new gf_multi();
    m->idx.assign((size_t)n_devices, nullptr);
    std::vector<int> rcs((size_t)n_devices, GF_OK);
    std::vector<std::string> errs((size_t)n_devices);
    std::vector<std::thread> th;
    for (int k = 0; k < n_devices; k++)
        th.emplace_back([&, k] {
            rcs[(size_t)k] = gf_index_create(genes, n_genes, params, devices[k], &m->idx[(size_t)k]);
            if (rcs[(size_t)k] != GF_OK) errs[(size_t)k] = gf_last_error();
        });
    for (auto& t : th) t.join();
    for (int k = 0; k < n_devices; k++)
        if (rcs[(size_t)k] != GF_OK) {
            int rc = rcs[(size_t)k];
            std::string e = errs[(size_t)k];
            for (gf_index* h : m->idx) if (h) gf_index_destroy(h);
            delete m;
            return fail(rc, "device " + std::to_string(devices[k]) + ": " + e);
        }
    *out = m;
    return GF_OK;
}

extern "C" void gf_multi_destroy(gf_multi* m) {
    if (!m) return;
    for (gf_index* h : m->idx) if (h) gf_index_destroy(h);
    delete m;
}

extern "C" int gf_multi_map_pairs(gf_multi* m, const gf_batch* in, gf_match* out, uint64_t out_cap, uint64_t* n_out) {
    if (!m || !n_out) return fail(GF_E_INVALID, "NULL argument");
    *n_out = 0;
    int rc0 = validate_batch(in);
    if (rc0 != GF_OK) return rc0;
    const size_t nd = m->idx.size();
    const uint64_t n = in->n;
    const bool pe = in->seq2 != nullptr;
    std::vector<std::vector<gf_match>> parts(nd);
    std::vector<int> rcs(nd, GF_OK);
    std::vector<std::string> errs(nd);
    std::vector<std::thread> th;
    for (size_t k = 0; k < nd; k++)
        th.emplace_back([&, k] {
            /* contiguous shard [lo, hi): sizes differ by at most one pair */
            const uint64_t base = n / nd, rem = n % nd;
            const uint64_t lo = k * base + std::min<uint64_t>(k, rem), hi = lo + base + (k < rem ? 1 : 0);
            if (hi == lo) return;
            gf_batch sb = *in;
            sb.n = hi - lo;
            sb.off1 = in->off1 + lo; /* offsets stay absolute into the shared arenas */
            sb.bytes1 = in->off1[hi] - in->off1[lo];
            if (pe) { sb.off2 = in->off2 + lo; sb.bytes2 = in->off2[hi] - in->off2[lo]; }
            uint64_t cap = std::max<uint64_t>(4096, sb.n / 64), got = 0; /* matches are << 1 % of pairs; grown on GF_E_CAPACITY */
            for (;;) {
                parts[k].resize(cap);
                int rc = gf_map_pairs(m->idx[k], &sb, parts[k].data(), cap, &got);
                if (rc == GF_E_CAPACITY) { cap = got; continue; }
                rcs[k] = rc;
                if (rc != GF_OK) errs[k] = gf_last_error();
                break;
            }
            parts[k].resize(rcs[k] == GF_OK || rcs[k] == GF_E_REF_PANIC ? got : 0);
            for (auto& r : parts[k]) r.pair_idx += lo;
        });
    for (auto& t : th) t.join();
    int rc = GF_OK;
    uint64_t total = 0;
    for (size_t k = 0; k < nd; k++) {
        if (rcs[k] != GF_OK && rcs[k] != GF_E_REF_PANIC) return fail(rcs[k], "shard " + std::to_string(k) + ": " + errs[k]);
        if (rcs[k] == GF_E_REF_PANIC) rc = GF_E_REF_PANIC;
        total += parts[k].size();
    }
    *n_out = total;
    if (total > out_cap) return fail(GF_E_CAPACITY, "out_cap too small; *n_out holds the required count");
    uint64_t w = 0;
    for (size_t k = 0; k < nd; k++) {
        if (!parts[k].empty()) memcpy(out + w, parts[k].data(), sizeof(gf_match) * parts[k].size());
        w += parts[k].size();
    }
    if (rc == GF_E_REF_PANIC) gf_set_error("a candidate needs an edit distance over more than 640 columns (reference panics)");
    return rc;
}

/* debug hook (not part of the ABI header): survivor list of the last mapping call on this handle */
extern "C" int gf_debug_get_survivors(gf_index* idx, uint32_t* out_pairs_meta, uint64_t cap, uint64_t* n) {
    std::lock_guard<std::mutex> lk(idx->mu);
    GF_CUDA_TRY(cudaSetDevice(idx->device));
    GF_CUDA_TRY(cudaDeviceSynchronize());
    GfMapCounters c;
    GF_CUDA_TRY(cudaMemcpy(&c, idx->ws_counters.p, sizeof(c), cudaMemcpyDeviceToHost));
    *n = c.n_survivors;
    uint64_t m = std::min<uint64_t>(cap, c.n_survivors);
    if (m) GF_CUDA_TRY(cudaMemcpy(out_pairs_meta, idx->ws_survivors.p, sizeof(uint32_t) * 2 * m, cudaMemcpyDeviceToHost));
    return GF_OK;
}

/* ---- the host packer on its own (include/genefuse_gpu.h); no device involved ---- */
extern "C" int gf_pack_supported(void) { return gf_pack_available() ? 1 : 0; }

extern "C" int gf_pack_reads(const uint8_t* seq, const uint64_t* off, uint64_t n, int mate2, uint32_t* words, uint32_t* woff,
                             uint32_t* xwords, uint32_t* xoff, uint64_t cap_words, uint64_t* n_words, uint64_t* n_xwords) {
    if (!off || !n_words || !n_xwords || (n && (!seq || !woff || !xoff))) return fail(GF_E_INVALID, "NULL argument");
    if (!gf_pack_available()) return fail(GF_E_INVALID, "the packed upload needs AVX-512BW on the host (or GF_HOST_PACK=0 is set)");
    uint64_t need = 0;
    for (uint64_t i = 0; i < n; i++) {
        if (off[i + 1] < off[i]) return fail(GF_E_INVALID, "offsets are not ascending");
        if (off[i + 1] - off[i] > 1024) return fail(GF_E_INVALID, "a read is longer than 1024 bases");
        need += 2 * ((off[i + 1] - off[i] + 31) >> 5);
    }
    *n_words = need;
    *n_xwords = 0;
    if (need > 0x7FFFFFFFull) return fail(GF_E_LIMIT, "more than 2^31 plane words: split the batch");
    if (need > cap_words) return fail(GF_E_CAPACITY, "cap_words too small; *n_words holds the required count");
    if (!n) return GF_OK;
    if (need && (!words || !xwords)) return fail(GF_E_INVALID, "NULL argument");
    GfPackMate pm{};
    pm.seq = seq;
    pm.off = off;
    pm.off_base = off[0];
    pm.n = n;
    pm.mate2 = mate2 != 0;
    pm.max_len = 1024;
    pm.words = words;
    pm.woff = woff;
    pm.xwords = xwords;
    pm.xoff = xoff;
    gf_pack_chunk(&pm, 1);
    /* the packing threads wrote their exception words into separate regions: close the gaps */
    uint64_t fill = 0;
    for (int t = 0; t < pm.n_threads; t++) {
        const uint64_t a = n * (uint64_t)t / pm.n_threads, b = n * (uint64_t)(t + 1) / pm.n_threads;
        const uint64_t shift = pm.xregion_start[t] - fill;
        if (pm.xregion_used[t] && shift) {
            memmove(xwords + fill, xwords + pm.xregion_start[t], sizeof(uint32_t) * pm.xregion_used[t]);
            for (uint64_t i = a; i < b; i++)
                if (xoff[i]) xoff[i] -= (uint32_t)shift;
        }
        fill += pm.xregion_used[t];
    }
    *n_xwords = fill;
    return GF_OK;
}
