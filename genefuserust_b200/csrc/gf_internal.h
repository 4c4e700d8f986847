/* gf_internal.h — host-side handle and helpers shared by the .cu translation units (not part of the ABI). */
#pragma once
#include <cuda_runtime.h>

#include <mutex>
#include <string>
#include <vector>

#include "../../include/genefuse_gpu.h"
#include "gf_device.cuh"
#include "gf_pack.h"

void gf_set_error(const std::string& msg);

#define GF_CUDA_TRY(expr)                                                                              \
    do {                                                                                               \
        cudaError_t _e = (expr);                                                                       \
        if (_e != cudaSuccess) {                                                                       \
            gf_set_error(std::string(#expr) + " failed: " + cudaGetErrorString(_e) + " (" + __FILE__ + \
                         ":" + std::to_string(__LINE__) + ")");                                        \
            return GF_E_CUDA;                                                                          \
        }                                                                                              \
    } while (0)

/* grow-only device buffer */
struct GfBuf {
    void* p = nullptr;
    size_t cap = 0;
    cudaError_t reserve(size_t bytes) {
        if (bytes <= cap) return cudaSuccess;
        if (p) cudaFree(p);
        p = nullptr;
        cap = 0;
        size_t want = bytes + bytes / 8 + 256;
        cudaError_t e = cudaMalloc(&p, want);
        if (e == cudaSuccess) cap = want;
        return e;
    }
    void release() {
        if (p) cudaFree(p);
        p = nullptr;
        cap = 0;
    }
    template <class T>
    T* as() const { return (T*)p; }
};

/* device-side counters of one mapping call (single 128-byte block, zeroed per call) */
struct GfMapCounters {
    unsigned long long n_sequences;   /* sequences screened */
    unsigned long long n_probes;      /* pass-1 probes issued by the screen */
    unsigned long long seq_bytes;     /* bytes of screened sequences */
    unsigned long long n_merged;      /* pairs merged */
    unsigned int n_survivors;         /* entries appended to the survivor list */
    unsigned int n_candidates;        /* candidates appended by the exact kernel */
    unsigned int n_ref_panic;         /* edit distances beyond the reference's 640-column limit */
    unsigned int error_flags;         /* bit 0: a read is longer than the kernel capacity; bit 1: survivor list overflow */
    unsigned long long n_survivors_total; /* survivors of the chunks before the current one (device batches run in chunks) */
    unsigned long long verify_from;       /* records [verify_from, *n_out) belong to the current chunk (k_verify's range) */
    unsigned long long pad[7];
};

/* grow-only pinned host buffer (contents are not kept when it grows) */
struct GfPinned {
    void* p = nullptr;
    size_t cap = 0;
    cudaError_t reserve(size_t bytes) {
        if (bytes <= cap) return cudaSuccess;
        if (p) cudaFreeHost(p);
        p = nullptr;
        cap = 0;
        size_t want = bytes + bytes / 8 + 4096;
        cudaError_t e = cudaMallocHost(&p, want);
        if (e == cudaSuccess) cap = want;
        return e;
    }
    void release() {
        if (p) cudaFreeHost(p);
        p = nullptr;
        cap = 0;
    }
    template <class T>
    T* as() const { return (T*)p; }
};

constexpr int GF_STAGES = 6;      /* chunks of a host batch in flight at once */
constexpr int GF_PACK_SETS = 6;   /* pinned buffer sets the packing threads fill (packed upload) */
constexpr int GF_SLOT_DEVICE = GF_STAGES;

struct GfStage { /* one in-flight chunk of a host batch */
    GfBuf seq1, qual1, off1, seq2, qual2, off2, out, nout;
    /* packed upload (gf_pack.cpp), per mate: plane words, their per-read offsets, exception words, per-read exception offsets —
     * built in a GfPackSet's pinned buffers by the host threads, copied to these device buffers */
    GfBuf pk[2], pko[2], pkx[2], pxo[2];
    GfBuf out2, keys; /* output mode != 0: compacted records + their order keys (nout holds two counters then) */
    cudaEvent_t copied = nullptr, done = nullptr;
    uint64_t n = 0, pair_base = 0, out_cap = 0;
};
struct GfPackSet { /* packed upload: what the packing threads build for one chunk; free again once it has been copied */
    GfPinned h_pk[2], h_pko[2], h_pkx[2], h_pxo[2];
    cudaEvent_t copied = nullptr;
};
struct GfHostSlot { /* pinned host memory the device writes results of one call/chunk into */
    GfMapCounters counters;
    unsigned long long n_out;
    unsigned long long n_out2; /* records left after the device-side filter (output mode != 0) */
    /* gf_map_fastq_text with the reads kept: pairs that have a record, the bytes of their lines (32-bit scan) and the same
     * bytes summed in 64 bits (they differ when a chunk's lines reach 2^32 bytes) */
    unsigned int n_read_pairs, read_bytes;
    unsigned long long read_bytes64;
    unsigned long long pad[12];
};

/* gf_fastq.cu: FASTQ text already on the device -> per-record start/end/quality-start tables */
struct GfFastqTable {
    uint64_t n_records = 0;
    uint32_t max_len = 0;
    GfBuf nl, s, e, qs; /* newline positions; sequence start / end; quality start (u64 each) */
    GfBuf cnt, off, tmp; /* per-tile newline counts, their exclusive scan, scan workspace (kept between calls) */
    void release() { nl.release(); s.release(); e.release(); qs.release(); cnt.release(); off.release(); tmp.release(); }
};

/* gf_fastq.cu: device workspace of gf_fastq_gather_reads (grow-only) */
struct GfFastqReadsWork {
    GfBuf mask, has, slot, bytes, off, tmp, total; /* per local pair: bit h = index h of the list has a record of it, 0/1 "has a
                                                      record", its slot, its bytes, its text offset; scan workspace */
    GfBuf pairs, pair_mask, text;             /* descriptors of the matched pairs and their masks (per pair of the chunk: their
                                                 count is known on the device only); their lines back to back (grow-only, sized
                                                 to the largest total seen) */
    const uint8_t *text1 = nullptr, *text2 = nullptr; /* the last gather: the chunk's text, its pairs, the arena bytes it could use */
    uint64_t n = 0, arena_used = 0;
    void release() {
        mask.release(); has.release(); slot.release(); bytes.release(); off.release(); tmp.release(); total.release();
        pairs.release(); pair_mask.release(); text.release();
    }
};
/* gf_map_fastq_text's optional output, per index: the lines of every pair that has a record of that index, in ascending pair
 * order (pair_idx counts from the start of the call's text, text_off into `text`) */
struct GfFastqReads {
    std::vector<gf_fastq_read_pair> pairs;
    std::vector<uint8_t> text;
};
/* indices one FASTQ stream maps against (one bit each in the per-pair masks of gf_fastq_gather_reads) */
constexpr uint32_t GF_FASTQ_LIST_MAX = 64;
/* the final record lists of a list's indices, as kernel parameters (device pointers; the counts are read on the device) */
struct GfRecordLists {
    const gf_match* rec[GF_FASTQ_LIST_MAX];
    const unsigned long long* n[GF_FASTQ_LIST_MAX];
};

struct GfChunkEvents { /* start, after k_prep, k_seed, k_diag, the whole screen, exact + verify */
    cudaEvent_t e[6] = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};
};

/* gf_fastq.cu: BGZF members of a .fq.gz chunk inflated on the device, one thread per member (csrc/gf_inflate.cuh) */
struct GfBgzfMember {
    uint64_t in_off;  /* raw DEFLATE payload inside the compressed buffer */
    uint64_t out_off; /* where its text goes */
    uint32_t clen, isize, crc, pad;
};
/* status[0]: OR of (1 << error code) over the members, status[1]: 1 + index of a failing member */
int gf_bgzf_inflate_device(const uint8_t* d_comp, const GfBgzfMember* d_members, uint32_t n, uint8_t* d_text, unsigned int* d_status,
                           cudaStream_t st);
/* per mate of gf_map_fastq_text: text that is partly on the host (`prefix` bytes, passed as fq1 / fq2) and partly still
 * compressed (BGZF members: their payloads back to back in `comp`, pinned host memory) */
struct GfFastqMembers {
    const uint8_t* comp = nullptr;
    uint64_t comp_bytes = 0;
    const GfBgzfMember* members = nullptr;
    uint32_t n_members = 0;
    uint64_t text_bytes = 0; /* sum of isize */
};

struct gf_index {
    int device = 0;
    gf_params params{};
    GfDevIndex dev{};
    gf_index_info info{};
    uint32_t n_genes = 0;
    std::vector<uint32_t> gene_start, gene_len;

    void *d_table = nullptr, *d_dupes = nullptr, *d_gene_ascii = nullptr, *d_gene_start = nullptr,
         *d_gene_len = nullptr, *d_gene_rev = nullptr, *d_planes = nullptr, *d_filter = nullptr, *d_granule = nullptr;

    std::mutex mu; /* serialises calls on one handle */
    cudaStream_t stream = nullptr, copy_stream = nullptr;
    cudaEvent_t ev_busy = nullptr; /* recorded at the end of every unsynchronised device-batch call (gf_map_pairs_device*):
                                      the next entry point that touches the handle's workspace waits for it on its stream */
    bool busy = false;
    cudaEvent_t ev_start = nullptr, ev_end = nullptr;  /* whole call */
    cudaEvent_t ev_ingest = nullptr;                   /* gf_map_fastq: end of the text ingest */
    std::vector<GfChunkEvents> chunk_events;           /* device-batch path: per chunk, between the launches (created on demand) */
    uint32_t n_chunks_timed = 0;                       /* chunks of the last device-batch call */
    bool split_events = false;                         /* the last device batch ran the split screen (prep / seed / diag / scan) */
    bool ev_valid = false;

    /* mapping workspace (grow-only) */
    GfBuf ws_survivors, ws_counters, ws_gtbl;
    GfFastqTable fq[2];
    GfFastqReadsWork fq_reads;
    GfBuf ws_seq_words, ws_seq_meta, ws_seq_seed, ws_seq_lists; /* split screen pipeline (gf_screen_split.cuh): sequence store
                                                                  (plane words, meta, seeds); counters + the two class lists */
    GfStage stage[GF_STAGES];
    GfPackSet pack_set[GF_PACK_SETS];
    GfBuf bgzf_comp[2], bgzf_members[2], bgzf_status; /* .fq.gz chunks inflated on the device */
    GfHostSlot* h_slots = nullptr; /* [GF_STAGES + 1]: the pipeline stages + the device-batch path (GF_SLOT_DEVICE) */
    bool stats_pending = false;    /* h_slots[2] is being written by an unsynchronised device-batch call */
    uint64_t pending_pairs = 0;
    gf_map_stats stats{};
    unsigned long long launches = 0;
    int sm_count = 148;
    uint32_t out_mode = 0; /* GF_OUT_* (gf_index_set_output_mode) */
};

/* gf_index.cu */
int gf_build_index_device(gf_index* idx, const gf_gene_span* genes, uint32_t n_genes);
int gf_lookup_device(gf_index* idx, const uint32_t* kmers, uint64_t n, gf_lookup* out);

size_t gf_scan_tmp_elems(uint64_t n);
cudaError_t gf_exclusive_scan_u32(const uint32_t* in, uint32_t* out, uint64_t n, uint32_t* tmp, cudaStream_t st);
uint32_t gf_scan_launches(uint64_t n); /* kernels gf_exclusive_scan_u32 launches for n elements */

/* final_chunk: the text ends the file (an unterminated last line is a line); otherwise it is ignored (streamed chunks) */
int gf_fastq_parse_device(const uint8_t* d_text, uint64_t bytes, GfFastqTable* out, cudaStream_t st, bool final_chunk = true);
/* gf_api.cu: gf_map_fastq's body, against the nh indices hs[] (all on one device, validated by the caller; all of them are
 * locked for the call).  The text is copied, inflated, split into records and converted once, in hs[0]'s workspace; every
 * index then screens and verifies it into its own record buffers.  out[h] / out_cap[h] / n_out[h] belong to hs[h]
 * (GF_E_CAPACITY when any out_cap[h] is too small: n_out[] holds the required counts, nothing is copied).  final_chunk = false
 * (gf_fastq_stream_*): only whole records are mapped and consumed[k] returns how many bytes of buffer k they covered (the caller
 * carries the rest over); pair_idx counts from 0.  GF_E_REF_PANIC when any index's records carry the reference's panic; then
 * panic[h] (when given) says which. */
int gf_map_fastq_text(gf_index* const* hs, uint32_t nh, const uint8_t* fq1, uint64_t bytes1, const uint8_t* fq2, uint64_t bytes2,
                      bool final_chunk, gf_match* const* out, const uint64_t* out_cap, uint64_t* n_out, uint64_t* n_records,
                      uint64_t consumed[2],
                      const GfFastqMembers* members = nullptr /* [2]: BGZF members that follow the host text, inflated on the device */,
                      GfFastqReads* reads = nullptr /* [nh]: the lines of the pairs that have a record (nullptr: nothing is gathered) */,
                      bool* panic = nullptr /* [nh] */,
                      std::vector<uint8_t>* tail = nullptr /* [2]: a mate with members gets its unconsumed text back here (the text
                                                               exists on the device only; copied while the indices are locked) */);
/* after the records of a FASTQ chunk are final (lists.rec[h][0 .. *lists.n[h]) for the nh indices of the list, local pair
 * indices): gather the lines of every pair that has a record of any of them from the chunk's text (text[1] = nullptr: single
 * end) into idx->fq_reads, with the mask of the indices it belongs to, and queue the copies of the totals into h
 * (n_read_pairs, read_bytes, read_bytes64).  n = records (pairs) of the chunk.  The lines are copied only when they fit the
 * arena as it is: once the totals have arrived, gf_fastq_regather_reads(idx, h->read_bytes64, st) grows it and copies them
 * when they did not (and returns at once when they did); the text and newline tables must still be resident. */
int gf_fastq_gather_reads(gf_index* idx, const uint8_t* const text[2], uint64_t n, const GfRecordLists& lists, uint32_t nh,
                          GfHostSlot* h, cudaStream_t st);
int gf_fastq_regather_reads(gf_index* idx, uint64_t bytes, cudaStream_t st);
/* gf_api.cu: the checks of gf_list_map_pairs on a list of handles (non-empty, no NULL, none twice, one device) */
int gf_validate_list(gf_index* const* hs, uint32_t nh);

/* gf_map.cu */
struct GfDevBatch {
    uint64_t n;
    const uint8_t *seq1, *qual1, *seq2, *qual2;
    /* per record: start / end of the sequence and start of the quality string, relative to base1/base2.
     * Arena batches: s = off, e = off + 1, qs = off.  FASTQ text: all three point into the parsed line table. */
    const uint64_t *s1, *e1, *qs1, *s2, *e2, *qs2;
    uint64_t base1, base2;   /* value subtracted from every offset (chunked host batches) */
    uint64_t bytes1, bytes2; /* readable extent of the seq/qual arenas (0 = unknown: no bounds guard) */
    uint64_t pair_base;      /* added to the local pair index in emitted records */
    uint32_t max_len;        /* upper bound of any read length (selects the kernel capacity) */
    /* packed upload (gf_pack.cpp; host batches in pinned memory, reads <= 256 bases): k_prep takes the plane words the host
     * built instead of converting the ASCII, and seq1 / seq2 are the MAPPED pinned arenas, read only by k_exact / k_verify
     * for the survivors.  pk == nullptr: convert from ASCII. */
    const uint32_t *pk1 = nullptr, *pk2 = nullptr;   /* plane words: per read nw x lo, nw x hi */
    const uint32_t *pko1 = nullptr, *pko2 = nullptr; /* per read: where its plane words start */
    const uint32_t *pkx1 = nullptr, *pkx2 = nullptr; /* exception words: per flagged read nw x valid, nw x aux */
    const uint32_t *pxo1 = nullptr, *pxo2 = nullptr; /* per read: 0 = every base upper-case ACGT, else 1 + start of its exception words */
};
/* store_owner != nullptr (list mode): reuse the sequence store `store_owner` filled for the SAME batch just before on the same
 * stream instead of running k_prep again (only taken on the split-screen path, reads <= 256 bases; ignored otherwise) */
/* ONE chunk.  first: zero the handle's counters and *d_n_out (later chunks of one call accumulate); ev: events to record
 * between the launches, or nullptr */
int gf_map_device_batch(gf_index* idx, const GfDevBatch& b, gf_match* d_out, uint64_t out_cap,
                        unsigned long long* d_n_out, cudaStream_t stream, GfChunkEvents* ev, bool first,
                        gf_index* store_owner = nullptr);
/* a device-resident batch of any size against nh indices (nh > 1 = list mode): cut into chunks whose workspace stays below
 * ~5 GB, every chunk converted once (hs[0]) and mapped against each index; records accumulate in d_outs[h] / d_n_outs[h] */
int gf_map_device_batches(gf_index* const* hs, uint32_t nh, const GfDevBatch& b, gf_match* const* d_outs, uint64_t out_cap,
                          unsigned long long* const* d_n_outs, cudaStream_t stream);
/* output mode: drop flagged records / compute the bucket-order keys of the records k_verify finished (d_in[0 .. *d_n_in)) */
int gf_finish_records_device(gf_index* idx, const gf_match* d_in, const unsigned long long* d_n_in, uint64_t in_cap,
                             gf_match* d_out2, unsigned long long* d_keys, unsigned long long* d_n_out2, uint32_t mode,
                             cudaStream_t stream);
int gf_fast_merge_device(gf_index* idx, const GfDevBatch& b, gf_merge_info* d_out, cudaStream_t stream);
int gf_adjust_break_device(gf_index* idx, const uint8_t* d_bytes, const gf_break_ref* d_refs, const gf_break_job* d_jobs,
                           uint64_t n_jobs, gf_break_out* d_out, unsigned int* d_n_flagged, cudaStream_t stream);
