/*
 * genefuse_gpu.h — C ABI of the B200-native fusion-matching hot path.
 *
 * This is the drop-in boundary for GeneFuseRust's per-read matching path.  The
 * reference has no FFI of its own (pure Rust); the two call sites this library
 * replaces are
 *
 *   Indexer::make_index            src/core/indexer.rs:122-177   -> gf_index_create
 *   PairEndScanner::scan_pair_end  src/core/pescanner.rs:427-518 -> gf_map_pairs
 *   SingleEndScanner::scan_single_end src/core/sescanner.rs:183-205 -> gf_map_pairs (seq2 == NULL)
 *
 * and the functions below them on the path (Indexer::map_read :252-538,
 * in_required_direction :541-608, FusionMapper::map_read / make_match /
 * calc_distance / calc_ed  src/core/fusion_mapper.rs:93-251, edit_distance
 * src/core/edit_distance.rs:164-197, SequenceReadPair::fast_merge
 * src/core/read.rs:313-440, reverse_complement src/core/sequence.rs:22-60).
 *
 * Everything is plain pointers and sizes.  All compute runs in hand-written
 * sm_100a CUDA kernels; there is no CPU fallback: every entry point fails with
 * GF_E_CUDA when no usable device is present.
 *
 * Threading: calls on DIFFERENT gf_index handles are independent.  Calls on
 * the same handle are serialised internally (one mutex per handle).
 */
#ifndef GENEFUSE_GPU_H
#define GENEFUSE_GPU_H

#include <stdint.h>
#include <stddef.h>

#ifdef __cplusplus
extern "C" {
#endif

#define GF_ABI_VERSION 2

/* status codes (0 = ok, negative = error; text via gf_last_error()) */
enum gf_status {
    GF_OK = 0,
    GF_E_INVALID = -1,   /* bad argument (NULL, inconsistent offsets, too long read, ...) */
    GF_E_CUDA = -2,      /* CUDA runtime error / no device */
    GF_E_CAPACITY = -3,  /* out_cap too small; *n_out = required count */
    GF_E_LIMIT = -4,     /* input exceeds a documented limit of the index layout */
    GF_E_REF_PANIC = -5  /* the reference would panic on this input (edit distance > 640 cols both sides,
                            src/core/edit_distance.rs:94-100,177-196) */
};

/* Limits.  FASTQ lines longer than 1000 bytes make the reference panic
 * (src/core/fastq_reader.rs:27, src/aux/limited_bufreader.rs:75-87). */
#define GF_MAX_READ_LEN 1000u
#define GF_MAX_SEQ_LEN 2048u /* >= 2*GF_MAX_READ_LEN - 30 (longest merged read) */
#define GF_KMER 16           /* src/core/indexer.rs:35 */

/* One fusion gene as Indexer::make_index sees it AFTER the host resolved the
 * chromosome name and sliced + upper-cased contig[m_start..m_end]
 * (src/core/indexer.rs:136-159).  len == 0 stands for an unresolved chromosome
 * (the gene keeps its contig id, :148-151). */
typedef struct gf_gene_span {
    const uint8_t* seq;   /* upper-cased gene bytes, may contain N / IUPAC */
    uint32_t len;
    uint8_t reversed;     /* Gene::is_reversed(), src/core/gene.rs:98-107 */
} gf_gene_span;

/* GlobalSettings fields read on the path (src/aux/global_settings.rs:15-29). */
typedef struct gf_params {
    int32_t skip_key_dup_threshold;      /* 5  */
    int32_t major_gene_key_requirement;  /* 40 */
    int32_t minor_gene_key_requirement;  /* 20 */
    int32_t mismatch_threshold;          /* 10 */
    int32_t deletion_threshold;          /* 50, CLI -d (src/argparse.rs:66-73); only used for GF_FILTER_INDEL */
} gf_params;

/* A batch of read pairs (PE) or reads (SE: seq2 == qual2 == off2 == NULL) as
 * byte arenas with n+1 offsets each.  Record i of arena k is
 * seqk[offk[i] .. offk[i+1]) and its quality string qualk[offk[i] .. offk[i+1])
 * (same offsets: FASTQ sequence and quality have equal length).
 * For gf_map_pairs the pointers are HOST pointers (pinned memory makes the
 * H2D copy faster but is not required); for gf_map_pairs_device they are
 * DEVICE pointers. */
typedef struct gf_batch {
    uint64_t n;
    const uint8_t* seq1;
    const uint8_t* qual1;
    const uint64_t* off1;
    const uint8_t* seq2;
    const uint8_t* qual2;
    const uint64_t* off2;
    uint64_t bytes1; /* == off1[n] - off1[0] */
    uint64_t bytes2; /* == off2[n] - off2[0] (0 for SE) */
    uint32_t max_len; /* hint: upper bound of any read's length in this batch, 0 = unknown.  Selects the
                         kernel capacity (<= 160 / <= 256: thread-per-pair kernels, else warp-per-pair).  A read longer
                         than the hint (or than 1024) makes the call fail with GF_E_INVALID; it is never truncated.
                         0: gf_map_pairs / gf_list_map_pairs find the longest read themselves (host offsets);
                         gf_map_pairs_device cannot without a synchronisation and takes the long-read kernels. */
    uint32_t reserved;
} gf_batch;

/* One fusion match = the integer content of a ReadMatch
 * (src/core/read_match.rs:17-30) plus where it came from.  The host rebuilds
 * the strings (fast_merge / reverse_complement on the few matched pairs).
 * Records are emitted sorted by (pair_idx, source). */
typedef struct gf_match {
    uint64_t pair_idx;   /* index into the batch */
    int32_t read_break;  /* m_read_break */
    int32_t l_pos;       /* m_left_gp.position  (after make_match's shift) */
    int32_t r_pos;       /* m_right_gp.position */
    int32_t gap;         /* m_gap */
    int32_t l_dist;      /* m_left_distance  (-1 / -2 sentinels of calc_ed kept) */
    int32_t r_dist;      /* m_right_distance */
    int32_t seq_len;     /* length of the sequence that matched (m_read.m_seq) */
    int16_t l_contig;    /* m_left_gp.contig */
    int16_t r_contig;    /* m_right_gp.contig */
    int16_t merge_olen;  /* overlap length of fast_merge, -1 when the pair did not merge */
    int16_t merge_diff;  /* the N of "merged_diff_N" (src/core/read.rs:372) */
    uint8_t source;      /* 0 = merged read, 1 = R1, 2 = R2 */
    uint8_t used_rc;     /* 1 = the match was found on the reverse complement (rc retry) */
    uint8_t reversed;    /* m_reversed: set only for R1/R2 rc matches (pescanner.rs:483,506), never for merged */
    uint8_t filter_flags; /* what FusionMapper::filter_matches would do with this record (src/core/fusion_mapper.rs:298-377):
                             GF_FILTER_COMPLEXITY | GF_FILTER_DISTANCE | GF_FILTER_INDEL; 0 = survives all three.
                             Records are never dropped by the library: the host filters run unchanged. */
} gf_match;
#define GF_FILTER_COMPLEXITY 1u /* remove_by_complexity: a side of the break is < 20 chars or has < 7 base changes */
#define GF_FILTER_DISTANCE 2u   /* remove_by_distance: l_dist + r_dist >= 5 */
#define GF_FILTER_INDEL 4u      /* remove_indels: same contig and |l_pos - r_pos| < deletion_threshold */

typedef struct gf_index gf_index; /* opaque */

typedef struct gf_index_info {
    uint64_t n_sites;        /* valid indexed k-mer occurrences (both strands) */
    uint64_t n_keys;         /* distinct k-mers (= set bits of the reference's bitmap) */
    uint64_t n_unique;       /* keys with one site */
    uint64_t n_normal;       /* keys with 2..skip_key_dup_threshold sites (DUPE_NORMAL_LEVEL) */
    uint64_t n_high;         /* keys with more (DUPE_HIGH_LEVEL) */
    uint64_t table_slots;    /* open-addressed slots allocated */
    uint64_t table_bytes;
    uint64_t max_displacement; /* worst (slot - home slot) */
    uint64_t gene_bytes;     /* Σ gene lengths */
    uint64_t device_bytes;   /* total HBM held by the handle */
    double build_ms;         /* device time of the build */
} gf_index_info;

/* Result of a debug/parity lookup of one 16-mer (A=0,T=1,C=2,G=3, first base in
 * the top bits; src/core/indexer.rs:852-913). */
typedef struct gf_lookup {
    int32_t kind;            /* 0 absent, 1 unique, 2 NORMAL dupe (sites sorted by contig, position), 3 HIGH */
    int32_t n_sites;
    int16_t contig[8];
    int32_t position[8];
} gf_lookup;

/* Result of the device fast_merge for one pair (parity hook). */
typedef struct gf_merge_info {
    int32_t merged;          /* 0 / 1 */
    int32_t olen;
    int32_t diff;
    int32_t merged_len;
} gf_merge_info;

/* Per-call device timing and counters of the last gf_map_pairs* on a handle. */
typedef struct gf_map_stats {
    uint64_t n_pairs;
    uint64_t n_sequences;    /* sequences screened (merged or R1+R2) */
    uint64_t n_probes_pass1; /* Σ P1(len) */
    uint64_t n_survivors;    /* sequences sent to the exact path */
    uint64_t n_matches;
    uint64_t seq_bytes;      /* Σ len of the screened sequences */
    uint64_t kernel_launches;
    float ms_total;          /* device time, events on the call's stream */
    float ms_merge;
    float ms_screen;
    float ms_exact;
    uint64_t h2d_bytes;      /* bytes gf_map_pairs copied host -> device (0 for gf_map_pairs_device) */
    uint64_t d2h_bytes;      /* bytes copied device -> host */
    uint32_t zero_copy_qual; /* 1 = the quality arenas were pinned host memory and were NOT copied: the kernels
                                read the few quality bytes fast_merge depends on directly over PCIe */
    uint32_t packed_upload;  /* != 0: sequence AND quality arenas were pinned host memory, reads <= 256 bases and the host has
                                AVX-512BW: for some (2) or all (1) pipeline chunks the host threads built the reads' 2-bit planes
                                and only those were copied (about a third of the bytes) while the copy engine was busy with
                                other chunks; the few reads that survive the screen are fetched from the pinned arenas on
                                demand.  GF_HOST_PACK=0 disables this, =1 packs every chunk; GF_PACK_THREADS sets the number of
                                packing threads. */
    /* the four launches ms_screen is made of (split screen, reads <= 256 bases; 0 otherwise).  gf_map_pairs (chunked
     * host path): the last chunk only, like every other ms_* field there. */
    float ms_prep;           /* k_prep: ASCII -> bit-planes, fast_merge, sequence store */
    float ms_seed;           /* k_seed: seed k-mers -> filter -> one table lookup, class lists */
    float ms_diag;           /* k_diag: seeded sequences against the gene planes */
    float ms_scan;           /* k_scan: unseeded sequences, filter probes */
    float ms_ingest;         /* gf_map_fastq only: H2D of the text + newline scan + record tables (before the mapping) */
    float ms_host_pack;      /* packed upload: host wall-clock milliseconds the packing threads took (sum over the chunks) */
} gf_map_stats;

const char* gf_last_error(void);
int gf_abi_version(void);
int gf_device_count(void);
void gf_default_params(gf_params* p);

/* Build the fusion-gene index on `device` (replaces Indexer::make_index rows:
 * index_contig fwd + reverse complement, dedup 1 / 2..5 / >=6, membership). */
int gf_index_create(const gf_gene_span* genes, uint32_t n_genes, const gf_params* params,
                    int device, gf_index** out);
void gf_index_destroy(gf_index* idx);
int gf_index_get_info(const gf_index* idx, gf_index_info* out);
int gf_index_lookup(gf_index* idx, const uint32_t* kmers, uint64_t n, gf_lookup* out);

/* Map a batch held in HOST memory: H2D copy, merge, screen, exact path,
 * verification, D2H of the match records.  SE when in->seq2 == NULL.
 * Returns GF_E_CAPACITY (and *n_out = needed) when out_cap is too small.
 * Pinned (page-locked) arenas make the copies asynchronous; when the quality
 * arenas are pinned and reads are <= 256 bases they are not copied at all
 * (fast_merge reads a quality byte only where R1 and rc(R2) disagree inside a
 * candidate overlap; those bytes are fetched on demand).  GF_ZEROCOPY_QUAL=0
 * in the environment disables this. */
int gf_map_pairs(gf_index* idx, const gf_batch* in, gf_match* out, uint64_t out_cap, uint64_t* n_out);

/* Same on a batch already resident in DEVICE memory of the index's device.
 * `d_out` / `d_n_out` are device pointers (capacity out_cap records / one
 * uint64).  Work is enqueued on `cuda_stream` (a cudaStream_t, NULL = legacy
 * default stream) and NOT synchronised: the caller owns the stream.  Records
 * are in arbitrary order here; gf_sort_matches orders a host copy.  *d_n_out
 * may exceed out_cap (records beyond the capacity are counted, not written).
 * Input errors detected on the device (a read longer than the capacity) are
 * reported by the next gf_get_map_stats on the handle. */
int gf_map_pairs_device(gf_index* idx, const gf_batch* in_dev, gf_match* d_out, uint64_t out_cap,
                        uint64_t* d_n_out, void* cuda_stream);
void gf_sort_matches(gf_match* m, uint64_t n); /* by (pair_idx, source), host */

/* Map reads given as raw FASTQ text in HOST memory (replaces FastqReader::read + the pack loop,
 * src/core/fastq_reader.rs:75-147, src/core/pescanner.rs:190-249): the text is copied to the device, split
 * into records there (four lines per record, one trailing '\n' stripped per line, nothing validated, an
 * incomplete trailing record is ignored) and mapped without repacking.  fq2 == NULL for single end; for pairs
 * the number of records is the smaller of the two files', like FastqReaderPair.  pair_idx in the output
 * counts records from the start of the buffers.  *n_records = records (pairs) mapped. */
int gf_map_fastq(gf_index* idx, const uint8_t* fq1, uint64_t bytes1, const uint8_t* fq2, uint64_t bytes2,
                 gf_match* out, uint64_t out_cap, uint64_t* n_out, uint64_t* n_records);

/* ---- post-filters and bucket order on the device (SURVEY 8(f) #3) ----
 * What the reference does with the records after the scan: add_match drops each into bucket n_genes * right.contig +
 * left.contig (src/core/fusion_mapper.rs:253-275), filter_matches removes records by three per-record predicates (:298-377,
 * = gf_match.filter_flags), sort_matches orders every bucket by read_break descending, read length ascending, read name
 * descending, stable (:379-385, src/core/read_match.rs:203-229).  With an output mode set, the HOST-batch entry points
 * (gf_map_pairs, gf_list_map_pairs, gf_map_fastq, gf_multi_map_pairs) do the first steps on the device, next to k_verify:
 *   GF_OUT_DROP_FILTERED  records with filter_flags != 0 are dropped before the device -> host copy;
 *   GF_OUT_BUCKET_ORDER   a 53-bit sort key (bucket, 2047 - read_break, seq_len) is computed per record on the device and the
 *                         records come back ordered by (key, pair_idx, source): bucket order, and inside a bucket the
 *                         reference's order up to the read-name tie-break.  Records with equal gf_match_order_key() form a
 *                         run in push order; the caller, who owns the names, orders such a run by name descending (stable).
 * Mode 0 (default): every record, ordered by (pair_idx, source).  gf_map_pairs_device* ignore the mode. */
#define GF_OUT_DROP_FILTERED 1u
#define GF_OUT_BUCKET_ORDER 2u
int gf_index_set_output_mode(gf_index* idx, uint32_t mode);
/* the key GF_OUT_BUCKET_ORDER sorts by (smaller first); n_genes = the index's gene count */
#ifdef __CUDACC__
#define GF_HOST_DEVICE __host__ __device__
#else
#define GF_HOST_DEVICE
#endif
static inline GF_HOST_DEVICE uint64_t gf_match_order_key(uint32_t n_genes, const gf_match* m) {
    const uint64_t bucket = (uint64_t)((int64_t)n_genes * m->r_contig + m->l_contig);
    const uint64_t brk = (uint64_t)(2047 - (m->read_break < 0 ? 0 : (m->read_break > 2047 ? 2047 : m->read_break)));
    return (bucket << 23) | (brk << 12) | (uint64_t)(m->seq_len & 0xFFF);
}

int gf_get_map_stats(const gf_index* idx, gf_map_stats* out);

/* Parity hook: run only the device fast_merge on a HOST batch. */
int gf_fast_merge(gf_index* idx, const gf_batch* in, gf_merge_info* out);

/* ---- report stage, per clustered match: FusionResult::adjust_fusion_break (src/core/fusion_result.rs:299-397) ----
 * SURVEY 8(f) #4.  After clustering, the reference slides every match's break point by -3..+3 and keeps the shift with
 * the smallest edit distance of the 20 bases on either side against FusionResult::m_left_ref / m_right_ref
 * (make_reference, :242-297 — built by the host exactly as today, get_ref_seq :770-798), 7 x 4 Levenshtein distances
 * per match; the winning shift's full-length left / right distances overwrite m_left_distance / m_right_distance.
 * `bytes` is one arena holding every read sequence and every reference string; jobs and refs index into it. */
typedef struct gf_break_ref {   /* one FusionResult */
    uint64_t left_off;          /* m_left_ref  = bytes[left_off  .. left_off  + left_len)  (may be empty) */
    uint64_t right_off;         /* m_right_ref = bytes[right_off .. right_off + right_len) */
    uint32_t left_len;
    uint32_t right_len;
} gf_break_ref;
typedef struct gf_break_job {   /* one ReadMatch of that FusionResult */
    uint64_t seq_off;           /* m_read.m_seq = bytes[seq_off .. seq_off + seq_len) */
    uint32_t seq_len;
    int32_t read_break;         /* m_read_break before the adjustment */
    uint32_t result;            /* index into refs */
    uint32_t reserved;
} gf_break_job;
typedef struct gf_break_out {
    int32_t shift;              /* add to m_read_break, m_left_gp.position and m_right_gp.position (:317-319) */
    int32_t left_distance;      /* new m_left_distance */
    int32_t right_distance;     /* new m_right_distance */
    int32_t status;             /* 0 ok; 1 = a shifted break lies outside the read (the reference's usize casts wrap there;
                                   not reachable from make_match's breaks) — shift / distances are 0; 2 = some shift's
                                   full-length left or right comparison is longer than 640 columns, where the reference's
                                   edit_distance panics (edit_distance.rs:94-100,177-196) — shift / distances are still the
                                   exact ones.  1 takes precedence over 2.  Any job with status != 0 makes the call return
                                   GF_E_REF_PANIC */
} gf_break_out;
int gf_adjust_fusion_break(gf_index* idx, const uint8_t* bytes, uint64_t n_bytes, const gf_break_ref* refs, uint32_t n_refs,
                           const gf_break_job* jobs, uint64_t n_jobs, gf_break_out* out);

/* ---- Matcher pass: FusionMapper::remove_alignables (src/core/fusion_mapper.rs:488-542), SURVEY 8(a) row M / 8(f) #4 ----
 * After the per-record filters the reference builds a `Matcher` over the WHOLE reference (Matcher::from_ref_and_seqs,
 * src/core/matcher.rs:44-169) and drops every match whose read `do_match`es it (:662-689).  As ported, the Matcher is
 * degenerate: its make_kmer* helpers `break` after the first base (:778-793,818-834,855-869), so a "k-mer" is the 2-bit code
 * of one base, the 512 MiB bloom array only ever has bits 0..3 of byte 0 set (:73-88), index_contig_bytes (:227-289) keeps a
 * reference position only where its rolling 32-bit value is < 4 (the start of every ACGT run, and any base preceded by
 * 15 'A's or by nothing but 'A's since the run start), and map_to_index (:388-529) can only return None or panic at
 * `.get(&kmer).unwrap()` (:490-491).  So remove_alignables removes nothing — but it costs one pass over the reference
 * (13-18 s of the reference's wall clock on hg19/hg38) and it can abort the run.  This call reproduces both observable
 * outcomes: the per-key position counts of m_kmer_positions and the panic pre-condition, from one streaming scan of the
 * reference on the GPU.
 *
 * gf_reference_create streams the contigs (host OR device pointers, ASCII, any case: to_ascii_uppercase, :143-148) through
 * the scan kernel once and keeps the result (4 counters and, for a key with <= 50 positions, the positions themselves) in
 * the handle; no reference bytes stay on the device.  List mode builds it once for all CSVs.  Contigs must be given in
 * FastaReader::m_all_contigs order (BTreeMap: ascending name), which defines the contig ids. */
typedef struct gf_ref_contig {
    const uint8_t* seq;
    uint64_t len;
} gf_ref_contig;
typedef struct gf_reference gf_reference; /* opaque */
typedef struct gf_reference_info {
    uint64_t n_contigs;
    uint64_t n_bases;
    uint64_t key_positions[4]; /* positions index_contig_bytes keeps for rolling key 0..3 (A, T, C, G) when the key's bloom
                                  bit is set */
    uint64_t short_contigs;    /* contigs shorter than 16 bases: Matcher::make_index panics on them (:240-243) */
    uint64_t h2d_bytes;        /* reference bytes copied host -> device (0 for device-resident contigs) */
    uint64_t kernel_launches;
    float ms_total;            /* device time of the whole pass (copies + scan), events on the handle's stream */
    float ms_scan;             /* scan kernels only */
} gf_reference_info;
int gf_reference_create(const gf_ref_contig* contigs, uint32_t n_contigs, int device, gf_reference** out);
void gf_reference_destroy(gf_reference* ref);
int gf_reference_get_info(const gf_reference* ref, gf_reference_info* out);

typedef struct gf_alignable_result {
    uint64_t key_positions[4]; /* Matcher::m_kmer_positions[k].len() for THIS set of sequences (0 when bloom bit k is unset) */
    uint64_t n_removed;        /* matches do_match returns Some for: always 0 (see above) */
    int64_t panic_seq;         /* index of the first sequence whose do_match panics, -1 = none */
    uint32_t bloom_bits;       /* m_bloom_filter_array[0] (bits 0..3 = base codes seen at a k-mer start of any sequence or
                                  of its reverse complement) */
    int32_t panic_stage;       /* 0 = the reference completes; 1 = Matcher::make_index panics (a contig shorter than 16
                                  bases); 2 / 3 = do_match panics in map_to_index of the sequence / of its reverse complement
                                  (:490-491); 4 = a sequence shorter than 15 bases (the reference's usize arithmetic wraps,
                                  :77, :414) */
} gf_alignable_result;
/* seqs[seq_off[j] .. seq_off[j+1]) = ReadMatch::get_read().m_seq of the j-th surviving match, in bucket order (the order
 * remove_alignables' retain() visits them).  alignable[j] = 1 where the match would be removed (always 0).  Returns GF_OK,
 * or GF_E_REF_PANIC when res->panic_stage != 0 (the result struct is still filled). */
int gf_alignable_filter(gf_reference* ref, const uint8_t* seqs, const uint64_t* seq_off, uint64_t n_seqs, uint8_t* alignable,
                        gf_alignable_result* res);

/* ---- list mode: the same reads against several fusion CSVs (src/core/fusion_scan.rs:62-188) ----
 * The reference scans its preloaded reads once per CSV with a fresh FusionMapper.  Here every CSV is one index handle, all on
 * one device, and one call maps a batch against all of them: the batch is uploaded ONCE and converted / merged ONCE
 * (fast_merge and the bit-plane conversion do not depend on the index), then seeded, screened and verified per index.
 * out[h] / out_cap[h] / n_out[h] belong to idx[h]; each output is identical to gf_map_pairs(idx[h], in, ...) on its own.
 * Returns the first error; GF_E_CAPACITY when any out_cap[h] is too small (n_out[] holds the required counts). */
int gf_list_map_pairs(gf_index* const* idx, uint32_t n_idx, const gf_batch* in, gf_match* const* out, const uint64_t* out_cap,
                      uint64_t* n_out);
/* the same on a DEVICE-resident batch, asynchronous on `cuda_stream` like gf_map_pairs_device (one capacity for all) */
int gf_map_pairs_device_list(gf_index* const* idx, uint32_t n_idx, const gf_batch* in_dev, gf_match* const* d_out,
                             uint64_t out_cap, uint64_t* const* d_n_out, void* cuda_stream);

/* ---- batched shim: packs in, large batches to the device (src/core/pescanner.rs:350-425, src/core/common.rs:20-23) ----
 * The reference's consumers call scan_pair_end once per pack of 1000 pairs.  A gf_stream takes the packs as they are — arrays
 * of pointers to the reads' sequence / quality strings with their lengths, which is what a ReadPairPack holds — copies them
 * into pinned arenas and maps them in batches of `batch_pairs` (0 = 2^20) pairs with gf_map_pairs.  Pair k of a push is
 * numbered first_pair + k in the records (the caller's own numbering, e.g. the running pair count of the producer), so
 * several consumer threads may push packs in any order.  Records of completed batches are collected with gf_stream_take
 * (sorted by (pair_idx, source), GF_E_CAPACITY protocol as in gf_map_pairs); gf_stream_flush maps what is still buffered
 * (end of input).  The strings may be released as soon as the push returns.  seq2 / qual2 / len2 = NULL for a single-end
 * stream.  Pushes on one stream are serialised internally. */
typedef struct gf_stream gf_stream;
int gf_stream_create(gf_index* idx, int paired, uint64_t batch_pairs, gf_stream** out);
void gf_stream_destroy(gf_stream* s);
int gf_stream_push(gf_stream* s, uint64_t first_pair, uint64_t n, const uint8_t* const* seq1, const uint8_t* const* qual1,
                   const uint32_t* len1, const uint8_t* const* seq2, const uint8_t* const* qual2, const uint32_t* len2);
int gf_stream_flush(gf_stream* s);
int gf_stream_take(gf_stream* s, gf_match* out, uint64_t out_cap, uint64_t* n_out);
int gf_stream_get_counts(const gf_stream* s, uint64_t* pairs_pushed, uint64_t* map_calls);

/* ---- FASTQ files as a byte stream, plain or gzip (src/core/fastq_reader.rs:39-69, 75-147, 149-179) ----
 * gf_map_fastq needs the whole text of both files in one buffer each.  A gf_fastq_stream is fed with the raw bytes of the
 * two files as they are read, in pieces that may end anywhere: whole records are mapped on the device as soon as
 * `chunk_bytes` (0 = 256 MiB) of text per mate have accumulated, the incomplete tail is carried over, and records are numbered
 * from the start of the files.  format = GF_FQ_GZIP (the caller decides from the file extension like FastqReader::new, :39-69):
 * the bytes are a gzip stream, possibly of several members (MultiGzDecoder, :49-55).  Blocked gzip (BGZF: what bgzip and
 * bcl2fastq write — members of <= 64 KB of text that say their own size in the header) is inflated ON THE DEVICE: only the
 * members' compressed payloads are copied, a warp per member decodes them, and a member whose sizes or CRC-32 do not come out
 * exactly fails the call (GF_E_INVALID); members that a fed piece cuts in two wait for their other half.  Any other gzip member
 * is inflated on the host (zlib, one thread per mate) into the pinned text buffers.  GF_BGZF_DEVICE=0 in the environment keeps
 * blocked gzip on the host threads too.  gf_fastq_stream_finish ends the files (a last line without '\n' counts,
 * an incomplete last record is dropped, the shorter file decides the pair count: FastqReaderPair); records are collected
 * with gf_fastq_stream_take at any time. */
#define GF_FQ_PLAIN 0
#define GF_FQ_GZIP 1
typedef struct gf_fastq_stream gf_fastq_stream;
int gf_fastq_stream_create(gf_index* idx, int paired, int format, uint64_t chunk_bytes, gf_fastq_stream** out);
void gf_fastq_stream_destroy(gf_fastq_stream* s);
int gf_fastq_stream_feed(gf_fastq_stream* s, const uint8_t* fq1, uint64_t n1, const uint8_t* fq2, uint64_t n2);
int gf_fastq_stream_finish(gf_fastq_stream* s);
int gf_fastq_stream_take(gf_fastq_stream* s, gf_match* out, uint64_t out_cap, uint64_t* n_out);
int gf_fastq_stream_get_counts(const gf_fastq_stream* s, uint64_t* records, uint64_t* text_bytes, uint64_t* map_calls);
/* Keeping the reads.  Everything after the scan needs the reads behind the records (ReadMatch::m_read and the original pair,
 * sort_matches' name tie-break, adjust_fusion_break, the reports), and on the stream's path their text exists only on the
 * device, only while its chunk is mapped.  gf_fastq_stream_keep_reads (before the first feed; GF_E_INVALID after it) makes the
 * stream gather, per mapped chunk and on the device, the four lines of both mates of every pair that has a record, and copy
 * them back with the records.  gf_fastq_stream_take_reads then returns what gf_fastq_stream_take would (same records, same
 * order, same GF_E_REF_PANIC rule) plus one gf_fastq_read_pair per distinct pair_idx among them, in ascending pair_idx, and
 * the text of their lines.  A capacity that is too small gives GF_E_CAPACITY with all three counts set and consumes nothing.
 * On a stream that keeps reads gf_fastq_stream_take fails with GF_E_INVALID (reads are never dropped silently); on one that
 * does not, gf_fastq_stream_take_reads does.  With GF_OUT_DROP_FILTERED only the pairs of surviving records come back. */
typedef struct gf_fastq_read_pair {
    uint64_t pair_idx;   /* as gf_match.pair_idx (counted from the start of the files) */
    uint64_t text_off;   /* mate 1's four lines start here in the text buffer, back to back, then mate 2's */
    uint32_t len[2][4];  /* [mate][name line, sequence, strand line, quality]; one trailing '\n' stripped, '\r' kept,
                            exactly the lines FastqReader::read yields (gf_fastq.cu's rule); mate 2 all 0 for single end */
} gf_fastq_read_pair;    /* 48 bytes */
int gf_fastq_stream_keep_reads(gf_fastq_stream* s);
int gf_fastq_stream_take_reads(gf_fastq_stream* s, gf_match* out, uint64_t out_cap, uint64_t* n_out,
                               gf_fastq_read_pair* pairs, uint64_t pairs_cap, uint64_t* n_pairs,
                               uint8_t* text, uint64_t text_cap, uint64_t* n_text);
/* One stream, several fusion CSVs (list mode on FASTQ input, src/core/fusion_scan.rs:62-188).  gf_fastq_stream_create_list
 * maps every chunk against the n_idx indices idx[]: the chunk is copied, inflated, split into records and converted ONCE, then
 * screened and verified per index.  The list is checked like gf_list_map_pairs checks it: non-empty, no NULL, no handle twice,
 * all handles on one device (GF_E_INVALID otherwise); more than 64 handles gives GF_E_LIMIT.  gf_fastq_stream_create(idx, ...)
 * is the list of one.  feed, finish, keep_reads and get_counts are unchanged; records are numbered from the start of the files,
 * the same for every index.
 * gf_fastq_stream_take_index(s, h, ...) returns exactly what gf_fastq_stream_take returns on a stream over idx[h] alone, fed the
 * same pieces with takes at the same points: the same records in the same order (idx[h]'s own output mode, bucket order when
 * idx[h] has it set), the same GF_E_CAPACITY protocol and the GF_E_REF_PANIC rule per index (only an index whose own records
 * carry the panic reports it).  gf_fastq_stream_take_reads_index is the same for gf_fastq_stream_take_reads: its records,
 * descriptors (text_off included) and text are byte-identical to the single-index stream's, so index h gets the pairs of its
 * own records only.  A take consumes only that index's records and lines.  On a stream with more than one index
 * gf_fastq_stream_take / take_reads fail with GF_E_INVALID; so does an index >= n_idx.
 * The handles must outlive the stream.  While a chunk is mapped all of them are locked (in address order, like
 * gf_list_map_pairs), after the stream's own lock.  Device memory: the chunk's text, its newline tables, the sequence store
 * and the gathered lines live in idx[0]'s workspace; every handle keeps its own record buffers for a chunk (up to 2 records
 * per pair: 48 B each, twice with an output mode, plus 8 B of sort key per record with one). */
int gf_fastq_stream_create_list(gf_index* const* idx, uint32_t n_idx, int paired, int format, uint64_t chunk_bytes,
                                gf_fastq_stream** out);
int gf_fastq_stream_take_index(gf_fastq_stream* s, uint32_t index, gf_match* out, uint64_t out_cap, uint64_t* n_out);
int gf_fastq_stream_take_reads_index(gf_fastq_stream* s, uint32_t index, gf_match* out, uint64_t out_cap, uint64_t* n_out,
                                     gf_fastq_read_pair* pairs, uint64_t pairs_cap, uint64_t* n_pairs,
                                     uint8_t* text, uint64_t text_cap, uint64_t* n_text);

/* ---- the packed upload, as a host-side utility ----
 * With all four arenas of a batch in pinned host memory (and reads <= 256 bases) gf_map_pairs / gf_list_map_pairs do not copy
 * the sequence bytes: the host threads turn them into the bit-planes the kernels work on — 2 bits per base — and only those
 * cross PCIe (gf_map_stats.packed_upload, csrc/gf_pack.cpp); the reads that survive the screen are fetched from the pinned
 * arenas on demand.  gf_pack_reads is that packer on its own (no device involved), for tests and for callers that want to
 * look at the format.  Per read i of `n` (bytes seq[off[i] - off[0] .. off[i + 1] - off[0])), with nw = ceil(len / 32):
 *   words[woff[i] ..]        nw words of the low code bit, nw words of the high code bit (A 0, T 1, C 2, G 3 = high:low; bit j
 *                            of word k = base 32 k + j), cleared where the base is not valid
 *   xoff[i] == 0             every base is upper-case ACGT; otherwise xwords[xoff[i] - 1 ..] = nw words `valid`, nw words `aux`:
 *                            mate2 == 0: valid = upper-case ACGT, aux = the byte is 'N';
 *                            mate2 != 0: valid = ACGT in either case, aux = upper-case ACGT.
 * words / xwords hold cap_words entries each, woff / xoff n; *n_words / *n_xwords = entries used (GF_E_CAPACITY: needed).
 * gf_pack_supported() == 0 (no AVX-512BW on this host, or GF_HOST_PACK=0): gf_pack_reads fails with GF_E_INVALID and
 * gf_map_pairs uploads the ASCII arenas as before. */
int gf_pack_supported(void);
int gf_pack_reads(const uint8_t* seq, const uint64_t* off, uint64_t n, int mate2, uint32_t* words, uint32_t* woff,
                  uint32_t* xwords, uint32_t* xoff, uint64_t cap_words, uint64_t* n_words, uint64_t* n_xwords);

/* ---- several GPUs of one box from ONE process (what the Rust binary needs; bench.py uses one process per GPU) ----
 * The index is replicated on every listed device (built there, ~19 ms each, in parallel); every batch is cut into
 * n_devices contiguous shards of pairs, each mapped by its own host thread on its own device (no device-to-device
 * traffic: reads are independent, map_read(&self), src/core/fusion_mapper.rs:93), and the records are gathered on
 * the host.  The result is identical to a single-device gf_map_pairs on the whole batch, including the order.
 * A device may be listed more than once (two streams of work on one GPU). */
typedef struct gf_multi gf_multi;
int gf_multi_create(const gf_gene_span* genes, uint32_t n_genes, const gf_params* params, const int* devices,
                    int n_devices, gf_multi** out);
void gf_multi_destroy(gf_multi* m);
int gf_multi_map_pairs(gf_multi* m, const gf_batch* in, gf_match* out, uint64_t out_cap, uint64_t* n_out);

#ifdef __cplusplus
}
#endif
#endif /* GENEFUSE_GPU_H */
