/*
 * gf_stream.cu — host-side staging in front of the mapping entry points (no kernels here):
 *
 *   gf_stream_*        the batched shim.  The reference's consumers call scan_pair_end once per pack of 1000 pairs
 *                      (/root/reference/src/core/pescanner.rs:350-425, src/core/common.rs:20-23); one gf_map_pairs call per
 *                      pack would pay 6 launches, 2 synchronisations and a tiny H2D for 1000 pairs.  A gf_stream takes packs
 *                      as they are (arrays of string pointers + lengths = what a ReadPairPack holds), copies them into
 *                      pinned arenas and maps them in batches of >= 2^20 pairs; records come back with the caller's own pair
 *                      numbering.
 *   gf_fastq_stream_*  SURVEY 8(f) #2: FastqReader / FastqReaderPair (src/core/fastq_reader.rs:39-69, 75-147, 149-179) as a
 *                      stream of raw file bytes: buffers may end anywhere (the incomplete tail is carried over), gzip input
 *                      (multi-member, like flate2's MultiGzDecoder, chosen by the caller from the file extension like
 *                      FastqReader::new) is inflated on host threads — one per mate — straight into the pinned text buffers,
 *                      and whole records are mapped on the device (gf_map_fastq_text: record splitting there too).
 *                      BGZF input (blocked gzip: what bcl2fastq / bgzip write — every member is <= 64 KB and says its own
 *                      compressed size in a 'BC' extra field and its uncompressed size in the trailer) is inflated by ALL
 *                      host threads: the members that lie completely in the fed piece go to their final place in the text
 *                      buffer side by side (the sizes give the offsets up front); a member cut by the end of the piece takes
 *                      the streaming path like any other gzip member.
 */
#include <zlib.h>

#include <algorithm>
#include <chrono>
#include <cstdio>
#include <cstring>
#include <memory>
#include <thread>
#include <vector>

#include "gf_internal.h"

namespace {

int sfail(int code, const std::string& msg) {
    gf_set_error(msg);
    return code;
}

/* grow-only pinned host buffer */
struct PinnedArena {
    uint8_t* p = nullptr;
    size_t cap = 0, fill = 0;
    ~PinnedArena() { if (p) cudaFreeHost(p); }
    cudaError_t reserve(size_t need) {
        if (need <= cap) return cudaSuccess;
        size_t want = std::max(need, cap * 2);
        uint8_t* q = nullptr;
        cudaError_t e = cudaMallocHost((void**)&q, want);
        if (e != cudaSuccess) return e;
        if (fill) memcpy(q, p, fill);
        if (p) cudaFreeHost(p);
        p = q;
        cap = want;
        return cudaSuccess;
    }
};

/* (pair_idx, source), or bucket order when the index's output mode asks for it (the same key the device computes) */
void sort_records(const gf_index* idx, std::vector<gf_match>& v) {
    if (!(idx->out_mode & GF_OUT_BUCKET_ORDER)) { gf_sort_matches(v.data(), v.size()); return; }
    const uint32_t ng = idx->n_genes;
    std::sort(v.begin(), v.end(), [ng](const gf_match& a, const gf_match& b) {
        const uint64_t ka = gf_match_order_key(ng, &a), kb = gf_match_order_key(ng, &b);
        if (ka != kb) return ka < kb;
        if (a.pair_idx != b.pair_idx) return a.pair_idx < b.pair_idx;
        return a.source < b.source;
    });
}

/* gf_map_pairs with the capacity protocol into a vector */
int map_into(gf_index* idx, const gf_batch* b, std::vector<gf_match>& tmp, uint64_t* n) {
    if (tmp.size() < 4096) tmp.resize(4096);
    for (;;) {
        int rc = gf_map_pairs(idx, b, tmp.data(), tmp.size(), n);
        if (rc == GF_E_CAPACITY) { tmp.resize(*n); continue; }
        return rc;
    }
}

}  // namespace

/* ================================================================================================== packs */
struct gf_stream {
    gf_index* idx = nullptr;
    uint64_t batch_pairs = 1u << 20;
    bool paired = true;
    PinnedArena seq[2], qual[2], off[2]; /* off: uint64 entries */
    std::vector<uint64_t> ids;           /* the caller's number of every buffered pair */
    uint32_t max_len = 0;
    std::vector<gf_match> done, tmp;
    uint64_t n_pushed = 0, n_calls = 0;
    bool panic = false;
    std::mutex mu;
};

namespace {

int stream_flush_locked(gf_stream* s) {
    const uint64_t n = s->ids.size();
    if (!n) return GF_OK;
    gf_batch b{};
    b.n = n;
    b.seq1 = s->seq[0].p; b.qual1 = s->qual[0].p; b.off1 = (const uint64_t*)s->off[0].p;
    b.bytes1 = s->seq[0].fill;
    if (s->paired) {
        b.seq2 = s->seq[1].p; b.qual2 = s->qual[1].p; b.off2 = (const uint64_t*)s->off[1].p;
        b.bytes2 = s->seq[1].fill;
    }
    b.max_len = std::max<uint32_t>(s->max_len, 1);
    uint64_t got = 0;
    int rc = map_into(s->idx, &b, s->tmp, &got);
    if (rc != GF_OK && rc != GF_E_REF_PANIC) return rc;
    if (rc == GF_E_REF_PANIC) s->panic = true;
    for (uint64_t i = 0; i < got; i++) {
        gf_match m = s->tmp[i];
        m.pair_idx = s->ids[m.pair_idx];
        s->done.push_back(m);
    }
    s->n_calls++;
    s->ids.clear();
    for (int k = 0; k < 2; k++) s->seq[k].fill = s->qual[k].fill = s->off[k].fill = 0;
    s->max_len = 0;
    return GF_OK;
}

}  // namespace

extern "C" {

int gf_stream_create(gf_index* idx, int paired, uint64_t batch_pairs, gf_stream** out) {
    if (!idx || !out) return sfail(GF_E_INVALID, "NULL argument");
    gf_stream* s = new gf_stream();
    s->idx = idx;
    s->paired = paired != 0;
    if (batch_pairs) s->batch_pairs = batch_pairs;
    *out = s;
    return GF_OK;
}

void gf_stream_destroy(gf_stream* s) { delete s; }

int gf_stream_push(gf_stream* s, uint64_t first_pair, uint64_t n, const uint8_t* const* seq1, const uint8_t* const* qual1,
                   const uint32_t* len1, const uint8_t* const* seq2, const uint8_t* const* qual2, const uint32_t* len2) {
    if (!s || (n && (!seq1 || !qual1 || !len1))) return sfail(GF_E_INVALID, "NULL argument");
    if (s->paired && n && (!seq2 || !qual2 || !len2)) return sfail(GF_E_INVALID, "a paired stream needs both mates");
    std::lock_guard<std::mutex> lk(s->mu);
    GF_CUDA_TRY(cudaSetDevice(s->idx->device));
    if (n && s->seq[0].cap == 0) {
        /* first pack: size the pinned arenas for a whole batch of reads like these, once (growing a pinned buffer means
         * cudaMallocHost + copy + cudaFreeHost, milliseconds each) */
        for (int k = 0; k < (s->paired ? 2 : 1); k++) {
            const uint32_t* ln = k ? len2 : len1;
            uint64_t sum = 0;
            for (uint64_t i = 0; i < n; i++) sum += ln[i];
            const uint64_t want = (sum / n + 8) * (s->batch_pairs + n) + (1u << 16);
            GF_CUDA_TRY(s->seq[k].reserve(want));
            GF_CUDA_TRY(s->qual[k].reserve(want));
            GF_CUDA_TRY(s->off[k].reserve(8 * (s->batch_pairs + n + 2)));
        }
        s->ids.reserve(s->batch_pairs + n);
    }
    for (uint64_t i = 0; i < n; i++) {
        const uint8_t* const* sq[2] = {seq1, seq2};
        const uint8_t* const* ql[2] = {qual1, qual2};
        const uint32_t* ln[2] = {len1, len2};
        for (int k = 0; k < (s->paired ? 2 : 1); k++) {
            const uint32_t L = ln[k][i];
            if (L > GF_MAX_READ_LEN + 24) return sfail(GF_E_INVALID, "a read is longer than the kernel capacity of 1024 bases");
            GF_CUDA_TRY(s->seq[k].reserve(s->seq[k].fill + L + 64));
            GF_CUDA_TRY(s->qual[k].reserve(s->qual[k].fill + L + 64));
            GF_CUDA_TRY(s->off[k].reserve(s->off[k].fill + 16));
            if (s->off[k].fill == 0) { ((uint64_t*)s->off[k].p)[0] = 0; s->off[k].fill = 8; }
            if (L) { memcpy(s->seq[k].p + s->seq[k].fill, sq[k][i], L); memcpy(s->qual[k].p + s->qual[k].fill, ql[k][i], L); }
            s->seq[k].fill += L;
            s->qual[k].fill += L;
            ((uint64_t*)s->off[k].p)[s->off[k].fill / 8] = s->seq[k].fill;
            s->off[k].fill += 8;
            s->max_len = std::max(s->max_len, L);
        }
        s->ids.push_back(first_pair + i);
        s->n_pushed++;
        if (s->ids.size() >= s->batch_pairs) {
            int rc = stream_flush_locked(s);
            if (rc != GF_OK) return rc;
        }
    }
    return GF_OK;
}

int gf_stream_flush(gf_stream* s) {
    if (!s) return sfail(GF_E_INVALID, "NULL argument");
    std::lock_guard<std::mutex> lk(s->mu);
    GF_CUDA_TRY(cudaSetDevice(s->idx->device));
    return stream_flush_locked(s);
}

int gf_stream_take(gf_stream* s, gf_match* out, uint64_t out_cap, uint64_t* n_out) {
    if (!s || !n_out) return sfail(GF_E_INVALID, "NULL argument");
    std::lock_guard<std::mutex> lk(s->mu);
    *n_out = s->done.size();
    if (s->done.size() > out_cap) return sfail(GF_E_CAPACITY, "out_cap too small; *n_out holds the required count");
    if (out_cap && !out && !s->done.empty()) return sfail(GF_E_INVALID, "out is NULL");
    sort_records(s->idx, s->done);
    if (!s->done.empty()) memcpy(out, s->done.data(), sizeof(gf_match) * s->done.size());
    s->done.clear();
    if (s->panic) {
        s->panic = false;
        return sfail(GF_E_REF_PANIC, "a candidate needs an edit distance over more than 640 columns (reference panics)");
    }
    return GF_OK;
}

int gf_stream_get_counts(const gf_stream* s, uint64_t* pairs_pushed, uint64_t* map_calls) {
    if (!s) return sfail(GF_E_INVALID, "NULL argument");
    if (pairs_pushed) *pairs_pushed = s->n_pushed;
    if (map_calls) *map_calls = s->n_calls;
    return GF_OK;
}

} /* extern "C" */

/* ================================================================================================== FASTQ text */
/* what one index of a FASTQ stream has mapped and not yet taken */
struct FqIndexOut {
    std::vector<gf_match> done, tmp;
    bool panic = false;
    std::vector<gf_fastq_read_pair> reads; /* ascending pair_idx, text_off into read_text */
    std::vector<uint8_t> read_text;
};

struct gf_fastq_stream {
    std::vector<gf_index*> idx; /* idx[0]'s workspace holds the text, the newline tables and the sequence store */
    std::vector<FqIndexOut> per; /* one per index */
    std::vector<GfFastqReads> chunk_reads; /* per index: what the last mapping call gathered (keep_reads) */
    bool paired = true;
    int format = GF_FQ_PLAIN;
    uint64_t chunk_bytes = 256ull << 20;
    PinnedArena text[2];
    /* blocked gzip, inflated on the device (GF_BGZF_DEVICE=0: on the host threads): the members' payloads back to back and their
     * descriptors; their text follows text[k].fill in the mate's logical text */
    bool device_inflate = true;
    PinnedArena comp[2];
    std::vector<GfBgzfMember> members[2];
    uint64_t pending_text[2] = {0, 0};
    std::vector<uint8_t> carry[2]; /* the first bytes of a BGZF member that the fed piece cut in two */
    z_stream z[2];
    bool z_open[2] = {false, false}, z_member_done[2] = {true, true};
    bool eof_seen[2] = {false, false};
    uint64_t records = 0, text_bytes = 0, n_calls = 0;
    uint64_t bgzf_blocks = 0; /* members inflated on the parallel path */
    double ms_bgzf = 0, ms_stream = 0, ms_map = 0; /* GF_DEBUG_TIMING: where the host time of the gzip path goes (mate 1's thread) */
    bool fed = false;
    bool keep_reads = false; /* gf_fastq_stream_keep_reads: the lines of the pairs behind each index's `done` */
    std::mutex mu;           /* taken before the indices' own locks */
    ~gf_fastq_stream() {
        for (int k = 0; k < 2; k++)
            if (z_open[k]) inflateEnd(&z[k]);
    }
};

namespace {

/* maps the whole records buffered so far against every index; final_chunk: the files have ended */
int fq_map_locked(gf_fastq_stream* s, bool final_chunk) {
    const int nm = s->paired ? 2 : 1;
    const uint32_t nh = (uint32_t)s->idx.size();
    const uint64_t total[2] = {s->text[0].fill + s->pending_text[0], s->text[1].fill + s->pending_text[1]};
    if (total[0] == 0 && (!s->paired || total[1] == 0)) return GF_OK;
    std::vector<gf_match*> outs(nh);
    std::vector<uint64_t> caps(nh), got(nh, 0);
    s->chunk_reads.resize(nh);
    std::unique_ptr<bool[]> panic(new bool[nh]);
    uint64_t nrec = 0, consumed[2] = {0, 0};
    std::vector<uint8_t> tail[2];
    int rc;
    const auto tm0 = std::chrono::steady_clock::now();
    GfFastqMembers mem[2];
    const bool have_members = !s->members[0].empty() || !s->members[1].empty();
    for (int k = 0; k < nm; k++) {
        mem[k].comp = s->comp[k].p;
        mem[k].comp_bytes = s->comp[k].fill;
        mem[k].members = s->members[k].data();
        mem[k].n_members = (uint32_t)s->members[k].size();
        mem[k].text_bytes = s->pending_text[k];
    }
    for (uint32_t h = 0; h < nh; h++)
        if (s->per[h].tmp.size() < 4096) s->per[h].tmp.resize(4096);
    for (;;) {
        for (uint32_t h = 0; h < nh; h++) { outs[h] = s->per[h].tmp.data(); caps[h] = s->per[h].tmp.size(); }
        rc = gf_map_fastq_text(s->idx.data(), nh, s->text[0].p, s->text[0].fill, s->paired ? s->text[1].p : nullptr,
                               s->paired ? s->text[1].fill : 0, final_chunk, outs.data(), caps.data(), got.data(), &nrec, consumed,
                               have_members ? mem : nullptr, s->keep_reads ? s->chunk_reads.data() : nullptr, panic.get(), tail);
        if (rc == GF_E_CAPACITY) {
            for (uint32_t h = 0; h < nh; h++) s->per[h].tmp.resize(std::max<uint64_t>(got[h], s->per[h].tmp.size()));
            continue;
        }
        break;
    }
    s->ms_map += std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - tm0).count();
    if (rc != GF_OK && rc != GF_E_REF_PANIC) return rc;
    for (uint32_t h = 0; h < nh; h++) {
        FqIndexOut& o = s->per[h];
        if (panic[h]) o.panic = true;
        for (uint64_t i = 0; i < got[h]; i++) {
            gf_match m = o.tmp[i];
            m.pair_idx += s->records;
            o.done.push_back(m);
        }
        if (s->keep_reads) { /* pair numbers and text offsets of the chunk -> the stream's */
            const uint64_t base = o.read_text.size();
            for (gf_fastq_read_pair p : s->chunk_reads[h].pairs) {
                p.pair_idx += s->records;
                p.text_off += base;
                o.reads.push_back(p);
            }
            o.read_text.insert(o.read_text.end(), s->chunk_reads[h].text.begin(), s->chunk_reads[h].text.end());
        }
    }
    s->records += nrec;
    s->n_calls++;
    for (int k = 0; k < nm; k++) {
        PinnedArena& t = s->text[k];
        const uint64_t c = std::min<uint64_t>(consumed[k], total[k]);
        s->text_bytes += c;
        if (final_chunk) {
            t.fill = 0;
        } else if (s->members[k].empty()) {
            memmove(t.p, t.p + c, t.fill - c);
            t.fill -= c;
        } else {
            /* the unconsumed tail (usually the last, incomplete record) came back from the device and opens the next chunk */
            if (t.reserve(tail[k].size() + 64) != cudaSuccess) return sfail(GF_E_CUDA, "pinned allocation failed");
            if (!tail[k].empty()) memcpy(t.p, tail[k].data(), tail[k].size());
            t.fill = tail[k].size();
        }
        s->members[k].clear();
        s->comp[k].fill = 0;
        s->pending_text[k] = 0;
    }
    return GF_OK;
}

/* BGZF member at p (n bytes available)?  Returns its total size and uncompressed size when the whole member is there. */
struct BgzfBlock { const uint8_t* data; uint32_t clen, isize, crc; uint64_t out; };
bool bgzf_block_at(const uint8_t* p, uint64_t n, uint32_t* total, BgzfBlock* b) {
    if (n < 18 || p[0] != 0x1f || p[1] != 0x8b || p[2] != 8 || !(p[3] & 4)) return false;
    const uint32_t xlen = p[10] | (p[11] << 8);
    if (n < 12 + (uint64_t)xlen) return false;
    uint32_t bsize = 0;
    bool found = false;
    for (uint32_t q = 12; q + 4 <= 12 + xlen;) { /* extra subfields: SI1 SI2 SLEN(2) data */
        const uint32_t slen = p[q + 2] | (p[q + 3] << 8);
        if (p[q] == 'B' && p[q + 1] == 'C' && slen == 2 && q + 6 <= 12 + xlen) { bsize = (p[q + 4] | (p[q + 5] << 8)) + 1u; found = true; }
        q += 4 + slen;
    }
    if (!found || (p[3] & ~4u) || bsize < 12 + xlen + 8 || n < bsize) return false; /* other header flags: streaming path */
    b->data = p + 12 + xlen;
    b->clen = bsize - (12 + xlen) - 8;
    b->crc = p[bsize - 8] | (p[bsize - 7] << 8) | (p[bsize - 6] << 16) | ((uint32_t)p[bsize - 5] << 24);
    b->isize = p[bsize - 4] | (p[bsize - 3] << 8) | (p[bsize - 2] << 16) | ((uint32_t)p[bsize - 1] << 24);
    if (b->isize > (1u << 16)) return false; /* not BGZF after all */
    *total = bsize;
    return true;
}
/* inflate blocks[lo, hi) to dst + blocks[i].out; false on a corrupt block */
bool bgzf_inflate_range(const std::vector<BgzfBlock>& blocks, size_t lo, size_t hi, uint8_t* dst) {
    z_stream z;
    memset(&z, 0, sizeof(z));
    if (inflateInit2(&z, -15) != Z_OK) return false;
    bool ok = true;
    for (size_t i = lo; i < hi && ok; i++) {
        const BgzfBlock& b = blocks[i];
        if (b.isize == 0) continue;
        z.next_in = const_cast<Bytef*>(b.data);
        z.avail_in = b.clen;
        z.next_out = dst + b.out;
        z.avail_out = b.isize;
        const int zr = inflate(&z, Z_FINISH);
        ok = zr == Z_STREAM_END && z.avail_out == 0 && (uint32_t)crc32(0L, dst + b.out, b.isize) == b.crc;
        inflateReset(&z);
    }
    inflateEnd(&z);
    return ok;
}

/* how long is the BGZF member that starts with these `have` bytes?  > 0: its size; 0: cannot tell yet (so far it may be one);
 * -1: not a BGZF member (some other gzip member: the streaming decoder takes it) */
int64_t bgzf_member_size(const uint8_t* p, uint64_t have) {
    static const uint8_t magic[3] = {0x1f, 0x8b, 8};
    for (uint64_t i = 0; i < 3 && i < have; i++)
        if (p[i] != magic[i]) return -1;
    if (have >= 4 && (p[3] != 4)) return -1; /* FEXTRA and nothing else (other flags: streaming path) */
    if (have < 12) return 0;
    const uint32_t xlen = p[10] | (p[11] << 8);
    if (have < 12 + (uint64_t)xlen) return 0;
    for (uint32_t q = 12; q + 4 <= 12 + xlen;) {
        const uint32_t slen = p[q + 2] | (p[q + 3] << 8);
        if (p[q] == 'B' && p[q + 1] == 'C' && slen == 2 && q + 6 <= 12 + xlen) {
            const int64_t bsize = (int64_t)(p[q + 4] | (p[q + 5] << 8)) + 1;
            return bsize >= 12 + (int64_t)xlen + 8 ? bsize : -1;
        }
        q += 4 + slen;
    }
    return -1;
}

/* append decoded text of mate k from `in`; returns the input bytes consumed.  Stops early when the chunk is full: the buffer
 * reached chunk_bytes, or (*full) the next BGZF member does not fit any more (the caller maps and calls again).
 *
 * Blocked gzip: whole members are never decoded here when the device inflates — only their payloads are kept, back to back in
 * pinned memory, with the sizes and CRC-32 from their headers and trailers; a member that a piece of input cuts in two waits in
 * `carry` for its other half, so the cut costs nothing.  Anything else (one big gzip member, members without the BGZF extra
 * field) goes through zlib's streaming decoder into the host text buffer. */
int fq_append(gf_fastq_stream* s, int k, const uint8_t* in, uint64_t n, uint64_t* used, bool* full, std::string* err) {
    PinnedArena& t = s->text[k];
    *used = 0;
    *full = false;
    const std::string corrupt = std::string("gzip stream of mate ") + (k ? "2" : "1") + " is corrupt";
    /* the text buffer is pinned once at its full size: growing a pinned buffer step by step (allocate, copy, free) costs more
     * than inflating what goes into it */
    const bool on_device = s->format == GF_FQ_GZIP && s->device_inflate; /* (then the host buffer holds little: the tail of the chunk before) */
    if (!on_device && t.cap < s->chunk_bytes + 64 && t.reserve(s->chunk_bytes + 64) != cudaSuccess) { *err = "pinned allocation failed"; return GF_E_CUDA; }
    if (on_device && (t.reserve(1u << 20) != cudaSuccess || /* (never NULL: a NULL second buffer means single-end to the mapping call) */
                      (s->comp[k].cap < s->chunk_bytes / 4 && s->comp[k].reserve(s->chunk_bytes / 4 + 64) != cudaSuccess))) {
        *err = "pinned allocation failed";
        return GF_E_CUDA;
    }
    if (s->format == GF_FQ_PLAIN) {
        const uint64_t room = t.fill < s->chunk_bytes ? s->chunk_bytes - t.fill : 0;
        const uint64_t c = std::min(n, room);
        if (c) {
            if (t.reserve(t.fill + c + 64) != cudaSuccess) { *err = "pinned allocation failed"; return GF_E_CUDA; }
            memcpy(t.p + t.fill, in, c);
            t.fill += c;
        }
        *used = c;
        return GF_OK;
    }
    z_stream& z = s->z[k];
    std::vector<uint8_t>& carry = s->carry[k];
    /* text of this mate that is waiting to be mapped: what lies in the host buffer + what the queued members will inflate to */
    auto logical_fill = [&]() { return (uint64_t)t.fill + s->pending_text[k]; };
    /* queued members -> host text (the streaming inflate below appends to the host buffer, so what was queued must be there first) */
    auto materialise = [&]() -> bool {
        if (s->members[k].empty()) return true;
        std::vector<BgzfBlock> blocks;
        for (const GfBgzfMember& m : s->members[k]) blocks.push_back(BgzfBlock{s->comp[k].p + m.in_off, m.clen, m.isize, m.crc, m.out_off});
        if (t.reserve(t.fill + s->pending_text[k] + 64) != cudaSuccess) return false;
        if (!bgzf_inflate_range(blocks, 0, blocks.size(), t.p + t.fill)) return false;
        t.fill += s->pending_text[k];
        s->members[k].clear();
        s->comp[k].fill = 0;
        s->pending_text[k] = 0;
        return true;
    };
    /* whole members (their `out` offsets count from the end of the text so far): queued for the device, or inflated here by
     * all host threads */
    auto take_members = [&](std::vector<BgzfBlock>& blocks, uint64_t out) -> int {
        if (s->device_inflate) {
            uint64_t cbytes = 0;
            for (const BgzfBlock& b : blocks) cbytes += b.clen;
            PinnedArena& c = s->comp[k];
            if (c.reserve(c.fill + cbytes + 64) != cudaSuccess) { *err = "pinned allocation failed"; return GF_E_CUDA; }
            for (const BgzfBlock& b : blocks) {
                if (b.isize == 0) continue; /* (the empty member that ends a BGZF file) */
                memcpy(c.p + c.fill, b.data, b.clen);
                s->members[k].push_back(GfBgzfMember{c.fill, s->pending_text[k], b.clen, b.isize, b.crc, 0u});
                c.fill += b.clen;
                s->pending_text[k] += b.isize;
            }
            if (k == 0) s->bgzf_blocks += blocks.size();
            return GF_OK;
        }
        const auto tb0 = std::chrono::steady_clock::now();
        if (t.reserve(t.fill + out + 64) != cudaSuccess) { *err = "pinned allocation failed"; return GF_E_CUDA; }
        const size_t nb = blocks.size();
        const unsigned want = s->paired ? std::max(1u, std::thread::hardware_concurrency() / 2) : std::max(1u, std::thread::hardware_concurrency());
        const size_t nt = std::max<size_t>(1, std::min<size_t>(want, (nb + 3) / 4));
        std::vector<char> okv(nt, 1);
        std::vector<std::thread> th;
        uint8_t* dst = t.p + t.fill;
        for (size_t u = 1; u < nt; u++)
            th.emplace_back([&, u] { okv[u] = bgzf_inflate_range(blocks, nb * u / nt, nb * (u + 1) / nt, dst) ? 1 : 0; });
        okv[0] = bgzf_inflate_range(blocks, 0, nb / nt, dst) ? 1 : 0;
        for (auto& x : th) x.join();
        for (char o : okv)
            if (!o) { *err = corrupt + " (BGZF block)"; return GF_E_INVALID; }
        t.fill += out;
        if (k == 0) { s->bgzf_blocks += nb; s->ms_bgzf += std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - tb0).count(); }
        return GF_OK;
    };
    if (!s->z_open[k]) {
        memset(&z, 0, sizeof(z));
        if (inflateInit2(&z, 15 + 32) != Z_OK) { *err = "inflateInit2 failed"; return GF_E_INVALID; }
        s->z_open[k] = true;
        s->z_member_done[k] = true;
    }
    uint64_t left = n;
    while (left && logical_fill() < s->chunk_bytes) {
        const uint8_t* zin = in + (n - left); /* what the streaming decoder would be given */
        uint64_t zn = left;
        bool from_carry = false;
        if (s->z_member_done[k]) {
            if (!carry.empty()) {
                /* the first bytes of a member came with the piece before: complete its header, then the member */
                int64_t sz = bgzf_member_size(carry.data(), carry.size());
                while (left && sz == 0) {
                    carry.push_back(in[n - left]);
                    left--;
                    sz = bgzf_member_size(carry.data(), carry.size());
                }
                if (sz == 0) break; /* (input used up) */
                if (sz > 0) {
                    const uint64_t more = std::min<uint64_t>(left, (uint64_t)sz > carry.size() ? (uint64_t)sz - carry.size() : 0);
                    carry.insert(carry.end(), in + (n - left), in + (n - left) + more);
                    left -= more;
                    if (carry.size() < (uint64_t)sz) break; /* (input used up) */
                    uint32_t total = 0;
                    BgzfBlock b;
                    if (!bgzf_block_at(carry.data(), carry.size(), &total, &b)) { *err = corrupt + " (BGZF header)"; return GF_E_INVALID; }
                    if (logical_fill() > 0 && logical_fill() + b.isize > s->chunk_bytes) { *full = true; break; } /* it opens the next chunk */
                    b.out = 0;
                    std::vector<BgzfBlock> one(1, b);
                    int r = take_members(one, b.isize);
                    if (r != GF_OK) return r;
                    carry.clear();
                    continue;
                }
                /* not BGZF after all: the streaming decoder gets the header bytes kept so far (they produce no text) */
                zin = carry.data();
                zn = carry.size();
                from_carry = true;
            } else {
                /* at a member boundary: as many whole BGZF members as lie in the piece and fit the chunk (a chunk holds at
                 * least one) */
                std::vector<BgzfBlock> blocks;
                uint64_t pos = n - left, out = 0;
                const uint64_t room = s->chunk_bytes - logical_fill();
                bool no_room = false;
                for (;;) {
                    uint32_t total = 0;
                    BgzfBlock b;
                    if (!bgzf_block_at(in + pos, n - pos, &total, &b)) break;
                    if (out + b.isize > room && (logical_fill() > 0 || out > 0)) { no_room = true; break; }
                    b.out = out;
                    out += b.isize;
                    pos += total;
                    blocks.push_back(b);
                }
                if (!blocks.empty()) {
                    int r = take_members(blocks, out);
                    if (r != GF_OK) return r;
                    left = n - pos;
                    if (no_room) { *full = true; break; }
                    continue;
                }
                if (no_room) { *full = true; break; }
                const int64_t sz = bgzf_member_size(in + pos, n - pos);
                if (sz == 0 || (sz > 0 && n - pos < (uint64_t)sz)) { /* a BGZF member the piece cuts in two: wait for the rest */
                    carry.assign(in + pos, in + n);
                    left = 0;
                    break;
                }
            }
        }
        if (!materialise()) { *err = corrupt + " (BGZF block)"; return GF_E_INVALID; }
        z.next_in = const_cast<Bytef*>(zin);
        if (t.reserve(std::min<uint64_t>(s->chunk_bytes, t.fill + (4u << 20)) + 64) != cudaSuccess) { *err = "pinned allocation failed"; return GF_E_CUDA; }
        const uint64_t room = std::min<uint64_t>(t.cap - 64, s->chunk_bytes) - t.fill;
        if (!room) break;
        z.avail_in = (uInt)std::min<uint64_t>(zn, 1u << 30);
        const uInt in0 = z.avail_in;
        z.next_out = t.p + t.fill;
        z.avail_out = (uInt)std::min<uint64_t>(room, 1u << 30);
        const uInt out0 = z.avail_out;
        s->z_member_done[k] = false;
        const auto ts0 = std::chrono::steady_clock::now();
        const int zr = inflate(&z, Z_NO_FLUSH);
        if (k == 0) s->ms_stream += std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - ts0).count();
        if (from_carry) {
            if (z.avail_in != 0) { *err = corrupt + " (gzip header)"; return GF_E_INVALID; } /* header bytes only: always taken whole */
            carry.clear();
        } else {
            left -= in0 - z.avail_in;
        }
        t.fill += out0 - z.avail_out;
        if (zr == Z_STREAM_END) { /* next member of a multi-member file (MultiGzDecoder, fastq_reader.rs:49-55) */
            s->z_member_done[k] = true;
            if (inflateReset(&z) != Z_OK) { *err = "inflateReset failed"; return GF_E_INVALID; }
        } else if (zr != Z_OK && zr != Z_BUF_ERROR) {
            *err = corrupt + ": " + (z.msg ? z.msg : "inflate error");
            return GF_E_INVALID;
        } else if (zr == Z_BUF_ERROR && in0 == z.avail_in && out0 == z.avail_out) {
            break; /* no progress possible with this input */
        }
    }
    *used = n - left;
    return GF_OK;
}

}  // namespace

extern "C" {

int gf_fastq_stream_create_list(gf_index* const* idx, uint32_t n_idx, int paired, int format, uint64_t chunk_bytes,
                                gf_fastq_stream** out) {
    if (!out) return sfail(GF_E_INVALID, "NULL argument");
    int rc = gf_validate_list(idx, n_idx);
    if (rc != GF_OK) return rc;
    if (n_idx > GF_FASTQ_LIST_MAX) return sfail(GF_E_LIMIT, "a FASTQ stream maps against at most 64 indices");
    if (format != GF_FQ_PLAIN && format != GF_FQ_GZIP) return sfail(GF_E_INVALID, "unknown FASTQ format");
    gf_fastq_stream* s = new gf_fastq_stream();
    s->idx.assign(idx, idx + n_idx);
    s->per.resize(n_idx);
    s->paired = paired != 0;
    s->format = format;
    if (chunk_bytes) s->chunk_bytes = std::max<uint64_t>(chunk_bytes, 4096);
    { const char* e = getenv("GF_BGZF_DEVICE"); s->device_inflate = !(e && atoi(e) == 0); }
    *out = s;
    return GF_OK;
}

int gf_fastq_stream_create(gf_index* idx, int paired, int format, uint64_t chunk_bytes, gf_fastq_stream** out) {
    if (!idx) return sfail(GF_E_INVALID, "NULL argument");
    return gf_fastq_stream_create_list(&idx, 1, paired, format, chunk_bytes, out);
}

void gf_fastq_stream_destroy(gf_fastq_stream* s) {
    if (s && getenv("GF_DEBUG_TIMING"))
        fprintf(stderr, "[gf_fastq_stream] records %llu, text bytes %llu, map calls %llu, BGZF members inflated side by side %llu; "
                "ms: side-by-side inflate %.1f, streaming inflate %.1f, mapping %.1f\n",
                (unsigned long long)s->records, (unsigned long long)s->text_bytes, (unsigned long long)s->n_calls,
                (unsigned long long)s->bgzf_blocks, s->ms_bgzf, s->ms_stream, s->ms_map);
    delete s;
}

int gf_fastq_stream_feed(gf_fastq_stream* s, const uint8_t* fq1, uint64_t n1, const uint8_t* fq2, uint64_t n2) {
    if (!s || (n1 && !fq1) || (n2 && !fq2)) return sfail(GF_E_INVALID, "NULL argument");
    if (!s->paired && n2) return sfail(GF_E_INVALID, "single-end stream fed with a second file");
    std::lock_guard<std::mutex> lk(s->mu);
    GF_CUDA_TRY(cudaSetDevice(s->idx[0]->device));
    s->fed = true;
    const uint8_t* in[2] = {fq1, fq2};
    uint64_t left[2] = {n1, n2};
    while (left[0] || left[1]) {
        /* decode both mates side by side (inflate is the host-side cost of .fq.gz input: one thread per mate) */
        uint64_t used[2] = {0, 0};
        bool fullf[2] = {false, false};
        int rcs[2] = {GF_OK, GF_OK};
        std::string errs[2];
        std::thread other;
        if (s->paired && left[1] && s->format == GF_FQ_GZIP)
            other = std::thread([&] { rcs[1] = fq_append(s, 1, in[1], left[1], &used[1], &fullf[1], &errs[1]); });
        else if (s->paired && left[1])
            rcs[1] = fq_append(s, 1, in[1], left[1], &used[1], &fullf[1], &errs[1]);
        if (left[0]) rcs[0] = fq_append(s, 0, in[0], left[0], &used[0], &fullf[0], &errs[0]);
        if (other.joinable()) other.join();
        for (int k = 0; k < 2; k++) {
            if (rcs[k] != GF_OK) return sfail(rcs[k], errs[k]);
            in[k] += used[k];
            left[k] -= used[k];
        }
        const uint64_t f0 = s->text[0].fill + s->pending_text[0], f1 = s->text[1].fill + s->pending_text[1];
        const bool full0 = f0 >= s->chunk_bytes || fullf[0], full1 = s->paired && (f1 >= s->chunk_bytes || fullf[1]);
        if (full0 || full1) {
            int rc = fq_map_locked(s, false);
            if (rc != GF_OK) return rc;
            if (s->text[0].fill == f0 && s->text[1].fill == f1) {
                /* a full buffer without one whole record in BOTH files (the other file is far behind, or a line is longer
                 * than the chunk): let the buffers grow instead of spinning */
                s->chunk_bytes *= 2;
            }
        } else if (!used[0] && !used[1]) {
            break; /* nothing could be consumed (cannot happen with room in the buffers) */
        }
    }
    return GF_OK;
}

int gf_fastq_stream_finish(gf_fastq_stream* s) {
    if (!s) return sfail(GF_E_INVALID, "NULL argument");
    std::lock_guard<std::mutex> lk(s->mu);
    GF_CUDA_TRY(cudaSetDevice(s->idx[0]->device));
    if (s->format == GF_FQ_GZIP)
        for (int k = 0; k < (s->paired ? 2 : 1); k++)
            if ((s->z_open[k] && !s->z_member_done[k]) || !s->carry[k].empty())
                return sfail(GF_E_INVALID, std::string("gzip stream of mate ") + (k ? "2" : "1") + " ends inside a member (truncated file)");
    return fq_map_locked(s, true);
}

int gf_fastq_stream_take_index(gf_fastq_stream* s, uint32_t index, gf_match* out, uint64_t out_cap, uint64_t* n_out) {
    if (!s || !n_out) return sfail(GF_E_INVALID, "NULL argument");
    std::lock_guard<std::mutex> lk(s->mu);
    if (index >= s->idx.size()) return sfail(GF_E_INVALID, "index out of range");
    if (s->keep_reads) return sfail(GF_E_INVALID, "the stream keeps reads: collect records with gf_fastq_stream_take_reads");
    FqIndexOut& o = s->per[index];
    *n_out = o.done.size();
    if (o.done.size() > out_cap) return sfail(GF_E_CAPACITY, "out_cap too small; *n_out holds the required count");
    if (!out && !o.done.empty()) return sfail(GF_E_INVALID, "out is NULL");
    sort_records(s->idx[index], o.done);
    if (!o.done.empty()) memcpy(out, o.done.data(), sizeof(gf_match) * o.done.size());
    o.done.clear();
    if (o.panic) {
        o.panic = false;
        return sfail(GF_E_REF_PANIC, "a candidate needs an edit distance over more than 640 columns (reference panics)");
    }
    return GF_OK;
}

int gf_fastq_stream_take(gf_fastq_stream* s, gf_match* out, uint64_t out_cap, uint64_t* n_out) {
    if (s && s->idx.size() != 1) return sfail(GF_E_INVALID, "the stream maps against several indices: use gf_fastq_stream_take_index");
    return gf_fastq_stream_take_index(s, 0, out, out_cap, n_out);
}

int gf_fastq_stream_keep_reads(gf_fastq_stream* s) {
    if (!s) return sfail(GF_E_INVALID, "NULL argument");
    std::lock_guard<std::mutex> lk(s->mu);
    if (s->fed) return sfail(GF_E_INVALID, "gf_fastq_stream_keep_reads after the first feed");
    s->keep_reads = true;
    return GF_OK;
}

int gf_fastq_stream_take_reads_index(gf_fastq_stream* s, uint32_t index, gf_match* out, uint64_t out_cap, uint64_t* n_out,
                                     gf_fastq_read_pair* pairs, uint64_t pairs_cap, uint64_t* n_pairs, uint8_t* text,
                                     uint64_t text_cap, uint64_t* n_text) {
    if (!s || !n_out || !n_pairs || !n_text) return sfail(GF_E_INVALID, "NULL argument");
    std::lock_guard<std::mutex> lk(s->mu);
    if (index >= s->idx.size()) return sfail(GF_E_INVALID, "index out of range");
    if (!s->keep_reads) return sfail(GF_E_INVALID, "the stream does not keep reads (gf_fastq_stream_keep_reads)");
    FqIndexOut& o = s->per[index];
    *n_out = o.done.size();
    *n_pairs = o.reads.size();
    *n_text = o.read_text.size();
    if (o.done.size() > out_cap || o.reads.size() > pairs_cap || o.read_text.size() > text_cap)
        return sfail(GF_E_CAPACITY, "a capacity is too small; *n_out, *n_pairs and *n_text hold the required counts");
    if ((!out && !o.done.empty()) || (!pairs && !o.reads.empty()) || (!text && !o.read_text.empty()))
        return sfail(GF_E_INVALID, "output buffer is NULL");
    sort_records(s->idx[index], o.done);
    if (!o.done.empty()) memcpy(out, o.done.data(), sizeof(gf_match) * o.done.size());
    if (!o.reads.empty()) memcpy(pairs, o.reads.data(), sizeof(gf_fastq_read_pair) * o.reads.size());
    if (!o.read_text.empty()) memcpy(text, o.read_text.data(), o.read_text.size());
    o.done.clear();
    o.reads.clear();
    o.read_text.clear();
    if (o.panic) {
        o.panic = false;
        return sfail(GF_E_REF_PANIC, "a candidate needs an edit distance over more than 640 columns (reference panics)");
    }
    return GF_OK;
}

int gf_fastq_stream_take_reads(gf_fastq_stream* s, gf_match* out, uint64_t out_cap, uint64_t* n_out, gf_fastq_read_pair* pairs,
                               uint64_t pairs_cap, uint64_t* n_pairs, uint8_t* text, uint64_t text_cap, uint64_t* n_text) {
    if (s && s->idx.size() != 1) return sfail(GF_E_INVALID, "the stream maps against several indices: use gf_fastq_stream_take_reads_index");
    return gf_fastq_stream_take_reads_index(s, 0, out, out_cap, n_out, pairs, pairs_cap, n_pairs, text, text_cap, n_text);
}

int gf_fastq_stream_get_counts(const gf_fastq_stream* s, uint64_t* records, uint64_t* text_bytes, uint64_t* map_calls) {
    if (!s) return sfail(GF_E_INVALID, "NULL argument");
    if (records) *records = s->records;
    if (text_bytes) *text_bytes = s->text_bytes;
    if (map_calls) *map_calls = s->n_calls;
    return GF_OK;
}

} /* extern "C" */
