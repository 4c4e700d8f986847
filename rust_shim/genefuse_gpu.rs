//! genefuse_gpu.rs — Rust FFI binding of include/genefuse_gpu.h.  SOURCE ONLY: this image has no cargo/rustc, so
//! the file is shipped for a maintainer to drop into GeneFuseRust as `src/core/genefuse_gpu.rs`
//! (add `pub(crate) mod genefuse_gpu;` to src/core/mod.rs and `println!("cargo:rustc-link-lib=genefuse_b200")`
//! + a search path to build.rs).  It replaces two call sites and nothing else:
//!   Indexer::make_index             src/core/indexer.rs:122-177      -> GpuIndex::build
//!   PairEndScanner::scan_pair_end   src/core/pescanner.rs:427-518    -> GpuIndex::map_pairs
//!   SingleEndScanner::scan_single_end src/core/sescanner.rs:183-205  -> GpuIndex::map_pairs (seq2 = null)
#![allow(non_camel_case_types, dead_code)]
use std::ffi::CStr;
use std::os::raw::{c_char, c_int, c_void};

#[repr(C)]
pub struct gf_gene_span { pub seq: *const u8, pub len: u32, pub reversed: u8 }

#[repr(C)]
#[derive(Clone, Copy)]
pub struct gf_params {
    pub skip_key_dup_threshold: i32,
    pub major_gene_key_requirement: i32,
    pub minor_gene_key_requirement: i32,
    pub mismatch_threshold: i32,
    pub deletion_threshold: i32,
}

#[repr(C)]
pub struct gf_batch {
    pub n: u64,
    pub seq1: *const u8, pub qual1: *const u8, pub off1: *const u64,
    pub seq2: *const u8, pub qual2: *const u8, pub off2: *const u64,
    pub bytes1: u64, pub bytes2: u64,
    pub max_len: u32, pub reserved: u32,
}

#[repr(C)]
#[derive(Clone, Copy, Default, Debug)]
pub struct gf_match {
    pub pair_idx: u64,
    pub read_break: i32, pub l_pos: i32, pub r_pos: i32, pub gap: i32,
    pub l_dist: i32, pub r_dist: i32, pub seq_len: i32,
    pub l_contig: i16, pub r_contig: i16, pub merge_olen: i16, pub merge_diff: i16,
    pub source: u8, pub used_rc: u8, pub reversed: u8, pub filter_flags: u8,
}

#[repr(C)] pub struct gf_index { _private: [u8; 0] }

extern "C" {
    fn gf_last_error() -> *const c_char;
    fn gf_index_create(genes: *const gf_gene_span, n_genes: u32, params: *const gf_params, device: c_int,
                       out: *mut *mut gf_index) -> c_int;
    fn gf_index_destroy(idx: *mut gf_index);
    fn gf_map_pairs(idx: *mut gf_index, batch: *const gf_batch, out: *mut gf_match, out_cap: u64,
                    n_out: *mut u64) -> c_int;
    fn gf_list_map_pairs(idx: *const *mut gf_index, n_idx: u32, batch: *const gf_batch, out: *const *mut gf_match,
                         out_cap: *const u64, n_out: *mut u64) -> c_int;
    fn gf_adjust_fusion_break(idx: *mut gf_index, bytes: *const u8, n_bytes: u64, refs: *const gf_break_ref, n_refs: u32,
                              jobs: *const gf_break_job, n_jobs: u64, out: *mut gf_break_out) -> c_int;
    fn gf_index_set_output_mode(idx: *mut gf_index, mode: u32) -> c_int;
    fn gf_stream_create(idx: *mut gf_index, paired: c_int, batch_pairs: u64, out: *mut *mut gf_stream) -> c_int;
    fn gf_stream_destroy(s: *mut gf_stream);
    fn gf_stream_push(s: *mut gf_stream, first_pair: u64, n: u64, seq1: *const *const u8, qual1: *const *const u8, len1: *const u32,
                      seq2: *const *const u8, qual2: *const *const u8, len2: *const u32) -> c_int;
    fn gf_stream_flush(s: *mut gf_stream) -> c_int;
    fn gf_stream_take(s: *mut gf_stream, out: *mut gf_match, out_cap: u64, n_out: *mut u64) -> c_int;
    fn gf_stream_get_counts(s: *const gf_stream, pairs_pushed: *mut u64, map_calls: *mut u64) -> c_int;
    fn gf_fastq_stream_create(idx: *mut gf_index, paired: c_int, format: c_int, chunk_bytes: u64,
                              out: *mut *mut gf_fastq_stream) -> c_int;
    fn gf_fastq_stream_destroy(s: *mut gf_fastq_stream);
    fn gf_fastq_stream_feed(s: *mut gf_fastq_stream, fq1: *const u8, n1: u64, fq2: *const u8, n2: u64) -> c_int;
    fn gf_fastq_stream_finish(s: *mut gf_fastq_stream) -> c_int;
    fn gf_fastq_stream_take(s: *mut gf_fastq_stream, out: *mut gf_match, out_cap: u64, n_out: *mut u64) -> c_int;
    fn gf_fastq_stream_get_counts(s: *const gf_fastq_stream, records: *mut u64, text_bytes: *mut u64, map_calls: *mut u64) -> c_int;
    fn gf_fastq_stream_keep_reads(s: *mut gf_fastq_stream) -> c_int;
    fn gf_fastq_stream_take_reads(s: *mut gf_fastq_stream, out: *mut gf_match, out_cap: u64, n_out: *mut u64,
                                  pairs: *mut gf_fastq_read_pair, pairs_cap: u64, n_pairs: *mut u64,
                                  text: *mut u8, text_cap: u64, n_text: *mut u64) -> c_int;
    fn gf_fastq_stream_create_list(idx: *const *mut gf_index, n_idx: u32, paired: c_int, format: c_int, chunk_bytes: u64,
                                   out: *mut *mut gf_fastq_stream) -> c_int;
    fn gf_fastq_stream_take_index(s: *mut gf_fastq_stream, index: u32, out: *mut gf_match, out_cap: u64, n_out: *mut u64) -> c_int;
    fn gf_fastq_stream_take_reads_index(s: *mut gf_fastq_stream, index: u32, out: *mut gf_match, out_cap: u64, n_out: *mut u64,
                                        pairs: *mut gf_fastq_read_pair, pairs_cap: u64, n_pairs: *mut u64,
                                        text: *mut u8, text_cap: u64, n_text: *mut u64) -> c_int;
    fn gf_reference_create(contigs: *const gf_ref_contig, n_contigs: u32, device: c_int, out: *mut *mut gf_reference) -> c_int;
    fn gf_reference_destroy(r: *mut gf_reference);
    fn gf_alignable_filter(r: *mut gf_reference, seqs: *const u8, seq_off: *const u64, n_seqs: u64, alignable: *mut u8,
                           res: *mut gf_alignable_result) -> c_int;
}

#[repr(C)] pub struct gf_stream { _private: [u8; 0] }
#[repr(C)] pub struct gf_reference { _private: [u8; 0] }
#[repr(C)] pub struct gf_fastq_stream { _private: [u8; 0] }
/// include/genefuse_gpu.h: the FASTQ lines of one matched pair inside the text that gf_fastq_stream_take_reads returns
#[repr(C)] #[derive(Clone, Copy, Default, Debug)]
pub struct gf_fastq_read_pair { pub pair_idx: u64, pub text_off: u64, pub len: [[u32; 4]; 2] }
pub const GF_FQ_PLAIN: c_int = 0;
pub const GF_FQ_GZIP: c_int = 1;
#[repr(C)] pub struct gf_ref_contig { pub seq: *const u8, pub len: u64 }
#[repr(C)] #[derive(Clone, Copy, Default, Debug)]
pub struct gf_alignable_result {
    pub key_positions: [u64; 4], pub n_removed: u64, pub panic_seq: i64, pub bloom_bits: u32, pub panic_stage: i32,
}
pub const GF_OUT_DROP_FILTERED: u32 = 1;
pub const GF_OUT_BUCKET_ORDER: u32 = 2;
pub const GF_E_REF_PANIC: c_int = -5;

/// include/genefuse_gpu.h: one FusionResult's m_left_ref / m_right_ref inside the byte arena
#[repr(C)] #[derive(Clone, Copy, Default)]
pub struct gf_break_ref { pub left_off: u64, pub right_off: u64, pub left_len: u32, pub right_len: u32 }
/// one ReadMatch of that FusionResult: m_read.m_seq inside the arena + m_read_break
#[repr(C)] #[derive(Clone, Copy, Default)]
pub struct gf_break_job { pub seq_off: u64, pub seq_len: u32, pub read_break: i32, pub result: u32, pub reserved: u32 }
#[repr(C)] #[derive(Clone, Copy, Default)]
pub struct gf_break_out { pub shift: i32, pub left_distance: i32, pub right_distance: i32, pub status: i32 }

pub const GF_E_CAPACITY: c_int = -3;

fn last_error() -> String {
    unsafe { CStr::from_ptr(gf_last_error()).to_string_lossy().into_owned() }
}

/// Owns one device index (one per FusionMapper; list mode: one per CSV, handles are independent).
pub struct GpuIndex { h: *mut gf_index }
unsafe impl Send for GpuIndex {}
unsafe impl Sync for GpuIndex {} // calls on one handle are serialised inside the library

impl GpuIndex {
    /// `genes[i]` = (upper-cased contig[m_start..m_end] or "" when the chromosome is unresolved, is_reversed),
    /// i.e. exactly what Indexer::make_index computes at src/core/indexer.rs:136-159 before index_contig.
    pub fn build(genes: &[(&[u8], bool)], params: gf_params, device: i32) -> Result<Self, String> {
        let spans: Vec<gf_gene_span> = genes.iter()
            .map(|(s, r)| gf_gene_span { seq: s.as_ptr(), len: s.len() as u32, reversed: *r as u8 }).collect();
        let mut h: *mut gf_index = std::ptr::null_mut();
        let rc = unsafe { gf_index_create(spans.as_ptr(), spans.len() as u32, &params, device, &mut h) };
        if rc != 0 { return Err(last_error()); }
        Ok(Self { h })
    }

    /// Maps a batch held in byte arenas (offsets have n+1 entries; seq and qual share them).
    pub fn map_pairs(&self, batch: &gf_batch) -> Result<Vec<gf_match>, String> {
        let mut cap = (batch.n as usize / 8).max(1024);
        loop {
            let mut out = vec![gf_match::default(); cap];
            let mut n: u64 = 0;
            let rc = unsafe { gf_map_pairs(self.h, batch, out.as_mut_ptr(), cap as u64, &mut n) };
            if rc == GF_E_CAPACITY { cap = n as usize; continue; }
            if rc != 0 { return Err(last_error()); } // upstream unwraps -> same abort behaviour as a panic
            out.truncate(n as usize);
            return Ok(out);
        }
    }
}

impl GpuIndex {
    /// FusionResult::adjust_fusion_break (src/core/fusion_result.rs:299-321) for every match of every result of one
    /// mapper: call it from cluster_matches right after fr.make_reference(..) (src/core/fusion_mapper.rs:438-456)
    /// instead of fr.adjust_fusion_break(); then for each match: m_read_break += shift, both positions += shift,
    /// m_left_distance / m_right_distance = the returned distances.  Where fr.adjust_fusion_break() would panic (a shifted
    /// break outside the read, or a distance over more than 640 columns: gf_break_out.status 1 / 2) the call returns
    /// GF_E_REF_PANIC and this Err(..).
    pub fn adjust_fusion_break(&self, arena: &[u8], refs: &[gf_break_ref], jobs: &[gf_break_job])
        -> Result<Vec<gf_break_out>, String> {
        let mut out = vec![gf_break_out::default(); jobs.len()];
        let rc = unsafe { gf_adjust_fusion_break(self.h, arena.as_ptr(), arena.len() as u64, refs.as_ptr(), refs.len() as u32,
                                                 jobs.as_ptr(), jobs.len() as u64, out.as_mut_ptr()) };
        if rc != 0 { return Err(last_error()); }
        Ok(out)
    }
}

/// List mode (src/core/fusion_scan.rs:62-188): one batch against every CSV's index in one call — one upload, one
/// conversion / fast_merge pass, then per-index seeding, screening and verification.  Returns one record vector per index,
/// each identical to `indices[h].map_pairs(batch)`.
pub fn list_map_pairs(indices: &[&GpuIndex], batch: &gf_batch) -> Result<Vec<Vec<gf_match>>, String> {
    let hs: Vec<*mut gf_index> = indices.iter().map(|g| g.h).collect();
    let mut caps: Vec<u64> = vec![(batch.n / 8).max(1024); hs.len()];
    loop {
        let mut bufs: Vec<Vec<gf_match>> = caps.iter().map(|c| vec![gf_match::default(); *c as usize]).collect();
        let ptrs: Vec<*mut gf_match> = bufs.iter_mut().map(|b| b.as_mut_ptr()).collect();
        let mut n = vec![0u64; hs.len()];
        let rc = unsafe { gf_list_map_pairs(hs.as_ptr(), hs.len() as u32, batch, ptrs.as_ptr(), caps.as_ptr(), n.as_mut_ptr()) };
        if rc == GF_E_CAPACITY { for (c, k) in caps.iter_mut().zip(&n) { *c = (*c).max(*k); } continue; }
        if rc != 0 { return Err(last_error()); }
        for (b, k) in bufs.iter_mut().zip(&n) { b.truncate(*k as usize); }
        return Ok(bufs);
    }
}

impl Drop for GpuIndex { fn drop(&mut self) { unsafe { gf_index_destroy(self.h) } } }


/// The batched shim (rust_shim/batched_consumer.patch.rs): packs in, large batches to the device.
pub struct PackStream { s: *mut gf_stream }
unsafe impl Send for PackStream {}
unsafe impl Sync for PackStream {} // pushes on one stream are serialised inside the library
impl PackStream {
    pub fn new(index: &GpuIndex, paired: bool, batch_pairs: u64) -> Result<Self, String> {
        let mut s: *mut gf_stream = std::ptr::null_mut();
        if unsafe { gf_stream_create(index.h, paired as c_int, batch_pairs, &mut s) } != 0 { return Err(last_error()); }
        Ok(Self { s })
    }
    pub fn push(&self, first_pair: u64, s1: &[*const u8], q1: &[*const u8], l1: &[u32], s2: &[*const u8], q2: &[*const u8],
                l2: &[u32]) -> Result<(), String> {
        let rc = unsafe { gf_stream_push(self.s, first_pair, s1.len() as u64, s1.as_ptr(), q1.as_ptr(), l1.as_ptr(),
                                         s2.as_ptr(), q2.as_ptr(), l2.as_ptr()) };
        if rc != 0 { Err(last_error()) } else { Ok(()) }
    }
    pub fn flush(&self) -> Result<(), String> { if unsafe { gf_stream_flush(self.s) } != 0 { Err(last_error()) } else { Ok(()) } }
    pub fn take(&self) -> Result<Vec<gf_match>, String> {
        let mut cap = 4096usize;
        loop {
            let mut out = vec![gf_match::default(); cap];
            let mut n = 0u64;
            let rc = unsafe { gf_stream_take(self.s, out.as_mut_ptr(), cap as u64, &mut n) };
            if rc == GF_E_CAPACITY { cap = n as usize; continue; }
            if rc != 0 { return Err(last_error()); }
            out.truncate(n as usize);
            return Ok(out);
        }
    }
    /// pairs that have gone through a mapping call (their packs can be released once their records were drained)
    pub fn pairs_mapped(&self) -> u64 {
        let (mut pushed, mut calls) = (0u64, 0u64);
        unsafe { gf_stream_get_counts(self.s, &mut pushed, &mut calls) };
        pushed // conservative: the caller releases packs only after take() returned their records
    }
}
impl Drop for PackStream { fn drop(&mut self) { unsafe { gf_stream_destroy(self.s) } } }

/// FastqReader / FastqReaderPair on raw file bytes (src/core/fastq_reader.rs:39-69,75-147,149-179): feed the files' bytes as
/// they are read (`.fq` plain, `.fq.gz` with gzip = true: BGZF members are inflated on the device); whole records are split and
/// mapped on the device.  With keep_reads the stream also returns the four lines of both mates of every matched pair, which is
/// all a ReadMatch needs (take_reads); without it, take() returns the records alone.
/// List mode (src/core/fusion_scan.rs:62-188 on FASTQ input): new_list maps every chunk against several indices — the chunk is
/// inflated, split and converted once — and take_index(h) / take_reads_index(h) return exactly what a stream over indices[h]
/// alone would.  The indices must outlive the stream.
pub struct FastqStream { s: *mut gf_fastq_stream, paired: bool }
unsafe impl Send for FastqStream {}
unsafe impl Sync for FastqStream {} // calls on one stream are serialised inside the library

/// (name, sequence, strand, quality) lines of one mate, as FastqReader::read yields them ('\n' stripped, '\r' kept)
pub type FastqLines<'a> = (&'a [u8], &'a [u8], &'a [u8], &'a [u8]);

/// what take_reads returns: the records and the lines of their pairs (ascending pair_idx)
pub struct FastqReads { pub records: Vec<gf_match>, pub pairs: Vec<gf_fastq_read_pair>, pub text: Vec<u8>, paired: bool }
impl FastqReads {
    /// mate 1's and (paired) mate 2's lines of self.pairs[k]
    pub fn lines(&self, k: usize) -> (FastqLines<'_>, Option<FastqLines<'_>>) {
        let p = &self.pairs[k];
        let mut pos = p.text_off as usize;
        let mut mate = |m: usize| {
            let mut l: [&[u8]; 4] = [&[]; 4];
            for j in 0..4 { let n = p.len[m][j] as usize; l[j] = &self.text[pos..pos + n]; pos += n; }
            (l[0], l[1], l[2], l[3])
        };
        let m1 = mate(0);
        let m2 = if self.paired { Some(mate(1)) } else { None };
        (m1, m2)
    }
    /// index into self.pairs of a record's pair
    pub fn find(&self, pair_idx: u64) -> Option<usize> { self.pairs.binary_search_by_key(&pair_idx, |p| p.pair_idx).ok() }
}

impl FastqStream {
    /// chunk_bytes = 0: 256 MiB of text per mate per mapping call
    pub fn new(index: &GpuIndex, paired: bool, gzip: bool, chunk_bytes: u64, keep_reads: bool) -> Result<Self, String> {
        Self::new_list(&[index], paired, gzip, chunk_bytes, keep_reads)
    }
    /// one stream against several indices (at most 64, all on one device, none twice)
    pub fn new_list(indices: &[&GpuIndex], paired: bool, gzip: bool, chunk_bytes: u64, keep_reads: bool) -> Result<Self, String> {
        let hs: Vec<*mut gf_index> = indices.iter().map(|g| g.h).collect();
        let mut s: *mut gf_fastq_stream = std::ptr::null_mut();
        let fmt = if gzip { GF_FQ_GZIP } else { GF_FQ_PLAIN };
        if unsafe { gf_fastq_stream_create_list(hs.as_ptr(), hs.len() as u32, paired as c_int, fmt, chunk_bytes, &mut s) } != 0 {
            return Err(last_error());
        }
        let st = Self { s, paired };
        if keep_reads && unsafe { gf_fastq_stream_keep_reads(st.s) } != 0 { return Err(last_error()); }
        Ok(st)
    }
    pub fn feed(&self, fq1: &[u8], fq2: &[u8]) -> Result<(), String> {
        let rc = unsafe { gf_fastq_stream_feed(self.s, fq1.as_ptr(), fq1.len() as u64, fq2.as_ptr(), fq2.len() as u64) };
        if rc != 0 { Err(last_error()) } else { Ok(()) }
    }
    /// end of the files: the last records are mapped
    pub fn finish(&self) -> Result<(), String> { if unsafe { gf_fastq_stream_finish(self.s) } != 0 { Err(last_error()) } else { Ok(()) } }
    /// the records of a one-index stream (take_index(0))
    pub fn take(&self) -> Result<Vec<gf_match>, String> { self.take_index(0) }
    /// the records of indices[index] mapped since its last take
    pub fn take_index(&self, index: u32) -> Result<Vec<gf_match>, String> {
        let mut cap = 4096usize;
        loop {
            let mut out = vec![gf_match::default(); cap];
            let mut n = 0u64;
            let rc = unsafe { gf_fastq_stream_take_index(self.s, index, out.as_mut_ptr(), cap as u64, &mut n) };
            if rc == GF_E_CAPACITY { cap = n as usize; continue; }
            if rc != 0 { return Err(last_error()); }
            out.truncate(n as usize);
            return Ok(out);
        }
    }
    /// the records (as take() would return them) and the lines of every pair among them, of a one-index stream
    pub fn take_reads(&self) -> Result<FastqReads, String> { self.take_reads_index(0) }
    /// take_reads for indices[index]: its records and the lines of its records' pairs only
    pub fn take_reads_index(&self, index: u32) -> Result<FastqReads, String> {
        let mut caps = [4096u64, 4096, 1 << 20];
        loop {
            let mut out = vec![gf_match::default(); caps[0] as usize];
            let mut pairs = vec![gf_fastq_read_pair::default(); caps[1] as usize];
            let mut text = vec![0u8; caps[2] as usize];
            let mut n = [0u64; 3];
            let rc = unsafe { gf_fastq_stream_take_reads_index(self.s, index, out.as_mut_ptr(), caps[0], &mut n[0], pairs.as_mut_ptr(),
                                                               caps[1], &mut n[1], text.as_mut_ptr(), caps[2], &mut n[2]) };
            if rc == GF_E_CAPACITY { for k in 0..3 { caps[k] = caps[k].max(n[k]); } continue; }
            if rc != 0 { return Err(last_error()); } // GF_E_REF_PANIC included: the reference aborts there
            out.truncate(n[0] as usize);
            pairs.truncate(n[1] as usize);
            text.truncate(n[2] as usize);
            return Ok(FastqReads { records: out, pairs, text, paired: self.paired });
        }
    }
    /// (records = pairs read so far, text bytes, mapping calls)
    pub fn counts(&self) -> (u64, u64, u64) {
        let (mut r, mut b, mut c) = (0u64, 0u64, 0u64);
        unsafe { gf_fastq_stream_get_counts(self.s, &mut r, &mut b, &mut c) };
        (r, b, c)
    }
}
impl Drop for FastqStream { fn drop(&mut self) { unsafe { gf_fastq_stream_destroy(self.s) } } }

/// The Matcher pass (src/core/fusion_mapper.rs:488-542, src/core/matcher.rs): the reference is scanned ONCE per FASTA.
pub struct GpuReference { r: *mut gf_reference }
unsafe impl Send for GpuReference {}
unsafe impl Sync for GpuReference {}
impl GpuReference {
    /// `contigs` = FastaReader::m_all_contigs values in BTreeMap (name) order
    pub fn build(contigs: &[&[u8]], device: i32) -> Result<Self, String> {
        let c: Vec<gf_ref_contig> = contigs.iter().map(|s| gf_ref_contig { seq: s.as_ptr(), len: s.len() as u64 }).collect();
        let mut r: *mut gf_reference = std::ptr::null_mut();
        if unsafe { gf_reference_create(c.as_ptr(), c.len() as u32, device, &mut r) } != 0 { return Err(last_error()); }
        Ok(Self { r })
    }
    /// `seqs` = ReadMatch::get_read().m_seq of every surviving match in bucket order (fusion_mapper.rs:496-500)
    pub fn alignable_filter(&self, seqs: &[&str]) -> Result<(Vec<u8>, gf_alignable_result), String> {
        let mut arena = Vec::new();
        let mut off = vec![0u64];
        for s in seqs { arena.extend_from_slice(s.as_bytes()); off.push(arena.len() as u64); }
        let mut flags = vec![0u8; seqs.len().max(1)];
        let mut res = gf_alignable_result::default();
        let rc = unsafe { gf_alignable_filter(self.r, arena.as_ptr(), off.as_ptr(), seqs.len() as u64, flags.as_mut_ptr(), &mut res) };
        if rc != 0 && rc != GF_E_REF_PANIC { return Err(last_error()); }
        flags.truncate(seqs.len());
        Ok((flags, res))
    }
}
impl Drop for GpuReference { fn drop(&mut self) { unsafe { gf_reference_destroy(self.r) } } }
