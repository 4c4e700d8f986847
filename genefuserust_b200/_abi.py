"""ctypes mirror of include/genefuse_gpu.h (the C ABI of the CUDA library).

Only plain structs live here; loading the product library is `load_library()`,
which fails loudly when the CUDA extension has not been built — there is no CPU
fallback anywhere in the package.
"""
import ctypes as C
import os

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "libgenefuse_b200.so")

GF_OK, GF_E_INVALID, GF_E_CUDA, GF_E_CAPACITY, GF_E_LIMIT, GF_E_REF_PANIC = 0, -1, -2, -3, -4, -5
GF_MAX_READ_LEN = 1000
GF_MAX_SEQ_LEN = 2048
GF_KMER = 16


class gf_gene_span(C.Structure):
    _fields_ = [("seq", C.c_void_p), ("len", C.c_uint32), ("reversed", C.c_uint8)]


class gf_params(C.Structure):
    _fields_ = [
        ("skip_key_dup_threshold", C.c_int32),
        ("major_gene_key_requirement", C.c_int32),
        ("minor_gene_key_requirement", C.c_int32),
        ("mismatch_threshold", C.c_int32),
        ("deletion_threshold", C.c_int32),
    ]

    @classmethod
    def default(cls):
        # src/aux/global_settings.rs:15-29
        return cls(5, 40, 20, 10, 50)


class gf_batch(C.Structure):
    _fields_ = [
        ("n", C.c_uint64),
        ("seq1", C.c_void_p),
        ("qual1", C.c_void_p),
        ("off1", C.c_void_p),
        ("seq2", C.c_void_p),
        ("qual2", C.c_void_p),
        ("off2", C.c_void_p),
        ("bytes1", C.c_uint64),
        ("bytes2", C.c_uint64),
        ("max_len", C.c_uint32),
        ("reserved", C.c_uint32),
    ]


class gf_match(C.Structure):
    _fields_ = [
        ("pair_idx", C.c_uint64),
        ("read_break", C.c_int32),
        ("l_pos", C.c_int32),
        ("r_pos", C.c_int32),
        ("gap", C.c_int32),
        ("l_dist", C.c_int32),
        ("r_dist", C.c_int32),
        ("seq_len", C.c_int32),
        ("l_contig", C.c_int16),
        ("r_contig", C.c_int16),
        ("merge_olen", C.c_int16),
        ("merge_diff", C.c_int16),
        ("source", C.c_uint8),
        ("used_rc", C.c_uint8),
        ("reversed", C.c_uint8),
        ("filter_flags", C.c_uint8),
    ]

    FIELDS = (
        "pair_idx", "source", "used_rc", "reversed", "read_break", "l_contig", "l_pos", "r_contig", "r_pos",
        "gap", "l_dist", "r_dist", "seq_len", "merge_olen", "merge_diff", "filter_flags",
    )

    def astuple(self):
        return tuple(int(getattr(self, f)) for f in self.FIELDS)


assert C.sizeof(gf_match) == 48


class gf_index_info(C.Structure):
    _fields_ = [
        ("n_sites", C.c_uint64),
        ("n_keys", C.c_uint64),
        ("n_unique", C.c_uint64),
        ("n_normal", C.c_uint64),
        ("n_high", C.c_uint64),
        ("table_slots", C.c_uint64),
        ("table_bytes", C.c_uint64),
        ("max_displacement", C.c_uint64),
        ("gene_bytes", C.c_uint64),
        ("device_bytes", C.c_uint64),
        ("build_ms", C.c_double),
    ]


class gf_lookup(C.Structure):
    _fields_ = [
        ("kind", C.c_int32),
        ("n_sites", C.c_int32),
        ("contig", C.c_int16 * 8),
        ("position", C.c_int32 * 8),
    ]


class gf_merge_info(C.Structure):
    _fields_ = [("merged", C.c_int32), ("olen", C.c_int32), ("diff", C.c_int32), ("merged_len", C.c_int32)]


class gf_map_stats(C.Structure):
    _fields_ = [
        ("n_pairs", C.c_uint64),
        ("n_sequences", C.c_uint64),
        ("n_probes_pass1", C.c_uint64),
        ("n_survivors", C.c_uint64),
        ("n_matches", C.c_uint64),
        ("seq_bytes", C.c_uint64),
        ("kernel_launches", C.c_uint64),
        ("ms_total", C.c_float),
        ("ms_merge", C.c_float),
        ("ms_screen", C.c_float),
        ("ms_exact", C.c_float),
        ("h2d_bytes", C.c_uint64),
        ("d2h_bytes", C.c_uint64),
        ("zero_copy_qual", C.c_uint32),
        ("packed_upload", C.c_uint32),
        ("ms_prep", C.c_float),
        ("ms_seed", C.c_float),
        ("ms_diag", C.c_float),
        ("ms_scan", C.c_float),
        ("ms_ingest", C.c_float),
        ("ms_host_pack", C.c_float),
    ]


class gf_break_ref(C.Structure):
    _fields_ = [("left_off", C.c_uint64), ("right_off", C.c_uint64), ("left_len", C.c_uint32), ("right_len", C.c_uint32)]


class gf_break_job(C.Structure):
    _fields_ = [("seq_off", C.c_uint64), ("seq_len", C.c_uint32), ("read_break", C.c_int32), ("result", C.c_uint32),
                ("reserved", C.c_uint32)]


class gf_break_out(C.Structure):
    _fields_ = [("shift", C.c_int32), ("left_distance", C.c_int32), ("right_distance", C.c_int32), ("status", C.c_int32)]


class gf_fastq_read_pair(C.Structure):
    _fields_ = [("pair_idx", C.c_uint64), ("text_off", C.c_uint64), ("len", (C.c_uint32 * 4) * 2)]


assert C.sizeof(gf_fastq_read_pair) == 48


class gf_ref_contig(C.Structure):
    _fields_ = [("seq", C.c_void_p), ("len", C.c_uint64)]


class gf_reference_info(C.Structure):
    _fields_ = [("n_contigs", C.c_uint64), ("n_bases", C.c_uint64), ("key_positions", C.c_uint64 * 4),
                ("short_contigs", C.c_uint64), ("h2d_bytes", C.c_uint64), ("kernel_launches", C.c_uint64),
                ("ms_total", C.c_float), ("ms_scan", C.c_float)]


class gf_alignable_result(C.Structure):
    _fields_ = [("key_positions", C.c_uint64 * 4), ("n_removed", C.c_uint64), ("panic_seq", C.c_int64),
                ("bloom_bits", C.c_uint32), ("panic_stage", C.c_int32)]

    def astuple(self):
        return (tuple(int(x) for x in self.key_positions), int(self.n_removed), int(self.panic_seq), int(self.bloom_bits),
                int(self.panic_stage))


# every symbol include/genefuse_gpu.h declares (tests check the .so exports all of them)
EXPORTS = (
    "gf_last_error", "gf_abi_version", "gf_device_count", "gf_default_params", "gf_index_create",
    "gf_index_destroy", "gf_index_get_info", "gf_index_lookup", "gf_map_pairs", "gf_map_pairs_device",
    "gf_sort_matches", "gf_get_map_stats", "gf_fast_merge", "gf_map_fastq", "gf_multi_create", "gf_multi_destroy",
    "gf_multi_map_pairs", "gf_adjust_fusion_break", "gf_list_map_pairs", "gf_map_pairs_device_list",
    "gf_reference_create", "gf_reference_destroy", "gf_reference_get_info", "gf_alignable_filter",
    "gf_index_set_output_mode",
    "gf_stream_create", "gf_stream_destroy", "gf_stream_push", "gf_stream_flush", "gf_stream_take", "gf_stream_get_counts",
    "gf_fastq_stream_create", "gf_fastq_stream_destroy", "gf_fastq_stream_feed", "gf_fastq_stream_finish",
    "gf_fastq_stream_take", "gf_fastq_stream_get_counts", "gf_fastq_stream_keep_reads", "gf_fastq_stream_take_reads",
    "gf_fastq_stream_create_list", "gf_fastq_stream_take_index", "gf_fastq_stream_take_reads_index",
    "gf_pack_supported", "gf_pack_reads",
)
GF_FQ_PLAIN, GF_FQ_GZIP = 0, 1
GF_OUT_DROP_FILTERED, GF_OUT_BUCKET_ORDER = 1, 2


def gf_match_order_key(n_genes, m):
    """static inline gf_match_order_key of the header"""
    bucket = n_genes * m.r_contig + m.l_contig
    brk = 2047 - min(max(m.read_break, 0), 2047)
    return (bucket << 23) | (brk << 12) | (m.seq_len & 0xFFF)

_lib = None


def load_library():
    """Load the CUDA library.  Raises (never falls back) when it is missing."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(
            f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "(nvcc, sm_100a).  There is no CPU fallback."
        )
    lib = C.CDLL(LIB_PATH)
    P = C.POINTER
    lib.gf_last_error.restype = C.c_char_p
    lib.gf_abi_version.restype = C.c_int
    lib.gf_device_count.restype = C.c_int
    lib.gf_default_params.argtypes = [P(gf_params)]
    lib.gf_default_params.restype = None
    lib.gf_index_create.argtypes = [P(gf_gene_span), C.c_uint32, P(gf_params), C.c_int, P(C.c_void_p)]
    lib.gf_index_create.restype = C.c_int
    lib.gf_index_destroy.argtypes = [C.c_void_p]
    lib.gf_index_destroy.restype = None
    lib.gf_index_get_info.argtypes = [C.c_void_p, P(gf_index_info)]
    lib.gf_index_get_info.restype = C.c_int
    lib.gf_index_lookup.argtypes = [C.c_void_p, C.c_void_p, C.c_uint64, P(gf_lookup)]
    lib.gf_index_lookup.restype = C.c_int
    lib.gf_map_pairs.argtypes = [C.c_void_p, P(gf_batch), P(gf_match), C.c_uint64, P(C.c_uint64)]
    lib.gf_map_pairs.restype = C.c_int
    lib.gf_map_pairs_device.argtypes = [C.c_void_p, P(gf_batch), C.c_void_p, C.c_uint64, C.c_void_p, C.c_void_p]
    lib.gf_map_pairs_device.restype = C.c_int
    lib.gf_sort_matches.argtypes = [P(gf_match), C.c_uint64]
    lib.gf_sort_matches.restype = None
    lib.gf_get_map_stats.argtypes = [C.c_void_p, P(gf_map_stats)]
    lib.gf_get_map_stats.restype = C.c_int
    lib.gf_map_fastq.argtypes = [C.c_void_p, C.c_char_p, C.c_uint64, C.c_char_p, C.c_uint64, P(gf_match), C.c_uint64,
                                 P(C.c_uint64), P(C.c_uint64)]
    lib.gf_map_fastq.restype = C.c_int
    lib.gf_multi_create.argtypes = [P(gf_gene_span), C.c_uint32, P(gf_params), P(C.c_int), C.c_int, P(C.c_void_p)]
    lib.gf_multi_create.restype = C.c_int
    lib.gf_multi_destroy.argtypes = [C.c_void_p]
    lib.gf_multi_destroy.restype = None
    lib.gf_multi_map_pairs.argtypes = [C.c_void_p, P(gf_batch), P(gf_match), C.c_uint64, P(C.c_uint64)]
    lib.gf_multi_map_pairs.restype = C.c_int
    lib.gf_fast_merge.argtypes = [C.c_void_p, P(gf_batch), P(gf_merge_info)]
    lib.gf_fast_merge.restype = C.c_int
    lib.gf_list_map_pairs.argtypes = [P(C.c_void_p), C.c_uint32, P(gf_batch), P(P(gf_match)), P(C.c_uint64), P(C.c_uint64)]
    lib.gf_list_map_pairs.restype = C.c_int
    lib.gf_map_pairs_device_list.argtypes = [P(C.c_void_p), C.c_uint32, P(gf_batch), P(C.c_void_p), C.c_uint64, P(C.c_void_p),
                                             C.c_void_p]
    lib.gf_map_pairs_device_list.restype = C.c_int
    lib.gf_adjust_fusion_break.argtypes = [C.c_void_p, C.c_char_p, C.c_uint64, P(gf_break_ref), C.c_uint32, P(gf_break_job),
                                           C.c_uint64, P(gf_break_out)]
    lib.gf_adjust_fusion_break.restype = C.c_int
    lib.gf_pack_supported.restype = C.c_int
    lib.gf_pack_reads.argtypes = [C.c_void_p, C.c_void_p, C.c_uint64, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                  C.c_uint64, P(C.c_uint64), P(C.c_uint64)]
    lib.gf_pack_reads.restype = C.c_int
    lib.gf_stream_create.argtypes = [C.c_void_p, C.c_int, C.c_uint64, P(C.c_void_p)]
    lib.gf_stream_create.restype = C.c_int
    lib.gf_stream_destroy.argtypes = [C.c_void_p]
    lib.gf_stream_destroy.restype = None
    lib.gf_stream_push.argtypes = [C.c_void_p, C.c_uint64, C.c_uint64, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                   C.c_void_p, C.c_void_p]
    lib.gf_stream_push.restype = C.c_int
    lib.gf_stream_flush.argtypes = [C.c_void_p]
    lib.gf_stream_flush.restype = C.c_int
    lib.gf_stream_take.argtypes = [C.c_void_p, P(gf_match), C.c_uint64, P(C.c_uint64)]
    lib.gf_stream_take.restype = C.c_int
    lib.gf_stream_get_counts.argtypes = [C.c_void_p, P(C.c_uint64), P(C.c_uint64)]
    lib.gf_stream_get_counts.restype = C.c_int
    lib.gf_fastq_stream_create.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_uint64, P(C.c_void_p)]
    lib.gf_fastq_stream_create.restype = C.c_int
    lib.gf_fastq_stream_destroy.argtypes = [C.c_void_p]
    lib.gf_fastq_stream_destroy.restype = None
    lib.gf_fastq_stream_feed.argtypes = [C.c_void_p, C.c_char_p, C.c_uint64, C.c_char_p, C.c_uint64]
    lib.gf_fastq_stream_feed.restype = C.c_int
    lib.gf_fastq_stream_finish.argtypes = [C.c_void_p]
    lib.gf_fastq_stream_finish.restype = C.c_int
    lib.gf_fastq_stream_take.argtypes = [C.c_void_p, P(gf_match), C.c_uint64, P(C.c_uint64)]
    lib.gf_fastq_stream_take.restype = C.c_int
    lib.gf_fastq_stream_get_counts.argtypes = [C.c_void_p, P(C.c_uint64), P(C.c_uint64), P(C.c_uint64)]
    lib.gf_fastq_stream_get_counts.restype = C.c_int
    lib.gf_fastq_stream_keep_reads.argtypes = [C.c_void_p]
    lib.gf_fastq_stream_keep_reads.restype = C.c_int
    lib.gf_fastq_stream_take_reads.argtypes = [C.c_void_p, P(gf_match), C.c_uint64, P(C.c_uint64), P(gf_fastq_read_pair), C.c_uint64,
                                               P(C.c_uint64), C.c_void_p, C.c_uint64, P(C.c_uint64)]
    lib.gf_fastq_stream_take_reads.restype = C.c_int
    lib.gf_fastq_stream_create_list.argtypes = [P(C.c_void_p), C.c_uint32, C.c_int, C.c_int, C.c_uint64, P(C.c_void_p)]
    lib.gf_fastq_stream_create_list.restype = C.c_int
    lib.gf_fastq_stream_take_index.argtypes = [C.c_void_p, C.c_uint32, P(gf_match), C.c_uint64, P(C.c_uint64)]
    lib.gf_fastq_stream_take_index.restype = C.c_int
    lib.gf_fastq_stream_take_reads_index.argtypes = [C.c_void_p, C.c_uint32, P(gf_match), C.c_uint64, P(C.c_uint64),
                                                     P(gf_fastq_read_pair), C.c_uint64, P(C.c_uint64), C.c_void_p, C.c_uint64,
                                                     P(C.c_uint64)]
    lib.gf_fastq_stream_take_reads_index.restype = C.c_int
    lib.gf_index_set_output_mode.argtypes = [C.c_void_p, C.c_uint32]
    lib.gf_index_set_output_mode.restype = C.c_int
    lib.gf_reference_create.argtypes = [P(gf_ref_contig), C.c_uint32, C.c_int, P(C.c_void_p)]
    lib.gf_reference_create.restype = C.c_int
    lib.gf_reference_destroy.argtypes = [C.c_void_p]
    lib.gf_reference_destroy.restype = None
    lib.gf_reference_get_info.argtypes = [C.c_void_p, P(gf_reference_info)]
    lib.gf_reference_get_info.restype = C.c_int
    lib.gf_alignable_filter.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint64, C.c_void_p, P(gf_alignable_result)]
    lib.gf_alignable_filter.restype = C.c_int
    _lib = lib
    return lib
