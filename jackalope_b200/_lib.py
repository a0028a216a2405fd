"""ctypes binding of the C ABI in include/jlp_b200.h (libjlp_b200.so, built
in-tree by jackalope_b200/build.py).  There is no fallback: if the library is
missing this module raises, and if no CUDA device is present jlp_ctx_create
fails."""
from __future__ import annotations

import ctypes as C
import os

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("JLP_B200_LIB") or os.path.join(HERE, "libjlp_b200.so")     # the override serves build-variant experiments

u8p, u32p, u64p, f64p = (C.POINTER(t) for t in (C.c_uint8, C.c_uint32, C.c_uint64, C.c_double))
ABORT_CB = C.CFUNCTYPE(C.c_int, C.c_void_p)
PROGRESS_CB = C.CFUNCTYPE(None, C.c_void_p, C.c_uint64)
CHUNK_CB = C.CFUNCTYPE(C.c_int, C.c_void_p, C.c_uint64, C.c_int, C.c_void_p, C.c_uint64)

JLP_OK, JLP_ERR_ARG, JLP_ERR_NO_DEVICE, JLP_ERR_CUDA, JLP_ERR_IO, JLP_ERR_ABORTED, JLP_ERR_UNSUPPORTED = 0, -1, -2, -3, -4, -5, -6


class Params(C.Structure):
    _fields_ = [
        ("paired", C.c_int), ("matepair", C.c_int), ("out_prefix", C.c_char_p), ("sep_files", C.c_int),
        ("compress", C.c_int), ("comp_method", C.c_char_p), ("n_reads", C.c_uint64), ("prob_dup", C.c_double),
        ("n_threads", C.c_uint64), ("show_progress", C.c_int), ("read_pool_size", C.c_uint64),
        ("haplotype_probs", f64p), ("frag_len_shape", C.c_double), ("frag_len_scale", C.c_double),
        ("frag_len_min", C.c_uint64), ("frag_len_max", C.c_uint64),
        ("ins_prob1", C.c_double), ("del_prob1", C.c_double), ("ins_prob2", C.c_double), ("del_prob2", C.c_double),
        ("barcodes", C.POINTER(C.c_char_p)), ("seed", C.c_uint64), ("batch_pairs", C.c_uint64),
        ("shard_index", C.c_uint32), ("shard_count", C.c_uint32),
        ("abort_cb", ABORT_CB), ("progress_cb", PROGRESS_CB), ("cb_user", C.c_void_p),
        ("comp_engine", C.c_int),
    ]


class PacbioParams(C.Structure):
    _fields_ = [
        ("out_prefix", C.c_char_p), ("sep_files", C.c_int), ("compress", C.c_int), ("comp_method", C.c_char_p),
        ("n_reads", C.c_uint64), ("n_threads", C.c_uint64), ("read_pool_size", C.c_uint64), ("haplotype_probs", f64p),
        ("prob_dup", C.c_double), ("scale", C.c_double), ("sigma", C.c_double), ("loc", C.c_double),
        ("min_read_len", C.c_double), ("read_probs", f64p), ("read_lens", u64p), ("n_custom", C.c_uint64),
        ("max_passes", C.c_uint64), ("chi2_params_n", C.c_double * 3), ("chi2_params_s", C.c_double * 5),
        ("sqrt_params", C.c_double * 2), ("norm_params", C.c_double * 2), ("prob_thresh", C.c_double),
        ("prob_ins", C.c_double), ("prob_del", C.c_double), ("prob_subst", C.c_double), ("seed", C.c_uint64),
        ("batch_reads", C.c_uint64), ("comp_engine", C.c_int), ("shard_index", C.c_uint32), ("shard_count", C.c_uint32),
        ("abort_cb", ABORT_CB), ("progress_cb", PROGRESS_CB), ("cb_user", C.c_void_p),
    ]


class RunStats(C.Structure):
    _fields_ = [
        ("pairs", C.c_uint64), ("bytes_out", C.c_uint64 * 2), ("batches", C.c_uint64),
        ("kernel_launches", C.c_uint64), ("device_ms", C.c_double), ("place_ms", C.c_double),
        ("reads_ms", C.c_double), ("d2h_bytes", C.c_uint64), ("h2d_bytes", C.c_uint64),
        ("run_ms", C.c_double), ("z_bytes", C.c_uint64 * 2), ("bgzf_ms", C.c_double),
    ]

    def as_dict(self):
        return dict(pairs=self.pairs, bytes_out=list(self.bytes_out), batches=self.batches,
                    kernel_launches=self.kernel_launches, device_ms=self.device_ms, place_ms=self.place_ms,
                    reads_ms=self.reads_ms, d2h_bytes=self.d2h_bytes, h2d_bytes=self.h2d_bytes, run_ms=self.run_ms,
                    z_bytes=list(self.z_bytes), bgzf_ms=self.bgzf_ms)


class MutationParams(C.Structure):
    _fields_ = [
        ("Q", C.c_double * 16), ("invariant", C.c_double), ("n_rates", C.c_uint32), ("rates", f64p),
        ("n_nodes", C.c_uint32), ("parent", C.POINTER(C.c_int32)), ("branch_len", f64p), ("n_tips", C.c_uint32),
        ("tip_node", u32p), ("tip_names", C.POINTER(C.c_char_p)), ("seed", C.c_uint64),
    ]


class MutationStats(C.Structure):
    _fields_ = [
        ("count_ms", C.c_double), ("scan_ms", C.c_double), ("write_ms", C.c_double), ("store_ms", C.c_double),
        ("total_ms", C.c_double), ("records", C.c_uint64), ("d2h_bytes", C.c_uint64), ("table_bytes", C.c_uint64),
        ("table_in_smem", C.c_int), ("max_slots", C.c_uint32),
    ]

    def as_dict(self):
        return {f: getattr(self, f) for f, _ in self._fields_}


# every symbol include/jlp_b200.h declares
SYMBOLS = [
    "jlp_ctx_create", "jlp_ctx_create_multi", "jlp_ctx_n_devices", "jlp_materialize_haplotypes", "jlp_ctx_destroy", "jlp_last_error", "jlp_set_genome", "jlp_set_genome_async", "jlp_genome_sync", "jlp_create_genome", "jlp_get_genome", "jlp_genome_draw", "jlp_clear_haplotypes",
    "jlp_add_haplotype", "jlp_get_haplotype_chrom", "jlp_create_haplotypes", "jlp_get_haplotype_muts", "jlp_transition_matrix", "jlp_set_profile", "jlp_illumina_ref", "jlp_illumina_hap",
    "jlp_illumina_to_memory", "jlp_illumina_stream", "jlp_illumina_device_only", "jlp_illumina_group_counts", "jlp_apportion", "jlp_shard_range", "jlp_deflate", "jlp_bgzf_device", "jlp_pacbio", "jlp_pacbio_to_memory", "jlp_pacbio_read_plan", "jlp_pacbio_sample", "jlp_reads_per_group", "jlp_alias_build",
    "jlp_threshold", "jlp_unif_expr", "jlp_frag_table", "jlp_philox4x32_10", "jlp_draw_pos", "jlp_draw_pair",
    "jlp_version",
]

_lib = None


def lib():
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(
            "jackalope_b200: %s is missing -- run `python -m jackalope_b200.build` "
            "(or __graft_entry__.build()); there is no CPU fallback" % LIB_PATH)
    L = C.CDLL(LIB_PATH)
    pp = C.POINTER(C.c_char_p)
    L.jlp_ctx_create.argtypes = [C.c_int, C.POINTER(C.c_void_p)]
    L.jlp_ctx_create_multi.argtypes = [C.c_int, C.POINTER(C.c_int), C.POINTER(C.c_void_p)]
    L.jlp_ctx_n_devices.argtypes = [C.c_void_p]
    L.jlp_materialize_haplotypes.argtypes = [C.c_void_p]
    L.jlp_ctx_destroy.argtypes = [C.c_void_p]
    L.jlp_ctx_destroy.restype = None
    L.jlp_last_error.argtypes = [C.c_void_p]
    L.jlp_last_error.restype = C.c_char_p
    L.jlp_set_genome.argtypes = [C.c_void_p, C.c_void_p, u64p, C.c_uint64, pp, C.c_char_p]
    L.jlp_set_genome_async.argtypes = L.jlp_set_genome.argtypes
    L.jlp_genome_sync.argtypes = [C.c_void_p]
    L.jlp_create_genome.argtypes = [C.c_void_p, C.c_uint64, u64p, f64p, C.c_uint64, pp, C.c_char_p]
    L.jlp_get_genome.argtypes = [C.c_void_p, C.c_void_p, C.c_uint64, u64p]
    L.jlp_genome_draw.argtypes = [C.c_uint64, C.c_uint32, C.c_uint64, C.c_int]
    L.jlp_genome_draw.restype = C.c_uint64
    L.jlp_clear_haplotypes.argtypes = [C.c_void_p]
    L.jlp_add_haplotype.argtypes = [C.c_void_p, C.c_char_p, u64p, C.POINTER(u64p), C.POINTER(u64p),
                                    C.POINTER(u64p), C.POINTER(C.c_void_p), u64p, u64p, u64p]
    L.jlp_get_haplotype_chrom.argtypes = [C.c_void_p, C.c_uint64, C.c_uint64, C.c_void_p, C.c_uint64, u64p]
    L.jlp_create_haplotypes.argtypes = [C.c_void_p, C.POINTER(MutationParams), C.POINTER(MutationStats)]
    L.jlp_get_haplotype_muts.argtypes = [C.c_void_p, C.c_uint64, C.c_uint64, u64p, u64p, u64p, C.c_void_p, C.c_uint64,
                                         C.c_uint64, u64p, u64p, u64p]
    L.jlp_transition_matrix.argtypes = [f64p, C.c_double, f64p]
    L.jlp_set_profile.argtypes = [C.c_void_p, C.c_int, C.c_uint64, u32p, f64p, u8p]
    L.jlp_illumina_ref.argtypes = [C.c_void_p, C.POINTER(Params), C.POINTER(RunStats)]
    L.jlp_illumina_hap.argtypes = [C.c_void_p, C.POINTER(Params), C.POINTER(RunStats)]
    L.jlp_illumina_to_memory.argtypes = [C.c_void_p, C.c_int, C.POINTER(Params), C.c_void_p, C.c_uint64, u64p,
                                         C.c_void_p, C.c_uint64, u64p, C.POINTER(RunStats)]
    L.jlp_illumina_stream.argtypes = [C.c_void_p, C.c_int, C.POINTER(Params), CHUNK_CB, C.c_void_p, C.POINTER(RunStats)]
    L.jlp_illumina_device_only.argtypes = [C.c_void_p, C.c_int, C.POINTER(Params), C.POINTER(RunStats)]
    L.jlp_illumina_group_counts.argtypes = [C.c_void_p, C.c_int, C.POINTER(Params), u64p, C.c_uint64, u64p]
    L.jlp_apportion.argtypes = [C.c_uint64, C.c_uint64, C.c_uint64, C.c_uint64, f64p, u64p, u64p]
    L.jlp_shard_range.argtypes = [C.c_uint64, C.c_uint64, C.c_uint32, C.c_uint32, u64p, u64p]
    L.jlp_deflate.argtypes = [C.c_int, C.c_int, C.c_void_p, C.c_uint64, C.c_void_p, C.c_uint64, u64p]
    L.jlp_bgzf_device.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_uint64, C.c_void_p, C.c_uint64, u64p]
    L.jlp_pacbio.argtypes = [C.c_void_p, C.c_int, C.POINTER(PacbioParams), C.POINTER(RunStats)]
    L.jlp_pacbio_to_memory.argtypes = [C.c_void_p, C.c_int, C.POINTER(PacbioParams), C.c_void_p, C.c_uint64, u64p, C.POINTER(RunStats)]
    L.jlp_pacbio_read_plan.argtypes = [C.c_void_p, C.c_int, C.POINTER(PacbioParams), u64p, u64p, u64p, f64p, f64p]
    L.jlp_pacbio_sample.argtypes = [C.POINTER(PacbioParams), C.c_uint64, C.c_uint64, u64p, u64p, f64p, f64p]
    L.jlp_reads_per_group.argtypes = [C.c_uint64, f64p, C.c_uint64, C.c_uint64, u64p]
    L.jlp_alias_build.argtypes = [f64p, C.c_uint64, f64p, u64p]
    L.jlp_threshold.argtypes = [C.c_int, C.c_double, u64p, C.POINTER(C.c_int)]
    L.jlp_unif_expr.argtypes = [C.c_int, C.c_uint64, C.c_double, C.c_uint64]
    L.jlp_unif_expr.restype = C.c_uint64
    L.jlp_frag_table.argtypes = [C.c_double, C.c_double, C.c_uint64, C.c_uint64, u64p, C.c_uint64, u64p]
    L.jlp_philox4x32_10.argtypes = [u32p, u32p, u32p]
    L.jlp_philox4x32_10.restype = None
    L.jlp_draw_pos.argtypes = [C.c_uint64, C.c_uint64, C.c_uint32, C.c_uint32, C.c_uint32]
    L.jlp_draw_pos.restype = C.c_uint64
    L.jlp_draw_pair.argtypes = [C.c_uint64, C.c_uint64, C.c_int]
    L.jlp_draw_pair.restype = C.c_uint64
    L.jlp_version.restype = C.c_char_p
    _lib = L
    return L
