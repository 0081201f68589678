"""ctypes binding of libpolyfasta_b200.so (include/polyfasta_b200.h).

The library is the product: there is no Python or CPU fallback.  If the shared object is missing, or no CUDA
device is present when a compute entry point is called, this module raises."""
import ctypes
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
SO_PATH = os.path.join(_HERE, "libpolyfasta_b200.so")

PFA_OK, PFA_ERR_CUDA, PFA_ERR_ARG, PFA_ERR_NOT_FASTA, PFA_ERR_RAGGED, PFA_ERR_IO, PFA_ERR_NOMEM, PFA_ERR_NON_ASCII = range(8)
PFA_CDS_LEN = 71
PFA_CDS_WIN_LEN = 72   # a codon window vector: the PFA_CDS_LEN words, then the site scan's S
PFA_BATCH_TOO_BIG = 100

# every symbol include/polyfasta_b200.h declares (tests check that the library exports all of them)
EXPORTS = [
    "pfa_version", "pfa_device_count", "pfa_global_error",
    "pfa_ctx_create", "pfa_ctx_destroy", "pfa_last_error", "pfa_ctx_sync", "pfa_ctx_trim", "pfa_ctx_set_stream", "pfa_ctx_launch_count",
    "pfa_ctx_set_host_threads", "pfa_ctx_ingest_stats", "pfa_ctx_last_kernel",
    "pfa_fasta_parse_file", "pfa_fasta_parse_buffer", "pfa_fasta_free", "pfa_fasta_nseq", "pfa_fasta_seqlen",
    "pfa_fasta_row_len", "pfa_fasta_header", "pfa_fasta_copy_row",
    "pfa_aln_from_fasta", "pfa_aln_from_rows", "pfa_aln_from_device_rows", "pfa_aln_synthetic", "pfa_synth_text_device", "pfa_aln_poke_gaps", "pfa_aln_force_validity", "pfa_aln_free",
    "pfa_aln_nseq", "pfa_aln_nsites", "pfa_aln_total_sites", "pfa_aln_num_escapes", "pfa_aln_packed_bytes", "pfa_aln_has_invalid", "pfa_aln_plane_alloc",
    "pfa_aln_copy_plane", "pfa_aln_read_probe", "pfa_aln_mask_words", "pfa_aln_set_pops", "pfa_aln_num_pops", "pfa_aln_pop_size",
    "pfa_site_len", "pfa_site_offset", "pfa_site_stats_device", "pfa_site_stats", "pfa_site_stats_hsite_device", "pfa_site_stats_hsite",
    "pfa_window_count", "pfa_site_windows_device", "pfa_site_windows", "pfa_cds_windows_device", "pfa_cds_windows",
    "pfa_divergence_device", "pfa_divergence_windows_device", "pfa_div_finalize", "pfa_divergence", "pfa_divergence_windows",
    "pfa_haplotypes_device", "pfa_haplotypes",
    "pfa_cds_stats_device", "pfa_cds_stats", "pfa_codon_pair_labels", "pfa_codon_set_labels", "pfa_codon_syn3",
    "pfa_codon_class", "pfa_pairwise_device", "pfa_pairwise", "pfa_finalize", "pfa_cds_ssites",
    "pfa_mask_words_for", "pfa_batch_create", "pfa_batch_destroy", "pfa_batch_clear", "pfa_batch_size", "pfa_batch_text_bytes",
    "pfa_batch_add", "pfa_batch_add_rows", "pfa_batch_add_synthetic", "pfa_batch_add_files", "pfa_batch_run", "pfa_batch_run_cds", "pfa_batch_stage", "pfa_batch_scan",
    "pfa_batch_release", "pfa_batch_kernel_ms", "pfa_batch_shape", "pfa_batch_num_pops", "pfa_batch_result", "pfa_batch_result_cds",
    "pfa_fasta_parse_files", "pfa_fasta_match_mask", "pfa_fasta_layout_bytes", "pfa_fasta_export_layout", "pfa_fasta_import_layout",
    "pfa_host_pack2", "pfa_host_pack2_rows", "pfa_host_pack3",
    "pfa_xchg_create", "pfa_xchg_destroy", "pfa_xchg_capacity", "pfa_xchg_export", "pfa_xchg_connect", "pfa_xchg_base",
    "pfa_xchg_connect_ptrs", "pfa_xchg_status", "pfa_xchg_set_timeout_ms", "pfa_xchg_stamps", "pfa_site_stats_xchg", "pfa_cds_stats_xchg", "pfa_site_cds_stats_xchg", "pfa_xchg_allreduce", "pfa_pairwise_xchg",
]


class FinalIn(ctypes.Structure):
    _fields_ = [("n", ctypes.c_int64), ("S", ctypes.c_int64), ("H", ctypes.c_int64), ("seqlen", ctypes.c_double),
                ("jc", ctypes.c_int32), ("pad", ctypes.c_int32)]


class FinalOut(ctypes.Structure):
    _fields_ = [("pi_site", ctypes.c_double), ("theta_site", ctypes.c_double), ("D", ctypes.c_double),
                ("D_is_NA", ctypes.c_int32), ("no_var", ctypes.c_int32)]


class DivIn(ctypes.Structure):
    _fields_ = [("n_x", ctypes.c_int64), ("n_y", ctypes.c_int64), ("D", ctypes.c_int64), ("seqlen", ctypes.c_double),
                ("pi_x", ctypes.c_double), ("pi_y", ctypes.c_double), ("jc", ctypes.c_int32), ("pad", ctypes.c_int32)]


class DivOut(ctypes.Structure):
    _fields_ = [("dxy", ctypes.c_double), ("da", ctypes.c_double), ("fst", ctypes.c_double),
                ("fst_is_NA", ctypes.c_int32), ("undefined", ctypes.c_int32)]


class PolyFastaError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__("polyfasta_b200 error %d: %s" % (code, msg))
        self.code = code


_lib = None


def lib():
    """the loaded shared object; raises if it has not been built (python -m polyfasta_b200.build)"""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(SO_PATH):
        raise ImportError("%s is missing: build it with `python -m polyfasta_b200.build` "
                          "(polyfasta_b200 has no CPU fallback)" % SO_PATH)
    L = ctypes.CDLL(SO_PATH)
    c = ctypes
    i64, p, sz = c.c_int64, c.c_void_p, c.c_size_t
    sig = {
        "pfa_version": (c.c_int, []),
        "pfa_device_count": (c.c_int, []),
        "pfa_global_error": (c.c_char_p, []),
        "pfa_ctx_create": (c.c_int, [c.c_int, c.POINTER(p)]),
        "pfa_ctx_destroy": (c.c_int, [p]),
        "pfa_last_error": (c.c_char_p, [p]),
        "pfa_ctx_sync": (c.c_int, [p]),
        "pfa_ctx_trim": (c.c_int, [p]),
        "pfa_ctx_set_stream": (c.c_int, [p, p]),
        "pfa_ctx_launch_count": (i64, [p]),
        "pfa_ctx_set_host_threads": (c.c_int, [p, c.c_int]),
        "pfa_ctx_ingest_stats": (c.c_int, [p, c.POINTER(i64)]),
        "pfa_fasta_parse_file": (c.c_int, [c.c_char_p, c.POINTER(p)]),
        "pfa_fasta_parse_buffer": (c.c_int, [p, sz, c.POINTER(p)]),
        "pfa_fasta_free": (None, [p]),
        "pfa_fasta_nseq": (i64, [p]),
        "pfa_fasta_seqlen": (i64, [p]),
        "pfa_fasta_row_len": (i64, [p, i64]),
        "pfa_fasta_header": (p, [p, i64, c.POINTER(i64)]),
        "pfa_fasta_copy_row": (c.c_int, [p, i64, p, i64]),
        "pfa_aln_from_fasta": (c.c_int, [p, p, i64, i64, c.POINTER(p)]),
        "pfa_aln_from_rows": (c.c_int, [p, p, i64, i64, i64, i64, i64, c.POINTER(p)]),
        "pfa_aln_from_device_rows": (c.c_int, [p, p, i64, i64, i64, i64, i64, c.POINTER(p)]),
        "pfa_aln_synthetic": (c.c_int, [p, i64, i64, c.c_uint64, c.c_uint32, c.c_uint32, i64, i64, c.POINTER(p)]),
        "pfa_synth_text_device": (c.c_int, [p, p, i64, i64, c.c_uint64, c.c_uint32, c.c_uint32, i64, i64]),
        "pfa_aln_force_validity": (c.c_int, [p, c.c_int]),
        "pfa_aln_free": (c.c_int, [p]),
        "pfa_aln_nseq": (i64, [p]),
        "pfa_aln_nsites": (i64, [p]),
        "pfa_aln_total_sites": (i64, [p]),
        "pfa_aln_num_escapes": (i64, [p]),
        "pfa_aln_packed_bytes": (i64, [p]),
        "pfa_aln_has_invalid": (c.c_int, [p]),
        "pfa_aln_plane_alloc": (c.c_int, [p]),
        "pfa_aln_poke_gaps": (c.c_int, [p, c.c_uint64, c.c_uint32]),
        "pfa_aln_copy_plane": (c.c_int, [p, c.c_int, p, sz]),
        "pfa_aln_read_probe": (c.c_int, [p, c.c_int, c.c_int, c.POINTER(c.c_double)]),
        "pfa_aln_mask_words": (i64, [p]),
        "pfa_aln_set_pops": (c.c_int, [p, p, c.c_int]),
        "pfa_aln_num_pops": (c.c_int, [p]),
        "pfa_aln_pop_size": (i64, [p, c.c_int]),
        "pfa_site_len": (i64, [p]),
        "pfa_site_offset": (i64, [p, c.c_int]),
        "pfa_site_stats_device": (c.c_int, [p, p, p]),
        "pfa_site_stats": (c.c_int, [p, p, p]),
        "pfa_site_stats_hsite_device": (c.c_int, [p, p, p, p]),
        "pfa_site_stats_hsite": (c.c_int, [p, p, p, p]),
        "pfa_window_count": (i64, [i64, i64, i64]),
        "pfa_site_windows_device": (c.c_int, [p, i64, i64, p]),
        "pfa_site_windows": (c.c_int, [p, i64, i64, p]),
        "pfa_cds_windows_device": (c.c_int, [p, i64, i64, p]),
        "pfa_cds_windows": (c.c_int, [p, i64, i64, p]),
        "pfa_divergence_device": (c.c_int, [p, p]),
        "pfa_divergence_windows_device": (c.c_int, [p, i64, i64, p]),
        "pfa_div_finalize": (c.c_int, [p, c.POINTER(DivIn), c.POINTER(DivOut), c.c_int]),
        "pfa_divergence": (c.c_int, [p, p]),
        "pfa_divergence_windows": (c.c_int, [p, i64, i64, p]),
        "pfa_haplotypes_device": (c.c_int, [p, i64, i64, p]),
        "pfa_haplotypes": (c.c_int, [p, i64, i64, p]),
        "pfa_cds_stats_device": (c.c_int, [p, p, p]),
        "pfa_cds_stats": (c.c_int, [p, p, p]),
        "pfa_codon_pair_labels": (c.c_int, [c.c_int, c.c_int]),
        "pfa_codon_set_labels": (c.c_int, [c.c_uint64]),
        "pfa_codon_syn3": (c.c_int, [c.c_int]),
        "pfa_codon_class": (c.c_int, [c.c_int]),
        "pfa_pairwise_device": (c.c_int, [p, p, p]),
        "pfa_pairwise": (c.c_int, [p, p, p]),
        "pfa_finalize": (c.c_int, [p, c.POINTER(FinalIn), c.POINTER(FinalOut), c.c_int]),
        "pfa_cds_ssites": (c.c_int, [p, p, p, c.c_int]),
        "pfa_mask_words_for": (i64, [i64]),
        "pfa_batch_create": (c.c_int, [p, c.POINTER(p)]),
        "pfa_batch_destroy": (c.c_int, [p]),
        "pfa_batch_clear": (c.c_int, [p]),
        "pfa_batch_size": (i64, [p]),
        "pfa_batch_text_bytes": (i64, [p]),
        "pfa_batch_add": (c.c_int, [p, p, p, c.c_int, c.POINTER(i64)]),
        "pfa_batch_add_rows": (c.c_int, [p, p, i64, i64, i64, p, c.c_int, c.POINTER(i64)]),
        "pfa_batch_add_synthetic": (c.c_int, [p, i64, i64, c.c_uint64, c.c_uint32, c.c_uint32, p, c.c_int, c.POINTER(i64)]),
        "pfa_batch_add_files": (c.c_int, [p, c.POINTER(c.c_char_p), c.c_int, c.POINTER(c.c_char_p), c.c_int, c.c_int,
                                          c.POINTER(c.c_int), c.POINTER(i64), c.POINTER(i64), c.POINTER(i64)]),
        "pfa_ctx_last_kernel": (c.c_char_p, [p]),
        "pfa_fasta_layout_bytes": (i64, [p]),
        "pfa_fasta_export_layout": (c.c_int, [p, p, i64]),
        "pfa_fasta_import_layout": (c.c_int, [c.c_char_p, p, i64, c.POINTER(p)]),
        "pfa_batch_run": (c.c_int, [p, c.c_int]),
        "pfa_batch_run_cds": (c.c_int, [p, c.c_int]),
        "pfa_batch_stage": (c.c_int, [p]),
        "pfa_batch_scan": (c.c_int, [p, c.c_int, c.c_int]),
        "pfa_batch_release": (c.c_int, [p]),
        "pfa_batch_kernel_ms": (c.c_int, [p, c.POINTER(c.c_double), c.POINTER(c.c_double)]),
        "pfa_batch_shape": (c.c_int, [p, c.POINTER(i64), c.POINTER(i64)]),
        "pfa_batch_result_cds": (c.c_int, [p, i64, c.c_int, p, c.POINTER(c.c_double), p]),
        "pfa_batch_num_pops": (c.c_int, [p, i64]),
        "pfa_batch_result": (c.c_int, [p, i64, c.c_int, c.POINTER(i64), p, c.POINTER(FinalOut)]),
        "pfa_fasta_parse_files": (c.c_int, [c.POINTER(c.c_char_p), c.c_int, c.c_int, c.POINTER(p), c.POINTER(c.c_int)]),
        "pfa_fasta_match_mask": (i64, [p, c.c_char_p, i64, p, i64]),
        "pfa_host_pack2": (c.c_int, [p, i64, p, c.c_int]),
        "pfa_host_pack2_rows": (i64, [p, i64, i64, i64, p, i64, c.c_int]),
        "pfa_host_pack3": (c.c_int, [p, i64, p, p, c.c_int]),
        "pfa_xchg_create": (c.c_int, [p, i64, c.POINTER(p)]),
        "pfa_xchg_destroy": (c.c_int, [p]),
        "pfa_xchg_capacity": (i64, [p]),
        "pfa_xchg_export": (c.c_int, [p, p]),
        "pfa_xchg_connect": (c.c_int, [p, c.c_int, c.c_int, p]),
        "pfa_xchg_base": (p, [p]),
        "pfa_xchg_connect_ptrs": (c.c_int, [p, c.c_int, c.c_int, c.POINTER(p)]),
        "pfa_xchg_status": (c.c_int, [p, c.POINTER(c.c_int)]),
        "pfa_xchg_set_timeout_ms": (c.c_int, [p, i64]),
        "pfa_xchg_stamps": (c.c_int, [p, c.POINTER(c.c_uint64)]),
        "pfa_site_stats_xchg": (c.c_int, [p, p, p, p]),
        "pfa_cds_stats_xchg": (c.c_int, [p, p, p, p]),
        "pfa_xchg_allreduce": (c.c_int, [p, p, i64]),
        "pfa_site_cds_stats_xchg": (c.c_int, [p, p, p, p, p]),
        "pfa_pairwise_xchg": (c.c_int, [p, p, p]),
    }
    for name, (res, args) in sig.items():
        fn = getattr(L, name)
        fn.restype = res
        fn.argtypes = args
    _lib = L
    return L


def check(rc, ctx=None):
    if rc != PFA_OK:
        L = lib()
        msg = (L.pfa_last_error(ctx) if ctx else L.pfa_global_error()) or b""
        raise PolyFastaError(rc, msg.decode("utf-8", "replace"))
