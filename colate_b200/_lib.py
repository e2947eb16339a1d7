"""ctypes loader for the in-tree C-ABI library (include/colate_b200.h).

The library is the product: there is no Python or CPU implementation behind it.  Loading
fails loudly if it has not been built (``python -c 'import __graft_entry__ as g; g.build()'``
or ``make -C colate_b200/csrc``), and every compute entry point fails with COLATE_ERR_CUDA
when no sm_100 GPU is usable.
"""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
# COLATE_B200_LIB: another build of the same library (kernel tuning variants, tools/sample_variants.py)
LIB_PATH = os.environ.get("COLATE_B200_LIB") or os.path.join(HERE, "libcolate_b200.so")

NBINS = 185
MAX_BLOCKS = 500
MT_WORDS = 624

_p = np.ctypeslib.ndpointer
f64 = _p(dtype=np.float64, flags="C_CONTIGUOUS")
f32 = _p(dtype=np.float32, flags="C_CONTIGUOUS")
i64 = _p(dtype=np.int64, flags="C_CONTIGUOUS")
i32 = _p(dtype=np.int32, flags="C_CONTIGUOUS")
u32 = _p(dtype=np.uint32, flags="C_CONTIGUOUS")
u16 = _p(dtype=np.uint16, flags="C_CONTIGUOUS")
VP = C.c_void_p


class Stage1Timing(C.Structure):
    _fields_ = [("join_ms", C.c_float), ("flags_ms", C.c_float), ("rng_ms", C.c_float), ("compact_ms", C.c_float),
                ("sample_ms", C.c_float), ("replay_ms", C.c_float), ("total_ms", C.c_float), ("n_site", C.c_int64),
                ("n_used", C.c_int64), ("rng_words", C.c_int64)]


class ColateError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__(f"colate_b200 error {code}: {msg}")
        self.code = code


# every symbol include/colate_b200.h declares: name -> (restype, argtypes)
SIGNATURES = {
    "colate_last_error": (C.c_char_p, []),
    "colate_version": (C.c_char_p, []),
    "colate_create": (C.c_int, [C.c_int, C.POINTER(VP)]),
    "colate_destroy": (None, [VP]),
    "colate_stream": (VP, [VP]),
    "colate_set_stream_cache": (C.c_int, [VP, C.c_int]),
    "colate_set_sites": (C.c_int, [VP, C.c_int, VP, VP, VP, VP, VP, C.c_int]),
    "colate_set_genome": (C.c_int, [VP, C.c_int, C.c_int64, VP, VP, VP, VP, VP, VP, C.c_int]),
    "colate_set_pileup": (C.c_int, [VP, C.c_int, VP, C.c_int]),
    "colate_set_row_counts": (C.c_int, [VP, C.c_int, VP, VP, C.c_int]),
    "colate_pileup_begin": (C.c_int, [VP, C.c_int]),
    "colate_pileup_reads": (C.c_int, [VP, C.c_int, C.c_int, C.c_int64, VP, VP, VP, VP, VP, VP, VP, C.c_int64, C.c_int, C.c_int, C.c_int]),
    "colate_pileup_end": (C.c_int, [VP, C.c_int, VP]),
    "colate_pileup_bam": (C.c_int, [VP, C.c_int, C.c_char_p, C.c_int, C.POINTER(C.c_char_p), C.POINTER(VP), VP, C.c_int, C.c_int, C.c_int, C.c_int64, VP]),
    "colate_last_bam_timing": (C.c_int, [VP, f64]),
    "colate_bam_scan": (C.c_int, [C.c_char_p, C.c_int, C.POINTER(C.c_char_p), C.c_int64, i64, i32, i32, i32]),
    "colate_rows_from_bcf": (C.c_int, [VP, C.c_int, C.c_int, C.c_int, C.POINTER(C.c_char_p), C.POINTER(C.c_char_p), VP, VP, C.c_int64, VP, VP]),
    "colate_rows_from_bcf_roles": (C.c_int, [VP, C.c_int, C.c_int, C.c_int, C.POINTER(C.c_char_p), C.POINTER(C.c_char_p), C.c_int, C.c_int64]),
    "colate_copy_genome": (C.c_int, [VP, C.c_int, C.c_int]),
    "colate_decode_bcf": (C.c_int, [VP, C.c_char_p, C.c_int64, VP, VP]),
    "colate_rows_from_bcf_genome": (C.c_int, [VP, C.c_int, C.c_int, C.c_int, C.POINTER(C.c_char_p), C.c_char_p, C.c_int, C.c_int64]),
    "colate_decode_bcf_genome": (C.c_int, [VP, C.c_char_p, C.c_int, C.POINTER(C.c_char_p), C.c_int64, VP, VP, VP]),
    "colate_bcf_genome_scan": (C.c_int, [C.c_char_p, C.c_int, C.POINTER(C.c_char_p), C.c_int64, VP, VP, VP, VP]),
    "colate_bcf_records": (C.c_int, [VP, C.c_int64, C.c_int64, VP, VP, VP, VP, VP]),
    "colate_last_bcf_timing": (C.c_int, [VP, f64]),
    "colate_bcf_scan": (C.c_int, [C.c_char_p, C.c_int64, VP, VP, VP, VP, VP, VP]),
    "colate_vcf_scan": (C.c_int, [C.c_char_p, C.c_int64, VP, VP, VP, VP, C.c_char_p, C.c_int64]),
    "colate_read_fasta": (C.c_int64, [C.c_char_p, C.POINTER(C.POINTER(C.c_uint8))]),
    "colate_free": (None, [VP]),
    "colate_set_mask": (C.c_int, [VP, C.c_int, VP, C.c_int]),
    "colate_stage1_flags": (C.c_int, [VP, C.c_int, C.c_int, VP, VP]),
    "colate_stage1_sample": (C.c_int, [VP, VP, C.c_int64, C.c_int, VP, VP, VP]),
    "colate_stage1": (C.c_int, [VP, C.c_int, C.c_int, VP, C.POINTER(C.c_int), VP, VP, C.POINTER(C.c_int64), VP]),
    "colate_stage2_bootstrap": (C.c_int, [VP, C.c_int, C.c_int, VP, VP, C.c_double, VP]),
    "colate_stage3_em": (C.c_int, [VP, C.c_int, C.c_int, VP, VP, VP, C.c_int, VP, VP, VP]),
    "colate_stage3_em_begin": (C.c_int, [VP, C.c_int, C.c_int, VP, VP, C.c_int]),
    "colate_stage3_em_end": (C.c_int, [VP, VP, VP, VP]),
    "colate_stage3_em_grids": (C.c_int, [VP, C.c_int, i32, C.c_int, i32, i64, f64, f64, f64, C.c_int, f64, i32, f64]),
    "colate_set_age_bins": (C.c_int, [VP, VP]),
    "colate_estep": (C.c_int, [VP, C.c_int, C.c_int, VP, VP, C.c_int, VP, VP, VP, VP]),
    "colate_libm_exact": (C.c_int, []),
    "colate_last_stage1_timing": (C.c_int, [VP, C.POINTER(Stage1Timing)]),
    "colate_set_option": (C.c_int, [VP, C.c_char_p, C.c_int64]),
    "colate_launch_count": (C.c_int64, [VP]),
    "colate_last_stage1_extra_words": (C.c_int64, [VP]),
    "colate_mt_seed": (None, [C.c_uint32, u32]),
    "colate_mt_generate": (None, [u32, C.c_int64, u32]),
    "colate_draw_block_weights": (None, [u32, C.c_int, C.c_int, i32]),
    "colate_age_bins": (None, [f64]),
    "colate_site_meta": (C.c_uint32, [C.c_int, C.c_int, C.c_float, C.c_float, C.c_char_p]),
    "colate_chr_ranges": (C.c_int, [C.c_int, C.c_int64, i32, i64, i64]),
    "colate_age_generations": (C.c_double, [C.c_char_p, C.c_char_p, C.c_int, C.c_float, C.POINTER(C.c_double)]),
    "colate_epochs_from_bins": (C.c_int, [C.c_char_p, C.c_double, C.c_double, f64, C.c_int, C.POINTER(C.c_int)]),
    "colate_epochs_from_coal_file": (C.c_int, [C.c_char_p, C.c_double, f64, f64, C.c_int]),
    "colate_ingest_begin": (C.c_int, [VP, C.c_int, C.c_int64]),
    "colate_ingest_mut_text": (C.c_int64, [VP, VP, C.c_int64, C.c_int]),
    "colate_ingest_mut_texts": (C.c_int, [VP, C.c_int, C.POINTER(VP), i64, C.c_int, VP]),
    "colate_ingest_end": (C.c_int, [VP]),
    "colate_ingest_colate_in": (C.c_int64, [VP, C.c_int, VP, C.c_int64, C.c_int, C.POINTER(C.c_char_p), C.c_int]),
    "colate_ingest_fetch": (C.c_int, [VP, C.c_int64, C.c_int64, VP, VP, VP, VP]),
    "colate_ingest_stats": (C.c_int, [VP, C.POINTER(C.c_double), C.POINTER(C.c_int64)]),
    "colate_read_mut": (C.c_int64, [C.c_char_p, C.c_int64, VP, VP, VP, VP]),
    "colate_read_colate_in": (C.c_int64, [C.c_char_p, C.c_int, C.POINTER(C.c_char_p), C.c_int64, VP, VP, VP, VP, VP]),
    "colate_mask_bits_from_fasta": (C.c_int, [C.c_char_p, C.c_int64, VP, C.c_int64, VP]),
    "colate_maketmp_table": (C.c_int64, [C.c_int, C.POINTER(C.c_char_p), C.POINTER(C.c_char_p), C.c_char_p, C.POINTER(C.c_char_p), C.c_int, C.c_char_p]),
    "colate_maketmp_records": (C.c_int64, [C.c_int, C.POINTER(C.c_char_p), C.POINTER(C.c_char_p), VP, VP, VP, VP, VP, VP, VP, C.POINTER(C.c_char_p), C.POINTER(C.c_char_p), C.c_char_p]),
    "colate_maketmp_pileup": (C.c_int64, [C.c_int, C.POINTER(C.c_char_p), C.POINTER(C.c_char_p), VP, C.c_int64, C.POINTER(C.c_char_p), C.c_char_p]),
    "colate_set_ref_genome": (C.c_int, [VP, C.c_int, C.POINTER(VP), VP]),
    "colate_maketmp_word": (C.c_uint32, [C.c_int, C.c_int, C.c_char_p]),
    "colate_read_mut_words": (C.c_int64, [C.c_char_p, C.c_int64, VP]),
    "colate_set_maketmp_words": (C.c_int, [VP, VP, C.c_int]),
    "colate_fetch_maketmp_words": (C.c_int, [VP, C.c_int64, C.c_int64, VP]),
    "colate_maketmp_mask_bits": (C.c_int, [C.c_char_p, C.c_int64, VP, C.c_int64, VP]),
    "colate_maketmp_write_pileup": (C.c_int64, [VP, C.c_int, C.c_int, C.POINTER(C.c_char_p), VP, C.c_char_p]),
    "colate_maketmp_write_bcf": (C.c_int64, [VP, C.c_int, C.POINTER(C.c_char_p), C.POINTER(C.c_char_p), VP, C.c_int64, C.c_char_p]),
    "colate_maketmp_write_bcf_genome": (C.c_int64, [VP, C.c_int, C.POINTER(C.c_char_p), C.c_char_p, VP, C.c_int64, C.c_char_p]),
    "colate_last_maketmp_timing": (C.c_int, [VP, f64]),
    "colate_upload_counts": (C.c_int, [VP, i64]),
    "colate_write_colate_mat": (C.c_int, [C.c_char_p, C.c_int, f64, f64]),
    "colate_write_coal": (C.c_int, [C.c_char_p, C.c_int, C.c_int, f64, f64, C.c_int, C.c_int]),
    "colate_write_bin": (C.c_int, [C.c_char_p, C.c_int, C.c_int, f64, f64, i32]),
}

TEST_HOOKS = {
    "colate_test_charpoly_terms": (C.c_int, [i32, C.c_int]),
    "colate_test_jump_window_host": (C.c_int, [u32, C.c_int, u32]),
    "colate_test_bin_thresholds": (C.c_int, [f64]),
    "colate_test_add_repeated": (C.c_double, [C.c_double, C.c_double, C.c_int]),
    "colate_test_stream_phys": (C.c_int64, [C.c_int64, C.c_int64]),
    "colate_test_colate_in_runs": (C.c_int64, [VP, C.c_int64, C.c_int, C.POINTER(C.c_char_p), C.c_int, i64, i64, i64]),
    "colate_test_libm": (C.c_int, [VP, C.c_int, C.c_int, f64, f64]),
    "colate_test_log1p_wide": (C.c_int, [C.c_int, f64, f64, i32]),
    "colate_test_em_prims": (C.c_int, [VP, C.c_int, C.c_int, f64, VP, f64, i32]),
    "colate_test_last_em": (C.c_int, [VP, C.POINTER(C.c_int), C.POINTER(C.c_int)]),
    "colate_test_last_vcf_paths": (C.c_int, [VP, C.POINTER(C.c_int64), C.POINTER(C.c_int64)]),
    "colate_test_bin_fast": (C.c_int, [VP, C.c_int, f64, i32, i32]),
    "colate_test_bin_sweep": (C.c_int, [VP, C.c_uint32, C.c_uint32, _p(dtype=np.uint64, flags="C_CONTIGUOUS")]),
    "colate_test_mt_stream": (C.c_int, [VP, u32, C.c_int64, C.c_int64, C.c_int, u32]),
}

_lib = None


def lib():
    """The loaded library.  Raises if it is missing -- there is no fallback implementation."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise ImportError(f"{LIB_PATH} is missing: build it with `make -C colate_b200/csrc` "
                              "(or __graft_entry__.build()); colate_b200 has no CPU fallback")
        L = C.CDLL(LIB_PATH)
        for table in (SIGNATURES, TEST_HOOKS):
            for name, (res, args) in table.items():
                f = getattr(L, name)
                f.restype = res
                f.argtypes = args
        _lib = L
    return _lib


def check(rc):
    if rc < 0:
        raise ColateError(rc, lib().colate_last_error().decode(errors="replace"))
    return rc


def ptr(a):
    """void* of a C-contiguous numpy array (or None)."""
    if a is None:
        return None
    assert a.flags["C_CONTIGUOUS"]
    return a.ctypes.data_as(VP)
