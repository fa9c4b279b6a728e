"""ctypes binding of libhkcsa.so (include/hkcsa.h).

The CUDA library is the only compute path: if it is missing or fails to load
this module raises -- there is no CPU or PyTorch fallback.
"""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libhkcsa.so")

MAX_LEVELS = 8
MAX_N = (1 << 30) - 2
BLOCK_BITS = 224
SUPER_BLOCKS = 65536
SELECT_SAMPLE = 4096
MAX_SLICES = 8
DSA_BUCKETS = 65536
DSA_MAX_RANKS = 8
DSA_MAX_N32 = (1 << 32) - 2
PROF_CLASSES = 16

OK, EINVAL, ECUDA, ESCRATCH, ERANGE = 0, -1, -2, -3, -4


class HkcsaError(RuntimeError):
    def __init__(self, code: int, msg: str):
        super().__init__(f"libhkcsa error {code}: {msg}")
        self.code = code


class SaStats(C.Structure):
    _fields_ = [
        ("rounds", C.c_uint32),
        ("bits_per_symbol", C.c_uint32),
        ("k0", C.c_uint32),
        ("sigma", C.c_uint32),
        ("sort_elem_passes", C.c_uint64),
        ("alg_bytes", C.c_uint64),
        ("round_elems", C.c_uint64 * 40),
        ("round_passes", C.c_uint32 * 40),
        ("byte_hist", C.c_uint64 * 256),
        ("key_bits0", C.c_uint32),
        ("bwt_carried", C.c_uint32),
        ("gram_k", C.c_uint32),
        ("lazy_ranks", C.c_uint32),
    ]


class WtPlan(C.Structure):
    _fields_ = [
        ("n", C.c_uint64),
        ("sigma", C.c_uint32),
        ("levels", C.c_uint32),
        ("sym_of_code", C.c_uint8 * 256),
        ("code_of_sym", C.c_uint16 * 256),
        ("cnt", C.c_uint64 * 256),
        ("C", C.c_uint64 * 257),
        ("depth", C.c_uint8 * 256),
        ("level_len", C.c_uint64 * MAX_LEVELS),
        ("level_nodes", C.c_uint32 * MAX_LEVELS),
        ("off_tables", C.c_uint64),
        ("off_blocks", C.c_uint64 * MAX_LEVELS),
        ("off_super", C.c_uint64 * MAX_LEVELS),
        ("off_select", C.c_uint64 * MAX_LEVELS),
        ("level_ones", C.c_uint64 * MAX_LEVELS),
        ("blob_bytes", C.c_uint64),
        ("scratch_bytes", C.c_uint64),
        ("node_start", (C.c_uint32 * 256) * MAX_LEVELS),
        ("node_bit", (C.c_uint8 * 256) * MAX_LEVELS),
        ("node_id", (C.c_uint8 * 256) * MAX_LEVELS),
    ]


class SsaPlan(C.Structure):
    _fields_ = [
        ("n", C.c_uint64),
        ("rate", C.c_uint32),
        ("n_samples", C.c_uint64),
        ("off_blocks", C.c_uint64),
        ("off_super", C.c_uint64),
        ("off_samples", C.c_uint64),
        ("blob_bytes", C.c_uint64),
        ("scratch_bytes", C.c_uint64),
    ]


class OccPlan(C.Structure):
    _fields_ = [
        ("n", C.c_uint64),
        ("sigma", C.c_uint32),
        ("shift", C.c_uint32),
        ("layout", C.c_uint32),
        ("reserved", C.c_uint32),
        ("off_bwt", C.c_uint64),
        ("rows", C.c_uint64),
        ("stride", C.c_uint64),
        ("blob_bytes", C.c_uint64),
        ("scratch_bytes", C.c_uint64),
    ]


class DsaPlan(C.Structure):
    _fields_ = [
        ("n", C.c_uint64),
        ("sigma", C.c_uint32),
        ("bits0", C.c_uint32),
        ("k0", C.c_uint32),
        ("passes0", C.c_uint32),
        ("b_fixed", C.c_uint32),
        ("wide", C.c_uint32),
        ("code", C.c_uint32 * 257),
        ("len", C.c_uint8 * 257),
        ("fixed_code", C.c_uint16 * 256),
    ]


class RrrPlan(C.Structure):
    _fields_ = [(k, C.c_uint64) for k in ("nbits", "nblocks", "nsuper", "ones", "stream_bits", "off_super",
                                          "off_classes", "off_stream", "blob_bytes")]


class ProfEntry(C.Structure):
    _fields_ = [
        ("name", C.c_char * 32),
        ("launches", C.c_uint64),
        ("ms", C.c_double),
        ("alg_bytes", C.c_uint64),
    ]


# name -> (restype, argtypes); every symbol include/hkcsa.h declares
_vp, _u64, _u32, _i32, _sz = C.c_void_p, C.c_uint64, C.c_uint32, C.c_int, C.c_size_t
SIGNATURES = {
    "hkcsa_abi_version": (_i32, []),
    "hkcsa_last_error": (C.c_char_p, []),
    "hkcsa_struct_size": (_sz, [_i32]),
    "hkcsa_gen_text": (_i32, [_i32, _u64, _u64, _vp, _vp]),
    "hkcsa_gen_pattern_lengths": (_i32, [_u64, _u64, _u32, _u32, _u64, _vp, _vp]),
    "hkcsa_gen_pattern_bytes": (_i32, [_u64, _u64, _vp, _u64, _vp, _u32, _vp, _vp, _vp]),
    "hkcsa_sa_scratch_bytes": (_sz, [_u64]),
    "hkcsa_sa_build": (_i32, [_vp, _u64, _vp, _vp, _sz, _vp, C.POINTER(SaStats)]),
    "hkcsa_sa_bwt_build": (_i32, [_vp, _u64, _vp, _vp, _vp, _sz, _vp, C.POINTER(SaStats)]),
    "hkcsa_wt_blob_bound": (_sz, [_u64]),
    "hkcsa_wt_scratch_bound": (_sz, [_u64]),
    "hkcsa_index_build": (_i32, [_vp, _u64, _vp, _vp, _vp, _sz, C.POINTER(WtPlan), _vp, _sz, _vp, _sz,
                                 C.POINTER(SsaPlan), _vp, _vp, _sz, _vp, _vp, _vp, C.POINTER(SaStats)]),
    "hkcsa_dsa_plan_make": (_i32, [C.POINTER(_u64), _u64, _i32, C.POINTER(DsaPlan)]),
    "hkcsa_dsa_bucket_hist": (_i32, [_vp, C.POINTER(DsaPlan), _u64, _u64, _vp, _vp]),
    "hkcsa_dsa_bucket_hist_sampled": (_i32, [_vp, C.POINTER(DsaPlan), _u64, _u64, C.c_uint32, _vp, _vp]),
    "hkcsa_dsa_dest_counts": (_i32, [_vp, C.POINTER(DsaPlan), _u64, _u64, C.c_uint32, C.POINTER(C.c_uint32), _vp, _vp]),
    "hkcsa_dsa_pack_exchange": (_i32, [_vp, C.POINTER(DsaPlan), _u64, _u64, _u32, C.POINTER(_u32), C.POINTER(_u64),
                                       C.POINTER(_u64), C.POINTER(_u64), _vp, _vp]),
    "hkcsa_dsa_state_bytes": (_sz, []),
    "hkcsa_dsa_scratch_bytes": (_sz, [_u64]),
    "hkcsa_dsa_begin": (_i32, [_vp, C.POINTER(DsaPlan), _vp, _vp, _vp, _vp, _vp, _u64, _u64, _vp, _sz, _vp]),
    "hkcsa_dsa_working_set": (_u64, [_vp]),
    "hkcsa_dsa_depth": (_u64, [_vp]),
    "hkcsa_dsa_slice": (_vp, [_vp]),
    "hkcsa_dsa_rounds": (_i32, [_vp, C.POINTER(_u32), C.POINTER(_u64), _u32]),
    "hkcsa_dsa_group_round": (_i32, [_vp, _vp]),
    "hkcsa_dsa_ext_round": (_i32, [_vp, _vp]),
    "hkcsa_dsa_isa_publish": (_i32, [_vp, _u32, C.POINTER(_u64), _u64, _u64, _i32, _vp]),
    "hkcsa_dsa_dbl_keys": (_i32, [_vp, _u32, C.POINTER(_u64), _u64, C.POINTER(_u64), C.POINTER(_u64), C.POINTER(_u64),
                                  C.POINTER(_u32), _vp]),
    "hkcsa_dsa_dbl_sort": (_i32, [_vp, _vp]),
    "hkcsa_dsa_gather_ids64": (_i32, [_vp, _vp, _vp, _vp]),
    "hkcsa_bwt_slice": (_i32, [_vp, _u64, _vp, _u64, _vp, _vp]),
    "hkcsa_bwt_slice64": (_i32, [_vp, _u64, _vp, _u64, _vp, _vp]),
    "hkcsa_ssa_build64": (_i32, [_vp, C.POINTER(SsaPlan), _vp, _vp, _sz, _vp]),
    "hkcsa_expand_ranges64": (_i32, [_vp, _vp, _vp, _u64, _vp, _vp]),
    "hkcsa_sort_scratch_bytes": (_sz, [_u64]),
    "hkcsa_sort_pairs_u64": (_i32, [_vp, _vp, _vp, _vp, _u64, _i32, _vp, _sz, _vp]),
    "hkcsa_bwt": (_i32, [_vp, _vp, _u64, _vp, _vp]),
    "hkcsa_byte_hist": (_i32, [_vp, _u64, _vp, _vp]),
    "hkcsa_wt_plan_from_hist": (_i32, [C.POINTER(_u64), C.POINTER(WtPlan)]),
    "hkcsa_wt_build": (_i32, [_vp, C.POINTER(WtPlan), _vp, _vp, _sz, _vp]),
    "hkcsa_bv_rank_batch": (_i32, [_vp, C.POINTER(WtPlan), _u32, _vp, _u64, _vp, _vp]),
    "hkcsa_bv_select_batch": (_i32, [_vp, C.POINTER(WtPlan), _u32, _vp, _u64, _vp, _vp]),
    "hkcsa_bv_unpack": (_i32, [_vp, C.POINTER(WtPlan), _u32, _u64, _u64, _vp, _vp]),
    "hkcsa_bv_rank_range": (_i32, [_vp, C.POINTER(WtPlan), _u32, _u64, _u64, _vp, _vp]),
    "hkcsa_bitvec_plan": (_i32, [_u64, C.POINTER(WtPlan)]),
    "hkcsa_bitvec_build": (_i32, [_vp, C.POINTER(WtPlan), _vp, _vp, _sz, _vp]),
    "hkcsa_partition_scratch_bytes": (_sz, [_u64]),
    "hkcsa_partition_bytes": (_i32, [_vp, _u64, C.POINTER(C.c_uint8), _vp, C.POINTER(_u64), _vp, _sz, _vp]),
    "hkcsa_wt_rank_batch": (_i32, [_vp, C.POINTER(WtPlan), _vp, _vp, _u64, _vp, _vp]),
    "hkcsa_wt_access_batch": (_i32, [_vp, C.POINTER(WtPlan), _vp, _u64, _vp, _vp]),
    "hkcsa_golomb_scratch_bytes": (_sz, [_u64]),
    "hkcsa_golomb_encode": (_i32, [_vp, C.POINTER(WtPlan), _u32, _u64, _u32, _vp, _u64, C.POINTER(_u64), _vp,
                                   _sz, _vp]),
    "hkcsa_count_batch": (_i32, [_vp, C.POINTER(WtPlan), _vp, _vp, _u64, _vp, _vp, _vp]),
    "hkcsa_occ_plan_make": (_i32, [_u64, _u32, _u32, _u32, C.POINTER(OccPlan)]),
    "hkcsa_occ_build": (_i32, [_vp, C.POINTER(WtPlan), _vp, C.POINTER(OccPlan), _vp, _vp, _sz, _vp]),
    "hkcsa_count_batch_occ": (_i32, [_vp, C.POINTER(WtPlan), _vp, C.POINTER(OccPlan), _vp, _u32, _vp, _vp, _u64,
                                     _vp, _vp, _vp]),
    "hkcsa_count_batch_peers": (_i32, [_vp, C.POINTER(WtPlan), _vp, C.POINTER(OccPlan), _vp, _u32, _vp, _vp, _u64, _u64,
                                       _u32, C.POINTER(_u64), C.POINTER(_u64), _vp]),
    "hkcsa_ranges_push_peers": (_i32, [_vp, _vp, _u64, _u64, _u32, C.POINTER(_u64), _u64, _vp]),
    "hkcsa_ranges_unpack": (_i32, [_vp, _u64, _vp, _vp, _vp]),
    "hkcsa_locate_rows_occ": (_i32, [_vp, C.POINTER(WtPlan), _vp, C.POINTER(OccPlan), _vp, C.POINTER(SsaPlan), _u32,
                                     _vp, _u64, _vp, _vp]),
    "hkcsa_isa_samples": (_i32, [_vp, C.POINTER(SsaPlan), _vp, _vp]),
    "hkcsa_extract_scratch_bytes": (_sz, [_u64]),
    "hkcsa_extract": (_i32, [_vp, C.POINTER(WtPlan), _vp, C.POINTER(OccPlan), _vp, _u32, _vp, _vp, _vp, _u64, _vp,
                             _vp, _sz, _vp]),
    "hkcsa_kmer_k": (_u32, [_u32]),
    "hkcsa_kmer_entries": (_u64, [_u32, _u32]),
    "hkcsa_kmer_scratch_bytes": (_sz, [_u32, _u32]),
    "hkcsa_kmer_table_build": (_i32, [_vp, C.POINTER(WtPlan), _u32, _vp, _vp, _sz, _vp]),
    "hkcsa_count_batch_kmer": (_i32, [_vp, C.POINTER(WtPlan), _vp, _u32, _vp, _vp, _u64, _vp, _vp, _vp]),
    "hkcsa_ssa_plan_make": (_i32, [_u64, _u32, C.POINTER(SsaPlan)]),
    "hkcsa_ssa_build": (_i32, [_vp, C.POINTER(SsaPlan), _vp, _vp, _sz, _vp]),
    "hkcsa_ssa_plan_make_slice": (_i32, [_u64, _u32, _u64, C.POINTER(SsaPlan)]),
    "hkcsa_multi_desc_bytes": (_sz, []),
    "hkcsa_multi_desc_build": (_i32, [_u32, C.POINTER(_vp), C.POINTER(C.POINTER(WtPlan)), C.POINTER(_u64),
                                      C.POINTER(_vp), C.POINTER(C.POINTER(SsaPlan)), _u64, _vp, _vp]),
    "hkcsa_multi_count_batch": (_i32, [_vp, _vp, _vp, _u64, _vp, _vp, _vp]),
    "hkcsa_multi_locate_rows": (_i32, [_vp, _vp, _u64, _vp, _vp]),
    "hkcsa_multi_isa_samples": (_i32, [_u32, C.POINTER(_vp), C.POINTER(C.POINTER(SsaPlan)), C.POINTER(_u64), _vp,
                                       _vp]),
    "hkcsa_multi_extract": (_i32, [_vp, _u64, _u32, _vp, _vp, _vp, _vp, _u64, _vp, _vp, _sz, _vp]),
    "hkcsa_expand_ranges": (_i32, [_vp, _vp, _vp, _u64, _vp, _vp]),
    "hkcsa_gather_u32": (_i32, [_vp, _vp, _u64, _vp, _vp]),
    "hkcsa_locate_rows": (_i32, [_vp, C.POINTER(WtPlan), _vp, C.POINTER(SsaPlan), _u32, _vp, _u64, _vp, _vp]),
    "hkcsa_symbol_positions_scratch_bytes": (_sz, [_u64]),
    "hkcsa_symbol_positions": (_i32, [_vp, _u64, _vp, _vp, _vp, _sz, _vp]),
    "hkcsa_rrr_tables_bytes": (_sz, []),
    "hkcsa_rrr_tables_init": (_i32, [_vp, _vp]),
    "hkcsa_rrr_scratch_bytes": (_sz, [_u64]),
    "hkcsa_rrr_encode": (_i32, [_vp, C.POINTER(WtPlan), _u32, _u64, _vp, C.POINTER(RrrPlan), _vp, _sz, _vp, _sz, _vp]),
    "hkcsa_rrr_rank_batch": (_i32, [_vp, C.POINTER(RrrPlan), _vp, _vp, _u64, _vp, _vp]),
    "hkcsa_rrr_unpack": (_i32, [_vp, C.POINTER(RrrPlan), _vp, _u64, _u64, _vp, _vp]),
    "hkcsa_wt_restore_begin": (_i32, [C.POINTER(WtPlan), _vp, _vp]),
    "hkcsa_rrr_restore_level": (_i32, [_vp, C.POINTER(RrrPlan), _vp, C.POINTER(WtPlan), _u32, _vp, _vp]),
    "hkcsa_wt_restore_finish": (_i32, [C.POINTER(WtPlan), _vp, _vp, _sz, _vp]),
    "hkcsa_entropy_scratch_bytes": (_sz, [_u64]),
    "hkcsa_entropy_from_sa": (_i32, [_vp, _u64, _vp, _u32, C.POINTER(C.c_double), _vp, _sz, _vp]),
    "hkcsa_lcp_scratch_bytes": (_sz, [_u64]),
    "hkcsa_lcp_build": (_i32, [_vp, _u64, _vp, _vp, _vp, _vp, _sz, C.POINTER(_u64), _vp]),
    "hkcsa_plcp_bits": (_i32, [_vp, _u64, _vp, _vp]),
    "hkcsa_launch_count": (C.c_ulonglong, []),
    "hkcsa_h2d_staged": (C.c_int, [C.c_void_p, C.c_void_p, C.c_size_t, C.c_int, C.c_void_p]),
    "hkcsa_d2h_staged": (C.c_int, [C.c_void_p, C.c_void_p, C.c_size_t, C.c_int, C.c_void_p]),
    "hkcsa_prof_enable": (_i32, [_i32]),
    "hkcsa_prof_enable_classes": (_i32, [_u32]),
    "hkcsa_prof_class_index": (_i32, [C.c_char_p]),
    "hkcsa_prof_reset": (_i32, []),
    "hkcsa_prof_read": (_i32, [C.POINTER(ProfEntry), _i32, C.POINTER(_i32)]),
    "hkcsa_prof_timeline": (_i32, [_vp, _vp, _vp, C.c_int, _vp]),
}

_lib = None


def load() -> C.CDLL:
    """Load libhkcsa.so; raises if the CUDA extension has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "(nvcc, sm_100a).  There is no CPU fallback.")
    L = C.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(L, name)     # AttributeError if the library lacks a declared symbol
        fn.restype = res
        fn.argtypes = args
    if L.hkcsa_abi_version() != 1:
        raise ImportError("libhkcsa.so ABI version mismatch")
    for idx, st in enumerate((SaStats, WtPlan, SsaPlan, ProfEntry, OccPlan, DsaPlan, RrrPlan)):
        if L.hkcsa_struct_size(idx) != C.sizeof(st):
            raise ImportError(f"struct layout mismatch for {st.__name__}: "
                              f"C {L.hkcsa_struct_size(idx)} vs ctypes {C.sizeof(st)}")
    _lib = L
    return L


def check(rc: int) -> None:
    if rc != OK:
        raise HkcsaError(rc, load().hkcsa_last_error().decode("utf-8", "replace"))
