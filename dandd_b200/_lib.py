"""ctypes binding of the C ABI in include/dandd_b200.h.

Loading fails loudly: if libdandd_b200.so has not been built, or there is no sm_100 device, an
exception is raised -- there is deliberately no slow path to fall back to."""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libdandd_b200.so")

DD_HIST_BINS = 64
DD_EXACT_BITMAP_MAXK = 16
DD_COVER_PART_BYTES = 64
ABI_VERSION = 2
DD_PACK_FLAG_OVERFLOW, DD_PACK_FLAG_FASTQ = 1, 2
DD_ERR_FORMAT = -5


class DandDError(RuntimeError):
    """A C-ABI call returned a negative status (message from dd_last_error())."""


class PackState(C.Structure):
    _fields_ = [("nsym", C.c_uint64), ("prev_nsym", C.c_uint64), ("in_header", C.c_uint32),
                ("last_byte", C.c_uint32), ("reserved", C.c_uint64)]


_vp, _sz, _i, _u32, _u64, _i64 = C.c_void_p, C.c_size_t, C.c_int, C.c_uint32, C.c_uint64, C.c_int64

# name -> (restype, argtypes); every symbol declared in include/dandd_b200.h
SIGNATURES = {
    "dd_last_error": (C.c_char_p, []),
    "dd_abi_version": (_i, []),
    "dd_kernel_launches": (C.c_ulonglong, []),
    "dd_init": (_i, [_i]),
    "dd_set_option": (_i, [C.c_char_p, C.c_long]),
    "dd_device_info": (_i, [_i, C.POINTER(_i), C.POINTER(_i), C.POINTER(_i), C.POINTER(_sz), C.POINTER(_sz)]),
    "dd_pack_codes_bytes": (_sz, [_sz]),
    "dd_pack_invalid_bytes": (_sz, [_sz]),
    "dd_pack_workspace_bytes": (_sz, [_sz]),
    "dd_pack_reset": (_i, [_vp, _sz, _vp, _sz, _vp, _vp]),
    "dd_pack_fasta": (_i, [_vp, _sz, _vp, _vp, _sz, _vp, _vp, _sz, _vp]),
    "dd_pack_polyt_sentinel": (_i, [_vp, _vp, _vp, _u64, _u64, _sz, _vp]),
    "dd_fastq_to_fasta_host": (_sz, [_vp, _sz, _vp]),
    "dd_fasta_first_record_host": (_sz, [_vp, _sz]),
    "dd_sketch_workspace_bytes": (_sz, [_i, _i]),
    "dd_sketch_begin": (_i, [_vp, _sz, _i, _i, _vp]),
    "dd_sketch_update": (_i, [_vp, _vp, _vp, _sz, _u32, _i, _i, _vp, _sz, _vp]),
    "dd_sketch_update_range": (_i, [_vp, _vp, _u64, _u64, _u32, _i, _i, _vp, _sz, _vp]),
    "dd_sketch_update_sched": (_i, [_vp, _vp, _vp, _u64, _u64, _sz, _u64, _u32, _i, _i, _vp, _sz, _vp]),
    "dd_sketch_refresh_floor": (_i, [_vp, _sz, _u32, _i, _vp]),
    "dd_sketch_end": (_i, [_vp, _sz, _i, _i, _vp, _vp, _vp, _vp]),
    "dd_card_ertl_mle": (_i, [_vp, _i, _i, _vp, _vp, _vp]),
    "dd_mle_from_hist": (_i, [_vp, _i, _i, _vp, _vp]),
    "dd_mle_from_hist_f64": (_i, [_vp, _i, _i, _vp, _vp]),
    "dd_union_max": (_i, [_vp, _i, _sz, _vp, _vp]),
    "dd_prefix_union_workspace_bytes": (_sz, [_i, _i, _i, _i, _i]),
    "dd_prefix_union_card": (_i, [_vp, _vp, _i, _i, _i, _i, _i, _i, _vp, _vp, _vp, _vp, _sz, _vp]),
    "dd_planes_bytes": (_sz, [_i64, _i]),
    "dd_to_planes": (_i, [_vp, _i64, _i, _vp, _vp]),
    "dd_prefix_union_card_planes": (_i, [_vp, _vp, _i, _i, _i, _i, _i, _i, _vp, _vp, _vp, _sz, _vp]),
    "dd_union_sets_card": (_i, [_vp, _i, _i, _i, _i, _vp, _vp, _vp, _vp]),
    "dd_pairwise_union_card": (_i, [_vp, _i, _i, _i, _vp, _i64, _vp, _vp, _vp, _sz, _vp]),
    "dd_pairwise_union_card_planes": (_i, [_vp, _i, _i, _i, _vp, _i64, _vp, _vp, _vp]),
    "dd_exact_workspace_bytes": (_sz, [_i, _u64]),
    "dd_exact_begin": (_i, [_vp, _sz, _i, _u64, _vp]),
    "dd_exact_insert": (_i, [_vp, _vp, _u64, _u64, _i, _i, _vp, _sz, _u64, _vp]),
    "dd_exact_insert_shard": (_i, [_vp, _vp, _u64, _u64, _i, _i, _vp, _sz, _u64, _u32, _u32, _vp]),
    "dd_exact_count": (_i, [_vp, _sz, _i, _u64, _vp, _vp]),
    "dd_exact_pairs_workspace_bytes": (_sz, [_i, _u64, _u64, _u32]),
    "dd_exact_pairs_begin": (_i, [_vp, _sz, _i, _u64, _u64, _u32, _vp]),
    "dd_exact_pairs_insert_shard": (_i, [_vp, _vp, _u64, _u64, _i, _i, _u32, _vp, _sz, _u64, _u64, _u32, _u32, _u32, _vp]),
    "dd_exact_pairs_accumulate": (_i, [_vp, _sz, _i, _u64, _u64, _u32, _i64, _vp, _vp]),
    "dd_exact_pair_popc": (_i, [_vp, _i64, _i, _vp, _i64, _i, _sz, _i, _i64, _vp, _vp]),
    "dd_exact_first_rank_hist": (_i, [_vp, _sz, _i, _u64, _u64, _u32, _i64, _vp, _i64, _vp, _vp]),
    "dd_exact_pairs_node_count": (_i, [_vp, _sz, _vp, _vp]),
    "dd_exact_occupancy_hist": (_i, [_vp, _sz, _i, _u64, _u64, _u32, _i64, _vp, _vp, _vp]),
    "dd_exact_query_counts": (_i, [_vp, _sz, _i, _u64, _u64, _u32, _i64, _i64, _vp, _vp, _vp, _vp]),
    "dd_exact_cover_count": (_i, [_vp, _sz, _i, _u64, _u64, _u32, _vp, _vp]),
    "dd_exact_cover_emit": (_i, [_vp, _sz, _i, _u64, _u64, _u32, _i64, _u64, _u64, _vp, _vp, _vp, _vp, _vp]),
    "dd_exact_cover_step": (_i, [_vp, _i, _i64, _i64, _vp, _sz, _vp]),
    "dd_leave_out_workspace_bytes": (_sz, [_i, _i]),
    "dd_leave_out_hist": (_i, [_vp, _i, _i, _i, _vp, _i, _u64, _u64, _vp, _vp, _sz, _vp]),
    "dd_register_spectrum_workspace_bytes": (_sz, [_i, _i]),
    "dd_register_spectrum": (_i, [_vp, _i, _i, _i, _u64, _u64, _vp, _vp, _sz, _vp]),
    "dd_greedy_workspace_bytes": (_sz, [_i]),
    "dd_greedy_dense_hist": (_i, [_vp, _i, _i, _i, _vp, _vp, _vp, _i, _vp, _vp, _vp, _sz, _vp]),
    "dd_greedy_compact": (_i, [_vp, _i, _i, _i, _vp, _vp, _i, _vp, _vp, _vp, _vp, _i64, _vp, _sz, _vp]),
    "dd_greedy_sparse_hist": (_i, [_vp, _i64, _vp, _vp, _i, _i, _i, _vp, _vp, _vp, _i, _vp, _vp, _vp, _sz, _vp]),
    "dd_sketch_fasta_host_workspace_bytes": (_sz, [_sz, _i, _i]),
    "dd_sketch_fasta_host": (_i, [_vp, _sz, _u32, _i, _i, _vp, _vp, _vp, _vp, _sz, _vp]),
    "dd_sketch_fasta_host_async": (_i, [_vp, _sz, _u32, _i, _i, _vp, _vp, _vp, _vp, _sz, _vp]),
}

_lib = None


def load():
    """dlopen the in-tree library and attach signatures.  Does not touch the GPU."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise DandDError(f"{LIB_PATH} is missing: run `python -m dandd_b200.build` "
                             "(or __graft_entry__.build()); there is no CPU fallback")
        L = C.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(L, name)            # AttributeError here == ABI drift, by design
            fn.restype, fn.argtypes = res, args
        if L.dd_abi_version() != ABI_VERSION:
            raise DandDError(f"ABI version mismatch: library {L.dd_abi_version()} != binding {ABI_VERSION}")
        _lib = L
    return _lib


def check(rc, what=""):
    if rc != 0:
        msg = load().dd_last_error().decode("utf-8", "replace")
        raise DandDError(f"{what or 'dandd_b200'} failed ({rc}): {msg}")
    return rc
