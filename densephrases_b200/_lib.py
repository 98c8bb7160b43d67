"""ctypes loader for libdph_b200.so (the C ABI declared in include/dph_b200.h).

There is NO CPU fallback: if the CUDA library is missing or a call fails, RuntimeError is raised
(the FAISS/SWIG convention the reference relies on, SURVEY.md 8b)."""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "lib", "libdph_b200.so")
_lib = None

MEM_HOST, MEM_DEVICE = 0, 1
SCAN_FAST, SCAN_EXACT, SCAN_PAIR, SCAN_SINGLE, SCAN_QUAD = 0, 1, 2, 3, 4

_vp, _i64, _i32, _u64, _f32 = C.c_void_p, C.c_int64, C.c_int, C.c_uint64, C.c_float
_SIGS = {
    "dph_last_error": (C.c_char_p, []),
    "dph_version": (_i32, []),
    "dph_index_create": (_i32, [C.POINTER(_vp), _i32, _i64, _i32, _i32, _i32]),
    "dph_index_free": (None, [_vp]),
    "dph_index_set_stream": (_i32, [_vp, _vp]),
    "dph_index_set_opq": (_i32, [_vp, _vp, _i32]),
    "dph_index_set_centroids": (_i32, [_vp, _vp, _i32]),
    "dph_index_set_pq": (_i32, [_vp, _vp, _i32]),
    "dph_index_gen_centroids": (_i32, [_vp, _u64, _f32]),
    "dph_index_gen_pq": (_i32, [_vp, _u64, _f32]),
    "dph_index_set_shard": (_i32, [_vp, _i64, _i64]),
    "dph_index_set_lists": (_i32, [_vp, _vp, _vp, _vp]),
    "dph_index_set_lists_synthetic": (_i32, [_vp, _vp, _u64]),
    "dph_index_ntotal": (_i64, [_vp]),
    "dph_index_ntotal_local": (_i64, [_vp]),
    "dph_index_d": (_i32, [_vp]),
    "dph_index_nlist": (_i64, [_vp]),
    "dph_index_nprobe": (_i32, [_vp]),
    "dph_index_set_nprobe": (_i32, [_vp, _i32]),
    "dph_index_set_scan_mode": (_i32, [_vp, _i32]),
    "dph_index_set_coarse_tc": (_i32, [_vp, _i32]),
    "dph_index_get_opq": (_i32, [_vp, _vp, _i32]),
    "dph_index_device_bytes": (_i64, [_vp]),
    "dph_index_set_profile": (_i32, [_vp, _i32]),
    "dph_index_last_scan_ms": (_i32, [_vp, C.POINTER(C.c_float)]),
    "dph_index_profile_scan_ms": (_i32, [_vp, _vp, _i32]),
    "dph_index_profile_count": (_i32, [_vp]),
    "dph_index_search": (_i32, [_vp, _vp, _i64, _i32, _vp, _vp, _i32]),
    "dph_index_search_partial": (_i32, [_vp, _vp, _i64, _i32, _vp, _vp, _vp]),
    "dph_index_coarse_local": (_i32, [_vp, _vp, _i64, _vp]),
    "dph_index_search_preassigned": (_i32, [_vp, _vp, _i32, _i64, _i32, _vp, _vp, _vp]),
    "dph_index_record_floats": (_i32, [_vp]),
    "dph_index_coarse_split": (_i32, [_vp, _vp, _i64, _vp]),
    "dph_index_search_assigned": (_i32, [_vp, _vp, _i64, _i32, _vp, _vp, _vp]),
    "dph_merge_shards": (_i32, [_vp, _vp, _vp, _i32, _i64, _i32, _vp, _vp, _vp]),
    "dph_pack_topk": (_i32, [_vp, _vp, _vp, _i64, _i32, _vp, _vp]),
    "dph_merge_shards_packed": (_i32, [_vp, _i32, _i64, _i32, _vp, _vp, _vp]),
    "dph_index_last_flags": (_vp, [_vp]),
    "dph_index_last_probes": (_vp, [_vp]),
    "dph_index_last_coarse": (_vp, [_vp]),
    "dph_index_last_xr": (_vp, [_vp]),
    "dph_index_last_used_pair_mode": (_i32, [_vp]),
    "dph_index_last_group_size": (_i32, [_vp]),
    "dph_index_copy_last": (_i32, [_vp, _i32, _vp, _i64]),
    "dph_index_reconstruct_batch": (_i32, [_vp, _vp, _i64, _vp, _vp, _i32]),
    "dph_encoder_create": (_i32, [C.POINTER(_vp), _i32, _i32, _i32, _i32]),
    "dph_encoder_free": (None, [_vp]),
    "dph_encoder_set_stream": (_i32, [_vp, _vp]),
    "dph_encoder_tower_floats": (_i64, [_vp]),
    "dph_encoder_load_tower": (_i32, [_vp, _i32, _vp, _i32]),
    "dph_encoder_embed_query": (_i32, [_vp, _vp, _vp, _vp, _i32, _i32, _vp, _vp, _i32]),
    "dph_encoder_load_filter": (_i32, [_vp, _vp, _vp, _i32]),
    "dph_encoder_embed_phrase": (_i32, [_vp, _vp, _vp, _vp, _i32, _i32, _vp, _vp, _vp, _vp, _f32, _f32, _i32]),
    "dph_sgemm_nt_seq": (_i32, [_vp, _i64, _vp, _i64, _i64, _vp, _vp]),
    "dph_gemm_tf32_nt": (_i32, [_vp, _vp, _vp, _vp, _vp, _i64, _i64, _i64, _i32, _i32, _vp]),
    "dph_encoder_set_precision": (_i32, [_vp, _i32]),
    "dph_gemm_tf32_set_mode": (_i32, [_i32]),
    "dph_set_tuning": (_i32, [_i32, _i32]),
    "dph_encoder_set_attention": (_i32, [_vp, _i32]),
    "dph_attention_bert": (_i32, [_vp, _vp, _i32, _i32, _vp, _i32, _vp]),
    "dph_index_window_scores": (_i32, [_vp, _vp, _vp, _i64, _i32, _vp, _i32]),
}
EXPORTS = tuple(_SIGS)


def lib():
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(f"{LIB_PATH} not built: run `make` (or __graft_entry__.build()). There is no CPU fallback.")
        L = C.CDLL(LIB_PATH)
        for name, (res, args) in _SIGS.items():
            fn = getattr(L, name)
            fn.restype, fn.argtypes = res, args
        _lib = L
    return _lib


def check(rc):
    if rc != 0:
        raise RuntimeError("libdph_b200: " + lib().dph_last_error().decode())
