"""ctypes binding of libgpcgc.so (the C ABI declared in include/gpcgc.h).

There is NO fallback: if the shared library is missing or a call fails, an exception is raised.
"""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("GPC_LIB_PATH", os.path.join(_HERE, "libgpcgc.so"))      # override: A/B builds of the same ABI (tools/)

c_vp, c_i64, c_int, c_sz, c_f32 = C.c_void_p, C.c_int64, C.c_int, C.c_size_t, C.c_float


class KeyXform(C.Structure):
    _fields_ = [("minx", C.c_uint32), ("miny", C.c_uint32), ("minz", C.c_uint32),
                ("sy", C.c_uint32), ("sz", C.c_uint32), ("total_bits", C.c_uint32)]


class GpcError(RuntimeError):
    pass


# name -> (restype, argtypes); every symbol include/gpcgc.h declares
SIGNATURES = {
    "gpc_last_error": (C.c_char_p, []),
    "gpc_version": (c_int, []),
    "gpc_launch_count": (C.c_uint64, []),
    "gpc_copy_async": (c_int, [c_vp, c_vp, c_i64, c_vp]),
    "gpc_pack_keys_f32": (c_int, [c_vp, c_i64, c_vp, c_vp, c_vp]),
    "gpc_pack_keys_i32": (c_int, [c_vp, c_i64, c_vp, c_vp, c_vp]),
    "gpc_unpack_keys_i32": (c_int, [c_vp, c_i64, c_vp, c_vp]),
    "gpc_unpack_keys_f32": (c_int, [c_vp, c_i64, c_f32, c_vp, c_vp]),
    "gpc_key_minmax": (c_int, [c_vp, c_i64, c_vp, c_vp]),
    "gpc_make_xform_h": (c_int, [c_vp, C.POINTER(KeyXform)]),
    "gpc_sort_workspace_bytes": (c_sz, [c_i64]),
    "gpc_sort_pairs": (c_int, [c_vp, c_vp, c_vp, c_vp, c_i64, KeyXform, c_vp, c_sz, c_vp]),
    "gpc_lexorder_workspace_bytes": (c_sz, [c_i64]),
    "gpc_lexorder_zyx": (c_int, [c_vp, c_int, c_i64, c_vp, c_vp, c_sz, c_vp]),
    "gpc_pyramid_workspace_bytes": (c_sz, [c_i64]),
    "gpc_unique_sorted": (c_int, [c_vp, c_i64, c_vp, c_vp, c_vp, c_sz, c_vp]),
    "gpc_pyramid_down": (c_int, [c_vp, c_i64, KeyXform, c_vp, c_vp, c_vp, c_vp, c_sz, c_vp]),
    "gpc_expand_workspace_bytes": (c_sz, [c_i64]),
    "gpc_expand_children": (c_int, [c_vp, c_vp, c_i64, c_i64, c_vp, c_vp, c_vp, c_sz, c_vp]),
    "gpc_expand_leaves_f32": (c_int, [c_vp, c_vp, c_i64, c_i64, c_f32, c_vp, c_vp, c_sz, c_vp]),
    "gpc_hash_capacity": (c_i64, [c_i64]),
    "gpc_hash_build": (c_int, [c_vp, c_i64, c_vp, c_i64, c_vp]),
    "gpc_hash_lookup": (c_int, [c_vp, c_i64, c_vp, c_i64, c_vp, c_vp]),
    "gpc_kmap_dense": (c_int, [c_vp, c_i64, c_vp, c_i64, c_vp, c_int, c_int, c_vp, c_vp]),
    "gpc_kmap_pairs_workspace_bytes": (c_sz, [c_i64, c_int]),
    "gpc_kmap_pairs_count": (c_int, [c_vp, c_i64, c_int, c_int, c_vp, c_vp, c_vp, c_sz, c_vp]),
    "gpc_kmap_pairs_fill": (c_int, [c_vp, c_i64, c_int, c_vp, c_vp, c_vp, c_vp, c_i64, c_vp]),
    "gpc_kmap_pairs_count_range": (c_int, [c_vp, c_i64, c_i64, c_i64, c_int, c_int, c_vp, c_vp, c_vp, c_sz, c_vp]),
    "gpc_kmap_pairs_fill_range": (c_int, [c_vp, c_i64, c_i64, c_i64, c_int, c_vp, c_vp, c_i64, c_vp]),
    "gpc_spconv_pack_weights_frag": (c_int, [c_vp, c_int, c_vp, c_vp]),
    "gpc_spconv_fwd_v6": (c_int, [c_vp, c_vp, c_vp, c_vp, c_i64, c_int, c_vp, c_int, c_vp, c_int, c_vp]),
    "gpc_spconv_fwd_v6_rows": (c_int, [c_vp, c_vp, c_vp, c_vp, c_i64, c_int, c_vp, c_int, c_vp, c_int, c_i64, c_i64, c_vp]),
    "gpc_spconv_fwd_v6_range": (c_int, [c_vp, c_vp, c_vp, c_vp, c_i64, c_i64, c_i64, c_int, c_vp, c_int, c_vp, c_int, c_vp]),
    "gpc_spconv_wgrad_workspace_bytes": (c_sz, [c_i64, c_int]),
    "gpc_spconv_wgrad_v6": (c_int, [c_vp, c_vp, c_vp, c_vp, c_i64, c_int, c_vp, c_vp, c_sz, c_vp]),
    "gpc_spconv_wgrad_balanced_workspace_bytes": (c_sz, [c_i64, c_int, c_i64]),
    "gpc_spconv_wgrad_v6_balanced": (c_int, [c_vp, c_vp, c_vp, c_vp, c_i64, c_int, c_i64, c_vp, c_vp, c_sz, c_vp]),
    "gpc_spconv_wgrad_um_workspace_bytes": (c_sz, [c_i64, c_int, c_i64]),
    "gpc_spconv_wgrad_um": (c_int, [c_vp, c_vp, c_vp, c_vp, c_vp, c_i64, c_int, c_i64, c_vp, c_vp, c_sz, c_vp]),
    "gpc_spconv_wgrad_sparse_workspace_bytes": (c_sz, [c_i64, c_i64]),
    "gpc_spconv_wgrad_sparse": (c_int, [c_vp, c_vp, c_vp, c_vp, c_vp, c_i64, c_i64, c_vp, c_vp, c_sz, c_vp]),
    "gpc_kmap_sparse_segments": (c_i64, [c_i64]),
    "gpc_kmap_sparse_workspace_bytes": (c_sz, [c_i64]),
    "gpc_kmap_sparse_count": (c_int, [c_vp, c_i64, c_vp, c_vp, c_vp, c_vp, c_sz, c_vp]),
    "gpc_kmap_sparse_fill": (c_int, [c_vp, c_i64, c_vp, c_vp, c_vp, c_vp, c_i64, c_vp]),
    "gpc_spconv_sparse_fwd": (c_int, [c_vp, c_vp, c_vp, c_vp, c_vp, c_i64, c_i64, c_vp, c_vp, c_int, c_vp, c_vp]),
    "gpc_spconv_sparse_fwd_rows": (c_int, [c_vp, c_vp, c_vp, c_vp, c_vp, c_i64, c_i64, c_vp, c_vp, c_int, c_vp, c_i64, c_i64, c_vp]),
    "gpc_kmap_sparse_count_range": (c_int, [c_vp, c_i64, c_i64, c_i64, c_vp, c_vp, c_vp, c_vp, c_sz, c_vp]),
    "gpc_kmap_sparse_fill_range": (c_int, [c_vp, c_i64, c_i64, c_i64, c_vp, c_vp, c_vp, c_vp, c_i64, c_vp]),
    "gpc_spconv_sparse_fwd_range": (c_int, [c_vp, c_vp, c_vp, c_vp, c_vp, c_i64, c_i64, c_i64, c_i64, c_vp, c_vp, c_int, c_vp, c_vp]),
    "gpc_rows_split": (c_int, [c_vp, c_i64, c_vp, c_vp]),
    "gpc_rows_join": (c_int, [c_vp, c_i64, c_vp, c_vp]),
    "gpc_debug_conv_um_profile": (c_int, [c_vp, c_int]),
    "gpc_kmap_um_workspace_bytes": (c_sz, [c_i64, c_int]),
    "gpc_kmap_um_count": (c_int, [c_vp, c_i64, c_int, c_vp, c_vp, c_vp, c_sz, c_vp]),
    "gpc_kmap_um_scan": (c_int, [c_vp, c_i64, c_int, c_vp, c_vp, c_vp, c_sz, c_vp]),
    "gpc_kmap_um_fill": (c_int, [c_vp, c_i64, c_int, c_vp, c_vp, c_vp, c_vp]),
    "gpc_spconv_pack_weights_um": (c_int, [c_vp, c_int, c_vp, c_vp]),
    "gpc_spconv_fwd_um": (c_int, [c_vp, c_vp, c_vp, c_vp, c_vp, c_i64, c_int, c_vp, c_vp, c_int, c_vp, c_vp, c_i64, c_i64, c_vp]),
    "gpc_kmap_um_count_range": (c_int, [c_vp, c_i64, c_i64, c_i64, c_int, c_vp, c_vp, c_vp, c_sz, c_vp]),
    "gpc_kmap_um_fill_range": (c_int, [c_vp, c_i64, c_i64, c_i64, c_int, c_vp, c_vp, c_vp, c_vp]),
    "gpc_spconv_fwd_um_range": (c_int, [c_vp, c_vp, c_vp, c_vp, c_vp, c_i64, c_i64, c_i64, c_vp, c_vp, c_int, c_vp, c_vp, c_vp]),
    "gpc_embed_rows": (c_int, [c_vp, c_i64, c_vp, c_vp, c_vp, c_vp]),
    "gpc_gather_parent_add_octant": (c_int, [c_vp, c_vp, c_vp, c_i64, c_vp, c_vp, c_vp, c_vp]),
    "gpc_add_ctx_embed": (c_int, [c_vp, c_vp, c_int, c_vp, c_i64, c_vp, c_vp, c_vp]),
    "gpc_head_cdf": (c_int, [c_vp, c_i64, c_vp, c_vp, c_vp, c_vp, c_int, c_vp, c_vp, c_vp]),
    "gpc_head_cdf_sym": (c_int, [c_vp, c_i64, c_vp, c_vp, c_vp, c_vp, c_int, c_vp, c_int, c_vp, c_vp, c_vp, c_vp]),
    "gpc_split_symbol": (c_int, [c_vp, c_i64, c_int, c_int, c_vp, c_vp]),
    "gpc_merge_symbol": (c_int, [c_vp, c_i64, c_int, c_vp, c_vp]),
    "gpc_ac_encode_h": (c_int, [c_vp, c_vp, c_i64, c_int, c_vp, c_i64, C.POINTER(c_i64)]),
    "gpc_ac_decode_h": (c_int, [c_vp, c_vp, c_i64, c_i64, c_int, c_vp]),
    "gpc_ac_decode_state_bytes": (c_i64, []),
    "gpc_ac_decode_begin_h": (c_int, [c_vp, c_vp, c_i64]),
    "gpc_ac_decode_more_h": (c_int, [c_vp, c_vp, c_i64, c_int, c_vp]),
    "gpc_ac_encode_lohi_h": (c_int, [c_vp, c_i64, c_vp, c_i64, C.POINTER(c_i64)]),
    "gpc_attr_calculate_cdf": (c_int, [c_vp, c_vp, c_vp, c_i64, c_int, c_int, c_vp, c_vp]),
    "gpc_attr_workspace_bytes": (c_sz, [c_i64, c_int]),
    "gpc_attr_encode_table": (c_int, [c_vp, c_vp, c_i64, c_int, c_int, c_vp, c_vp, c_vp, c_sz, c_vp]),
    "gpc_attr_encode_gaussian": (c_int, [c_vp, c_vp, c_vp, c_vp, c_i64, c_int, c_int, c_int, c_vp, c_vp, c_vp, c_sz, c_vp]),
    "gpc_attr_merge_chunks": (c_int, [c_vp, c_i64, c_int, c_vp, c_vp, c_vp]),
    "gpc_attr_decode_table": (c_int, [c_vp, c_vp, c_vp, c_i64, c_int, c_int, c_vp, c_vp, c_sz, c_vp]),
    "gpc_mixture_encode": (c_int, [c_vp, c_vp, c_vp, c_vp, c_vp, c_i64, c_int, c_int, c_int, c_int, c_vp, c_vp, c_vp, c_sz, c_vp]),
    "gpc_mixture_decode": (c_int, [c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_i64, c_int, c_int, c_int, c_int, c_vp, c_vp, c_sz, c_vp]),
    "gpc_row_encode": (c_int, [c_vp, c_vp, c_i64, c_int, c_int, c_vp, c_vp, c_vp, c_sz, c_vp]),
    "gpc_row_decode": (c_int, [c_vp, c_vp, c_vp, c_i64, c_int, c_int, c_vp, c_vp, c_sz, c_vp]),
    "gpc_chunk_workspace_bytes": (c_sz, [c_int, c_int]),
    "gpc_chunk_encode_lohi": (c_int, [c_vp, c_vp, c_int, c_int, c_vp, c_vp, c_vp, c_sz, c_vp]),
    "gpc_chunk_merge": (c_int, [c_vp, c_int, c_int, c_vp, c_vp, c_vp]),
    "gpc_chunk_decode_u16": (c_int, [c_vp, c_vp, c_vp, c_i64, c_int, c_int, c_vp, c_vp]),
    "gpc_chunk_decode_u16_ranges": (c_int, [c_vp, c_int, c_vp, c_vp, c_vp, c_int, c_i64, c_vp, c_vp]),
    "gpc_attr_decode_gaussian": (c_int, [c_vp, c_vp, c_vp, c_vp, c_vp, c_i64, c_int, c_int, c_int, c_vp, c_vp, c_sz, c_vp]),
    "gpc_ply_format_workspace_bytes": (c_sz, [c_i64]),
    "gpc_ply_format_f32": (c_int, [c_vp, c_i64, c_vp, C.c_uint64, C.POINTER(C.c_uint64), c_vp, c_sz, c_vp]),
    "gpc_text_parse_workspace_bytes": (c_sz, [C.c_uint64]),
    "gpc_text_parse_xyz": (c_int, [c_vp, C.c_uint64, c_vp, C.POINTER(C.c_uint32), c_vp, C.POINTER(C.c_uint32), c_vp, c_sz, c_vp]),
}

_lib = None


def load():
    """Load libgpcgc.so; raise if it is not built (python __graft_entry__.py build / make -C gauspcc_b200/csrc)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise GpcError(
            f"{LIB_PATH} is missing: the CUDA library is not built. Run `make -C gauspcc_b200/csrc` "
            "(or `python -c 'import __graft_entry__ as g; g.build()'`). There is no CPU fallback.")
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)           # AttributeError if the library does not export a declared symbol
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def check(rc: int, what: str = ""):
    if rc != 0:
        msg = load().gpc_last_error()
        raise GpcError(f"libgpcgc {what} failed rc={rc}: {msg.decode() if msg else ''}")
