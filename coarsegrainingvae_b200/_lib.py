"""ctypes binding of libcgvae_sm100.so (the C ABI declared in include/cgvae_b200.h).

This is the reference-side binding a maintainer would add (INTEGRATION.md): plain pointers and
sizes, no torch types cross the boundary.  There is NO fallback: if the library is missing or no
CUDA device is present the product fails loudly.
"""
import ctypes
import os
import re

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libcgvae_sm100.so")
HEADER_PATH = os.path.join(_HERE, "..", "include", "cgvae_b200.h")

_lib = None

_P = ctypes.c_void_p
_I64 = ctypes.c_int64
_INT = ctypes.c_int
_F32 = ctypes.c_float
_SZ = ctypes.c_size_t

# name -> (restype, argtypes); mirrors include/cgvae_b200.h one to one
SIGNATURES = {
    "cgvae_abi_version": (_INT, []),
    "cgvae_last_error": (ctypes.c_char_p, []),
    "cgvae_launch_count": (ctypes.c_ulonglong, []),
    "cgvae_set_error_flags": (_INT, [_INT, _P]),
    "cgvae_radius_graph_ws_bytes": (_SZ, [_I64, _I64]),
    "cgvae_radius_graph_count": (_INT, [_P, _I64, _P, _I64, _F32, _INT, _INT, _P, _P, _SZ, _P]),
    "cgvae_radius_graph_fill": (_INT, [_P, _I64, _P, _I64, _F32, _INT, _INT, _P, _P, _P, _SZ, _P]),
    "cgvae_exclusive_scan": (_INT, [_P, _I64, _P, _P]),
    "cgvae_edge_orientation": (_INT, [_P, _I64, _P, _P]),
    "cgvae_csr_count": (_INT, [_P, _I64, _P, _INT, _I64, _I64, _P, _P, _P]),
    "cgvae_scan_i32": (_INT, [_P, _I64, _P, _P]),
    "cgvae_csr_fill": (_INT, [_P, _I64, _P, _INT, _I64, _I64, _P, _P, _P, _P, _P, _P, _P, _P]),
    "cgvae_segment_count": (_INT, [_P, _I64, _I64, _P, _P]),
    "cgvae_segment_rank": (_INT, [_P, _I64, _I64, _P, _P, _P, _P, _P, _P]),
    "cgvae_edge_geometry": (_INT, [_P, _P, _P, _P, _P, _I64, _I64, _P, _INT, _INT, _F32, _P, _P, _P, _P, _P]),
    "cgvae_edge_geometry_bwd": (_INT, [_P, _P, _P, _P, _P, _I64, _I64, _P, _INT, _INT, _F32, _P, _P, _P, _P, _P, _P]),
    "cgvae_edge_coord_reduce": (_INT, [_P, _P, _I64, _P, _P, _I64, _INT, _P, _P, _P]),
    "cgvae_gemm": (_INT, [_INT, _P, _I64, _P, _I64, _P, _I64, _I64, _I64, _I64, _P, _INT, _P, _P, _INT, _P, _P, _SZ, _P, _INT, _P]),
    "cgvae_dense_pair_fwd": (_INT, [_P, _I64, _P, _I64, _I64, _I64, _I64, _I64, _P, _P, _P]),
    "cgvae_colsum": (_INT, [_P, _I64, _I64, _I64, _P, _P]),
    "cgvae_wgrad_grouped": (_INT, [_P, _INT, _P]),
    "cgvae_message_fwd": (_INT, [_INT, _P, _P, _P, _P, _P, _P, _P, _P, _P, _I64, _I64, _INT, _INT, _INT, _P, _P, _INT,
                                 _P, _P, _P, _P]),
    "cgvae_message_bwd_ws_bytes": (_SZ, [_INT, _INT, _INT, _I64]),
    "cgvae_message_bwd": (_INT, [_INT, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _I64, _I64, _INT, _INT, _INT, _P, _P,
                                 _INT, _INT, _P, _P, _P, _P, _P, _SZ, _P]),
    "cgvae_message_geom_bwd": (_INT, [_INT, _P, _P, _P, _P, _P, _I64, _I64, _P, _P, _P, _P, _INT, _INT, _INT, _P, _P, _INT, _P,
                                      _P, _P]),
    "cgvae_msg_tiles_batches_cap": (_I64, [_I64, _I64, _I64, _INT]),
    "cgvae_msg_tiles_rec_bytes": (_SZ, []),
    "cgvae_msg_tiles_build": (_INT, [_P, _P, _P, _I64, _I64, _I64, _P, _P, _INT, _INT, _P, _P, _P, _P, _I64, _P]),
    "cgvae_message_tc_ws_bytes": (_SZ, [_INT, _INT, _I64, _INT]),
    "cgvae_message_tc_fwd": (_INT, [_INT, _P, _P, _P, _P, _P, _P, _I64, _INT, _P, _P, _I64, _INT, _INT, _P, _P, _INT, _P, _P, _P,
                                    _P, _SZ, _P]),
    "cgvae_message9_fwd": (_INT, [_P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _I64, _INT, _INT, _INT, _INT, _P, _P, _P, _P, _P]),
    "cgvae_message9_bwd": (_INT, [_P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _I64, _I64, _INT, _INT, _INT, _INT,
                                  _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P]),
    "cgvae_update_norm_fwd": (_INT, [_P, _P, _I64, _INT, _P, _P]),
    "cgvae_update_combine_fwd": (_INT, [_P, _P, _P, _P, _P, _I64, _INT, _INT, _P, _P, _P]),
    "cgvae_update_combine_bwd": (_INT, [_P, _P, _P, _P, _P, _I64, _INT, _P, _P, _P, _P]),
    "cgvae_update_norm_bwd": (_INT, [_P, _P, _P, _P, _I64, _INT, _INT, _P, _P, _P]),
    "cgvae_update_combine_bwd_ld": (_INT, [_P, _P, _P, _P, _P, _I64, _INT, _P, _P, _P, _I64, _P]),
    "cgvae_update_norm_bwd_ld": (_INT, [_P, _P, _P, _P, _I64, _INT, _INT, _P, _P, _I64, _P]),
    "cgvae_segment_reduce_fwd": (_INT, [_P, _P, _P, _I64, _I64, _INT, _P, _P]),
    "cgvae_segment_reduce_bwd": (_INT, [_P, _P, _P, _I64, _I64, _INT, _P, _P]),
    "cgvae_gather_rows": (_INT, [_P, _P, _I64, _I64, _I64, _P, _P]),
    "cgvae_lift_fwd": (_INT, [_P, _P, _P, _P, _P, _P, _P, _I64, _I64, _INT, _INT, _P, _P]),
    "cgvae_lift_bwd": (_INT, [_P, _P, _P, _P, _P, _P, _I64, _I64, _INT, _INT, _P, _P]),
    "cgvae_adam_ws_bytes": (_SZ, []),
    "cgvae_adam_clip_step": (_INT, [_P, _P, _P, _P, _I64, _F32, _F32, _F32, _F32, _F32, _F32, _P, _P, _P, _F32, _F32, _P,
                                    _P, _SZ, _P]),
    "cgvae_bond_graph": (_INT, [_P, _P, _I64, _F32, _P, _P]),
    "cgvae_sample_quality": (_INT, [_P, _P, _P, _P, _I64, _I64, _F32, _P, _P, _P]),
    "cgvae_set_pdl": (_INT, [_INT]),
    "cgvae_set_matmul_precision": (_INT, [_INT]),
    "cgvae_get_matmul_precision": (_INT, []),
    "cgvae_register_const_range": (_INT, [_P, _SZ]),
    "cgvae_grad_sumsq": (_INT, [_P, _I64, _P, _P, _SZ, _P]),
    "cgvae_adam_apply": (_INT, [_P, _P, _P, _P, _I64, _F32, _F32, _F32, _F32, _F32, _F32, _P, _P, _INT, _F32, _F32, _P, _P, _SZ, _P]),
    "cgvae_dihedral_loss_fwd": (_INT, [_P, _P, _P, _I64, _P, _P, _P, _P, _P, _SZ, _P]),
    "cgvae_dihedral_loss_bwd": (_INT, [_P, _P, _P, _P, _I64, _I64, _P, _P, _P, _P]),
    "cgvae_pin_mask": (_INT, [_P, _I64, _P, _I64, _P, _SZ, _P]),
    "cgvae_vae_latent_fwd": (_INT, [_P, _P, _P, _I64, _P, _P, _P]),
    "cgvae_vae_latent_bwd": (_INT, [_P, _P, _P, _P, _I64, _P, _P, _P]),
    "cgvae_std_logvar_fwd": (_INT, [_P, _I64, _F32, _P, _P]),
    "cgvae_std_logvar_bwd": (_INT, [_P, _P, _I64, _F32, _P, _P]),
    "cgvae_loss_ws_bytes": (_SZ, []),
    "cgvae_loss_fwd": (_INT, [_P, _P, _I64, _P, _P, _P, _P, _P, _P, _I64, _INT, _P, _F32, _F32, _P, _P, _SZ, _P]),
    "cgvae_loss_bwd": (_INT, [_P, _P, _P, _I64, _P, _P, _P, _P, _P, _P, _I64, _INT, _P, _F32, _F32, _P, _P, _P, _P, _P, _P]),
    "cgvae_loss_bwd_target": (_INT, [_P, _P, _P, _I64, _P, _P, _P, _F32, _P, _P]),
    "cgvae_fill": (_INT, [_P, _I64, _F32, _P]),
    "cgvae_vec_to_planar": (_INT, [_P, _I64, _INT, _P, _P]),
    "cgvae_vec_from_planar": (_INT, [_P, _I64, _INT, _P, _P]),
    "cgvae_collate_plan_bytes": (_SZ, []),
    "cgvae_collate": (_INT, [_P, _P]),
}


def header_symbols():
    """every function name declared in include/cgvae_b200.h (used by the CPU test-suite)."""
    with open(HEADER_PATH) as fh:
        text = fh.read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(cgvae_[a-z0-9_]+)\s*\(", text)))


def load():
    """dlopen the library and attach prototypes.  Raises if it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(
            "libcgvae_sm100.so not built (%s): run `python -m coarsegrainingvae_b200.build`; "
            "there is no CPU or PyTorch fallback" % LIB_PATH)
    lib = ctypes.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)
        fn.restype = res
        fn.argtypes = args
    if lib.cgvae_abi_version() != 1:
        raise RuntimeError("libcgvae_sm100.so ABI version mismatch")
    _lib = lib
    return lib


def last_error():
    return load().cgvae_last_error().decode("utf-8", "replace")


def launch_count():
    return int(load().cgvae_launch_count())


def check(rc, what):
    if rc != 0:
        raise RuntimeError("%s failed (code %d): %s" % (what, rc, last_error()))
