"""ctypes binding of libgccvae.so (include/gccvae.h).  There is NO fallback: if the library is
missing or fails to load, every op raises."""
from __future__ import annotations

import ctypes as C
import os
import threading

_HERE = os.path.dirname(os.path.abspath(__file__))
# GCCVAE_LIB selects another build of the same library in csrc/ (libgccvae_tl.so: timeline hooks compiled in)
LIB_PATH = os.path.join(_HERE, "csrc", os.environ.get("GCCVAE_LIB", "libgccvae.so"))

ACT_NONE, ACT_RELU, ACT_SIGMOID, ACT_ACCUMULATE = 0, 1, 2, 0x100
OUT_S2D, MASK_S2D, TAP_HALO = 0x10, 0x20, 0x40   # layout flags OR-ed into `act` (include/gccvae.h)
GATE_WS_FLOATS = 7 * 324 + 32
LATENT_PARTIAL_FLOATS = 5 * 324 + 32
RESULT_SLOT_FLOATS = 328


class Geom(C.Structure):
    """gccvae_geom: the L<->S relation of one layer (include/gccvae.h)."""
    _fields_ = [(n, C.c_int) for n in ("batch", "HL", "WL", "CL", "HS", "WS", "CS", "KH", "KW", "stride", "pad")]



class LatentFwdArgs(C.Structure):
    _fields_ = [
        ("batch", C.c_int), ("batch_global", C.c_int), ("supervised", C.c_int), ("K", C.c_int),
        ("loc_pre", C.c_void_p), ("scale_pre", C.c_void_p), ("y", C.c_void_p), ("eps", C.c_void_p),
        ("eps_k", C.c_void_p), ("U_y", C.c_void_p), ("seed", C.c_uint64), ("offset", C.c_uint64),
        ("step_dev", C.c_void_p), ("gate_ws", C.c_void_p), ("ld_pre", C.c_int), ("loc", C.c_void_p),
        ("scale", C.c_void_p), ("z", C.c_void_p),
        ("terms", C.c_void_p), ("logits", C.c_void_p), ("y_out", C.c_void_p), ("z16", C.c_void_p),
    ]


GEN_GENERATE, GEN_RECONSTRUCT, GEN_INTERVENE = 1, 2, 3


class GenLatentArgs(C.Structure):
    """gccvae_gen_latent_args (include/gccvae.h)."""
    _fields_ = [
        ("batch", C.c_int), ("mode", C.c_int), ("sample", C.c_int), ("ld_pre", C.c_int), ("n_labels", C.c_int),
        ("labels", C.c_int * 18), ("n_alpha", C.c_int), ("alphas", C.c_void_p), ("row0", C.c_int), ("rows", C.c_int),
        ("loc_pre", C.c_void_p), ("scale_pre", C.c_void_p), ("y_tgt", C.c_void_p), ("y_src", C.c_void_p),
        ("eps", C.c_void_p), ("seed", C.c_uint64), ("offset", C.c_uint64), ("step_dev", C.c_void_p),
        ("gate_ws", C.c_void_p), ("z", C.c_void_p), ("z16", C.c_void_p), ("y_src_out", C.c_void_p),
        ("n_dims", C.c_int), ("dims", C.c_int * 45), ("pair", C.c_int), ("mix_lo", C.c_int), ("mix_hi", C.c_int),
    ]


class IwLatentArgs(C.Structure):
    """gccvae_iw_latent_args (include/gccvae.h)."""
    _fields_ = [
        ("batch", C.c_int), ("K", C.c_int), ("k0", C.c_int), ("kc", C.c_int), ("labelled", C.c_int), ("ld_pre", C.c_int),
        ("loc_pre", C.c_void_p), ("scale_pre", C.c_void_p), ("y", C.c_void_p), ("eps", C.c_void_p), ("U_y", C.c_void_p),
        ("seed", C.c_uint64), ("offset", C.c_uint64), ("step_dev", C.c_void_p), ("gate_ws", C.c_void_p),
        ("lw_part", C.c_void_p), ("z", C.c_void_p), ("z16", C.c_void_p),
    ]


class LatentBwdArgs(C.Structure):
    _fields_ = [
        ("batch", C.c_int), ("batch_global", C.c_int), ("supervised", C.c_int), ("K", C.c_int),
        ("loc_pre", C.c_void_p), ("scale_pre", C.c_void_p), ("y", C.c_void_p), ("eps", C.c_void_p),
        ("eps_k", C.c_void_p), ("seed", C.c_uint64), ("offset", C.c_uint64), ("step_dev", C.c_void_p),
        ("gate_ws", C.c_void_p),
        ("terms", C.c_void_p), ("log_pxz", C.c_void_p), ("dz", C.c_void_p), ("dloc_pre", C.c_void_p),
        ("dscale_pre", C.c_void_p), ("ld_pre", C.c_int), ("ld_dz", C.c_int), ("dpre16", C.c_void_p),
        ("db_loc", C.c_void_p), ("db_scale", C.c_void_p),
        ("partials", C.c_void_p), ("n_partials", C.c_int), ("loss_out", C.c_void_p),
    ]


class ChainFwdArgs(C.Structure):
    """gccvae_chain_fwd_args (include/gccvae.h)."""
    _fields_ = [
        ("batch", C.c_int), ("batch_global", C.c_int), ("supervised", C.c_int), ("K", C.c_int),
        ("rows_per_cta", C.c_int), ("pad_", C.c_int),
        ("h5", C.c_void_p), ("w_heads", C.c_void_p), ("b_heads", C.c_void_p), ("w_fc1", C.c_void_p),
        ("b_fc1", C.c_void_p), ("w_conv1t", C.c_void_p), ("b_conv1t", C.c_void_p),
        ("y", C.c_void_p), ("eps", C.c_void_p), ("eps_k", C.c_void_p), ("U_y", C.c_void_p),
        ("seed", C.c_uint64), ("offset", C.c_uint64), ("step_dev", C.c_void_p), ("gate_ws", C.c_void_p),
        ("pre", C.c_void_p), ("loc", C.c_void_p), ("scale", C.c_void_p), ("z", C.c_void_p), ("terms", C.c_void_p),
        ("logits", C.c_void_p), ("y_out", C.c_void_p), ("z16", C.c_void_p), ("g0", C.c_void_p), ("g1", C.c_void_p),
    ]


class ChainBwdArgs(C.Structure):
    """gccvae_chain_bwd_args (include/gccvae.h)."""
    _fields_ = [
        ("batch", C.c_int), ("batch_global", C.c_int), ("supervised", C.c_int), ("K", C.c_int),
        ("rows_per_cta", C.c_int), ("n_partials", C.c_int),
        ("dg1", C.c_void_p), ("g0", C.c_void_p), ("h5", C.c_void_p), ("pre", C.c_void_p), ("y", C.c_void_p),
        ("eps", C.c_void_p), ("eps_k", C.c_void_p), ("seed", C.c_uint64), ("offset", C.c_uint64),
        ("step_dev", C.c_void_p), ("gate_ws", C.c_void_p), ("terms", C.c_void_p), ("log_pxz", C.c_void_p),
        ("w_conv1t_t", C.c_void_p), ("w_fc1_t", C.c_void_p), ("w_heads_t", C.c_void_p),
        ("dg0", C.c_void_p), ("dpre16", C.c_void_p), ("dh5", C.c_void_p), ("partials", C.c_void_p),
        ("db_loc", C.c_void_p), ("db_scale", C.c_void_p), ("db_fc1", C.c_void_p), ("db_conv1t", C.c_void_p),
        ("db_conv5", C.c_void_p),
    ]


DP_MAX_RANKS, DP_SYNC_WORDS = 16, 32


class DpArgs(C.Structure):
    """gccvae_dp_args (include/gccvae.h)."""
    _fields_ = [
        ("world", C.c_int), ("rank", C.c_int), ("grad", C.c_void_p * DP_MAX_RANKS), ("sync", C.c_void_p * DP_MAX_RANKS),
        ("param", C.c_void_p), ("m", C.c_void_p), ("v", C.c_void_p), ("i0", C.c_longlong), ("n", C.c_longlong),
        ("n_zero", C.c_longlong), ("loss_index", C.c_longlong), ("lr", C.c_float), ("beta1", C.c_float),
        ("beta2", C.c_float), ("eps", C.c_float), ("step_state", C.c_void_p), ("publish", C.c_int),
        ("ring_slots", C.c_int), ("result_loss", C.c_void_p), ("result_c", C.c_void_p), ("result_ring", C.c_void_p),
        ("push", C.c_int), ("pad_", C.c_int), ("recv_stride", C.c_longlong), ("recv", C.c_void_p * DP_MAX_RANKS),
    ]


class PackJob(C.Structure):
    _fields_ = [("kind", C.c_int), ("taps", C.c_int), ("CL", C.c_int), ("CS", C.c_int), ("W", C.c_void_p),
                ("out", C.c_void_p), ("sr", C.c_int), ("sk", C.c_int), ("ld_out", C.c_int), ("row_off", C.c_int),
                ("col_off", C.c_int), ("pad_", C.c_int)]


class WgSeg(C.Structure):
    _fields_ = [("col0", C.c_int), ("ncols", C.c_int), ("ld", C.c_int), ("pad_", C.c_int), ("dst", C.c_void_p)]


class WgOut(C.Structure):
    _fields_ = [("n_seg", C.c_int), ("m_valid", C.c_int), ("seg", WgSeg * 2)]


_P, _I, _F, _LL, _SZ, _U64 = C.c_void_p, C.c_int, C.c_float, C.c_longlong, C.c_size_t, C.c_uint64
_G = C.POINTER(Geom)

# name -> (restype, argtypes); mirrors include/gccvae.h one to one
SIGNATURES = {
    "gccvae_abi_version": (_I, []),
    "gccvae_last_error": (C.c_char_p, []),
    "gccvae_arch_check": (_I, [_I]),
    "gccvae_launch_count": (_LL, []),
    "gccvae_reset_launch_count": (None, []),
    "gccvae_add_launch_count": (None, [_LL]),
    "gccvae_ls_f32": (_I, [_G, _P, _P, _P, _I, _P, _P, _P]),
    "gccvae_sl_f32": (_I, [_G, _P, _P, _P, _I, _P, _P, _P]),
    "gccvae_wg_f32_workspace_bytes": (_SZ, [_G]),
    "gccvae_wg_f32": (_I, [_G, _P, _P, _P, _P, _SZ, _P]),
    "gccvae_colsum_f32_workspace_bytes": (_SZ, [_LL, _I]),
    "gccvae_colsum_f32": (_I, [_P, _LL, _I, _P, _P, _SZ, _P]),
    "gccvae_packed_weight_elems": (_SZ, [_G, _I]),
    "gccvae_pack_jobs_bf16": (_I, [C.POINTER(PackJob), _I, _P]),
    "gccvae_pack_weights_bf16": (_I, [_G, _P, _P, _P, _P]),
    "gccvae_ls_bf16": (_I, [_G, _P, _P, _P, _I, _P, _P, _I, _P]),
    "gccvae_sl_bf16": (_I, [_G, _P, _P, _P, _I, _P, _P, _I, _P]),
    "gccvae_wg_bf16": (_I, [_G, _P, _P, _P, _P]),
    "gccvae_colsum_bf16": (_I, [_P, _LL, _I, _I, _P, _P]),
    "gccvae_gemm_bf16": (_I, [_LL, _I, _I, _P, _P, _P, _I, _I, _I, _P, _P, _I, _P]),
    "gccvae_gemm_tn_bf16": (_I, [_LL, _I, _I, _P, _P, C.POINTER(WgOut), _P]),
    "gccvae_sl_halo_supported": (_I, [_G]),
    "gccvae_sl_halo_bf16": (_I, [_G, _P, _P, _P, _I, _P, _P, _I, _P]),
    "gccvae_cast_f32_to_bf16": (_I, [_P, _LL, _P, _P]),
    "gccvae_cast_bf16_to_f32": (_I, [_P, _LL, _P, _P]),
    "gccvae_prep_x2_bf16": (_I, [_P, _I, _I, _P, _P, _P]),
    "gccvae_tap4_ls_bf16": (_I, [_I, _I, _I, _I, _P, _P, _I, _P, _I, _P, _P, _P]),
    "gccvae_c3conv_bf16": (_I, [_I, _P, _P, _I, _P, _I, _P, _P, _P]),
    "gccvae_wg_s2d_bf16": (_I, [_I, _I, _I, _I, _P, _P, _I, _P, _P]),
    "gccvae_tap4_wg_bf16": (_I, [_I, _P, _P, _I, _P, _P, _P]),
    "gccvae_convt_recon_bf16": (_I, [_I, _P, _P, _P, _P, _I, _P, _P, _P, _P, _P, _I, _P]),
    "gccvae_convt_image_bf16": (_I, [_I, _P, _P, _P, _P, _I, _P]),
    "gccvae_convt_complete_bf16": (_I, [_I, _P, _P, _P, _P, _P, _P]),
    "gccvae_convt_ll_bf16": (_I, [_I, _I, _P, _P, _P, _P, _I, _P, _P]),
    "gccvae_fill_f32": (_I, [_P, _LL, _F, _P]),
    "gccvae_gate_fwd": (_I, [_P, _P, _P, _P, _U64, _U64, _P, _F, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P]),
    "gccvae_latent_fwd": (_I, [C.POINTER(LatentFwdArgs), _P]),
    "gccvae_latent_bwd_partials": (_I, [_I]),
    "gccvae_gen_latent": (_I, [C.POINTER(GenLatentArgs), _P]),
    "gccvae_iw_latent": (_I, [C.POINTER(IwLatentArgs), _P]),
    "gccvae_iw_accumulate": (_I, [_I, _I, _I, _I, _P, _P, _P, _P, _I, _I, _P, _P, _P]),
    "gccvae_latent_bwd": (_I, [C.POINTER(LatentBwdArgs), _P]),
    "gccvae_chain_rows": (_I, [_I]),
    "gccvae_chain_partials": (_I, [_I]),
    "gccvae_chain_fwd": (_I, [C.POINTER(ChainFwdArgs), _P]),
    "gccvae_chain_bwd": (_I, [C.POINTER(ChainBwdArgs), _P]),
    "gccvae_gate_bwd": (_I, [_P, _I, _P, _P, _P, _P, _P, _P, _P, _F, _F, _P, _P, _P, _P, _P, _P, _P, _P, _P]),
    "gccvae_recon_f32": (_I, [_P, _P, _I, _I, _P, _P, _P, _P]),
    "gccvae_adam_f32": (_I, [_P, _P, _P, _P, _LL, _F, _F, _F, _F, _I, _P, _P]),
    "gccvae_adam_fused_f32": (_I, [_P, _P, _P, _P, _LL, _LL, _LL, _F, _F, _F, _F, _P, _I, _P, _P, _P, _I, _P]),
    "gccvae_dp_reduce_adam_f32": (_I, [C.POINTER(DpArgs), _P]),
    "gccvae_elbo_loss_f32": (_I, [_P, _P, _I, _I, _I, _P, _F, _P, _P]),
    "gccvae_draw_noise_f32": (_I, [_I, _U64, _U64, _I, _I, _P, _P]),
    "gccvae_head_act_f32": (_I, [_P, _P, _LL, _P, _P, _P]),
    "gccvae_accuracy_f32": (_I, [_P, _P, _I, _P, _P]),
    "gccvae_classifier_tiled_f32": (_I, [_P, _LL, _LL, _LL, _I, _P, _P, _P, _P, _P]),
    "gccvae_cond_prior_tiled_f32": (_I, [_P, _LL, _LL, _LL, _I, _P, _P, _P, _P, _P, _P, _P, _P]),
    "gccvae_gaussian_kl_f32": (_I, [_P, _P, _P, _P, _I, _I, _P, _P]),
}


# development aids (include/gccvae_debug.h): not part of the drop-in boundary
DEBUG_SIGNATURES = {
    "gccvae_debug_set_timeline": (None, [_P]),
    "gccvae_debug_mark": (_I, [_P, _I, _P]),
    "gccvae_debug_tma4d": (_I, [_P] + [_I] * 13 + [_P, _I, _P]),
}


class GccvaeError(RuntimeError):
    pass


_lock = threading.Lock()
_lib = None


def load():
    """Load (once) and return the ctypes library.  Raises GccvaeError if it is not built."""
    global _lib
    with _lock:
        if _lib is not None:
            return _lib
        if not os.path.exists(LIB_PATH):
            raise GccvaeError(
                "libgccvae.so is not built ({}).  Run `python __graft_entry__.py build` (needs nvcc). "
                "There is no CPU or PyTorch fallback for the Gated-CCVAE kernels.".format(LIB_PATH))
        # the library links the CUDA runtime dynamically (libcudart.so.12): import torch first, so that the loader
        # binds it to the runtime torch has already mapped instead of bringing a second one into the process
        import torch  # noqa: F401
        lib = C.CDLL(LIB_PATH)
        for name, (res, args) in list(SIGNATURES.items()) + list(DEBUG_SIGNATURES.items()):
            try:
                fn = getattr(lib, name)
            except AttributeError as e:
                raise GccvaeError("libgccvae.so does not export {} (stale build?)".format(name)) from e
            fn.restype = res
            fn.argtypes = args
        if lib.gccvae_abi_version() != 1:
            raise GccvaeError("libgccvae.so ABI version mismatch")
        _lib = lib
        return lib


def check(rc: int, what: str = ""):
    if rc != 0:
        msg = load().gccvae_last_error()
        raise GccvaeError("{} failed (status {}): {}".format(what or "gccvae call", rc, (msg or b"").decode()))


def ptr(t):
    """Device pointer of a torch tensor (None -> NULL)."""
    return None if t is None else t.data_ptr()
