"""ctypes binding of ``libscann_b200.so`` (declared in ``include/scann_b200.h``).

There is no CPU fallback: importing this module without the built library, or calling a
compute entry point without a CUDA device, raises.  Build with ``python -m scann_b200.build``
(or ``__graft_entry__.build()``).
"""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
# (development: SCANN_B200_LIB selects another build of the same library, e.g. an A/B variant)
LIB_PATH = os.environ.get("SCANN_B200_LIB") or os.path.join(_HERE, "libscann_b200.so")

vp = C.c_void_p
ci = C.c_int

# name -> (restype, argtypes).  Mirrors include/scann_b200.h exactly; tests/test_abi.py checks
# that every symbol declared in the header is exported and listed here.
PROTOTYPES = {
    "scann_last_error": (C.c_char_p, []),
    "scann_version": (ci, []),
    "scann_device_sm_count": (ci, []),
    "scann_device_cc": (ci, []),
    "scann_set_pdl": (ci, [ci]),
    "scann_set_la_groups4": (ci, [ci]),
    "scann_plan_build": (ci, [vp, vp, vp, vp, ci, ci, ci, ci, ci, ci] + [vp] * 13 + [vp, ci, vp, vp]),
    "scann_pack_batch": (ci, [vp] + [C.c_longlong] * 8 + [ci, ci, ci] + [vp] * 8 + [vp]),
    "scann_embed_forward": (ci, [vp, vp, ci, ci, ci] + [vp] * 7 + [vp, vp, vp, vp]),
    "scann_cgcnn_embed_forward": (ci, [vp, vp, vp, ci, ci, ci, vp, vp]),
    "scann_cgcnn_embed_backward": (ci, [vp, vp, vp, ci, ci, ci] + [vp] * 12 + [vp, vp]),
    "scann_embed_backward": (ci, [vp, vp, ci, ci, ci] + [vp] * 12 + [vp, vp]),
    "scann_geom_init_forward": (ci, [vp, ci, ci] + [vp] * 10 + [vp]),
    "scann_geom_init_backward": (ci, [vp, ci, ci] + [vp] * 14 + [vp]),
    "scann_dense_forward": (ci, [vp, ci, vp, vp, ci, ci, ci, vp, ci, ci, vp, ci, vp, vp, vp, vp, vp]),
    "scann_dense_forward_tc": (ci, [vp, ci, vp, vp, ci, ci, ci, vp, ci, ci, vp, ci, vp, vp, vp, vp, vp]),
    "scann_dense_chain": (ci, [vp, ci, ci, vp]),
    "scann_dense_chain2": (ci, [vp, ci, ci, vp, vp]),
    "scann_dense_chain2_max_rows": (ci, []),
    "scann_weight_images": (ci, [vp, vp, ci, vp, vp]),
    "scann_dense_wgrad": (ci, [vp, ci, vp, ci, ci, ci, ci, vp, vp, vp]),
    "scann_layernorm_backward": (ci, [vp, vp, vp, ci, vp, vp, ci, vp, vp, vp]),
    "scann_la_nopair_forward": (ci, [vp, vp, ci, vp, vp, vp, vp, vp]),
    "scann_transpose_blocks": (ci, [vp, vp, vp, ci, vp]),
    "scann_la_forward": (ci, [ci] + [vp] * 21 + [vp]),
    "scann_la_forward_tc": (ci, [ci, ci, ci] + [vp] * 23 + [vp, ci, vp]),
    "scann_la_forward_noupdate_tc": (ci, [ci, ci, ci] + [vp] * 23 + [vp, ci, vp]),
    "scann_la_forward_pipe": (ci, [ci, C.c_longlong, ci] + [vp] * 19 + [vp, ci, vp, vp]),
    "scann_la_backward_noupdate_tc": (ci, [ci, ci, ci] + [vp] * 17 + [vp, ci, vp]),
    "scann_noupdate_geom_forward": (ci, [vp, ci, ci] + [vp] * 7 + [vp]),
    "scann_noupdate_geom_backward": (ci, [vp, ci, ci] + [vp] * 9 + [vp]),
    "scann_la_backward": (ci, [ci] + [vp] * 28 + [vp]),
    "scann_la_backward_tc": (ci, [ci, ci, ci] + [vp] * 18 + [ci] + [vp] * 9 + [vp, ci, vp]),
    "scann_la_backward_tc_part": (ci, [ci, ci, ci, ci] + [vp] * 18 + [ci] + [vp] * 9 + [vp, ci, vp]),
    "scann_la_backward_pipe": (ci, [ci, C.c_longlong, ci] + [vp] * 14 + [ci] + [vp] * 8 + [vp, ci, vp, vp]),
    "scann_la_wgrad_tc": (ci, [ci, ci] + [vp] * 9 + [vp]),
    "scann_wgrad_batch_tc": (ci, [ci, vp, ci, vp, ci, vp, vp, vp, vp, vp, vp]),
    "scann_la_wpart_reduce": (ci, [vp, vp, ci, ci, vp, vp, vp]),
    "scann_ga_head_forward": (ci, [vp, vp, ci, ci, ci, vp, vp, vp, vp, ci, vp, vp, vp, vp, vp]),
    "scann_ga_head_backward": (ci, [vp, vp, ci, ci, ci, vp, vp, vp, vp, vp, vp, vp, vp, vp]),
    "scann_rmse_prepare": (ci, [vp, vp, ci, vp, vp, vp]),
    "scann_adam_step": (ci, [vp, vp, vp, vp, vp, ci, vp, vp, vp, ci, vp]),
    "scann_loss_value": (ci, [vp, vp, ci, vp, C.c_float, C.c_float, vp, vp]),
    "scann_voronoi_neighbors": (ci, [vp] * 6 + [ci, ci, ci, vp, vp, vp, vp, vp, vp]),
    "scann_allreduce_unique_id": (ci, [vp]),
    "scann_allreduce_init": (ci, [vp, ci, ci]),
    "scann_allreduce_sum": (ci, [vp, C.c_longlong, vp]),
    "scann_allreduce_world": (ci, []),
    "scann_allreduce_destroy": (ci, []),
    "scann_p2p_alloc": (ci, [C.c_longlong, C.POINTER(vp)]),
    "scann_p2p_free": (ci, [vp]),
    "scann_p2p_export": (ci, [vp, vp]),
    "scann_p2p_import": (ci, [vp, C.POINTER(vp)]),
    "scann_p2p_close": (ci, [vp]),
    "scann_p2p_begin_step": (ci, [vp, vp, vp]),
    "scann_adam_p2p_step": (ci, [vp, vp, vp, vp, ci, vp, vp, vp, vp, ci, vp]),
}

# development probes: exported only by builds with -DSCANN_DEV_PROBES (bound when present)
DEV_PROTOTYPES = {
    "scann_tc_probe": (ci, [vp, vp, vp, ci, ci, vp]),
    "scann_tc_time": (ci, [vp, ci, ci, ci, vp]),
    "scann_debug_clocks": (ci, [vp]),
    "scann_debug_clocks_dense": (ci, [vp]),
    "scann_debug_clocks_chain": (ci, [vp]),
    "scann_debug_clocks_chain2": (ci, [vp]),
    "scann_pipe_clocks": (ci, [vp]),
    "scann_pipe_clocks_bwd": (ci, [vp]),
}


class ChainStep(C.Structure):
    """``ScannChainStep`` of include/scann_b200.h (one step of ``scann_dense_chain``)."""
    _fields_ = ([("A", vp * 3), ("W", vp * 3)] +
                [(n, vp) for n in ("bias", "resid", "pre_in", "pre_out", "gamma", "beta", "dgamma", "dbeta", "C", "C2",
                                   "cnt", "np_ctx", "np_out", "drop")] +
                [(n, ci) for n in ("lda", "ldres", "ldpre", "ldc", "ldc2", "kblk", "mode", "to_image", "drop_site", "pad")])


def chain_step(A=(), W=(), bias=0, resid=0, ldres=128, pre_in=0, pre_out=0, ldpre=128, gamma=0, beta=0, dgamma=0,
               dbeta=0, C_=0, ldc=128, C2=0, ldc2=128, cnt=0, np_ctx=0, np_out=0, lda=128, mode=0, to_image=False,
               drop=0, drop_site=0):
    """Builds one ChainStep from integer device addresses (0 = NULL).  ``A`` empty: the operand is the image
    left in shared memory by the previous step."""
    st = ChainStep()
    for i, p in enumerate(A):
        st.A[i] = p or None
    for i, p in enumerate(W):
        st.W[i] = p or None
    st.kblk = len(W)
    for name, val in (("bias", bias), ("resid", resid), ("pre_in", pre_in), ("pre_out", pre_out), ("gamma", gamma),
                      ("beta", beta), ("dgamma", dgamma), ("dbeta", dbeta), ("C", C_), ("C2", C2), ("cnt", cnt),
                      ("np_ctx", np_ctx), ("np_out", np_out), ("drop", drop)):
        setattr(st, name, val or None)
    st.lda, st.ldres, st.ldpre, st.ldc, st.ldc2 = lda, ldres, ldpre, ldc, ldc2
    st.mode, st.to_image, st.drop_site, st.pad = mode, 1 if to_image else 0, drop_site, 0
    return st


class WgradProblem(C.Structure):
    """``ScannWgradProblem`` of include/scann_b200.h (one dW += X^T Y problem of ``scann_wgrad_batch_tc``)."""
    _fields_ = [("X", vp), ("Y", vp), ("xg", vp), ("dW", vp), ("db", vp), ("ldx", ci), ("ldy", ci), ("rows", ci),
                ("pad", ci)]


class ScannAbiError(RuntimeError):
    pass


def _load():
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            f"{LIB_PATH} is missing: the sm_100a extension has not been built "
            "(run `python -m scann_b200.build`). There is no CPU fallback.")
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in PROTOTYPES.items():
        fn = getattr(lib, name)
        fn.restype = res
        fn.argtypes = args
    for name, (res, args) in DEV_PROTOTYPES.items():
        if hasattr(lib, name):
            fn = getattr(lib, name)
            fn.restype = res
            fn.argtypes = args
    return lib


lib = _load()


def last_error() -> str:
    return lib.scann_last_error().decode()


def check(status: int, what: str = "") -> None:
    if status != 0:
        raise ScannAbiError(f"{what or 'scann'} failed (status {status}): {last_error()}")


def require_gpu() -> int:
    """Number of SMs of the current device; raises when no CUDA device is usable."""
    sms = lib.scann_device_sm_count()
    if sms <= 0:
        raise ScannAbiError("scann_b200 needs a CUDA device (sm_100a); no CPU fallback exists: " + last_error())
    return sms


def ptr_array(ptrs):
    """A C array of pointers (``const float* const*``) from ints / None."""
    arr = (vp * len(ptrs))()
    for i, p in enumerate(ptrs):
        arr[i] = p if p else None
    return arr
