"""ctypes binding of liblvae_b200.so (the C-ABI declared in include/lvae_b200.h).

There is NO fallback: if the shared library is missing or a call fails, a RuntimeError is
raised.  PyTorch is used only for device memory, streams and torch.distributed.
"""
from __future__ import annotations

import ctypes
import os
from ctypes import c_int, c_longlong, c_ulonglong, c_float, c_void_p, c_char_p

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "liblvae_b200.so")

_lib = None

P, I, L, U, F = c_void_p, c_int, c_longlong, c_ulonglong, c_float

# name -> argtypes (every function returns int except the few listed in _SPECIAL)
_SIGNATURES = {
    "lvae_conv2d_gather": [P, P, P, P, P, P, P, P, I, I, I, I, I, I, I, I, I, I, I, I, I, I, I, P],
    "lvae_conv2d_wgrad": [P, P, P, P, P, P, P, I, I, I, I, I, I, I, I, I, I, I, I, I, P],
    "lvae_pack_weights": [P, I, P],
    "lvae_conv2d_tc": [P, P, P, P, P, P, P, P, I, I, I, I, I, I, I, I, I, P],
    "lvae_conv2d_tc_ex": [P, P, P, P, P, P, P, P, I, I, I, I, I, I, I, I, I, P, P],
    "lvae_conv2d_tc_s2": [P, P, P, P, P, I, I, I, I, I, P],
    "lvae_conv_gate_tc": [P, P, P, P, P, P, P, P, P, P, P, I, I, I, I, P],
    "lvae_conv3x3_narrow": [P, P, P, P, I, I, I, I, I, P],
    "lvae_conv3x3_narrow_ex": [P, P, P, P, I, I, I, I, I, I, L, P],
    "lvae_channel_scale": [P, P, P, I, I, I, I, P],
    "lvae_conv2d_wgrad_tc": [P, P, P, P, P, P, I, I, I, I, I, I, I, I, I, P],
    "lvae_conv2d_wgrad_tc_ex": [P, P, P, P, P, P, I, I, I, I, I, I, I, I, I, I, I, P],
    "lvae_conv2d_wgrad_tc_acc": [P, P, P, P, I, I, I, I, I, I, I, P],
    "lvae_conv2d_wgrad_tc_s2_acc": [P, P, P, I, I, I, P],
    "lvae_conv2d_wgrad_tc_s2": [P, P, P, P, P, I, I, I, P],
    "lvae_wgrad_unpack_desc": [P, P, P, P, I, I, I, I, I, I],
    "lvae_wgrad_unpack_batched": [P, I, I, P],
    "lvae_colsum": [P, P, P, I, I, I, I, P],
    "lvae_bn_stats": [P, P, L, I, I, P],
    "lvae_bn_finalize": [P, P, P, P, P, P, L, I, F, F, P],
    "lvae_bn_eval_prepare": [P, P, P, P, I, F, P],
    "lvae_bn_act_fwd": [P, P, P, P, P, P, L, I, I, I, I, P],
    "lvae_bn_act_bwd": [P, P, P, P, P, P, P, P, P, P, L, I, I, I, I, P],
    "lvae_bn_act_fwd2": [P, P, P, P, P, P, P, P, P, L, I, I, I, F, F, I, I, P],
    "lvae_bn_act_bwd2": [P, P, P, P, P, P, P, P, P, P, P, L, I, I, I, I, I, I, P],
    "lvae_bn_act_bwd2_gate": [P, P, P, P, P, P, P, P, P, P, P, P, P, L, I, I, I, I, I, P],
    "lvae_gate_fwd_stats": [P, P, P, P, L, I, I, I, P],
    "lvae_gate_fwd": [P, P, P, L, I, I, I, P],
    "lvae_gate_bwd": [P, P, P, L, I, I, I, P],
    "lvae_upsample2x_fwd": [P, P, I, I, I, I, I, P],
    "lvae_upsample2x_bwd": [P, P, I, I, I, I, I, P],
    "lvae_copy_window": [P, P, I, I, I, I, I, I, I, I, I, I, I, I, I, I, I, I, P],
    "lvae_dropout_masks": [P, L, F, P, U, P],
    "lvae_rng_advance": [P, U, P],
    "lvae_sum_batch": [P, P, I, L, I, P],
    "lvae_stoch_fwd": [P, P, I, P, P, P, U, P, P, I, P, P, P, P, I, I, I, I, I, P, P],
    "lvae_stoch_bwd": [P, P, I, P, P, P, P, P, P, P, P, I, I, I, I, I, P],
    "lvae_stoch_bwd_ex": [P, P, I, P, P, P, P, P, P, P, P, P, P, I, I, I, I, I, P],
    "lvae_kl_bookkeeping": [P, P, I, I, F, P, P, P, P, P],
    "lvae_kl_bookkeeping_bwd": [P, P, P, P, I, I, P, P, P],
    "lvae_bernoulli_fwd": [P, P, P, P, I, I, I, P],
    "lvae_bernoulli_bwd": [P, P, P, P, P, I, I, I, P],
    "lvae_bernoulli_sample": [P, P, I, I, I, P, U, P],
    "lvae_dmol_fwd": [P, P, P, I, I, P],
    "lvae_dmol_bwd": [P, P, P, P, P, I, I, P],
    "lvae_dmol_sample": [P, P, I, I, P, U, P],
    "lvae_adamax_step": [P, P, P, P, L, F, F, F, F, F, P, F, P, P],
    "lvae_adamax_step_l2": [P, P, P, P, L, F, F, F, F, F, P, F, P, P, P, P],
    "lvae_l2_norm": [P, L, P, P, P],
    "lvae_iw_lse_update": [P, P, P, I, I, P],
    "lvae_iw_lse_combine": [P, P, I, I, I, P],
}
_SPECIAL = {
    "lvae_last_error": ([], c_char_p),
    "lvae_abi_version": ([], c_int),
    "lvae_launch_count": ([], c_ulonglong),
    "lvae_reset_launch_count": ([], None),
    "lvae_device_check": ([], c_int),
    "lvae_pack_desc_size": ([], c_int),
    "lvae_set_pdl": ([c_int], None),
    "lvae_conv2d_tc_debug": ([c_void_p], None),
    "lvae_conv_gate_tc_debug": ([c_void_p], None),
    "lvae_get_pdl": ([], c_int),
    "lvae_wgrad_tc_workspace": ([I, I, I, I, I, I], c_longlong),
    "lvae_wgrad_tc_packed_size": ([I, I, I], c_longlong),
    "lvae_conv2d_tc_plan": ([I, I, I, I, I, I, I], c_int),
    "lvae_wgrad_unpack_desc_size": ([], c_int),
    "lvae_stoch_ws_bytes": ([I], c_longlong),
}


class ConvFuse(ctypes.Structure):
    """LvaeConvFuse of include/lvae_b200.h."""
    _fields_ = [("stats_acc", c_void_p), ("bnb_x", c_void_p), ("bnb_save", c_void_p), ("bnb_gamma", c_void_p),
                ("bnb_beta", c_void_p), ("bnb_acc", c_void_p), ("bnb_act", c_int), ("gate_x", c_void_p),
                ("gate_out", c_void_p), ("gate_act", c_int), ("gate_skip_h", c_int), ("fold_gamma", c_void_p),
                ("fold_beta", c_void_p), ("fold_mean", c_void_p), ("fold_var", c_void_p), ("fold_eps", ctypes.c_float),
                ("fold_act", c_int), ("pre_gamma", c_void_p), ("pre_beta", c_void_p), ("pre_mean", c_void_p), ("pre_var", c_void_p),
                ("pre_eps", ctypes.c_float)]


def exported_symbols():
    return sorted(list(_SIGNATURES) + list(_SPECIAL))


def lib():
    """Load the shared library (once).  Raises if it has not been built."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(
                "lvae_b200: %s is missing -- build it with `python ladder-vae-pytorch_b200/build.py` "
                "(there is no CPU or PyTorch fallback)" % LIB_PATH)
        l = ctypes.CDLL(LIB_PATH)
        for name, argtypes in _SIGNATURES.items():
            fn = getattr(l, name)
            fn.argtypes = argtypes
            fn.restype = c_int
        for name, (argtypes, restype) in _SPECIAL.items():
            fn = getattr(l, name)
            fn.argtypes = argtypes
            fn.restype = restype
        if os.environ.get("LVAE_PDL", "1") == "0":
            l.lvae_set_pdl(0)
        _lib = l
    return _lib


def call(name, *args):
    """Invoke a C-ABI entry point; nonzero return -> RuntimeError(lvae_last_error())."""
    l = lib()
    rc = getattr(l, name)(*args)
    if rc != 0:
        raise RuntimeError("%s failed (code %d): %s" % (name, rc, l.lvae_last_error().decode()))


def launch_count() -> int:
    return int(lib().lvae_launch_count())


def reset_launch_count() -> None:
    lib().lvae_reset_launch_count()


def device_check() -> None:
    l = lib()
    rc = l.lvae_device_check()
    if rc != 0:
        raise RuntimeError("lvae_b200: " + l.lvae_last_error().decode())
