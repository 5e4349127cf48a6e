"""ctypes binding of libb200seg.so (the C ABI declared in include/b200seg.h).

The library is built in-tree by ``__graft_entry__.build()`` / ``make -C csrc`` and loaded from ``b200seg/lib``.
There is deliberately no fallback: if the shared object is missing, using a kernel-backed op raises.
"""
import ctypes
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
# B200SEG_LIB_VARIANT=<tag> loads lib/libb200seg_<tag>.so (A/B of compile-time switches, csrc/Makefile); default: the product
_VARIANT = os.environ.get("B200SEG_LIB_VARIANT", "")
LIB_PATH = os.path.join(_HERE, "lib", "libb200seg%s.so" % (("_" + _VARIANT) if _VARIANT else ""))

c_int32 = ctypes.c_int32
c_int64 = ctypes.c_int64
c_float = ctypes.c_float
c_void_p = ctypes.c_void_p
c_size_t = ctypes.c_size_t
P32 = ctypes.POINTER(c_int32)


class ConvDesc(ctypes.Structure):
    _fields_ = [(n, c_int32) for n in (
        "n", "h", "w", "cin", "cout", "ksize", "stride", "pad", "x_ld", "y_ld",
        "out_fp32", "has_bias", "emit_stats", "reserved", "dilation")]


class FuseTerm(ctypes.Structure):
    _fields_ = [("x", c_void_p), ("scale", c_void_p), ("shift", c_void_p),
                ("ld", c_int32), ("h", c_int32), ("w", c_int32), ("reserved", c_int32)]


class FuseDesc(ctypes.Structure):
    _fields_ = [("term", FuseTerm * 4), ("nterms", c_int32), ("n", c_int32), ("h", c_int32), ("w", c_int32),
                ("c", c_int32), ("relu", c_int32), ("reserved", c_int32 * 2)]


class MscaleDesc(ctypes.Structure):
    _fields_ = [("n", c_int32), ("h", c_int32), ("w", c_int32), ("hq", c_int32), ("wq", c_int32),
                ("hm", c_int32), ("wm", c_int32), ("hl", c_int32), ("wl", c_int32), ("nheads", c_int32),
                ("w_head0", c_float), ("w_head1", c_float), ("sup_wt", c_float), ("ignore_index", c_int32),
                ("loss_kind", c_int32), ("reserved", c_int32)]


class BnSync(ctypes.Structure):
    _fields_ = [("mail_peers", c_void_p), ("flag_peers", c_void_p), ("step", c_void_p), ("mail_offset", c_int64),
                ("parity_stride", c_int64), ("flag_offset", c_int32), ("world", c_int32), ("rank", c_int32),
                ("reserved", c_int32), ("beacon", c_void_p)]


class BnFold(ctypes.Structure):
    _fields_ = [("accum", c_void_p), ("counter", c_void_p), ("gamma", c_void_p), ("beta", c_void_p),
                ("scale", c_void_p), ("shift", c_void_p), ("mean", c_void_p), ("invstd", c_void_p),
                ("batch_stats_out", c_void_p), ("running_mean", c_void_p), ("running_var", c_void_p),
                ("num_batches_tracked", c_void_p), ("eps", c_float), ("momentum", c_float), ("count", c_float),
                ("c", c_int32)]


class AugGeom(ctypes.Structure):
    _fields_ = [(n, c_int32) for n in ("src_h", "src_w", "out_h", "out_w", "win_y0", "win_x0", "n_y", "n_x", "ksize_v",
                                       "ksize_h", "flip", "ignore_label")]


class AugColor(ctypes.Structure):
    _fields_ = [("n_ops", c_int32), ("kind", c_int32 * 4), ("factor", c_float * 4), ("hue_shift", c_int32 * 4),
                ("mean", c_float * 3), ("std", c_float * 3)]


class ProbeOperand(ctypes.Structure):
    _fields_ = [(n, c_int32) for n in (
        "rows", "cols", "box_cols", "box_rows", "nboxes", "c0", "r0", "dcol", "drow", "smem_stride",
        "swizzle_bytes")]


class ProbeDesc(ctypes.Structure):
    _fields_ = [("a", ProbeOperand), ("b", ProbeOperand)] + [(n, c_int32) for n in (
        "M", "N", "ksteps",
        "a_off", "a_lbo", "a_sbo", "a_layout", "a_base", "a_major", "a_kstep",
        "b_off", "b_lbo", "b_sbo", "b_layout", "b_base", "b_major", "b_kstep")]


# name -> (restype, argtypes). Must list every symbol include/b200seg.h declares (tests/test_abi.py checks this).
V, I32, I64, F = c_void_p, c_int32, c_int64, c_float
SIGNATURES = {
    "b200seg_abi_version": (ctypes.c_int, []),
    "b200seg_build_info": (ctypes.c_char_p, []),
    "b200seg_conv2d_stats_elems": (c_size_t, [ctypes.POINTER(ConvDesc)]),
    "b200seg_conv2d_plan_info": (c_int32, [ctypes.POINTER(ConvDesc), c_int32, P32]),
    "b200seg_debug_occupancy": (c_int32, [c_int32, c_int32, c_int32]),
    "b200seg_debug_occupancy_report": (None, []),
    "b200seg_conv2d_fwd": (ctypes.c_int, [ctypes.POINTER(ConvDesc), V, V, V, V, V, P32, V]),
    "b200seg_set_smem_reserve": (ctypes.c_int, [I32]),
    "b200seg_conv2d_fwd_bn": (ctypes.c_int, [ctypes.POINTER(ConvDesc), V, V, V, V, ctypes.POINTER(BnFold), V]),
    "b200seg_conv2d_fwd_add": (ctypes.c_int, [ctypes.POINTER(ConvDesc), V, V, V, V, I32, V, V, P32, V]),
    "b200seg_conv2d_fwd_affine": (ctypes.c_int, [ctypes.POINTER(ConvDesc), V, V, V, V, I32, V, I32, V, V]),
    "b200seg_pack_weight": (ctypes.c_int, [V, I32, I32, I32, V, V, I32, V]),
    "b200seg_pack_chunk": (I32, []),
    "b200seg_pack_weights": (ctypes.c_int, [V, V, V, I32, I32, V]),
    "b200seg_conv2d_dgrad": (ctypes.c_int, [ctypes.POINTER(ConvDesc), V, I32, V, V, I32, V, I32, V]),
    "b200seg_conv2d_wgrad_ws_bytes": (c_size_t, [ctypes.POINTER(ConvDesc)]),
    "b200seg_conv2d_wgrad_launches": (I32, [ctypes.POINTER(ConvDesc)]),
    "b200seg_conv2d_wgrad": (ctypes.c_int, [ctypes.POINTER(ConvDesc), V, V, I32, V, V, c_size_t, V]),
    "b200seg_grad_fold_chunk": (I32, []),
    "b200seg_grad_fold": (ctypes.c_int, [V, V, V, V, V, V, I32, I32, V]),
    "b200seg_bn_finalize": (ctypes.c_int, [V, I32, I32, I32, F, V, V, F, F, V, V, V, V, V, V, V, V,
                                           ctypes.POINTER(BnSync), V]),
    "b200seg_p2p_alloc": (ctypes.c_int, [c_size_t, ctypes.POINTER(c_void_p), ctypes.POINTER(ctypes.c_uint8)]),
    "b200seg_p2p_open": (ctypes.c_int, [ctypes.POINTER(ctypes.c_uint8), ctypes.POINTER(c_void_p)]),
    "b200seg_p2p_close": (ctypes.c_int, [V]),
    "b200seg_p2p_free": (ctypes.c_int, [V]),
    "b200seg_bn_running_update": (ctypes.c_int, [V, V, V, I64, F, V, I32, I32, V]),
    "b200seg_accum_f32": (ctypes.c_int, [V, V, I64, V]),
    "b200seg_publish_grads": (ctypes.c_int, [V, V, I64, V, F, I32, V]),
    "b200seg_sgd_chunk": (I32, []),
    "b200seg_sgd_step": (ctypes.c_int, [V, V, V, I32, F, F, F, F, I32, I32, V]),
    "b200seg_bn_eval_params": (ctypes.c_int, [I32, V, V, F, V, V, V, V, V]),
    "b200seg_bn_apply": (ctypes.c_int, [V, I32, V, V, V, I32, V, I32, V, I32, I64, I32, I32, V]),
    "b200seg_bn_apply_cells": (ctypes.c_int, [V, I32, ctypes.POINTER(BnFold), V, I32, V, I32, V, I32, I64, I32, I32, V]),
    "b200seg_bn_bwd_grid": (I32, [I64, I32]),
    "b200seg_bn_bwd_reduce": (ctypes.c_int, [V, I32, V, I32, V, V, I32, V, V, I64, I32, I32, V, V]),
    "b200seg_bn_bwd_finalize": (ctypes.c_int, [V, I32, I32, F, V, V, V, V, ctypes.POINTER(BnSync), V]),
    "b200seg_bn_bwd_reduce_finalize": (ctypes.c_int, [V, I32, V, I32, V, V, I32, V, V, I64, I32, I32, V, V, V, V, V, V,
                                                      V]),
    "b200seg_bn_bwd_apply": (ctypes.c_int, [V, I32, V, I32, V, V, I32, V, V, V, V, V, V, I32, V, I32, I32, I64, I32,
                                            I32, V]),
    "b200seg_bn_bwd_cells": (ctypes.c_int, [V, I32, V, I32, V, V, I32, V, V, V, V, V, V, V, I32, V, I32, I32, I64, I32,
                                            I32, V]),
    "b200seg_masked_accum": (ctypes.c_int, [V, I32, V, I32, V, I32, I32, I64, I32, V]),
    "b200seg_fuse_fwd": (ctypes.c_int, [ctypes.POINTER(FuseDesc), V, I32, V]),
    "b200seg_upsample_adjoint": (ctypes.c_int, [V, I32, V, I32, I32, I32, I32, I32, V, I32, I32, I32, I32, V]),
    "b200seg_image_prep": (ctypes.c_int, [V, I32, I32, I32, V, I32, I32, V]),
    "b200seg_spatial_softmax_blocks": (I32, [I32]),
    "b200seg_spatial_softmax_fwd": (ctypes.c_int, [V, I32, I32, I32, I32, V, V, V, V]),
    "b200seg_spatial_softmax_bwd": (ctypes.c_int, [V, I32, V, I32, I32, I32, V, V, I32, V]),
    "b200seg_class_softmax_fwd": (ctypes.c_int, [V, I32, I64, I32, F, V, V]),
    "b200seg_class_softmax_bwd": (ctypes.c_int, [V, I32, V, I64, I32, F, V, V]),
    "b200seg_transpose_pad": (ctypes.c_int, [V, I32, I32, I32, I32, V, I32, V]),
    "b200seg_cast_rows": (ctypes.c_int, [V, I32, V, I32, I64, I32, I32, V]),
    "b200seg_bias_grad_blocks": (I32, [I64]),
    "b200seg_bias_grad": (ctypes.c_int, [V, I32, I64, I32, V, V, V]),
    "b200seg_count_valid": (ctypes.c_int, [V, I64, I32, I32, V, V, V]),
    "b200seg_rmi_pool": (ctypes.c_int, [ctypes.POINTER(MscaleDesc), V, V, V, V, V, V]),
    "b200seg_rmi_ws_bytes": (c_size_t, [I32]),
    "b200seg_rmi_solve_grad": (ctypes.c_int, [I32, I32, I32, V, V, F, V, c_size_t, V, V, V, V]),
    "b200seg_mscale_mid_fwd": (ctypes.c_int, [ctypes.POINTER(MscaleDesc), V, V, V, V, V, V]),
    "b200seg_mscale_loss_blocks": (I32, [ctypes.POINTER(MscaleDesc)]),
    "b200seg_mscale_loss_fwd": (ctypes.c_int, [ctypes.POINTER(MscaleDesc), V, V, V, V, V, V, V, V, V, V, V, V, V, I32,
                                               V]),
    "b200seg_mscale_hi_bwd": (ctypes.c_int, [ctypes.POINTER(MscaleDesc), V, V, V, V]),
    "b200seg_mscale_lo_bwd": (ctypes.c_int, [ctypes.POINTER(MscaleDesc), V, V, V, V, V, V, V, V, V, V, V]),
    "b200seg_resize_to_nchw": (ctypes.c_int, [V, I32, I32, I32, I32, I32, I32, V, I32, I32, V]),
    "b200seg_resize_nchw": (ctypes.c_int, [V, I32, I32, I32, V, I32, I32, V]),
    "b200seg_blend": (ctypes.c_int, [V, V, V, V, I32, I32, I64, I32, V]),
    "b200seg_maxpool3x3s2_fwd": (ctypes.c_int, [V, I32, I32, I32, I32, I32, V, I32, V]),
    "b200seg_maxpool3x3s2_bwd": (ctypes.c_int, [V, I32, V, I32, I32, I32, I32, I32, V, I32, I32, V]),
    "b200seg_channel_stats_grid": (I32, [I64, I32]),
    "b200seg_channel_stats": (ctypes.c_int, [V, I32, I64, I32, V, V]),
    "b200seg_spatial_sum_splits": (I32, [I32]),
    "b200seg_spatial_sum": (ctypes.c_int, [V, I32, I32, I32, I32, F, V, V, I32, I32, V]),
    "b200seg_broadcast_pixels": (ctypes.c_int, [V, I32, I32, I32, I32, F, V, I32, I32, V]),
    "b200seg_accum_pred": (ctypes.c_int, [V, V, I32, I32, I32, I32, I32, I32, V]),
    "b200seg_aug_resize_crop": (ctypes.c_int, [ctypes.POINTER(AugGeom), V, V, V, V, V, V, V, V, V, V, V, V]),
    "b200seg_aug_color_normalize": (ctypes.c_int, [ctypes.POINTER(AugColor), V, I32, I32, V, V, V]),
    "b200seg_argmax_hist": (ctypes.c_int, [V, I32, I32, I64, F, V, V, V, V, V]),
}
# test-only entry points (csrc/probe.h, libb200seg_test.so), not part of include/b200seg.h / the product library
PROBE_SIGNATURES = {
    "b200seg_conv2d_fwd_direct": (ctypes.c_int, [ctypes.POINTER(ConvDesc), V, V, V, V, V]),
    "b200seg_umma_probe": (ctypes.c_int, [ctypes.POINTER(ProbeDesc), V, V, V, V]),
}

_lib = None


class B200SegError(RuntimeError):
    pass


def lib():
    """Load (once) and return the shared library; raises if it has not been built."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise B200SegError(
                "libb200seg.so not found at %s - run `python -c 'import __graft_entry__ as g; g.build()'` "
                "(there is no CPU / PyTorch fallback for the hot path)" % LIB_PATH)
        L = ctypes.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(L, name)
            fn.restype = res
            fn.argtypes = args
        _lib = L
    return _lib


TEST_LIB_PATH = os.path.join(_HERE, "lib", "libb200seg_test.so")
_test_lib = None


def test_lib():
    """The test-only library (direct cross-check convolution, descriptor probe); never loaded by the product path."""
    global _test_lib
    if _test_lib is None:
        if not os.path.exists(TEST_LIB_PATH):
            raise B200SegError("libb200seg_test.so not found at %s (make -C csrc)" % TEST_LIB_PATH)
        L = ctypes.CDLL(TEST_LIB_PATH)
        for name, (res, args) in PROBE_SIGNATURES.items():
            fn = getattr(L, name)
            fn.restype = res
            fn.argtypes = args
        _test_lib = L
    return _test_lib


KERNEL_LAUNCHES = 0   # running count of kernels launched through the ABI by this process (bench.py reports it)


def check(rc, what, launches=1):
    global KERNEL_LAUNCHES
    if rc != 0:
        raise B200SegError("%s failed with status %d" % (what, rc))
    KERNEL_LAUNCHES += launches


def ptr(t):
    """Raw device pointer of a torch tensor (or None)."""
    return None if t is None else t.data_ptr()


def stream_ptr():
    import torch
    return torch.cuda.current_stream().cuda_stream
