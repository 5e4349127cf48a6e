"""Functional (no-autograd) wrappers: torch tensors in, C-ABI calls on the current CUDA stream, torch tensors out.

Activations are NHWC bf16 tensors (or channel-slice views of wider NHWC buffers: ``t.stride(3) == 1`` and
``t.stride(2)`` is the pixel pitch). PyTorch only provides device memory and streams here.
"""
import ctypes

import torch

from ._lib import AugColor, AugGeom, BnFold, ConvDesc, FuseDesc, MscaleDesc, check, lib, ptr, stream_ptr

BF16 = torch.bfloat16
F32 = torch.float32

# Step-scoped keep-alive: a training step runs on several streams (scale passes, HRNet branches, weight-gradient side
# streams); the caching allocator hands a freed block back to the stream that allocated it, which may overwrite it while
# another stream still reads it. While KEEP is a list every tensor allocated here stays referenced until the step's final
# join clears it (the step is static, so nothing is ever needed twice; costs memory, not time).
KEEP = None


def _new(*a, **k):
    t = torch.empty(*a, **k)
    if KEEP is not None:
        KEEP.append(t)
    return t


def _newz(*a, **k):
    t = torch.zeros(*a, **k)
    if KEEP is not None:
        KEEP.append(t)
    return t


def _new_like(x):
    t = torch.empty_like(x)
    if KEEP is not None:
        KEEP.append(t)
    return t


def _ld(t):
    assert t.stride(-1) == 1, "channel dimension must be contiguous"
    return t.stride(-2)


def _dev(t):
    return t.device


def empty_act(n, h, w, c, device, dtype=BF16):
    return _new((n, h, w, c), dtype=dtype, device=device)


# ----------------------------------------------------------------------------------------------- convolution
def pack_weight(w_oihw, want_dgrad=True):
    """fp32 OIHW master weight -> (bf16 [O][k*k][I], bf16 [I][k*k flipped][roundup8(O)])."""
    assert w_oihw.is_cuda and w_oihw.dtype == F32 and w_oihw.is_contiguous()
    o, i, k, _ = w_oihw.shape
    o_pad = (o + 7) // 8 * 8
    w_f = _new((o, k * k, i), dtype=BF16, device=w_oihw.device)
    w_d = _newz((i, k * k, o_pad), dtype=BF16, device=w_oihw.device) if want_dgrad else None
    check(lib().b200seg_pack_weight(ptr(w_oihw), o, i, k, ptr(w_f), ptr(w_d), o_pad, stream_ptr()), "pack_weight")
    return w_f, w_d


def pack_weight_into(w_oihw, w_f, w_d):
    o, i, k, _ = w_oihw.shape
    o_pad = w_d.shape[2] if w_d is not None else 0
    check(lib().b200seg_pack_weight(ptr(w_oihw), o, i, k, ptr(w_f), ptr(w_d), o_pad, stream_ptr()), "pack_weight")


def pack_table(entries, device):
    """entries: list of (w_oihw fp32 tensor, w_f, w_d) -> device tables for pack_weights (one launch for all of them).
    The table stores raw pointers: rebuild it when a parameter's storage moves."""
    import numpy as np
    chunk = lib().b200seg_pack_chunk()
    items, blk_item, blk_start = [], [], []
    for idx, (w, w_f, w_d) in enumerate(entries):
        o, i, k, _ = w.shape
        i_dst = w_f.shape[2]
        assert w.is_contiguous() and w.dtype == F32
        items.append((w.data_ptr(), w_f.data_ptr(), w_d.data_ptr() if w_d is not None else 0, o, i, i_dst, k,
                      w_d.shape[2] if w_d is not None else 0, 0))
        for st in range(0, w.numel(), chunk):
            blk_item.append(idx)
            blk_start.append(st)
    it_np = np.array(items, dtype=np.dtype([("w", "<u8"), ("f", "<u8"), ("d", "<u8"), ("o", "<i4"), ("i", "<i4"),
                                            ("i_dst", "<i4"), ("k", "<i4"), ("o_pad", "<i4"), ("r", "<i4")]))
    return dict(items=torch.from_numpy(it_np.view(np.uint8).copy()).to(device),
                blk_item=torch.tensor(blk_item, dtype=torch.int32, device=device),
                blk_start=torch.tensor(blk_start, dtype=torch.int32, device=device), n_blocks=len(blk_item),
                ptrs=tuple(e[0].data_ptr() for e in entries))


def pack_weights(table, which=3):
    """which: 1 forward operands, 2 data-gradient operands, 3 both."""
    check(lib().b200seg_pack_weights(ptr(table["items"]), ptr(table["blk_item"]), ptr(table["blk_start"]),
                                     table["n_blocks"], which, stream_ptr()), "pack_weights")


def conv_desc(n, h, w, cin, cout, ksize, stride, x_ld, y_ld, out_fp32=False, has_bias=False, emit_stats=False,
              force_kc=0, dilation=1):
    d = ConvDesc()
    d.n, d.h, d.w, d.cin, d.cout = n, h, w, cin, cout
    d.ksize, d.stride, d.pad = ksize, stride, (dilation if ksize == 3 else 0)
    d.x_ld, d.y_ld = x_ld, y_ld
    d.out_fp32, d.has_bias, d.emit_stats, d.reserved = int(out_fp32), int(has_bias), int(emit_stats), force_kc
    d.dilation = dilation
    return d


def out_hw(h, w, ksize, stride, dilation=1):
    pad = dilation if ksize == 3 else 0
    span = dilation * (ksize - 1) + 1
    return (h + 2 * pad - span) // stride + 1, (w + 2 * pad - span) // stride + 1


def conv2d_fwd(x, w_ohwi, bias=None, stride=1, out=None, out_fp32=False, emit_stats=False, force_kc=0,
               direct=False, out_ld=None, dilation=1, addend=None):
    """x: [N,H,W,Cin] bf16; w_ohwi: [Cout][k*k][Cin] bf16. Returns y (and with emit_stats the per-CTA partials
    [grid][2][cout_pad] fp32)."""
    assert x.is_cuda and x.dtype == BF16
    cout, taps, cin = w_ohwi.shape
    assert cin == x.shape[3], (cin, x.shape)
    ksize = 3 if taps == 9 else 1
    n, h, w, _ = x.shape
    ho, wo = out_hw(h, w, ksize, stride, dilation)
    if out is None:
        width = cout if out_ld is None else out_ld
        buf = _new((n, ho, wo, width), dtype=F32 if out_fp32 else BF16, device=x.device)
        out = buf[..., :cout] if width != cout else buf
    d = conv_desc(n, h, w, cin, cout, ksize, stride, _ld(x), _ld(out), out_fp32, bias is not None, emit_stats,
                  force_kc, dilation)
    if direct:
        from ._lib import test_lib        # test-only library (tests/test_gpu_ops.py cross-check)
        check(test_lib().b200seg_conv2d_fwd_direct(ctypes.byref(d), ptr(x), ptr(w_ohwi), ptr(bias), ptr(out),
                                              stream_ptr()), "conv2d_fwd_direct")
        return out
    stats = None
    grid = ctypes.c_int32(0)
    if emit_stats:
        nelem = lib().b200seg_conv2d_stats_elems(ctypes.byref(d))
        stats = _new(nelem, dtype=F32, device=x.device)
    if addend is not None:      # y = conv(x) + addend (identity-mapping residual sum in the convolution epilogue)
        check(lib().b200seg_conv2d_fwd_add(ctypes.byref(d), ptr(x), ptr(w_ohwi), ptr(bias), ptr(addend), _ld(addend),
                                           ptr(out), ptr(stats), ctypes.byref(grid), stream_ptr()), "conv2d_fwd_add")
    else:
        check(lib().b200seg_conv2d_fwd(ctypes.byref(d), ptr(x), ptr(w_ohwi), ptr(bias), ptr(out), ptr(stats),
                                       ctypes.byref(grid), stream_ptr()), "conv2d_fwd")
    if emit_stats:
        cout_pad = (cout + 15) // 16 * 16
        return out, (stats, grid.value, cout_pad)
    return out


def conv2d_fwd_bn(x, w_ohwi, bias, stride, gamma, beta, eps, momentum, accum, counter, batch_out=None,
                  running_mean=None, running_var=None, nbt=None, out=None, dilation=1):
    """Convolution + training-mode BatchNorm statistics finalised inside the launch (b200seg_conv2d_fwd_bn): returns
    (y, params fp32 [4, cout] = scale, shift, mean, invstd). accum (fp64 [2*roundup16(cout)]) / counter (int32 [1]) are
    the layer's private, self-clearing reduction cells."""
    assert x.is_cuda and x.dtype == BF16
    cout, taps, cin = w_ohwi.shape
    assert cin == x.shape[3], (cin, x.shape)
    ksize = 3 if taps == 9 else 1
    n, h, w, _ = x.shape
    ho, wo = out_hw(h, w, ksize, stride, dilation)
    if out is None:
        out = _new((n, ho, wo, cout), dtype=BF16, device=x.device)
    d = conv_desc(n, h, w, cin, cout, ksize, stride, _ld(x), _ld(out), False, bias is not None, True,
                  dilation=dilation)
    par = _new((4, cout), dtype=F32, device=x.device)
    f = BnFold()
    f.accum, f.counter = ptr(accum), ptr(counter)
    f.gamma, f.beta = ptr(gamma), ptr(beta)
    f.scale, f.shift, f.mean, f.invstd = ptr(par[0]), ptr(par[1]), ptr(par[2]), ptr(par[3])
    f.batch_stats_out = ptr(batch_out)
    f.running_mean, f.running_var, f.num_batches_tracked = ptr(running_mean), ptr(running_var), ptr(nbt)
    f.eps, f.momentum, f.count, f.c = eps, momentum, float(n * ho * wo), cout
    check(lib().b200seg_conv2d_fwd_bn(ctypes.byref(d), ptr(x), ptr(w_ohwi), ptr(bias), ptr(out), ctypes.byref(f),
                                      stream_ptr()), "conv2d_fwd_bn")
    return out, par


def conv2d_fwd_affine(x, w_ohwi, scale, shift, relu, stride=1, addend=None, out=None, dilation=1):
    """Evaluation: y = relu?(conv(x) * scale + shift (+ addend)) in one launch (BatchNorm from running statistics)."""
    assert x.is_cuda and x.dtype == BF16
    cout, taps, cin = w_ohwi.shape
    assert cin == x.shape[3], (cin, x.shape)
    ksize = 3 if taps == 9 else 1
    n, h, w, _ = x.shape
    ho, wo = out_hw(h, w, ksize, stride, dilation)
    if out is None:
        out = _new((n, ho, wo, cout), dtype=BF16, device=x.device)
    d = conv_desc(n, h, w, cin, cout, ksize, stride, _ld(x), _ld(out), dilation=dilation)
    check(lib().b200seg_conv2d_fwd_affine(ctypes.byref(d), ptr(x), ptr(w_ohwi), ptr(scale), ptr(shift), int(relu),
                                          ptr(addend), _ld(addend) if addend is not None else 0, ptr(out),
                                          stream_ptr()), "conv2d_fwd_affine")
    return out


def _cells_fold(cells, par, gamma, beta, eps, momentum, count, c, batch_out, running_mean, running_var, nbt):
    f = BnFold()
    f.accum, f.counter = ptr(cells), None          # counter NULL = deferred finalisation (csrc/bn_fold.cuh)
    f.gamma, f.beta = ptr(gamma), ptr(beta)
    f.scale, f.shift, f.mean, f.invstd = ptr(par[0]), ptr(par[1]), ptr(par[2]), ptr(par[3])
    f.batch_stats_out = ptr(batch_out)
    f.running_mean, f.running_var, f.num_batches_tracked = ptr(running_mean), ptr(running_var), ptr(nbt)
    f.eps, f.momentum, f.count, f.c = eps, momentum, float(count), c
    return f


def conv2d_fwd_cells(x, w_ohwi, bias, stride, cells, out=None, dilation=1):
    """Convolution whose epilogue adds the batch statistics of the stored output to `cells` (fp64 [2*roundup16(cout)],
    zero at the start of the step) and nothing else: the consuming bn_apply_cells finalises them. Returns y."""
    assert x.is_cuda and x.dtype == BF16
    cout, taps, cin = w_ohwi.shape
    assert cin == x.shape[3], (cin, x.shape)
    ksize = 3 if taps == 9 else 1
    n, h, w, _ = x.shape
    ho, wo = out_hw(h, w, ksize, stride, dilation)
    if out is None:
        out = _new((n, ho, wo, cout), dtype=BF16, device=x.device)
    d = conv_desc(n, h, w, cin, cout, ksize, stride, _ld(x), _ld(out), False, bias is not None, True,
                  dilation=dilation)
    f = BnFold()
    f.accum, f.counter, f.c = ptr(cells), None, cout
    check(lib().b200seg_conv2d_fwd_bn(ctypes.byref(d), ptr(x), ptr(w_ohwi), ptr(bias), ptr(out), ctypes.byref(f),
                                      stream_ptr()), "conv2d_fwd_bn(cells)")
    return out


def bn_apply_cells(y, cells, par, gamma, beta, eps, momentum, res=None, post_scale=None, relu=True, out=None,
                   batch_out=None, running_mean=None, running_var=None, nbt=None):
    """bn_apply as the consumer of conv2d_fwd_cells: finalises the statistics in its prologue and fills par (fp32
    [4, c] = scale, shift, mean, invstd) and the batch / running statistics."""
    n, h, w, c = y.shape
    if out is None:
        out = _new((n, h, w, c), dtype=BF16, device=y.device)
    f = _cells_fold(cells, par, gamma, beta, eps, momentum, n * h * w, c, batch_out, running_mean, running_var, nbt)
    check(lib().b200seg_bn_apply_cells(ptr(y), _ld(y), ctypes.byref(f), ptr(res), _ld(res) if res is not None else 0,
                                       ptr(post_scale), int(relu), ptr(out), _ld(out), n * h * w, h * w, c,
                                       stream_ptr()), "bn_apply_cells")
    return out


def conv2d_dgrad(dy, w_dgrad, x_shape, ksize, stride, addend=None, out=None, force_kc=0, dilation=1):
    """dy: [N,Ho,Wo,roundup8(Cout)] bf16; w_dgrad: [Cin][k*k][roundup8(Cout)]; x_shape = (N,H,W,Cin)."""
    n, h, w, cin = x_shape
    cout_pad = w_dgrad.shape[2]
    assert dy.shape[3] >= cout_pad or dy.shape[3] == cout_pad, (dy.shape, w_dgrad.shape)
    if out is None:
        if addend is not None:
            out = addend
        elif ksize == 1 and stride == 2:     # only the even lattice is written by the kernel
            out = _newz((n, h, w, cin), dtype=BF16, device=dy.device)
        else:
            out = _new((n, h, w, cin), dtype=BF16, device=dy.device)
    d = conv_desc(n, h, w, cin, cout_pad, ksize, stride, _ld(out), _ld(out), force_kc=force_kc, dilation=dilation)
    check(lib().b200seg_conv2d_dgrad(ctypes.byref(d), ptr(dy), _ld(dy), ptr(w_dgrad), ptr(addend),
                                     _ld(addend) if addend is not None else 0, ptr(out), _ld(out), stream_ptr()),
          "conv2d_dgrad", (4 if ksize == 3 else 1) if stride == 2 else 1)
    return out


def conv2d_wgrad(x, dy, dw_ohwi, cout, ksize, stride, ws_holder=None, dilation=1):
    """dw_ohwi (fp32 accumulator [Cout][k*k][Cin], contiguous; a [Cout,Cin,1,1] tensor is the same memory for 1x1)
    += sum_pixels dy x shifted(x). Returns the workspace tensor (keep it alive while the launch is in flight).
    ws_holder: optional one-element list holding a reusable workspace of the calling stream (grown on demand): all
    weight gradients of one side stream run back to back, so they can share one slab buffer."""
    n, h, w, cin = x.shape
    assert dw_ohwi.is_contiguous() and dw_ohwi.dtype == F32 and dw_ohwi.numel() == cout * cin * ksize * ksize
    d = conv_desc(n, h, w, cin, cout, ksize, stride, _ld(x), _ld(dy), dilation=dilation)
    L = lib()
    nbytes = L.b200seg_conv2d_wgrad_ws_bytes(ctypes.byref(d))
    need = max(nbytes, 16) // 4
    if ws_holder is not None:
        if ws_holder[0] is None or ws_holder[0].numel() < need:
            ws_holder[0] = _new((need,), dtype=F32, device=x.device)
        ws = ws_holder[0]
    else:
        ws = _new((need,), dtype=F32, device=x.device)
    check(L.b200seg_conv2d_wgrad(ctypes.byref(d), ptr(x), ptr(dy), _ld(dy), ptr(dw_ohwi), ptr(ws), nbytes,
                                 stream_ptr()), "conv2d_wgrad", L.b200seg_conv2d_wgrad_launches(ctypes.byref(d)))
    return ws


def ohwi_to_oihw(dw_ohwi, ksize):
    """[O][k*k][I] accumulator -> the nn.Parameter .grad layout [O,I,k,k] (a permuted view)."""
    o, taps, i = dw_ohwi.shape
    return dw_ohwi.view(o, ksize, ksize, i).permute(0, 3, 1, 2)


def grad_fold_table(segs, device):
    """segs: list of (dst offset, accumulator offset, cout, cin, taps, accumulator cin) -> device tables for grad_fold."""
    import numpy as np
    chunk = lib().b200seg_grad_fold_chunk()
    blk_seg, blk_start = [], []
    for si, (_off, _soff, cout, cin, taps, _scin) in enumerate(segs):
        numel = cout * cin * taps
        for st in range(0, numel, chunk):
            blk_seg.append(si)
            blk_start.append(st)
    seg_np = np.array(segs, dtype=np.dtype([("offset", "<i8"), ("src_offset", "<i8"), ("cout", "<i4"), ("cin", "<i4"),
                                            ("taps", "<i4"), ("src_cin", "<i4")]))
    return dict(segs=torch.from_numpy(seg_np.view(np.uint8).copy()).to(device),
                blk_seg=torch.tensor(blk_seg, dtype=torch.int32, device=device),
                blk_start=torch.tensor(blk_start, dtype=torch.int32, device=device), n_blocks=len(blk_seg))


def grad_fold(dst, acc_a, acc_b, table, clear=False, overwrite=False):
    check(lib().b200seg_grad_fold(ptr(dst), ptr(acc_a), ptr(acc_b), ptr(table["segs"]), ptr(table["blk_seg"]),
                                  ptr(table["blk_start"]), table["n_blocks"], int(clear) | (int(overwrite) << 1),
                                  stream_ptr()), "grad_fold")


def publish_grads(dst, src, scale_dev=None, scale_const=1.0, accumulate=False):
    """dst = (accumulate ? dst : 0) + (*scale_dev * scale_const) * src over flat fp32 buffers of equal size."""
    assert dst.numel() == src.numel() and dst.dtype == F32 and src.dtype == F32
    if scale_dev is not None:
        assert scale_dev.dtype == F32 and scale_dev.numel() == 1 and scale_dev.is_cuda
    check(lib().b200seg_publish_grads(ptr(dst), ptr(src), dst.numel(), ptr(scale_dev), float(scale_const),
                                      int(accumulate), stream_ptr()), "publish_grads")


# ----------------------------------------------------------------------------------------------- batch norm
def _sync_ref(sync):
    return ctypes.byref(sync) if sync is not None else None


def bn_finalize(stats, count, gamma, beta, eps, momentum, running_mean, running_var, nbt, c, batch_out=None, sync=None):
    """batch_out (fp32 [2*c], optional): receives [mean | unbiased var] for a deferred bn_running_update; pass
    running_mean = running_var = nbt = None with it. sync (BnSync, optional): SyncBN exchange descriptor."""
    buf, grid, cpad = stats
    out = _new((4, c), dtype=F32, device=buf.device)   # scale, shift, mean, invstd
    check(lib().b200seg_bn_finalize(ptr(buf), grid, c, cpad, float(count), ptr(gamma), ptr(beta), eps, momentum,
                                    ptr(running_mean), ptr(running_var), ptr(nbt), ptr(out[0]), ptr(out[1]),
                                    ptr(out[2]), ptr(out[3]), ptr(batch_out), _sync_ref(sync), stream_ptr()),
          "bn_finalize")
    return out


def bn_running_update(running, batch0, batch1, momentum, nbt, n_passes):
    check(lib().b200seg_bn_running_update(ptr(running), ptr(batch0), ptr(batch1), running.numel(), momentum, ptr(nbt),
                                          nbt.numel() if nbt is not None else 0, n_passes, stream_ptr()),
          "bn_running_update")


def accum_f32(dst, src):
    assert dst.numel() == src.numel() and dst.dtype == F32 and src.dtype == F32
    check(lib().b200seg_accum_f32(ptr(dst), ptr(src), dst.numel(), stream_ptr()), "accum_f32")


def bn_eval_params(gamma, beta, eps, running_mean, running_var):
    c = gamma.shape[0]
    out = _new((2, c), dtype=F32, device=gamma.device)
    check(lib().b200seg_bn_eval_params(c, ptr(gamma), ptr(beta), eps, ptr(running_mean), ptr(running_var), ptr(out[0]),
                                       ptr(out[1]), stream_ptr()), "bn_eval_params")
    return out


def bn_apply(y, scale, shift, res=None, post_scale=None, relu=True, out=None):
    n, h, w, c = y.shape
    if out is None:
        out = _new((n, h, w, c), dtype=BF16, device=y.device)
    check(lib().b200seg_bn_apply(ptr(y), _ld(y), ptr(scale), ptr(shift), ptr(res), _ld(res) if res is not None else 0,
                                 ptr(post_scale), int(relu), ptr(out), _ld(out), n * h * w, h * w, c, stream_ptr()),
          "bn_apply")
    return out


def bn_bwd(dz, mask, post_scale, y, mean, invstd, gamma, dgamma, dbeta, g_out=None, g_accumulate=False, dy_out=None,
           sync=None, fold=None, cells=None):
    """Returns dy (gradient w.r.t. the BN input). dgamma/dbeta (fp32 views) are accumulated into. fold = (fp64
    accumulator [2*c], int32 ticket): finalise inside the reduce launch (per-GPU statistics, no bn_bwd_finalize).
    cells (fp64 [2*c], zero at the start of the step): deferred finalisation inside the gradient pass (two launches)."""
    n, h, w, c = y.shape
    npix = n * h * w
    L = lib()
    if cells is not None and sync is None:
        dy = dy_out if dy_out is not None else _new((n, h, w, c), dtype=BF16, device=y.device)
        check(L.b200seg_bn_bwd_cells(ptr(dz), _ld(dz), ptr(mask), _ld(mask) if mask is not None else 0, ptr(post_scale),
                                     ptr(y), _ld(y), ptr(mean), ptr(invstd), ptr(gamma), ptr(dgamma), ptr(dbeta),
                                     ptr(cells), ptr(dy), _ld(dy), ptr(g_out), _ld(g_out) if g_out is not None else 0,
                                     int(g_accumulate), npix, h * w, c, stream_ptr()), "bn_bwd_cells", launches=2)
        return dy
    cc = _new((2, c), dtype=F32, device=y.device)
    if fold is not None and sync is None:
        check(L.b200seg_bn_bwd_reduce_finalize(ptr(dz), _ld(dz), ptr(mask), _ld(mask) if mask is not None else 0,
                                               ptr(post_scale), ptr(y), _ld(y), ptr(mean), ptr(invstd), npix, h * w, c,
                                               ptr(fold[0]), ptr(fold[1]), ptr(dgamma), ptr(dbeta), ptr(cc[0]),
                                               ptr(cc[1]), stream_ptr()), "bn_bwd_reduce_finalize")
    else:
        grid = L.b200seg_bn_bwd_grid(npix, c)
        partials = _new((grid, 2, c), dtype=F32, device=y.device)
        check(L.b200seg_bn_bwd_reduce(ptr(dz), _ld(dz), ptr(mask), _ld(mask) if mask is not None else 0,
                                      ptr(post_scale), ptr(y), _ld(y), ptr(mean), ptr(invstd), npix, h * w, c,
                                      ptr(partials), stream_ptr()), "bn_bwd_reduce")
        check(L.b200seg_bn_bwd_finalize(ptr(partials), grid, c, float(npix), ptr(dgamma), ptr(dbeta), ptr(cc[0]),
                                        ptr(cc[1]), _sync_ref(sync), stream_ptr()), "bn_bwd_finalize")
    dy = dy_out if dy_out is not None else _new((n, h, w, c), dtype=BF16, device=y.device)
    check(L.b200seg_bn_bwd_apply(ptr(dz), _ld(dz), ptr(mask), _ld(mask) if mask is not None else 0, ptr(post_scale),
                                 ptr(y), _ld(y), ptr(mean), ptr(invstd), ptr(gamma), ptr(cc[0]), ptr(cc[1]), ptr(dy),
                                 _ld(dy), ptr(g_out), _ld(g_out) if g_out is not None else 0, int(g_accumulate), npix,
                                 h * w, c, stream_ptr()), "bn_bwd_apply")
    return dy


def masked_accum(src, mask, dst, accumulate):
    n, h, w, c = src.shape
    check(lib().b200seg_masked_accum(ptr(src), _ld(src), ptr(mask), _ld(mask) if mask is not None else 0, ptr(dst),
                                     _ld(dst), int(accumulate), n * h * w, c, stream_ptr()), "masked_accum")
    return dst


# ----------------------------------------------------------------------------------------------- resampling
def fuse_fwd(terms, n, h, w, c, relu, out=None):
    """terms: list of (x [N,hj,wj,C], scale or None, shift or None)."""
    d = FuseDesc()
    d.nterms = len(terms)
    d.n, d.h, d.w, d.c, d.relu = n, h, w, c, int(relu)
    for i, (x, sc, sh) in enumerate(terms):
        t = d.term[i]
        t.x, t.scale, t.shift = ptr(x), ptr(sc), ptr(sh)
        t.ld, t.h, t.w = _ld(x), x.shape[1], x.shape[2]
    if out is None:
        out = _new((n, h, w, c), dtype=BF16, device=terms[0][0].device)
    check(lib().b200seg_fuse_fwd(ctypes.byref(d), ptr(out), _ld(out), stream_ptr()), "fuse_fwd")
    return out


def upsample_adjoint(g, mask, h, w, out=None, accumulate=False):
    n, H, W, c = g.shape
    if out is None:
        out = _new((n, h, w, c), dtype=BF16, device=g.device)
    check(lib().b200seg_upsample_adjoint(ptr(g), _ld(g), ptr(mask), _ld(mask) if mask is not None else 0, n, H, W, c,
                                         ptr(out), _ld(out), h, w, int(accumulate), stream_ptr()), "upsample_adjoint")
    return out


def image_prep(images_nchw, h, w):
    n, three, H, W = images_nchw.shape
    assert three == 3 and images_nchw.dtype == F32 and images_nchw.is_contiguous()
    out = _new((n, h, w, 16), dtype=BF16, device=images_nchw.device)
    check(lib().b200seg_image_prep(ptr(images_nchw), n, H, W, ptr(out), h, w, stream_ptr()), "image_prep")
    return out


# ----------------------------------------------------------------------------------------------- OCR glue
def spatial_softmax_fwd(logits, K):
    """logits fp32 [N,P,ld] -> probs bf16 [N,P,32] (softmax over P)."""
    n, P, ld = logits.shape
    L = lib()
    B = L.b200seg_spatial_softmax_blocks(P)
    ws = _new((n * B * 32 * 2,), dtype=F32, device=logits.device)
    probs = _new((n, P, 32), dtype=BF16, device=logits.device)
    check(L.b200seg_spatial_softmax_fwd(ptr(logits), ld, n, P, K, ptr(ws), ptr(probs), None, stream_ptr()),
          "spatial_softmax_fwd", 2)
    return probs


def spatial_softmax_bwd(dprobs, probs, K, dlogit, accumulate):
    n, P, ldd = dprobs.shape
    L = lib()
    B = L.b200seg_spatial_softmax_blocks(P)
    ws = _new((n * B * 32,), dtype=F32, device=dprobs.device)
    check(L.b200seg_spatial_softmax_bwd(ptr(dprobs), ldd, ptr(probs), n, P, K, ptr(ws), ptr(dlogit), int(accumulate),
                                        stream_ptr()), "spatial_softmax_bwd", 2)
    return dlogit


def class_softmax_fwd(x, K, scale):
    P, ld = x.shape
    sim = _new((P, 32), dtype=BF16, device=x.device)
    check(lib().b200seg_class_softmax_fwd(ptr(x), ld, P, K, scale, ptr(sim), stream_ptr()), "class_softmax_fwd")
    return sim


def class_softmax_bwd(dsim, sim, K, scale):
    P, ld = dsim.shape
    ds = _new((P, 32), dtype=BF16, device=dsim.device)
    check(lib().b200seg_class_softmax_bwd(ptr(dsim), ld, ptr(sim), P, K, scale, ptr(ds), stream_ptr()),
          "class_softmax_bwd")
    return ds


def transpose_pad(src, rpad):
    """src [R][C] (bf16 or fp32, row pitch = stride(0)) -> bf16 [C][rpad] zero padded."""
    R, C = src.shape
    dst = _new((C, rpad), dtype=BF16, device=src.device)
    check(lib().b200seg_transpose_pad(ptr(src), int(src.dtype == F32), R, C, src.stride(0), ptr(dst), rpad,
                                      stream_ptr()), "transpose_pad")
    return dst


def cast_rows(src, dst, C, accumulate=False):
    rows = src.shape[0]
    check(lib().b200seg_cast_rows(ptr(src), src.stride(0), ptr(dst), dst.stride(0), rows, C, int(accumulate),
                                  stream_ptr()), "cast_rows")
    return dst


def bias_grad(dy, C, db):
    rows = dy.numel() // dy.shape[-1]
    L = lib()
    partials = _new(L.b200seg_bias_grad_blocks(rows) * 32, dtype=F32, device=dy.device)
    check(L.b200seg_bias_grad(ptr(dy), _ld(dy), rows, C, ptr(partials), ptr(db), stream_ptr()), "bias_grad", launches=2)


# ----------------------------------------------------------------------------------------------- mscale + loss
RMI_LAMBDA = 0.5   # RMILoss(loss_weight_lambda=0.5), loss/rmi.py:48


def mscale_desc(n, h, w, hq, wq, hm=0, wm=0, hl=0, wl=0, nheads=2, w0=1.0, w1=0.4, sup_wt=0.0, ignore_index=255,
                loss_kind=0):
    """loss_kind 0: CrossEntropyLoss2d heads; 1: RMILoss criterion (sigmoid BCE heads + RMI on head 0)."""
    d = MscaleDesc()
    d.n, d.h, d.w, d.hq, d.wq, d.hm, d.wm, d.hl, d.wl = n, h, w, hq, wq, hm, wm, hl, wl
    d.nheads, d.w_head0, d.w_head1, d.sup_wt, d.ignore_index = nheads, w0, w1, sup_wt, ignore_index
    d.loss_kind = loss_kind
    return d


def count_valid(labels, ignore_index=255, plus_one=False):
    """-> fp32 [1] = 1 / (#valid labels (+1 for the RMILoss normalisation, loss/rmi.py:95))."""
    ws = _new((1,), dtype=torch.int64, device=labels.device)
    inv = _new((1,), dtype=F32, device=labels.device)
    check(lib().b200seg_count_valid(ptr(labels), labels.numel(), ignore_index, int(plus_one), ptr(ws), ptr(inv),
                                    stream_ptr()), "count_valid", 2)
    return inv


def rmi_head(d, labels, hi_cls, mid):
    """RMI term of head 0 (loss/rmi.py rmi_lower_bound): -> (dpr fp32 [n,h/4+1,w/4+1,20], rmi_terms fp32 [n*19])."""
    dev = hi_cls.device
    n, hp, wp = d.n, d.h // 4 + 1, d.w // 4 + 1
    L = lib()
    pr = _new((n, hp, wp, 20), dtype=F32, device=dev)
    la = _new((n, hp, wp, 20), dtype=F32, device=dev)
    check(L.b200seg_rmi_pool(ctypes.byref(d), ptr(labels), ptr(hi_cls), ptr(mid), ptr(pr), ptr(la), stream_ptr()),
          "rmi_pool")
    nbytes = L.b200seg_rmi_ws_bytes(n)
    ws = _new((nbytes // 8,), dtype=torch.float64, device=dev)
    G = _new((n, 19, 180), dtype=torch.float64, device=dev)
    terms = _new((n * 19,), dtype=F32, device=dev)
    dpr = _new((n, hp, wp, 20), dtype=F32, device=dev)
    scale = d.w_head0 * (1.0 - RMI_LAMBDA) / (n * 9.0)
    check(L.b200seg_rmi_solve_grad(n, d.h, d.w, ptr(pr), ptr(la), scale, ptr(ws), nbytes, ptr(G), ptr(terms), ptr(dpr),
                                   stream_ptr()), "rmi_solve_grad", 3)
    return dpr, terms


def mscale_mid_fwd(d, lo_cls, lo_aux, lo_attn):
    dev = lo_cls.device
    mid = _new((d.n, d.hm, d.wm, 40), dtype=F32, device=dev)
    mid_sup = _new((d.n, d.hm, d.wm, 20), dtype=F32, device=dev) if d.sup_wt != 0.0 else None
    check(lib().b200seg_mscale_mid_fwd(ctypes.byref(d), ptr(lo_cls), ptr(lo_aux), ptr(lo_attn), ptr(mid), ptr(mid_sup),
                                       stream_ptr()), "mscale_mid_fwd")
    return mid, mid_sup


def mscale_loss_fwd(d, labels, inv_count, hi_cls, hi_aux, mid, mid_sup, rmi_dpr=None, rmi_terms=None):
    dev = hi_cls.device
    L = lib()
    nb = L.b200seg_mscale_loss_blocks(ctypes.byref(d))
    npix = d.n * d.h * d.w
    g_hi = _new((npix, 40), dtype=BF16, device=dev)
    g_lo = _new((npix, 40), dtype=BF16, device=dev) if d.hm > 0 else None
    g_sup = _new((npix, 40), dtype=BF16, device=dev) if (d.hm > 0 and d.sup_wt != 0.0) else None
    ws = _new((nb * 4,), dtype=F32, device=dev)
    loss = _newz((8,), dtype=F32, device=dev)   # total, 4 pointwise means, RMI term, 2 pad
    check(L.b200seg_mscale_loss_fwd(ctypes.byref(d), ptr(labels), ptr(inv_count), ptr(hi_cls), ptr(hi_aux), ptr(mid),
                                    ptr(mid_sup), ptr(g_hi), ptr(g_lo), ptr(g_sup), ptr(ws), ptr(loss), ptr(rmi_dpr),
                                    ptr(rmi_terms), rmi_terms.numel() if rmi_terms is not None else 0, stream_ptr()),
          "mscale_loss_fwd", 2)
    return loss, g_hi, g_lo, g_sup


def mscale_hi_bwd(d, g_hi):
    dev = g_hi.device
    d_cls = _new((d.n, d.hq, d.wq, 32), dtype=BF16, device=dev)
    d_aux = _new((d.n, d.hq, d.wq, 32), dtype=BF16, device=dev) if d.nheads > 1 else None
    check(lib().b200seg_mscale_hi_bwd(ctypes.byref(d), ptr(g_hi), ptr(d_cls), ptr(d_aux), stream_ptr()),
          "mscale_hi_bwd")
    return d_cls, d_aux


def mscale_lo_bwd(d, g_lo, g_sup, lo_cls, lo_aux, lo_attn, mid):
    dev = g_lo.device
    ws = _new((d.n, d.hm, d.wm, 40), dtype=F32, device=dev)
    d_cls = _new((d.n, d.hl, d.wl, 32), dtype=BF16, device=dev)
    d_aux = _new((d.n, d.hl, d.wl, 32), dtype=BF16, device=dev) if d.nheads > 1 else None
    d_attn = _new((d.n, d.hl, d.wl, 8), dtype=BF16, device=dev)
    check(lib().b200seg_mscale_lo_bwd(ctypes.byref(d), ptr(g_lo), ptr(g_sup), ptr(lo_cls), ptr(lo_aux), ptr(lo_attn),
                                      ptr(mid), ptr(ws), ptr(d_cls), ptr(d_aux), ptr(d_attn), stream_ptr()),
          "mscale_lo_bwd", 2)
    return d_cls, d_aux, d_attn


# ----------------------------------------------------------------------------------------------- eval-mode assembly
def resize_to_nchw(src_nhwc, C, H, W, apply_sigmoid=False):
    """fp32 NHWC [n,h,w,ld] -> fp32 NCHW [n,C,H,W] (bilinear, align_corners=False)."""
    n, h, w, _ = src_nhwc.shape
    dst = _new((n, C, H, W), dtype=F32, device=src_nhwc.device)
    check(lib().b200seg_resize_to_nchw(ptr(src_nhwc), _ld(src_nhwc), n, h, w, C, int(apply_sigmoid), ptr(dst), H, W,
                                       stream_ptr()), "resize_to_nchw")
    return dst


def resize_nchw(src, H, W):
    n, c, h, w = src.shape
    if (h, w) == (H, W):
        return src
    dst = _new((n, c, H, W), dtype=F32, device=src.device)
    check(lib().b200seg_resize_nchw(ptr(src), n * c, h, w, ptr(dst), H, W, stream_ptr()), "resize_nchw")
    return dst


def blend(a, x, y, mode):
    """mode 0: a*x + (1-a)*y; 1: x + (1-a)*y; 2: a*x   (a [n,1,H,W]; x,y [n,C,H,W])."""
    n, c, h, w = x.shape
    out = _new_like(x)
    check(lib().b200seg_blend(ptr(a), ptr(x), ptr(y), ptr(out), n, c, h * w, mode, stream_ptr()), "blend")
    return out


# ----------------------------------------------------------------------------------------------- evaluation tail
def accum_pred(pred, out=None, flip=False):
    """out (+)= pred [n,c,h,w] fp32 (mirrored along w when flip); allocates out on the first call."""
    n, c, h, w = pred.shape
    acc = out is not None
    if out is None:
        out = _new_like(pred)
    check(lib().b200seg_accum_pred(ptr(pred), ptr(out), n, c, h, w, int(flip), int(acc), stream_ptr()), "accum_pred")
    return out


def argmax_hist(pred, labels=None, scale=1.0, hist=None):
    """-> (argmax int64 [n,h,w], max softmax prob fp32 [n,h,w], hist int64 [c,c] (accumulated) or None)."""
    n, c, h, w = pred.shape
    assert pred.dtype == F32 and pred.is_contiguous()
    pm = _new((n, h, w), dtype=torch.int64, device=pred.device)
    mp = _new((n, h, w), dtype=F32, device=pred.device)
    if labels is not None and hist is None:
        hist = _newz((c, c), dtype=torch.int64, device=pred.device)
    check(lib().b200seg_argmax_hist(ptr(pred), n, c, h * w, float(scale), ptr(labels), ptr(pm), ptr(mp), ptr(hist),
                                    stream_ptr()), "argmax_hist")
    return pm, mp, hist


# ----------------------------------------------------------------------------------------------- pooling / broadcast (f2)
def maxpool3x3s2(x):
    n, h, w, c = x.shape
    ho, wo = (h - 1) // 2 + 1, (w - 1) // 2 + 1
    y = _new((n, ho, wo, c), dtype=BF16, device=x.device)
    check(lib().b200seg_maxpool3x3s2_fwd(ptr(x), _ld(x), n, h, w, c, ptr(y), _ld(y), stream_ptr()), "maxpool_fwd")
    return y


def maxpool3x3s2_bwd(x, dy, out=None, accumulate=False):
    n, h, w, c = x.shape
    if out is None:
        out = _new((n, h, w, c), dtype=BF16, device=x.device)
    check(lib().b200seg_maxpool3x3s2_bwd(ptr(x), _ld(x), ptr(dy), _ld(dy), n, h, w, c, ptr(out), _ld(out),
                                         int(accumulate), stream_ptr()), "maxpool_bwd")
    return out


def channel_stats(x):
    """-> (partials, grid, cpad) in the layout bn_finalize consumes (statistics of an activation that did not come out
    of a convolution epilogue)."""
    n, h, w, c = x.shape
    npix = n * h * w
    grid = lib().b200seg_channel_stats_grid(npix, c)
    partials = _new((grid * 2 * c,), dtype=F32, device=x.device)
    check(lib().b200seg_channel_stats(ptr(x), _ld(x), npix, c, ptr(partials), stream_ptr()), "channel_stats")
    return partials, grid, c


def spatial_sum(x, scale, out=None, accumulate=False):
    """x [n,h,w,c] -> [n,1,1,c] bf16: scale * sum over pixels (per image)."""
    n, h, w, c = x.shape
    L = lib()
    ws = _new((n * L.b200seg_spatial_sum_splits(h * w) * c,), dtype=F32, device=x.device)
    if out is None:
        out = _new((n, 1, 1, c), dtype=BF16, device=x.device)
    check(L.b200seg_spatial_sum(ptr(x), _ld(x), n, h * w, c, float(scale), ptr(ws), ptr(out), out.stride(0),
                                int(accumulate), stream_ptr()), "spatial_sum", 2)
    return out


def broadcast_pixels(v, h, w, out=None, scale=1.0, accumulate=False):
    """v [n,1,1,c] -> out [n,h,w,c] (=|+=) scale * v at every pixel."""
    n, _, _, c = v.shape
    if out is None:
        assert not accumulate
        out = _new((n, h, w, c), dtype=BF16, device=v.device)
    check(lib().b200seg_broadcast_pixels(ptr(v), v.stride(0), n, h * w, c, float(scale), ptr(out), _ld(out),
                                         int(accumulate), stream_ptr()), "broadcast_pixels")
    return out


# ----------------------------------------------------------------------------------------------- input pipeline (f4)
def augment(image_u8, mask_u8, p, t, id_lut, ignore_label, mean, std, out_image=None, out_label=None):
    """b200seg.augment.DeviceTrainTransform: resize + crop + flip (uint8), colour jitter + ToTensor + Normalize.
    p: AugParams, t: the window tables of DeviceTrainTransform.tables. Returns (fp32 [3,th,tw], int64 [th,tw])."""
    import numpy as np
    dev = image_u8.device
    h, w = image_u8.shape[:2]
    th, tw = t["th"], t["tw"]
    g = AugGeom()
    g.src_h, g.src_w, g.out_h, g.out_w = h, w, th, tw
    g.win_y0, g.win_x0 = t["lo_y"] - (p.y1 - p.pad_y), t["lo_x"] - (p.x1 - p.pad_x)
    g.n_y, g.n_x = t["n_y"], t["n_x"]
    g.ksize_v, g.ksize_h = t["kv"].shape[1], t["kh"].shape[1]
    g.flip, g.ignore_label = int(bool(p.flip)), int(ignore_label)
    # one upload for all six tables
    parts = [t["kh"].ravel(), t["bh"].ravel(), t["kv"].ravel(), t["bv"].ravel(), t["nx"].ravel(), t["ny"].ravel()]
    flat = torch.from_numpy(np.concatenate(parts).astype(np.int32)).to(dev, non_blocking=True)
    offs = np.cumsum([0] + [x.size for x in parts])
    tab = [flat[offs[i]:offs[i + 1]] for i in range(6)]
    rgb = _new((th, tw, 3), dtype=torch.uint8, device=dev)
    if out_label is None:
        out_label = _new((th, tw), dtype=torch.int64, device=dev)
    check(lib().b200seg_aug_resize_crop(ctypes.byref(g), ptr(image_u8), ptr(mask_u8), ptr(tab[0]), ptr(tab[1]),
                                        ptr(tab[2]), ptr(tab[3]), ptr(tab[4]), ptr(tab[5]), ptr(id_lut), ptr(rgb),
                                        ptr(out_label), stream_ptr()), "aug_resize_crop")
    c = AugColor()
    c.n_ops = len(p.ops)
    has_contrast = False
    for i, (kind, factor) in enumerate(p.ops):
        c.kind[i], c.factor[i] = kind, factor
        if kind == 3:          # transforms.py:289-290: np_h += np.uint8(hue_factor * 255): C cast (truncate, wrap mod 256)
            c.hue_shift[i] = int(factor * 255) & 0xFF
        has_contrast |= kind == 1
    for i in range(3):
        c.mean[i], c.std[i] = mean[i], std[i]
    ws = _new((1,), dtype=torch.int64, device=dev) if has_contrast else None
    if out_image is None:
        out_image = _new((3, th, tw), dtype=F32, device=dev)
    check(lib().b200seg_aug_color_normalize(ctypes.byref(c), ptr(rgb), th, tw, ptr(ws), ptr(out_image), stream_ptr()),
          "aug_color_normalize", launches=2 if has_contrast else 1)
    return out_image, out_label, rgb
