"""Op-level parity of every CUDA kernel against plain PyTorch fp32 on the same (bf16-rounded) inputs.

All calls go through the C ABI (ctypes wrappers in b200seg.raw). Tolerances: outputs stored in bf16 are compared at
bf16 resolution (2^-8 relative to the tensor scale), fp32 outputs at 1e-4.
"""
import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu

BF16_TOL = 1.0 / 128


def _setup():
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    from b200seg import raw
    return raw


def rnd(shape, seed, scale=1.0, dtype=torch.bfloat16):
    g = torch.Generator(device="cuda").manual_seed(seed)
    return (torch.randn(shape, generator=g, device="cuda") * scale).to(dtype)


def close(a, b, tol, what=""):
    a, b = a.float(), b.float()
    scale = b.abs().max().item() + 1e-12
    err = (a - b).abs().max().item()
    assert err <= tol * scale, "%s max err %.3e vs scale %.3e (tol %.1e)" % (what, err, scale, tol)


CONV_CASES = [
    # n, h, w, cin, cout, k, s, bias, kc
    (1, 8, 16, 64, 64, 1, 1, False, 0), (1, 16, 32, 64, 64, 3, 1, False, 0), (2, 24, 40, 128, 96, 3, 1, True, 0),
    (1, 16, 32, 32, 32, 3, 1, False, 32), (1, 16, 32, 48, 48, 3, 1, False, 16), (1, 16, 32, 48, 48, 3, 1, False, 0),
    (1, 32, 64, 96, 96, 3, 1, False, 0), (1, 32, 64, 192, 192, 3, 1, False, 0), (1, 16, 32, 384, 384, 3, 1, False, 0),
    (1, 32, 64, 720, 512, 3, 1, True, 0), (1, 32, 64, 720, 720, 1, 1, True, 0), (1, 32, 64, 64, 64, 3, 2, False, 0),
    (1, 32, 64, 48, 96, 3, 2, False, 0), (1, 30, 52, 96, 192, 3, 2, False, 0), (1, 19, 1, 512, 256, 1, 1, False, 0),
    (2, 33, 47, 16, 64, 3, 2, False, 0), (1, 9, 7, 256, 48, 3, 1, False, 0),
    # weight-gradient decompositions: split-over-pixels + reduce (narrow, many pixels) and single-owner units (wide)
    (1, 128, 256, 48, 48, 3, 1, False, 0), (1, 64, 64, 192, 192, 3, 1, False, 0), (2, 16, 32, 384, 384, 3, 1, False, 0),
    (1, 64, 128, 720, 256, 1, 1, False, 0),
]


@pytest.mark.parametrize("case", CONV_CASES)
def test_conv_fwd_dgrad_wgrad(case):
    raw = _setup()
    n, h, w, cin, cout, k, s, bias, kc = case
    x = rnd((n, h, w, cin), 1)
    wt = rnd((cout, cin, k, k), 2, scale=(cin * k * k) ** -0.5, dtype=torch.float32).contiguous()
    b = rnd((cout,), 3, dtype=torch.float32) if bias else None
    w_f, w_d = raw.pack_weight(wt)
    xr = x.float().permute(0, 3, 1, 2).requires_grad_(True)
    wr = wt.to(torch.bfloat16).float().requires_grad_(True)
    ref = F.conv2d(xr, wr, b, stride=s, padding=1 if k == 3 else 0)
    y, stats = raw.conv2d_fwd(x, w_f, b, stride=s, emit_stats=True, force_kc=kc)
    close(y, ref.permute(0, 2, 3, 1), BF16_TOL, "fwd")
    buf, grid, cpad = stats
    tot = buf[: grid * 2 * cpad].view(grid, 2, cpad).sum(0)[:, :cout]
    yr = y.float().reshape(-1, cout)
    close(tot[0], yr.sum(0), 1e-3 * max(1.0, yr.shape[0] ** 0.5), "stats sum")
    close(tot[1], (yr * yr).sum(0), 1e-3, "stats sumsq")
    # direct kernel cross-check (bit-level agreement is not expected: different summation order)
    yd = raw.conv2d_fwd(x, w_f, b, stride=s, direct=True)
    close(y, yd, BF16_TOL, "direct")
    # backward
    ho, wo = y.shape[1:3]
    dy = rnd((n, ho, wo, cout), 4)
    ref.backward(dy.float().permute(0, 3, 1, 2))
    dx = raw.conv2d_dgrad(dy, w_d, (n, h, w, cin), k, s, force_kc=kc) if cout % 8 == 0 else None
    if dx is not None:
        close(dx, xr.grad.permute(0, 2, 3, 1), BF16_TOL, "dgrad")
        add = rnd((n, h, w, cin), 5)
        dx2 = raw.conv2d_dgrad(dy, w_d, (n, h, w, cin), k, s, addend=add.clone(), force_kc=kc)
        close(dx2, xr.grad.permute(0, 2, 3, 1) + add.float(), BF16_TOL, "dgrad+addend")
    if cin % 16 == 0:
        dw = torch.zeros((cout, k * k, cin), dtype=torch.float32, device="cuda")    # kernel-layout accumulator
        raw.conv2d_wgrad(x, dy, dw, cout, k, s)
        raw.conv2d_wgrad(x, dy, dw, cout, k, s)        # accumulates
        close(raw.ohwi_to_oihw(dw, k), 2 * wr.grad, 2e-3, "wgrad")


@pytest.mark.parametrize("case", [(1, 64, 96, 48, 48, 3, 1, False), (2, 40, 72, 64, 64, 3, 1, False),
                                  (1, 32, 64, 720, 512, 3, 1, True), (1, 32, 64, 96, 48, 1, 1, False),
                                  (1, 64, 128, 48, 96, 3, 2, False), (1, 19, 1, 512, 256, 1, 1, False),
                                  (1, 256, 512, 48, 48, 3, 1, False)])
def test_conv_with_in_launch_bn_finalize(case):
    """b200seg_conv2d_fwd_bn (statistics finalised by the last CTA, csrc/bn_fold.cuh) against the two-launch path
    (conv2d_fwd partials + bn_finalize): same output bits, same scale / shift / mean / invstd / batch statistics /
    running statistics, reduction cells left clean (three launches in a row share them), and against F.batch_norm."""
    raw = _setup()
    n, h, w, cin, cout, k, s, bias = case
    x = rnd((n, h, w, cin), 1)
    wt = rnd((cout, cin, k, k), 2, scale=(cin * k * k) ** -0.5, dtype=torch.float32).contiguous()
    b = rnd((cout,), 3, dtype=torch.float32) if bias else None
    gamma = 1.0 + 0.1 * rnd((cout,), 4, dtype=torch.float32)
    beta = 0.1 * rnd((cout,), 5, dtype=torch.float32)
    w_f, _ = raw.pack_weight(wt, want_dgrad=False)
    y0, stats = raw.conv2d_fwd(x, w_f, b, stride=s, emit_stats=True)
    npix = y0.shape[0] * y0.shape[1] * y0.shape[2]
    rm0, rv0 = torch.zeros(cout, device="cuda"), torch.ones(cout, device="cuda")
    nbt0 = torch.zeros((), dtype=torch.long, device="cuda")
    par0 = raw.bn_finalize(stats, npix, gamma, beta, 1e-5, 0.1, rm0, rv0, nbt0, cout)
    cpad = (cout + 15) // 16 * 16
    acc = torch.zeros(2 * cpad, dtype=torch.float64, device="cuda")
    ticket = torch.zeros(1, dtype=torch.int32, device="cuda")
    rm1, rv1 = torch.zeros(cout, device="cuda"), torch.ones(cout, device="cuda")
    nbt1 = torch.zeros((), dtype=torch.long, device="cuda")
    for rep in range(3):
        batch = torch.zeros(2 * cout, device="cuda")
        if rep == 0:
            y1, par1 = raw.conv2d_fwd_bn(x, w_f, b, s, gamma, beta, 1e-5, 0.1, acc, ticket, running_mean=rm1,
                                         running_var=rv1, nbt=nbt1)
        else:
            y1, par1 = raw.conv2d_fwd_bn(x, w_f, b, s, gamma, beta, 1e-5, 0.1, acc, ticket, batch_out=batch)
        torch.cuda.synchronize()
        assert torch.equal(y1, y0)
        assert float(acc.abs().max()) == 0.0 and int(ticket) == 0, rep
        for i, name in enumerate(("scale", "shift", "mean", "invstd")):
            close(par1[i], par0[i], 2e-6, name)
        if rep:
            close(batch[:cout], par0[2], 2e-6, "batch mean")
    close(rm1, rm0, 2e-6, "running mean")
    close(rv1, rv0, 2e-6, "running var")
    assert int(nbt1) == int(nbt0) == 1
    yr = y0.float().reshape(-1, cout)
    ref = F.batch_norm(yr, None, None, gamma, beta, training=True, eps=1e-5)
    close(yr * par1[0] + par1[1], ref, 2e-5, "affine vs F.batch_norm")


@pytest.mark.parametrize("case", [(1, 64, 96, 48, 48, 3, 1, False), (2, 40, 72, 64, 64, 3, 1, False),
                                  (1, 32, 64, 720, 512, 3, 1, True), (1, 32, 64, 96, 48, 1, 1, False),
                                  (1, 64, 128, 48, 96, 3, 2, False), (1, 256, 512, 48, 48, 3, 1, False)])
@pytest.mark.parametrize("res,relu", [(True, True), (False, False)])
def test_conv_with_deferred_bn_finalize(case, res, relu):
    """Deferred finalisation (the training default): conv2d_fwd_cells adds its statistics to fp64 cells, bn_apply_cells
    folds them in its prologue. Against the three-launch path (conv2d_fwd partials + bn_finalize + bn_apply): same conv
    bits, same z bits up to one bf16 ulp, same scale / shift / mean / invstd / batch + running statistics."""
    raw = _setup()
    n, h, w, cin, cout, k, s, bias = case
    x = rnd((n, h, w, cin), 1)
    wt = rnd((cout, cin, k, k), 2, scale=(cin * k * k) ** -0.5, dtype=torch.float32).contiguous()
    b = rnd((cout,), 3, dtype=torch.float32) if bias else None
    gamma = 1.0 + 0.1 * rnd((cout,), 4, dtype=torch.float32)
    beta = 0.1 * rnd((cout,), 5, dtype=torch.float32)
    w_f, _ = raw.pack_weight(wt, want_dgrad=False)
    y0, stats = raw.conv2d_fwd(x, w_f, b, stride=s, emit_stats=True)
    npix = y0.shape[0] * y0.shape[1] * y0.shape[2]
    rm0, rv0 = torch.zeros(cout, device="cuda"), torch.ones(cout, device="cuda")
    nbt0 = torch.zeros((), dtype=torch.long, device="cuda")
    par0 = raw.bn_finalize(stats, npix, gamma, beta, 1e-5, 0.1, rm0, rv0, nbt0, cout)
    r = rnd(tuple(y0.shape), 6) if res else None
    z0 = raw.bn_apply(y0, par0[0], par0[1], r, None, relu)
    cpad = (cout + 15) // 16 * 16
    rm1, rv1 = torch.zeros(cout, device="cuda"), torch.ones(cout, device="cuda")
    nbt1 = torch.zeros((), dtype=torch.long, device="cuda")
    for rep in range(2):
        cells = torch.zeros(2 * cpad, dtype=torch.float64, device="cuda")
        par1 = torch.full((4, cout), float("nan"), device="cuda")
        batch = torch.zeros(2 * cout, device="cuda")
        y1 = raw.conv2d_fwd_cells(x, w_f, b, s, cells)
        if rep == 0:
            z1 = raw.bn_apply_cells(y1, cells, par1, gamma, beta, 1e-5, 0.1, r, None, relu, running_mean=rm1,
                                    running_var=rv1, nbt=nbt1)
        else:
            z1 = raw.bn_apply_cells(y1, cells, par1, gamma, beta, 1e-5, 0.1, r, None, relu, batch_out=batch)
        torch.cuda.synchronize()
        assert torch.equal(y1, y0)
        yr = y0.double().reshape(-1, cout)
        close(cells[:cout].float(), yr.sum(0).float(), 1e-5, "cell sums")
        close(cells[cpad:cpad + cout].float(), (yr * yr).sum(0).float(), 1e-5, "cell sums of squares")
        for i, name in enumerate(("scale", "shift", "mean", "invstd")):
            close(par1[i], par0[i], 2e-6, name)
        close(z1, z0, 2.0 ** -8, "z")
        if rep:
            close(batch[:cout], par0[2], 2e-6, "batch mean")
            var_b = yr.var(0, unbiased=True).float()
            close(batch[cout:], var_b, 1e-4, "batch var")
    close(rm1, rm0, 2e-6, "running mean")
    close(rv1, rv0, 2e-6, "running var")
    assert int(nbt1) == int(nbt0) == 1


def test_grad_fold_layouts_and_clearing():
    """End-of-step fold: OHWI accumulators of two passes -> OIHW gradient (+= or overwrite), vectors of both passes, the
    stem accumulating on 16 padded input channels at its own accumulator offset, accumulators cleared on request."""
    import numpy as np
    raw = _setup()
    shapes = [(48, 32, 3, 3), (19, 512, 1, 1), (96,), (64, 16, 3, 3), (7,), (96, 96, 3, 3), (64, 3, 3, 3)]
    offs, off = [], 0
    for shp in shapes:
        offs.append(off)
        off += (int(np.prod(shp)) + 63) // 64 * 64
    stem_src = off                        # padded stem accumulator [64][9][16] behind the flat layout
    acc_len = off + 64 * 9 * 16
    g = torch.Generator(device="cuda").manual_seed(0)
    for overwrite in (False, True):
        dst = torch.randn(off, generator=g, device="cuda")
        a = torch.randn(acc_len, generator=g, device="cuda")
        b = torch.randn(acc_len, generator=g, device="cuda")
        want = torch.zeros_like(dst) if overwrite else dst.clone()
        untouched = dst.clone()
        segs = []
        for shp, o_ in zip(shapes, offs):
            n = int(np.prod(shp))
            if len(shp) == 4 and shp[1] == 3:
                co, ci, k, _ = shp
                src = (a[stem_src:] + b[stem_src:]).view(co, k * k, 16)[:, :, :ci]
                want[o_:o_ + n] += src.permute(0, 2, 1).reshape(-1)
                segs.append((o_, stem_src, co, ci, k * k, 16))
            elif len(shp) == 4:
                co, ci, k, _ = shp
                src = (a[o_:o_ + n] + b[o_:o_ + n]).view(co, k * k, ci)
                want[o_:o_ + n] += src.permute(0, 2, 1).reshape(-1)
                segs.append((o_, o_, co, ci, k * k, ci))
            else:
                want[o_:o_ + n] += a[o_:o_ + n] + b[o_:o_ + n]
                segs.append((o_, o_, 1, n, 1, n))
        table = raw.grad_fold_table(segs, "cuda")
        a0 = a.clone()
        raw.grad_fold(dst, a, b, table, clear=False, overwrite=overwrite)
        torch.cuda.synchronize()
        assert torch.equal(a, a0)                                           # not cleared unless asked
        for shp, o_ in zip(shapes, offs):
            n = int(np.prod(shp))
            assert torch.allclose(dst[o_:o_ + n], want[o_:o_ + n], rtol=0, atol=2e-6), (shp, overwrite)
            pad_end = o_ + (n + 63) // 64 * 64
            assert torch.equal(dst[o_ + n:pad_end], untouched[o_ + n:pad_end])   # alignment gaps are not written
        raw.grad_fold(dst, a, b, table, clear=True, overwrite=True)
        torch.cuda.synchronize()
        for shp, o_ in zip(shapes, offs):
            n = int(np.prod(shp))
            if not (len(shp) == 4 and shp[1] == 3):
                assert float(a[o_:o_ + n].abs().max()) == 0.0 and float(b[o_:o_ + n].abs().max()) == 0.0
        assert float(a[stem_src:].view(64, 9, 16)[:, :, :3].abs().max()) == 0.0


def test_publish_grads_scales_and_accumulates():
    """Gradient publish: dst = (accumulate ? dst : 0) + (*scale_dev * scale_const) * src."""
    raw = _setup()
    g = torch.Generator(device="cuda").manual_seed(1)
    n = 64 * 1000 + 64
    src = torch.randn(n, generator=g, device="cuda")
    dst = torch.randn(n, generator=g, device="cuda")
    d0 = dst.clone()
    sc = torch.tensor(0.25, device="cuda")
    raw.publish_grads(dst, src, sc, 0.5, accumulate=True)
    assert torch.allclose(dst, d0 + 0.125 * src, rtol=0, atol=1e-6)
    raw.publish_grads(dst, src, None, 1.0, accumulate=False)
    assert torch.equal(dst, src)


def test_conv_logit_head_fp32_and_padded_grads():
    raw = _setup()
    n, h, w, cin, cout = 2, 32, 64, 512, 19
    x = rnd((n, h, w, cin), 1)
    wt = rnd((cout, cin, 1, 1), 2, scale=cin ** -0.5, dtype=torch.float32).contiguous()
    b = rnd((cout,), 3, dtype=torch.float32)
    w_f, w_d = raw.pack_weight(wt)
    y = raw.conv2d_fwd(x, w_f, b, out_fp32=True, out_ld=20)
    assert y.shape == (n, h, w, 19) and y.stride(2) == 20
    xr = x.float().permute(0, 3, 1, 2).requires_grad_(True)
    wr = wt.to(torch.bfloat16).float().requires_grad_(True)
    ref = F.conv2d(xr, wr, b)
    close(y, ref.permute(0, 2, 3, 1), 2e-5, "logits")
    dl = torch.zeros((n, h, w, 32), dtype=torch.bfloat16, device="cuda")
    dl[..., :19] = rnd((n, h, w, 19), 4)
    ref.backward(dl[..., :19].float().permute(0, 3, 1, 2))
    dx = raw.conv2d_dgrad(dl[..., :24], w_d, (n, h, w, cin), 1, 1)
    close(dx, xr.grad.permute(0, 2, 3, 1), BF16_TOL, "head dgrad")
    dw = torch.zeros_like(wt)
    raw.conv2d_wgrad(x, dl, dw, cout, 1, 1)
    close(dw, wr.grad, 2e-3, "head wgrad")
    db = torch.zeros(19, device="cuda")
    raw.bias_grad(dl, 19, db)
    close(db, dl[..., :19].float().sum((0, 1, 2)), 1e-3, "bias grad")
    # at the head's full-resolution size every block of the reduction is busy; its partial sums are combined in a fixed
    # order, so repeated calls give the same gradient bit for bit
    big = torch.randn((1, 256, 512, 24), device="cuda").to(torch.bfloat16)
    runs = []
    for _ in range(3):
        d = torch.zeros(19, device="cuda")
        raw.bias_grad(big, 19, d)
        runs.append(d)
    assert all(torch.equal(runs[0], d) for d in runs[1:]), runs
    close(runs[0], big[..., :19].float().sum((0, 1, 2)), 1e-3, "bias grad, 131072 rows")


@pytest.mark.parametrize("c,res,relu,size", [(48, True, True, (2, 24, 40)), (96, False, True, (2, 24, 40)),
                                             (720, False, False, (2, 24, 40)), (256, True, True, (2, 24, 40)),
                                             # many pixels per thread: the multi-vector (unrolled) paths of the passes
                                             (48, True, True, (1, 256, 512)), (96, False, True, (1, 131, 257)),
                                             (192, True, False, (2, 64, 128))])
def test_batchnorm_train_fwd_bwd(c, res, relu, size):
    raw = _setup()
    n, h, w = size
    x = rnd((n, h, w, 64), 1)
    wt = rnd((c, 64, 1, 1), 2, scale=0.2, dtype=torch.float32).contiguous()
    w_f, _ = raw.pack_weight(wt, want_dgrad=False)
    y, stats = raw.conv2d_fwd(x, w_f, emit_stats=True)
    gamma = (1 + 0.1 * rnd((c,), 3, dtype=torch.float32)).contiguous()
    beta = (0.1 * rnd((c,), 4, dtype=torch.float32)).contiguous()
    rm, rv = torch.zeros(c, device="cuda"), torch.ones(c, device="cuda")
    nbt = torch.zeros((), dtype=torch.long, device="cuda")
    par = raw.bn_finalize(stats, n * h * w, gamma, beta, 1e-5, 0.1, rm, rv, nbt, c)
    r = rnd((n, h, w, c), 5) if res else None
    ps = torch.ones((n, c), device="cuda")
    ps[0, ::3] = 0.0
    ps = ps / 0.95
    z = raw.bn_apply(y, par[0], par[1], r, ps, relu)
    # torch reference on the stored bf16 conv output
    yr = y.float().permute(0, 3, 1, 2).requires_grad_(True)
    g_t, b_t = gamma.clone().requires_grad_(True), beta.clone().requires_grad_(True)
    rm2, rv2 = torch.zeros(c, device="cuda"), torch.ones(c, device="cuda")
    o = F.batch_norm(yr, rm2, rv2, g_t, b_t, training=True, momentum=0.1, eps=1e-5)
    rr = r.float().permute(0, 3, 1, 2).requires_grad_(True) if res else None
    if res:
        o = o + rr
    if relu:
        o = F.relu(o)
    o = o * ps[:, :, None, None]
    close(z, o.permute(0, 2, 3, 1), BF16_TOL, "bn fwd")
    close(rm, rm2, 1e-4, "running mean")
    close(rv, rv2, 1e-4, "running var")
    assert int(nbt) == 1
    dz = rnd((n, h, w, c), 6)
    o.backward(dz.float().permute(0, 3, 1, 2))
    dgamma, dbeta = torch.zeros(c, device="cuda"), torch.zeros(c, device="cuda")
    g_out = torch.empty((n, h, w, c), dtype=torch.bfloat16, device="cuda") if res else None
    dy = raw.bn_bwd(dz, z if relu else None, ps, y, par[2], par[3], gamma, dgamma, dbeta, g_out=g_out)
    close(dy, yr.grad.permute(0, 2, 3, 1), 2 * BF16_TOL, "bn dx")
    close(dgamma, g_t.grad, 5e-3, "dgamma")
    close(dbeta, b_t.grad, 5e-3, "dbeta")
    if res:
        close(g_out, rr.grad.permute(0, 2, 3, 1), BF16_TOL, "residual grad")
    # the in-launch finalisation of the reduce (no bn_bwd_finalize launch) gives the same gradients and leaves its
    # reduction cells clean (two launches in a row share them)
    acc = torch.zeros(2 * ((c + 15) // 16 * 16), dtype=torch.float64, device="cuda")
    ticket = torch.zeros(1, dtype=torch.int32, device="cuda")
    for _ in range(2):
        dgamma2, dbeta2 = torch.zeros(c, device="cuda"), torch.zeros(c, device="cuda")
        dy2 = raw.bn_bwd(dz, z if relu else None, ps, y, par[2], par[3], gamma, dgamma2, dbeta2, fold=(acc, ticket))
        torch.cuda.synchronize()
        close(dy2, dy, 2.0 ** -8, "fused dx")            # the mean terms may differ in the last fp32 bit -> <= 1 bf16 ulp
        close(dgamma2, dgamma, 1e-5, "fused dgamma")
        close(dbeta2, dbeta, 1e-5, "fused dbeta")
        assert float(acc.abs().max()) == 0.0 and int(ticket) == 0
    # deferred finalisation (the training default): the reduce only adds to the cells, the gradient pass folds them
    cells = torch.zeros(2 * c, dtype=torch.float64, device="cuda")
    dgamma3, dbeta3 = torch.zeros(c, device="cuda"), torch.zeros(c, device="cuda")
    g_out3 = torch.empty((n, h, w, c), dtype=torch.bfloat16, device="cuda") if res else None
    dy3 = raw.bn_bwd(dz, z if relu else None, ps, y, par[2], par[3], gamma, dgamma3, dbeta3, g_out=g_out3, cells=cells)
    torch.cuda.synchronize()
    close(dy3, dy, 2.0 ** -8, "deferred dx")
    close(dgamma3, dgamma, 1e-5, "deferred dgamma")
    close(dbeta3, dbeta, 1e-5, "deferred dbeta")
    if res:
        assert torch.equal(g_out3, g_out)
    close(cells[:c].float(), dbeta, 1e-5, "cells hold the sums")


def test_fuse_and_upsample_adjoint():
    raw = _setup()
    n, H, W, c = 2, 32, 48, 48
    x0 = rnd((n, H, W, c), 1)
    x1 = rnd((n, H // 2, W // 2, c), 2)
    x2 = rnd((n, H // 4, W // 4, c), 3)
    x3 = rnd((n, H, W, c), 4)
    sc = [(1 + 0.1 * rnd((c,), 10 + i, dtype=torch.float32)).contiguous() for i in range(3)]
    sh = [(0.1 * rnd((c,), 20 + i, dtype=torch.float32)).contiguous() for i in range(3)]
    z = raw.fuse_fwd([(x0, None, None), (x1, sc[0], sh[0]), (x2, sc[1], sh[1]), (x3, sc[2], sh[2])], n, H, W, c, True)
    t = [v.float().permute(0, 3, 1, 2).requires_grad_(True) for v in (x0, x1, x2, x3)]
    aff = lambda v, i: v * sc[i][None, :, None, None] + sh[i][None, :, None, None]
    ref = t[0] + F.interpolate(aff(t[1], 0), size=(H, W), mode="bilinear", align_corners=False) \
        + F.interpolate(aff(t[2], 1), size=(H, W), mode="bilinear", align_corners=False) + aff(t[3], 2)
    ref = F.relu(ref)
    close(z, ref.permute(0, 2, 3, 1), BF16_TOL, "fuse fwd")
    dz = rnd((n, H, W, c), 5)
    ref.backward(dz.float().permute(0, 3, 1, 2))
    for v, tt, i in ((x1, t[1], 0), (x2, t[2], 1)):
        gl = raw.upsample_adjoint(dz, z, v.shape[1], v.shape[2])
        want = tt.grad.permute(0, 2, 3, 1) / sc[i][None, None, None, :]
        close(gl, want, BF16_TOL, "upsample adjoint")
    # x8 and odd sizes, no mask, accumulate
    g = rnd((1, 40, 72, 16), 7)
    small = torch.zeros((1, 5, 9, 16), device="cuda", requires_grad=True)
    F.interpolate(small.permute(0, 3, 1, 2), size=(40, 72), mode="bilinear", align_corners=False) \
        .backward(g.float().permute(0, 3, 1, 2))
    base = rnd((1, 5, 9, 16), 8)
    got = raw.upsample_adjoint(g, None, 5, 9, out=base.clone(), accumulate=True)
    close(got, small.grad + base.float(), BF16_TOL, "adjoint x8 accumulate")


def test_image_prep():
    raw = _setup()
    img = torch.randn((2, 3, 64, 96), device="cuda")
    full = raw.image_prep(img, 64, 96)
    close(full[..., :3], img.permute(0, 2, 3, 1), BF16_TOL / 2, "image copy")
    assert float(full[..., 3:].abs().max()) == 0.0
    half = raw.image_prep(img, 32, 48)
    ref = F.interpolate(img, scale_factor=0.5, mode="bilinear", align_corners=False, recompute_scale_factor=True)
    close(half[..., :3], ref.permute(0, 2, 3, 1), BF16_TOL / 2, "ResizeX 0.5")


def test_ocr_softmax_glue():
    raw = _setup()
    n, P, K = 2, 1000, 19
    logits = torch.randn((n, P, 20), device="cuda") * 3
    probs = raw.spatial_softmax_fwd(logits, K)
    lr = logits[..., :K].clone().requires_grad_(True)
    ref = F.softmax(lr, dim=1)
    close(probs[..., :K], ref, BF16_TOL, "spatial softmax")
    assert float(probs[..., K:].abs().max()) == 0.0
    dpr = torch.randn((n, P, 20), device="cuda")
    probs_f = probs.float()[..., :K].detach()
    want = probs_f * (dpr[..., :K] - (probs_f * dpr[..., :K]).sum(1, keepdim=True))
    dl = torch.zeros((n, P, 32), dtype=torch.bfloat16, device="cuda")
    raw.spatial_softmax_bwd(dpr, probs, K, dl, True)
    close(dl[..., :K], want, BF16_TOL, "spatial softmax bwd")
    x = torch.randn((P, 20), device="cuda") * 8
    sim = raw.class_softmax_fwd(x, K, 1.0 / 16)
    close(sim[:, :K], F.softmax(x[:, :K] / 16, dim=1), BF16_TOL, "class softmax")
    dsim = torch.randn((P, 20), device="cuda")
    s = sim.float()[:, :K]
    want = (s * (dsim[:, :K] - (s * dsim[:, :K]).sum(1, keepdim=True))) / 16
    close(raw.class_softmax_bwd(dsim, sim, K, 1.0 / 16)[:, :K], want, BF16_TOL, "class softmax bwd")
    m = rnd((19, 256), 3)
    tp = raw.transpose_pad(m, 24)
    assert tp.shape == (256, 24) and torch.equal(tp[:, :19], m.t()) and float(tp[:, 19:].abs().max()) == 0.0


@pytest.mark.parametrize("two_scale,sup", [(True, 0.0), (True, 0.05), (False, 0.0)])
def test_mscale_loss_fwd_bwd(two_scale, sup):
    raw = _setup()
    n, H, W = 2, 64, 96
    hq, wq = H // 4, W // 4
    hm, wm, hl, wl = (H // 2, W // 2, H // 8, W // 8) if two_scale else (0, 0, 0, 0)
    g = torch.Generator(device="cuda").manual_seed(0)
    mk = lambda *s: torch.randn(s, generator=g, device="cuda")
    hi_cls, hi_aux = torch.zeros((n, hq, wq, 20), device="cuda"), torch.zeros((n, hq, wq, 20), device="cuda")
    hi_cls[..., :19], hi_aux[..., :19] = mk(n, hq, wq, 19) * 2, mk(n, hq, wq, 19) * 2
    gts = torch.randint(0, 19, (n, H, W), generator=g, device="cuda")
    gts[:, :5] = 255
    d = raw.mscale_desc(n, H, W, hq, wq, hm, wm, hl, wl, 2, 1.0, 0.4, sup)
    leaves = [hi_cls[..., :19].permute(0, 3, 1, 2).clone().requires_grad_(True),
              hi_aux[..., :19].permute(0, 3, 1, 2).clone().requires_grad_(True)]
    up = lambda t, size: F.interpolate(t, size=size, mode="bilinear", align_corners=False)
    ce = lambda t: F.nll_loss(F.log_softmax(t, dim=1), gts, ignore_index=255)
    if two_scale:
        lo_cls, lo_aux = torch.zeros((n, hl, wl, 20), device="cuda"), torch.zeros((n, hl, wl, 20), device="cuda")
        lo_cls[..., :19], lo_aux[..., :19] = mk(n, hl, wl, 19) * 2, mk(n, hl, wl, 19) * 2
        lo_attn = mk(n, hl, wl, 1).contiguous()
        leaves += [lo_cls[..., :19].permute(0, 3, 1, 2).clone().requires_grad_(True),
                   lo_aux[..., :19].permute(0, 3, 1, 2).clone().requires_grad_(True),
                   lo_attn.permute(0, 3, 1, 2).clone().requires_grad_(True)]
        a = up(torch.sigmoid(leaves[4]), (hm, wm))
        p_lo = up(a * up(leaves[2], (hm, wm)), (H, W))
        aux_lo = up(a * up(leaves[3], (hm, wm)), (H, W))
        a_up = up(a, (H, W))
        joint = p_lo + (1 - a_up) * up(leaves[0], (H, W))
        joint_aux = aux_lo + (1 - a_up) * up(leaves[1], (H, W))
        ref = 0.4 * ce(joint_aux) + ce(joint)
        if sup:
            ref = ref + sup * ce(up(up(leaves[2], (hm, wm)), (H, W))) + sup * ce(up(leaves[0], (H, W)))
        mid, mid_sup = raw.mscale_mid_fwd(d, lo_cls, lo_aux, lo_attn)
    else:
        ref = 0.4 * ce(up(leaves[1], (H, W))) + ce(up(leaves[0], (H, W)))
        mid = mid_sup = None
    ref.backward()
    inv = raw.count_valid(gts)
    loss, g_hi, g_lo, g_sup = raw.mscale_loss_fwd(d, gts, inv, hi_cls, hi_aux, mid, mid_sup)
    assert abs(float(loss[0]) - float(ref)) <= 2e-5 * abs(float(ref)), (float(loss[0]), float(ref))
    d_cls, d_aux = raw.mscale_hi_bwd(d, g_hi)
    gscale = max(leaves[0].grad.abs().max().item(), 1e-12)
    close(d_cls[..., :19], leaves[0].grad.permute(0, 2, 3, 1), 2 * BF16_TOL, "d hi cls")
    close(d_aux[..., :19], leaves[1].grad.permute(0, 2, 3, 1), 2 * BF16_TOL, "d hi aux")
    assert float(d_cls[..., 19:].abs().max()) == 0.0 and gscale > 0
    if two_scale:
        dl_cls, dl_aux, dl_attn = raw.mscale_lo_bwd(d, g_lo, g_sup, lo_cls, lo_aux, lo_attn, mid)
        close(dl_cls[..., :19], leaves[2].grad.permute(0, 2, 3, 1), 2 * BF16_TOL, "d lo cls")
        close(dl_aux[..., :19], leaves[3].grad.permute(0, 2, 3, 1), 2 * BF16_TOL, "d lo aux")
        close(dl_attn[..., :1], leaves[4].grad.permute(0, 2, 3, 1), 2 * BF16_TOL, "d lo attn logit")


@pytest.mark.parametrize("two_scale,sup", [(True, 0.0), (True, 0.05), (False, 0.0)])
def test_rmi_criterion_fwd_bwd(two_scale, sup):
    """RMILoss criterion (loss/rmi.py) on the blended logits: sigmoid-BCE heads + the region-mutual-information term of
    the main head, against the oracle's fp64 restatement (pinned to the reference by tests/golden) with autograd."""
    from oracle import seg_oracle as O
    raw = _setup()
    n, H, W = 2, 64, 96
    hq, wq = H // 4, W // 4
    hm, wm, hl, wl = (H // 2, W // 2, H // 8, W // 8) if two_scale else (0, 0, 0, 0)
    g = torch.Generator(device="cuda").manual_seed(0)
    mk = lambda *s: torch.randn(s, generator=g, device="cuda")
    hi_cls, hi_aux = torch.zeros((n, hq, wq, 20), device="cuda"), torch.zeros((n, hq, wq, 20), device="cuda")
    hi_cls[..., :19], hi_aux[..., :19] = mk(n, hq, wq, 19) * 2, mk(n, hq, wq, 19) * 2
    gts = torch.randint(0, 19, (n, H, W), generator=g, device="cuda")
    gts[:, :5] = 255
    gts[:, 20:30, 40:50] = 3          # a coherent region: non-trivial label covariance
    d = raw.mscale_desc(n, H, W, hq, wq, hm, wm, hl, wl, 2, 1.0, 0.4, sup, loss_kind=1)
    # contiguous NCHW leaves, like the reference network's logits: torch's CUDA avg_pool2d backward gives different
    # (wrong) gradients for channels-last strided inputs (checked against the CPU and against the closed form)
    nchw = lambda t: t.permute(0, 3, 1, 2).contiguous().clone().requires_grad_(True)
    leaves = [nchw(hi_cls[..., :19]), nchw(hi_aux[..., :19])]
    up = lambda t, size: F.interpolate(t, size=size, mode="bilinear", align_corners=False)
    crit = lambda t, do_rmi: O.rmi_loss(t, gts, do_rmi=do_rmi)
    if two_scale:
        lo_cls, lo_aux = torch.zeros((n, hl, wl, 20), device="cuda"), torch.zeros((n, hl, wl, 20), device="cuda")
        lo_cls[..., :19], lo_aux[..., :19] = mk(n, hl, wl, 19) * 2, mk(n, hl, wl, 19) * 2
        lo_attn = mk(n, hl, wl, 1).contiguous()
        leaves += [nchw(lo_cls[..., :19]), nchw(lo_aux[..., :19]), nchw(lo_attn)]
        a = up(torch.sigmoid(leaves[4]), (hm, wm))
        p_lo = up(a * up(leaves[2], (hm, wm)), (H, W))
        aux_lo = up(a * up(leaves[3], (hm, wm)), (H, W))
        a_up = up(a, (H, W))
        joint = p_lo + (1 - a_up) * up(leaves[0], (H, W))
        joint_aux = aux_lo + (1 - a_up) * up(leaves[1], (H, W))
        ref = 0.4 * crit(joint_aux, False) + crit(joint, True)
        if sup:
            ref = ref + sup * crit(up(up(leaves[2], (hm, wm)), (H, W)), False) + sup * crit(up(leaves[0], (H, W)), False)
        mid, mid_sup = raw.mscale_mid_fwd(d, lo_cls, lo_aux, lo_attn)
    else:
        ref = 0.4 * crit(up(leaves[1], (H, W)), False) + crit(up(leaves[0], (H, W)), True)
        mid = mid_sup = None
    ref.backward()
    inv = raw.count_valid(gts, plus_one=True)
    dpr, terms = raw.rmi_head(d, gts, hi_cls, mid)
    loss, g_hi, g_lo, g_sup = raw.mscale_loss_fwd(d, gts, inv, hi_cls, hi_aux, mid, mid_sup, dpr, terms)
    # the RMI value alone, against the oracle evaluated on the same blended logits
    with torch.no_grad():
        jt = joint if two_scale else up(leaves[0], (H, W))
        rmi_ref = 2.0 * (O.rmi_loss(jt, gts, do_rmi=True) - 0.5 * O.rmi_loss(jt, gts, do_rmi=False)) * 0.5
    assert abs(float(loss[5]) - float(rmi_ref)) <= 1e-4 * abs(float(rmi_ref)) + 1e-6, (float(loss[5]), float(rmi_ref))
    assert abs(float(loss[0]) - float(ref)) <= 1e-4 * abs(float(ref)), (float(loss[0]), float(ref))
    d_cls, d_aux = raw.mscale_hi_bwd(d, g_hi)
    close(d_cls[..., :19], leaves[0].grad.permute(0, 2, 3, 1), 2 * BF16_TOL, "d hi cls (rmi)")
    close(d_aux[..., :19], leaves[1].grad.permute(0, 2, 3, 1), 2 * BF16_TOL, "d hi aux (bce)")
    if two_scale:
        dl_cls, dl_aux, dl_attn = raw.mscale_lo_bwd(d, g_lo, g_sup, lo_cls, lo_aux, lo_attn, mid)
        close(dl_cls[..., :19], leaves[2].grad.permute(0, 2, 3, 1), 2 * BF16_TOL, "d lo cls (rmi)")
        close(dl_aux[..., :19], leaves[3].grad.permute(0, 2, 3, 1), 2 * BF16_TOL, "d lo aux (bce)")
        close(dl_attn[..., :1], leaves[4].grad.permute(0, 2, 3, 1), 2 * BF16_TOL, "d lo attn logit (rmi)")


def test_eval_tail_argmax_confusion_and_flip_average():
    """Device evaluation tail vs the reference's host-side softmax / max / fast_hist (utils/misc.py:50-85)."""
    raw = _setup()
    n, c, h, w = 2, 19, 37, 53
    g = torch.Generator(device="cuda").manual_seed(0)
    p0 = torch.randn((n, c, h, w), generator=g, device="cuda") * 3
    p1 = torch.randn((n, c, h, w), generator=g, device="cuda") * 3
    gts = torch.randint(0, 19, (n, h, w), generator=g, device="cuda")
    gts[:, :4] = 255
    out = raw.accum_pred(p0, None, flip=False)
    out = raw.accum_pred(p1, out, flip=True)
    ref_out = p0 + torch.flip(p1, dims=[3])
    assert torch.equal(out, ref_out)
    pm, mp, hist = raw.argmax_hist(out, gts, 0.5)
    sm = F.softmax(ref_out * 0.5, dim=1)
    rmax, rarg = sm.max(1)
    assert torch.equal(pm, rarg)                                   # bit-exact class map
    assert float((mp - rmax).abs().max()) <= 1e-6
    mask = (gts >= 0) & (gts < c)
    ref_hist = torch.bincount(c * gts[mask] + rarg[mask], minlength=c * c).view(c, c)
    assert torch.equal(hist, ref_hist)
    _, _, hist2 = raw.argmax_hist(out, gts, 0.5, hist)             # accumulates
    assert torch.equal(hist2, 2 * ref_hist)


def test_fused_sgd_matches_torch_sgd():
    """b200seg.optim.FusedSGD vs torch.optim.SGD (the optimizer of loss/optimizer.py:43-60) over several steps."""
    _setup()
    from b200seg.optim import FusedSGD
    g = torch.Generator(device="cuda").manual_seed(0)
    shapes = [(48, 32, 3, 3), (96,), (19, 512, 1, 1), (5000,)]
    pa = [torch.randn(s, generator=g, device="cuda").requires_grad_(True) for s in shapes]
    pb = [p.detach().clone().requires_grad_(True) for p in pa]
    oa = torch.optim.SGD(pa, lr=0.05, momentum=0.9, weight_decay=1e-4)
    ob = FusedSGD(pb, lr=0.05, momentum=0.9, weight_decay=1e-4)
    for step in range(4):
        for x, y in zip(pa, pb):
            gr = torch.randn(x.shape, generator=g, device="cuda")
            x.grad, y.grad = gr.clone(), (gr.clone() if y.grad is None else y.grad.copy_(gr))
        for grp in ob.param_groups:
            grp["lr"] = 0.05 * (1 - 0.1 * step)          # scheduler-style LR change
        for grp in oa.param_groups:
            grp["lr"] = 0.05 * (1 - 0.1 * step)
        oa.step()
        ob.step()
    for x, y in zip(pa, pb):
        assert float((x - y).abs().max()) <= 1e-6 * (1 + float(x.abs().max()))
        assert float((oa.state[x]["momentum_buffer"] - ob.state[y]["momentum_buffer"]).abs().max()) <= 1e-5
