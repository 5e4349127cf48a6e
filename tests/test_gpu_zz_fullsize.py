"""BASELINE.json's full configuration (HRNet-W48 + OCR + two-scale attention, one 1024x2048 crop) through properties that
need no CPU restatement at that size (the oracle takes minutes per step there; it is compared at reduced width / size in
test_gpu_model.py):

  * idempotence: the captured step replayed twice on the same batch gives the same loss and the same flat gradient, and
    the eager warm-up step agrees with the replays;
  * loss bookkeeping: total = main + OCR_ALPHA * aux (loss/utils + network/ocrnet.py:303-318);
  * softmax cross-entropy is shift invariant per pixel, so the gradient of a CE-only logit head (cls_head) sums to zero
    over the classes - for the bias (sum over pixels of sum_c dlogit_c) and for every input channel of the weight (the
    aux head also feeds the soft-region softmax over pixels: only its bias keeps the invariant). This goes
    through the attention blend, both bilinear upsampling adjoints, the bf16 logit gradients, the bias column sum and
    the weight-gradient GEMM at full size;
  * BatchNorm bookkeeping: every layer saw two forward passes per step (0.5x and 1.0x), statistics finite and positive;
  * every parameter receives a finite gradient.
Runs last (file name) because it holds ~40 GB of activations and graph pools while it runs."""
import os
import sys

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "semantic-segmentation_b200"))

pytestmark = pytest.mark.gpu


@pytest.mark.timeout(600)
def test_full_size_two_scale_step_properties():
    from b200seg.module import B200SegModule
    torch.manual_seed(0)
    net = B200SegModule("ocrnet.HRNet_Mscale", 19, ocfg=None).cuda().train()
    with torch.no_grad():       # He initialisation of the trunk (the reference's N(0, 1e-3) underflows without a checkpoint)
        for n_, p_ in net.named_parameters():
            if p_.dim() == 4 and n_.startswith("backbone"):
                p_.normal_(0, (2.0 / (p_.shape[1] * p_.shape[2] * p_.shape[3])) ** 0.5)
    g = torch.Generator().manual_seed(11)
    images = torch.randn((1, 3, 1024, 2048), generator=g).cuda()
    gts = torch.randint(0, 19, (1, 1024, 2048), generator=g)
    gts[:, :8] = 255
    gts = gts.cuda()
    drop = net.ocfg["dropout"]
    net.ocfg["dropout"] = 0.0          # identical steps: no fresh Dropout2d mask per call

    def step():
        net.zero_grad(set_to_none=True)
        loss = net({"images": images, "gts": gts})
        loss.backward()
        torch.cuda.synchronize()
        return float(loss), net._flat_grad.clone(), net.last_loss_terms.clone()

    l_eager, g_eager, _ = step()               # eager warm-up
    l_a, g_a, terms = step()                   # capture + first replay
    l_b, g_b, _ = step()                       # second replay
    net.ocfg["dropout"] = drop
    assert all(map(lambda v: v == v and abs(v) < 1e4, (l_eager, l_a, l_b))), (l_eager, l_a, l_b)

    def rel(a, b):
        return float((a.double() - b.double()).norm() / (b.double().norm() + 1e-30))

    assert abs(l_a - l_b) <= 1e-6 * abs(l_a), (l_a, l_b)
    assert rel(g_a, g_b) <= 1e-5
    assert abs(l_eager - l_a) <= 1e-4 * abs(l_a), (l_eager, l_a)
    assert rel(g_eager, g_a) <= 1e-3

    total, main, aux = (float(terms[i]) for i in range(3))
    assert abs(total - (main + net.ocr_alpha * aux)) <= 1e-5 * abs(total), (total, main, aux)
    assert abs(total - l_a) <= 1e-6 * abs(total)

    # cls_head feeds only the CE losses: shift invariance holds per pixel, so the bias gradient AND every weight column
    # sum to zero over the classes. aux_head.2 additionally feeds SpatialGather's softmax over PIXELS (the reference does
    # not detach aux_out, network/ocrnet.py:88-89): that path's gradient sums to zero over the pixels of a class, so only
    # the bias (sum over pixels AND classes) keeps the invariant, a weight column does not.
    for head, columns in (("ocr.cls_head", True), ("ocr.aux_head.2", False)):
        gb = net.get_parameter(head + ".bias").grad.double()
        gw = net.get_parameter(head + ".weight").grad.double().flatten(1)        # [19, Cin]
        assert gb.abs().sum() > 0 and gw.abs().sum() > 0, head
        assert abs(float(gb.sum())) <= 2e-3 * float(gb.abs().sum()), (head, gb)
        if columns:
            col = gw.sum(0).abs().sum() / gw.abs().sum()
            assert float(col) <= 2e-3, (head, float(col))

    n_nonfinite = 0
    for name, p in net.named_parameters():
        assert p.grad is not None, name
        n_nonfinite += int((~torch.isfinite(p.grad)).sum())
    assert n_nonfinite == 0
    assert float(g_a.norm()) > 0

    sd = net.state_dict()
    nbt = {int(v) for k, v in sd.items() if k.endswith("num_batches_tracked")}
    assert nbt == {6}, nbt                      # 3 steps x 2 scale passes (the reference's BN modules run twice per step)
    for k, v in sd.items():
        if k.endswith("running_var"):
            assert bool(torch.isfinite(v).all()) and float(v.min()) > 0, k
        elif k.endswith("running_mean"):
            assert bool(torch.isfinite(v).all()), k


def _dump(name, obj):
    import json
    out = os.path.join(ROOT, "gpurun_out")
    try:
        os.makedirs(out, exist_ok=True)
        with open(os.path.join(out, name), "w") as f:
            json.dump(obj, f, indent=1)
    except OSError:
        pass


@pytest.mark.timeout(900)
def test_full_size_value_parity_vs_gpu_oracle():
    """VALUE parity at the BASELINE configuration (HRNet-W48 + OCR + two-scale attention, one 1024x2048 crop): the fused
    step against the oracle run on the same GPU through stock PyTorch (fp32 cuDNN, TF32 off, bf16-storage emulation):
      * loss to 5e-3 relative;
      * every per-tensor gradient (955 tensors: stem, every stage, OCR, attention) within the oracle's own noise floor
        under a one-bf16-ulp input perturbation (tests/_parity.py explains why that is the meaningful bar), at least 24
        named tensors spanning the depth reported, the tensors next to the loss to cosine >= 0.99;
      * running statistics of all 316 BatchNorm layers after the step;
      * eval mode (running statistics, no batch-statistics feedback): 'pred' to 3 % L2, argmax agreement >= 99.9 % and
        bit-exact wherever the oracle's top-2 margin exceeds 2 % of the logit range."""
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import _parity as P
    from oracle import seg_oracle as O
    from b200seg.module import B200SegModule
    arch, hcfg = "ocrnet.HRNet_Mscale", O.HRNET_W48
    sd0 = O.synth_state_dict(arch, hcfg, seed=3)
    images, gts = O.synth_batch(1, 1024, 2048, seed=5)
    sd_ref, loss_ref = P.oracle_train_step(O, arch, hcfg, sd0, images, gts)
    ref_grads = {k: v.grad.detach().clone() for k, v in sd_ref.items() if v.grad is not None}
    ref_run = {k: v.detach().clone() for k, v in sd_ref.items() if "running" in k}

    class _G:       # gradient / value holder standing in for the oracle's autograd leaves (frees its graph)
        def __init__(self, g):
            self.grad = g
    sd_ref = {k: _G(ref_grads.get(k)) for k in sd_ref}
    torch.cuda.empty_cache()
    # noise floor: the oracle against itself, input moved by one bf16 ulp
    sd_p, _ = P.oracle_train_step(O, arch, hcfg, sd0, P.ulp_perturbed(images), gts)
    floor = {n: P.cos_rel(sd_p[n].grad, g) for n, g in ref_grads.items() if float(g.abs().max()) >= 1e-12}
    run_floor = {k: float((sd_p[k].detach() - v).abs().max() / (v.abs().max() + 1e-6)) for k, v in ref_run.items()}
    del sd_p
    torch.cuda.empty_cache()
    net, lv = P.product_train_step(B200SegModule, O, arch, hcfg, sd0, images, gts)
    assert abs(lv - loss_ref) <= 5e-3 * abs(loss_ref), (lv, loss_ref)
    skip = ("ocr.conv3x3_ocr.0.bias", "ocr.aux_head.0.bias")      # bias in front of a training-mode BN: exactly zero here
    rep = {k: v for k, v in P.grad_report(net, sd_ref).items() if k not in skip}
    run_rep = {}
    for k, v in net.state_dict().items():
        if k in ref_run and not k.endswith("num_batches_tracked"):
            run_rep[k] = float((v - ref_run[k]).abs().max() / (ref_run[k].abs().max() + 1e-6))
    bad, summary = P.check_against_floor(rep, floor, run_rep, run_floor)
    names = list(rep)
    sampled = {k: dict(cos=round(rep[k][0], 4), rel=round(rep[k][1], 4), floor_cos=round(floor[k][0], 4),
                       floor_rel=round(floor[k][1], 4)) for k in names[:: max(1, len(names) // 30)]}
    near_loss = {k: rep[k][0] for k in ("ocr.cls_head.bias", "ocr.aux_head.2.bias", "ocr.cls_head.weight")}
    _dump("parity_fullsize_train.json", dict(loss=lv, loss_ref=loss_ref, summary=summary, sampled=sampled,
                                              near_loss=near_loss, running_max=max(run_rep.values()),
                                              running_floor_max=max(run_floor.values()), violations=bad[:20]))
    assert len(sampled) >= 24
    assert not bad, (summary, bad[:8])
    assert min(near_loss.values()) >= 0.99, near_loss
    assert len(run_rep) == 2 * 316
    del net
    torch.cuda.empty_cache()

    # ---- eval mode at full size
    from test_gpu_model import _condition_eval_weights
    P._tf32_off()
    g = torch.Generator().manual_seed(9)
    for k in sd0:
        if k.endswith("running_mean"):
            sd0[k] = 0.1 * torch.randn(sd0[k].shape, generator=g)
        elif k.endswith("running_var"):
            sd0[k] = 0.5 + torch.rand(sd0[k].shape, generator=g)
    _condition_eval_weights(sd0)
    net = B200SegModule(arch, 19, hcfg=hcfg)
    net.load_state_dict(sd0)
    net = net.cuda().eval()
    got = net({"images": images.cuda()})
    sd = {k: v.clone().cuda() for k, v in sd0.items()}
    with torch.no_grad():
        ref = O.mscale_two_scale(O.Ctx(sd, training=False, emulate_bf16=True), images.cuda(), hcfg=hcfg)
    assert sorted(got.keys()) == sorted(ref.keys())
    res = {}
    for k in ref:
        res[k] = P.cos_rel(got[k], ref[k])[1]
        assert res[k] <= 0.03, (k, res[k])
    a, b = got["pred"], ref["pred"]
    same = a.argmax(1) == b.argmax(1)
    top2 = b.topk(2, dim=1).values
    confident = (top2[:, 0] - top2[:, 1]) > 0.02 * float(b.abs().max())
    res.update(argmax_agree=float(same.float().mean()), confident=float(confident.float().mean()),
               confident_agree=float((same | ~confident).float().mean()))
    _dump("parity_fullsize_eval.json", res)
    assert res["argmax_agree"] >= 0.999, res
    assert res["confident"] >= 0.99 and res["confident_agree"] == 1.0, res


def test_w48_step_against_the_committed_reference_vectors(golden):
    """The W48 model on the 64x128 crop the golden script fed to the UNMODIFIED reference (tests/golden/make_golden.py ->
    'ocrnet.HRNet_Mscale/ce/w48'): loss, and the eval-mode prediction / attention samples, against the reference's own
    fp32 numbers (bf16 storage vs fp32: percent-level bounds; the matched-precision bounds are in the tests above)."""
    from oracle import seg_oracle as O
    from b200seg.module import B200SegModule
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import _parity as P
    g = golden["ocrnet.HRNet_Mscale/ce/w48"]
    arch, hcfg = "ocrnet.HRNet_Mscale", O.HRNET_W48
    sd0 = O.synth_state_dict(arch, hcfg, seed=0)
    images, gts = O.synth_batch(1, 64, 128, seed=7)
    net, lv = P.product_train_step(B200SegModule, O, arch, hcfg, sd0, images, gts)
    assert abs(lv - float(g["loss"])) <= 2e-2 * float(g["loss"]), (lv, float(g["loss"]))
    assert len(net.state_dict()) == g["nkeys"] and sum(p.numel() for p in net.parameters()) == g["nparams"]
    c, r = P.cos_rel(O.sample_like(net.get_parameter("ocr.cls_head.weight").grad), g["grad_cls"])
    assert c >= 0.9, (c, r)
    cls_cos = c
    net.eval()
    out = net({"images": images.cuda()})
    # untrained synthetic heads put soft-region logits at +-150 in front of a softmax (see _condition_eval_weights in
    # test_gpu_model.py): bf16-vs-fp32 eval maps of THIS weight set agree only coarsely; recorded, loosely bounded
    _, r_pred = P.cos_rel(O.sample_like(out["pred"]), g["eval_pred_sample"])
    _, r_attn = P.cos_rel(O.sample_like(out["attn_05x"]), g["eval_attn_sample"])
    _dump("parity_w48_golden.json", dict(loss=lv, loss_ref=float(g["loss"]), cls_grad_cos=cls_cos, pred_rel=r_pred,
                                         attn_rel=r_attn))
    # measured: attention 0.12, prediction 0.74 (dominated by the saturated soft-region softmax of these weights; the
    # well-conditioned eval comparison is test_full_size_value_parity_vs_gpu_oracle: 1.3 % / 99.99 % argmax)
    assert r_attn <= 0.3 and r_pred <= 1.0, (r_pred, r_attn)


def _seeded_training_run(steps):
    from b200seg.module import B200SegModule
    from b200seg.optim import FusedSGD
    torch.manual_seed(0)
    net = B200SegModule("ocrnet.HRNet_Mscale", 19).cuda().train()
    with torch.no_grad():
        for n_, p_ in net.named_parameters():
            if p_.dim() == 4 and n_.startswith("backbone"):
                p_.normal_(0, (2.0 / (p_.shape[1] * p_.shape[2] * p_.shape[3])) ** 0.5)
    opt = FusedSGD(net.parameters(), lr=1e-3, momentum=0.9, weight_decay=1e-4)
    g = torch.Generator().manual_seed(1)
    images = torch.randn((1, 3, 1024, 2048), generator=g).cuda()
    gts = torch.randint(0, 19, (1, 1024, 2048), generator=g)
    gts[:, :8] = 255
    gts = gts.cuda()
    losses = []
    for _ in range(steps):                     # eager warm-up, capture, replays; Dropout2d on, masks from the seed
        opt.zero_grad(set_to_none=True)
        loss = net({"images": images, "gts": gts})
        loss.backward()
        opt.step()
        losses.append(loss.detach().clone())
    torch.cuda.synchronize()
    out = dict(loss=torch.stack(losses).cpu(),
               grad=torch.cat([p.grad.reshape(-1) for p in net.parameters()]).cpu(),
               param=torch.cat([p.detach().reshape(-1) for p in net.parameters()]).cpu(),
               running=torch.cat([b.reshape(-1).float() for n, b in net.named_buffers() if "running_" in n]).cpu())
    del net, opt
    torch.cuda.empty_cache()
    return out


@pytest.mark.timeout(600)
def test_seeded_full_size_training_is_bit_identical():
    """bench.py's training loop (two-scale 1024x2048 step, Dropout2d on, FusedSGD) run twice from the same seed gives the
    same losses, gradients, parameters and BatchNorm running statistics bit for bit: no reduction of the step depends on
    the order in which blocks or streams finish. Otherwise a one-ulp difference grows over a few steps of training into
    different gradients, and two runs of the benchmark cannot be compared output for output."""
    a, b = _seeded_training_run(5), _seeded_training_run(5)
    for k in a:
        diff = int((a[k] != b[k]).sum())
        assert diff == 0, (k, diff, float((a[k] - b[k]).abs().max()))
