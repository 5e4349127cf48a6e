"""Boundary proof (SURVEY.md §8b): the calls the reference's train.py makes on the `network` package, made in the same
order on the overlay (semantic-segmentation_b200/network + shims/runx) with the reference's --test_mode
--dataset nullloader settings: network.get_net(args, criterion) with a criterion of the reference's class name,
wrap_network_in_dataparallel, SGD on ordinary param.grad tensors over 2 epochs x 11 iterations of the constant
nullloader batch (the running-average loss is finite and does not increase), validate() on the eval-mode 'pred' after
every epoch (confusion matrix -> mean IoU), the checkpoint logx.save_model writes, and its restore (the reference's
--snapshot path: torch.load on the host, load_state_dict into a freshly built wrapped network) giving the same
prediction."""
import math
import os
import sys
import types

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SHIMS = os.path.join(ROOT, "semantic-segmentation_b200", "shims")
if SHIMS not in sys.path:
    sys.path.append(SHIMS)


class CrossEntropyLoss2d(torch.nn.Module):
    """Stands in for loss/utils.py's criterion: the overlay picks its fused loss by the criterion's class name."""


def _validate(net, images, gts, num_classes=19):
    net.eval()
    with torch.no_grad():
        out = net({"images": images})
    net.train()
    pred = out["pred"]
    assert tuple(pred.shape) == (images.shape[0], num_classes) + tuple(images.shape[2:]), pred.shape
    assert bool(torch.isfinite(pred).all())
    p = pred.argmax(1).cpu().numpy().ravel()
    g = gts.cpu().numpy().ravel()
    hist = np.bincount(num_classes * g + p, minlength=num_classes ** 2).reshape(num_classes, num_classes)
    with np.errstate(divide="ignore", invalid="ignore"):
        iu = np.diag(hist) / (hist.sum(1) + hist.sum(0) - np.diag(hist))
    return pred, float(np.nanmean(iu))


@pytest.mark.timeout(600)
@pytest.mark.parametrize("arch,crop", [("ocrnet.HRNet_Mscale", "256,512"), ("basic.HRNet", "256,512"),
                                       ("mscale.HRNet", "128,256")])
def test_train_loop_runs_on_the_overlay(tmp_path, capsys, arch, crop):
    import network
    from runx.logx import logx

    logdir = str(tmp_path / "logs")
    logx.initialize(logdir=logdir, global_rank=0)
    args = types.SimpleNamespace(arch=arch, apex=False)
    criterion = CrossEntropyLoss2d()
    net = network.wrap_network_in_dataparallel(network.get_net(args, criterion), args.apex)
    assert "Model params" in capsys.readouterr().out
    optim = torch.optim.SGD(net.parameters(), lr=0.002, momentum=0.9, weight_decay=1e-4)
    h, w = (int(v) for v in crop.split(","))
    images = torch.zeros((1, 3, h, w), device="cuda")        # datasets/nullloader.py: zero image, zero mask
    gts = torch.zeros((1, h, w), dtype=torch.long, device="cuda")

    net.train()
    averages = []
    total = 0.0
    for epoch in range(2):
        for i in range(11):
            optim.zero_grad()
            main_loss = net({"images": images, "gts": gts})
            main_loss.backward()
            optim.step()
            total += main_loss.item()
            averages.append(total / (len(averages) + 1))
        pred, mean_iu = _validate(net, images, gts)
        assert 0.0 <= mean_iu <= 1.0, mean_iu
        logx.save_model({"state_dict": net.state_dict(), "optimizer": optim.state_dict(), "epoch": epoch,
                         "mean_iu": mean_iu}, metric=mean_iu, epoch=epoch)
    assert all(math.isfinite(v) for v in averages), averages
    assert averages[-1] <= averages[0] + 1e-3, averages       # running average on a constant batch: no increase
    assert all(p.grad is not None for p in net.parameters())

    ckpts = sorted(f for f in os.listdir(logdir) if f.endswith(".pth"))
    assert ckpts == ["last_checkpoint_ep0.pth", "last_checkpoint_ep1.pth"], ckpts
    checkpoint = torch.load(os.path.join(logdir, ckpts[-1]), map_location=torch.device("cpu"), weights_only=False)
    restored = network.wrap_network_in_dataparallel(network.get_net(args, criterion), args.apex)
    restored.load_state_dict(checkpoint["state_dict"])
    optim2 = torch.optim.SGD(restored.parameters(), lr=0.002, momentum=0.9, weight_decay=1e-4)
    optim2.load_state_dict(checkpoint["optimizer"])
    pred2, mean_iu2 = _validate(restored, images, gts)
    rel = float((pred2.double() - pred.double()).norm() / (pred.double().norm() + 1e-30))
    assert rel <= 1e-4, rel
    assert abs(mean_iu2 - checkpoint["mean_iu"]) <= 1e-3, (mean_iu2, checkpoint["mean_iu"])
