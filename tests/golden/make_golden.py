"""Generate the golden fixtures by running the UNMODIFIED reference.

    python tests/golden/make_golden.py <reference checkout>

It imports ``networks.vgg_osvos`` and ``layers.osvos_layers`` from the
reference checkout (no edits), feeds them the seeded synthetic inputs/weights of
``oracle.osvos_oracle`` and stores what the reference returns.  The fixtures
pin the oracle (tests/test_oracle.py) and, through it, the CUDA path.

Only outputs are stored: inputs and weights are regenerated from their seeds
(torch's CPU generator is deterministic for a given torch version; the version
used is recorded in the fixture).  Of the 240x427 logit maps a seeded sample of
SAMPLED_PIXELS pixels is kept (``<case>.idx`` = flat indices into the
(n, 1, h, w) map, ``<case>.absmax<i>`` = max |logit| over the whole map), which
keeps the fixture well under 1 MB.
"""
import contextlib
import io
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
if __name__ == "__main__":
    if len(sys.argv) != 2:
        sys.exit(__doc__)
    sys.path.insert(0, os.path.abspath(sys.argv[1]))

import networks.vgg_osvos as ref_net          # noqa: E402  (reference, unmodified)
import layers.osvos_layers as ref_layers      # noqa: E402  (reference, unmodified)
from oracle import osvos_oracle as oc         # noqa: E402

SAMPLED_PIXELS = {"fwd_240x427": 8192}


def build_reference(params):
    with contextlib.redirect_stdout(io.StringIO()):
        net = ref_net.OSVOS(pretrained=0)
    sd = net.state_dict()
    for k, v in params.items():
        assert sd[k].shape == v.shape, k
        sd[k] = v.clone()
    net.load_state_dict(sd)
    return net


def grads_summary(net):
    out = {}
    for name, p in net.named_parameters():
        if p.grad is None:
            out[name] = None
        else:
            g = p.grad.detach().double().flatten()
            idx = torch.linspace(0, g.numel() - 1, steps=min(8, g.numel())).long()
            out[name] = dict(norm=float(g.norm()), sum=float(g.sum()), idx=idx.numpy(), val=g[idx].numpy())
    return out


def main():
    torch.set_num_threads(max(1, os.cpu_count() or 1))
    fx = {"torch_version": torch.__version__}
    params = oc.he_params(seed=0)
    net = build_reference(params)

    # ---- forward cases (He weights, seeded frames) -------------------------
    for tag, (n, h, w, seed) in {"fwd_48x70": (1, 48, 70, 11), "fwd_33x45_n2": (2, 33, 45, 12),
                                 "fwd_240x427": (1, 240, 427, 1234)}.items():
        x, _ = oc.synthetic_frame(n, h, w, seed)
        with torch.no_grad():
            outs = net(x)
        assert len(outs) == 5
        keep = SAMPLED_PIXELS.get(tag)
        if keep:
            fx[f"{tag}.idx"] = np.sort(np.random.default_rng(seed).choice(n * h * w, keep, replace=False)).astype(np.int32)
        for i, o in enumerate(outs):
            assert tuple(o.shape) == (n, 1, h, w)
            a = o.numpy().astype(np.float32)
            if keep:
                fx[f"{tag}.absmax{i}"] = np.array(np.abs(a).max())
                a = a.reshape(-1)[fx[f"{tag}.idx"]]
            fx[f"{tag}.out{i}"] = a

    # ---- config 1 of BASELINE.json: stock pretrained=0 init on CPU ----------
    torch.manual_seed(7)
    with contextlib.redirect_stdout(io.StringIO()):
        net0 = ref_net.OSVOS(pretrained=0)
    x, gt = oc.synthetic_frame(1, 240, 427, 1234)
    with torch.no_grad():
        outs0 = net0(x)
    loss0 = ref_layers.class_balanced_cross_entropy_loss(outs0[-1], gt, size_average=False)
    fx["cfg1.shapes"] = np.array([list(o.shape) for o in outs0])
    fx["cfg1.absmax"] = np.array([float(o.abs().max()) for o in outs0])
    fx["cfg1.loss"] = np.array(float(loss0))

    # ---- loss known-answer values from the reference ------------------------
    g = torch.Generator().manual_seed(5)
    lo = torch.randn(2, 1, 9, 13, generator=g) * 4.0
    la = torch.rand(2, 1, 9, 13, generator=g)
    fx["loss.rand.sa"] = np.array(float(ref_layers.class_balanced_cross_entropy_loss(lo, la)))
    fx["loss.rand.ba"] = np.array(float(ref_layers.class_balanced_cross_entropy_loss(lo, la, size_average=False)))
    fx["loss.rand.none"] = np.array(float(ref_layers.class_balanced_cross_entropy_loss(
        lo, la, size_average=False, batch_average=False)))
    lo_g = lo.clone().requires_grad_(True)
    ref_layers.class_balanced_cross_entropy_loss(lo_g, la, size_average=False).backward()
    fx["loss.rand.grad"] = lo_g.grad.numpy()
    z = torch.zeros(1, 1, 4, 5)
    lab = torch.zeros(1, 1, 4, 5)
    lab.view(-1)[:10] = 1.0
    fx["loss.zero.ba"] = np.array(float(ref_layers.class_balanced_cross_entropy_loss(z, lab, size_average=False)))
    fx["loss.zero.sa"] = np.array(float(ref_layers.class_balanced_cross_entropy_loss(z, lab)))
    fx["loss.m100"] = np.array(float(ref_layers.class_balanced_cross_entropy_loss(
        torch.full((1, 1, 2, 2), -100.0), torch.tensor([1.0, 0, 0, 0]).view(1, 1, 2, 2), size_average=False)))
    fx["loss.p100"] = np.array(float(ref_layers.class_balanced_cross_entropy_loss(
        torch.full((1, 1, 2, 2), 100.0), torch.ones(1, 1, 2, 2), size_average=False)))
    fx["loss.nopos"] = np.array(float(ref_layers.class_balanced_cross_entropy_loss(
        torch.randn(1, 1, 3, 3, generator=g), torch.zeros(1, 1, 3, 3), size_average=False)))

    # ---- helper tables -------------------------------------------------------
    for s in (4, 8, 16, 32):
        fx[f"upsample_filt.{s}"] = ref_layers.upsample_filt(s)
    crops = []
    for (h, w) in ((240, 427), (480, 854), (720, 1280), (1080, 1920), (33, 45), (48, 70)):
        row = [h, w]
        hh, ww = h, w
        for i in range(4):
            hh, ww = (hh + 1) // 2, (ww + 1) // 2
            s = 2 ** (i + 1)
            t = torch.zeros(1, 1, (hh + 1) * s, (ww + 1) * s)
            t[0, 0] = torch.arange(t.shape[2]).view(-1, 1) * 10000 + torch.arange(t.shape[3]).view(1, -1)
            c = ref_layers.center_crop(t, h, w)
            assert tuple(c.shape[2:]) == (h, w)
            row += [int(c[0, 0, 0, 0]) // 10000, int(c[0, 0, 0, 0]) % 10000]
        crops.append(row)
    fx["crop_table"] = np.array(crops)

    # ---- forward + backward (both objectives), 40x56, He weights -----------
    x, gt = oc.synthetic_frame(1, 40, 56, 21)
    for tag in ("online", "parent"):
        net.zero_grad()
        xin = x.clone().requires_grad_(True)       # train_online.py:121
        outs = net(xin)
        if tag == "online":
            loss = ref_layers.class_balanced_cross_entropy_loss(outs[-1], gt, size_average=False)
        else:
            ls = [ref_layers.class_balanced_cross_entropy_loss(o, gt, size_average=False) for o in outs]
            loss = 0.75 * sum(ls[:-1]) + ls[-1]     # train_parent.py:143-147 at epoch/nEpochs = .25
        loss.backward()
        fx[f"bwd.{tag}.loss"] = np.array(float(loss))
        fx[f"bwd.{tag}.xgrad"] = xin.grad.numpy().astype(np.float32)
        for name, s in grads_summary(net).items():
            if s is None:
                fx[f"bwd.{tag}.none.{name}"] = np.array(1)
            else:
                fx[f"bwd.{tag}.norm.{name}"] = np.array(s["norm"])
                fx[f"bwd.{tag}.sum.{name}"] = np.array(s["sum"])
                fx[f"bwd.{tag}.idx.{name}"] = s["idx"]
                fx[f"bwd.{tag}.val.{name}"] = s["val"]

    # ---- batch semantics of the loss counts (global over the tensor) -------
    x2, gt2 = oc.synthetic_frame(3, 24, 40, 31)
    with torch.no_grad():
        o2 = net(x2)[-1]
    fx["batch3.loss"] = np.array(float(ref_layers.class_balanced_cross_entropy_loss(o2, gt2, size_average=False)))
    fx["batch3.per_sample"] = np.array([float(ref_layers.class_balanced_cross_entropy_loss(
        o2[i:i + 1], gt2[i:i + 1], size_average=False)) for i in range(3)])

    path = os.path.join(HERE, "reference_outputs.npz")
    np.savez_compressed(path, **fx)
    print("wrote", path, os.path.getsize(path) // 1024, "KiB,", len(fx), "arrays")


if __name__ == "__main__":
    main()
