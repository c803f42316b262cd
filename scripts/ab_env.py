"""A/B of a per-launch environment switch of the library inside ONE process - development aid.

    python scripts/ab_env.py OSVOS_SPLITACC128 1 0 [H W] [--train]

For each value: the engine's CUDA graphs are dropped and re-captured, 480x854 inference is replayed 200 times over
four rotating frames (CUDA events), and the five output maps are compared with the first value's.
"""
import os
import sys
os.environ.setdefault("OSVOS_ENV_RELOAD", "1")   # the library re-reads its switches on every launch (csrc/runtime.cu)
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
torch.set_grad_enabled(False)
from oracle import osvos_oracle as oc
from osvos_pytorch_b200.networks.vgg_osvos import OSVOS, he_init_

train = "--train" in sys.argv
argv = [a for a in sys.argv if a != "--train"]
var, values = argv[1], argv[2:4]
h, w = (int(argv[4]), int(argv[5])) if len(argv) > 5 else (480, 854)
net = he_init_(OSVOS(pretrained=0, verbose=False)).cuda().eval()
xs = [oc.synthetic_frame(1, h, w, 1234 + i)[0].cuda() for i in range(4)]
ref = None
for rnd in range(2):                      # two rounds: the second repeats the measurement in reverse order
    for v in (values if rnd == 0 else values[::-1]):
        os.environ[var] = v
        net._engine._graphs.clear()
        for i in range(8):
            net(xs[i % 4])
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(200):
            net(xs[i % 4])
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / 200
        outs = [o.clone() for o in net(xs[0])]
        if ref is None:
            ref = outs
        err = max(float((a - b).abs().max() / b.abs().max()) for a, b in zip(outs, ref))
        print(f"{var}={v}: {ms:.4f} ms/frame = {1000 / ms:.1f} fps   max-rel difference to the first variant {err:.2e}")

if train:
    # the fwd + online loss + bwd micro-batch graph (dgrad with ReLU masks, wgrad, unpool ...), re-captured per value
    torch.set_grad_enabled(True)
    from osvos_pytorch_b200.layers.osvos_layers import class_balanced_cross_entropy_loss as cbce
    from osvos_pytorch_b200.training import GraphedTrainStep
    net.train()
    gts = [oc.synthetic_frame(1, h, w, 1234 + i)[1].cuda() for i in range(4)]
    gref = None
    for v in values + values[::-1]:
        os.environ[var] = v
        net._engine.drop_derived_caches()
        step = GraphedTrainStep(net, lambda o, gt: cbce(o[-1], gt, size_average=False), {"image": xs[0], "gt": gts[0]})
        for i in range(5):
            step({"image": xs[i % 4], "gt": gts[i % 4]})
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(60):
            step({"image": xs[i % 4], "gt": gts[i % 4]})
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / 60
        step.zero_grads()
        step({"image": xs[0], "gt": gts[0]})
        torch.cuda.synchronize()
        grads = {n: p.grad.detach().clone() for n, p in net.named_parameters() if p.grad is not None}
        if gref is None:
            gref = grads
        worst = max(float((grads[n] - gref[n]).norm() / (gref[n].norm() + 1e-30)) for n in gref)
        print(f"{var}={v}: fwd+bwd {ms:.4f} ms = {1000 / ms:.1f} fps   worst per-parameter gradient difference to the "
              f"first variant {worst:.2e}")
