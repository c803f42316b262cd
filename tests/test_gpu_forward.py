"""Whole-path forward parity: CUDA OSVOS.forward vs the oracle and vs the golden outputs of the
unmodified reference.  Tolerance (BASELINE.json north_star): max|a-b| / max|b| <= 1e-3 per logit map in
exact mode; masks (logit > 0) must agree wherever |logit| exceeds that error bound."""
import numpy as np
import pytest
import torch

from oracle import osvos_oracle as oc
from gpu_util import golden_map, maxrel, rmsrel

pytestmark = pytest.mark.gpu

LOGIT_TOL = 1e-3


@pytest.fixture(scope="module")
def net():
    assert torch.cuda.is_available()
    from osvos_pytorch_b200.networks.vgg_osvos import OSVOS
    m = OSVOS(pretrained=0, verbose=False)
    m.load_state_dict(oc.he_params(seed=0), strict=False)
    return m.cuda().eval()


def mask_report(got, ref, tol, scale=None):
    got = got.detach().cpu().numpy() if isinstance(got, torch.Tensor) else np.asarray(got)
    ref = np.asarray(ref)
    flips = (got > 0) != (ref > 0)
    band = np.abs(ref) <= tol * (np.abs(ref).max() if scale is None else scale)
    inter = ((got > 0) & (ref > 0)).sum()
    union = ((got > 0) | (ref > 0)).sum()
    return int(flips.sum()), int((flips & ~band).sum()), float(inter / max(union, 1))


@pytest.mark.parametrize("tag,n,h,w,seed", [("fwd_48x70", 1, 48, 70, 11), ("fwd_33x45_n2", 2, 33, 45, 12),
                                            ("fwd_240x427", 1, 240, 427, 1234)])
def test_forward_vs_reference_golden(net, golden, tag, n, h, w, seed):
    """Of the 240x427 maps the fixture keeps a seeded sample of pixels: there the whole maps are also held to the
    oracle, which tests/test_oracle.py pins to the reference."""
    x, _ = oc.synthetic_frame(n, h, w, seed)
    with torch.no_grad():
        outs = net(x.cuda())
    assert isinstance(outs, list) and len(outs) == 5
    for i, o in enumerate(outs):
        assert tuple(o.shape) == (n, 1, h, w) and o.dtype == torch.float32 and o.is_cuda
        got, ref, scale = golden_map(golden, tag, i, o)
        err = maxrel(got, ref, scale)
        flips, hard_flips, iou = mask_report(got, ref, LOGIT_TOL, scale)
        print(f"{tag} out{i}: maxrel {err:.2e} rmsrel {rmsrel(got, ref):.2e} flips {flips} (outside band {hard_flips}) IoU {iou:.6f}")
        assert err <= LOGIT_TOL
        assert hard_flips == 0
        assert iou > 0.999
    if f"{tag}.idx" in golden:
        with torch.no_grad():
            full = oc.osvos_forward(oc.he_params(seed=0), x)
        for i, (o, r) in enumerate(zip(outs, full)):
            flips, hard_flips, iou = mask_report(o, r.numpy(), LOGIT_TOL)
            assert maxrel(o, r) <= LOGIT_TOL and hard_flips == 0 and iou > 0.999, i


def test_forward_stagewise_vs_oracle(net):
    """Localises an error: every stage output and side feature against the oracle."""
    from osvos_pytorch_b200 import ops
    x, _ = oc.synthetic_frame(1, 40, 56, 21)
    params = oc.he_params(seed=0)
    with torch.no_grad():
        stages = oc.trunk_forward(params, x)
        ref_outs, ref_feats = oc.osvos_forward(params, x, return_side_feats=True)
        outs, inter = net._engine.forward_inference(x.cuda(), return_intermediates=True)
    for i in range(5):
        got = ops.act_to_nchw(inter[f"stage{i}"]).cpu()
        assert maxrel(got, stages[i]) < 2e-4, (i, maxrel(got, stages[i]))
    for i in range(4):
        got = inter[f"side{i + 1}"].permute(0, 3, 1, 2).cpu()
        assert maxrel(got, ref_feats[i]) < 3e-4, (i, maxrel(got, ref_feats[i]))
    for o, r in zip(outs, ref_outs):
        assert maxrel(o, r) < LOGIT_TOL


def test_forward_simt_path_agrees(net):
    x, _ = oc.synthetic_frame(1, 24, 40, 31)
    with torch.no_grad():
        a = net._engine.forward_inference(x.cuda())
        b = net._engine.forward_inference(x.cuda(), simt=True)
    for u, v in zip(a, b):
        assert maxrel(u, v) < 1e-4


def test_forward_full_resolution_480p(net):
    """BASELINE.json configs[1] shape: 480x854, batch 1, against the oracle run on the host CPU."""
    x, _ = oc.synthetic_frame(1, 480, 854, 1234)
    params = oc.he_params(seed=0)
    with torch.no_grad():
        ref = oc.osvos_forward(params, x)
        outs = net(x.cuda())
    for i, (o, r) in enumerate(zip(outs, ref)):
        err = maxrel(o, r)
        flips, hard_flips, iou = mask_report(o, r.numpy(), LOGIT_TOL)
        print(f"480p out{i}: maxrel {err:.2e} flips {flips} (outside band {hard_flips}) IoU {iou:.6f}")
        assert err <= LOGIT_TOL and hard_flips == 0 and iou > 0.999
    # input must not be mutated, outputs are fresh tensors
    x2 = x.cuda()
    keep = x2.clone()
    with torch.no_grad():
        o1 = net(x2)
        o2 = net(x2)
    assert torch.equal(x2, keep) and o1[4].data_ptr() != o2[4].data_ptr() and torch.equal(o1[4], o2[4])


def test_fast_mode_reports_its_error(net):
    x, _ = oc.synthetic_frame(1, 240, 427, 1234)
    params = oc.he_params(seed=0)
    net.precision = "fast"
    try:
        with torch.no_grad():
            outs = net(x.cuda())
            ref = oc.osvos_forward(params, x)
    finally:
        net.precision = "exact"
    err = maxrel(outs[4], ref[4])
    flips, _, iou = mask_report(outs[4], ref[4].numpy(), LOGIT_TOL)
    print(f"fast mode 240x427 fused: maxrel {err:.2e} flips {flips} IoU {iou:.5f}")
    assert err < 5e-2 and iou > 0.97


@pytest.mark.parametrize("n,h,w", [(1, 720, 1280), (1, 1080, 1920), (3, 97, 131), (1, 17, 9)])
def test_forward_other_resolutions_vs_oracle(net, n, h, w):
    """BASELINE.json configs[4] shapes (720p, 1080p), a ragged batch, and a frame smaller than one tile at every stage."""
    x, _ = oc.synthetic_frame(n, h, w, 99)
    params = oc.he_params(seed=0)
    with torch.no_grad():
        ref = oc.osvos_forward(params, x)
        outs = net(x.cuda())
    for i, (o, r) in enumerate(zip(outs, ref)):
        err = maxrel(o, r)
        flips, hard_flips, iou = mask_report(o, r.numpy(), LOGIT_TOL)
        print(f"{n}x{h}x{w} out{i}: maxrel {err:.2e} flips {flips} (outside band {hard_flips}) IoU {iou:.6f}")
        assert err <= LOGIT_TOL and hard_flips == 0


def test_forward_is_deterministic_and_graph_equals_eager(net):
    x, _ = oc.synthetic_frame(1, 96, 160, 5)
    xc = x.cuda()
    with torch.no_grad():
        a = net(xc)
        b = net(xc)
        net._engine.use_cuda_graph = False
        try:
            c = net(xc)
        finally:
            net._engine.use_cuda_graph = True
    for u, v, z in zip(a, b, c):
        assert torch.equal(u, v) and torch.equal(u, z)


def test_direct_graph_on_a_returning_buffer(net):
    """An input buffer that comes back gets a graph captured on the buffer itself (engine._forward_graphed): the replay must
    read the buffer's CURRENT contents, give what the eager pass gives, still hand back fresh tensors, and the view form
    (fresh_outputs=False, used by SequenceSegmenter) must alias the static output."""
    eng = net._engine
    was = eng.use_cuda_graph
    try:
        eng.use_cuda_graph = True
        eng._graphs.clear()
        eng._buffers_seen.clear()
        buf = torch.empty(1, 3, 40, 56, device="cuda")
        frames = [oc.synthetic_frame(1, 40, 56, 300 + i)[0].cuda() for i in range(4)]
        with torch.no_grad():
            outs = []
            for f in frames:
                buf.copy_(f)
                outs.append([o.clone() for o in net(buf)])
            direct = [k for k in eng._graphs if len(k) == 4 and k[-1] == buf.data_ptr()]
            assert len(direct) == 1                                   # second call on: a graph bound to the buffer
            assert eng._graphs[direct[0]][1] is None                  # ... without a static input copy
            eng.use_cuda_graph = False
            for f, got in zip(frames, outs):
                want = net(f)
                for a, b in zip(got, want):
                    assert torch.equal(a, b)
            eng.use_cuda_graph = True
            buf.copy_(frames[0])
            fresh = net(buf)
            view = eng.forward(buf, fresh_outputs=False)
            assert fresh[4].data_ptr() != view[4].data_ptr() and torch.equal(fresh[4], view[4])
            buf.copy_(frames[1])
            eng.forward(buf, fresh_outputs=False)                     # replays the same entry: the view now shows frame 1
            assert torch.equal(view[4], outs[1][4]) and torch.equal(fresh[4], outs[0][4])
            # a non-contiguous / other-dtype input still goes through the generic entry
            odd = frames[2].double()
            assert torch.equal(net(odd)[4], outs[2][4])
            # the number of buffer-bound graphs is capped: further buffers use the generic entry, nothing is evicted
            eng.max_direct_graphs = 2
            more = [frames[i].clone() for i in range(3)]
            for _ in range(3):
                for i, t in enumerate(more):
                    assert torch.equal(net(t)[4], outs[i][4])
            assert sum(1 for k in eng._graphs if len(k) == 4) == 2
            # a parameter update drops every graph
            with torch.no_grad():
                net.fuse.bias.add_(1.0)
            shifted = net(buf)
            assert all(len(k) == 3 for k in eng._graphs) and not torch.equal(shifted[4], view[4])
            with torch.no_grad():
                net.fuse.bias.sub_(1.0)
    finally:
        eng.use_cuda_graph = was
        eng.max_direct_graphs = 12
        eng._graphs.clear()
