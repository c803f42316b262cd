"""Pins oracle/osvos_oracle.py against outputs of the unmodified reference
(tests/golden/reference_outputs.npz, made by tests/golden/make_golden.py) and
against the analytic known-answer values of SURVEY.md section 8c."""
import math

import numpy as np
import pytest
import torch

from gpu_util import golden_map
from oracle import osvos_oracle as oc


def maxrel(a, b):
    a, b = np.asarray(a, dtype=np.float64), np.asarray(b, dtype=np.float64)
    return float(np.abs(a - b).max() / max(np.abs(b).max(), 1e-30))


@pytest.fixture(scope="module")
def params():
    return oc.he_params(seed=0)


# ---- KAT 1/2: bilinear taps and interp_surgery ------------------------------
def test_upsample_filt_kat(golden):
    np.testing.assert_allclose(oc.upsample_filt(4), np.outer([.25, .75, .75, .25], [.25, .75, .75, .25]))
    np.testing.assert_allclose(oc.upsample_filt(8)[3] / oc.upsample_filt(8)[3].max() * .765625,
                               [.109375, .328125, .546875, .765625, .765625, .546875, .328125, .109375])
    for s in (4, 8, 16, 32):
        np.testing.assert_array_equal(oc.upsample_filt(s), golden[f"upsample_filt.{s}"])
        np.testing.assert_allclose(np.outer(oc.upsample_taps_1d(s // 2), oc.upsample_taps_1d(s // 2)),
                                   golden[f"upsample_filt.{s}"], rtol=0, atol=1e-15)


def test_interp_weight_is_diagonal():
    w = oc.interp_weight(16, 4)
    assert tuple(w.shape) == (16, 16, 8, 8)
    for i in range(16):
        for j in range(16):
            if i == j:
                np.testing.assert_allclose(w[i, j].numpy(), oc.upsample_filt(8).astype(np.float32))
            else:
                assert float(w[i, j].abs().max()) == 0.0


def test_upsample_closed_form_matches_conv_transpose():
    g = torch.Generator().manual_seed(3)
    for s, (h, w) in ((2, (5, 7)), (4, (3, 4)), (8, (2, 3)), (16, (2, 2))):
        x = torch.randn(2, 3, h, w, generator=g, dtype=torch.float64)
        ref = torch.nn.functional.conv_transpose2d(x, oc.interp_weight(3, s, torch.float64), stride=s)
        got = oc.upsample_zero_padded(x, s)
        assert got.shape == ref.shape == (2, 3, (h + 1) * s, (w + 1) * s)
        assert maxrel(got, ref) < 1e-14
    # border attenuation of a constant-1 input (SURVEY.md 8a a6)
    for s, corner in ((2, .5625), (4, .390625), (8, .31640625), (16, .2822265625)):
        one = torch.ones(1, 1, 4, 4, dtype=torch.float64)
        up = oc.upsample_zero_padded(one, s)
        crop = up[0, 0, s // 2:, s // 2:]
        assert abs(float(crop[0, 0]) - corner) < 1e-12
        assert abs(float(up[0, 0, 2 * s, 2 * s]) - 1.0) < 1e-12


# ---- KAT 6: crop offsets / pooled sizes --------------------------------------
def test_crop_table_and_pooled_sizes(golden):
    for row in golden["crop_table"]:
        h, w = int(row[0]), int(row[1])
        hh, ww = h, w
        for i in range(4):
            hh, ww = oc.pooled_size(hh), oc.pooled_size(ww)
            s = 2 ** (i + 1)
            top, _ = oc.crop_offsets((hh + 1) * s, h)
            left, _ = oc.crop_offsets((ww + 1) * s, w)
            assert (top, left) == (int(row[2 + 2 * i]), int(row[3 + 2 * i]))
    sizes = [854]
    for _ in range(4):
        sizes.append(oc.pooled_size(sizes[-1]))
    assert sizes == [854, 427, 214, 107, 54]
    assert oc.pooled_size(54) == 27
    # the table of SURVEY.md 8a a7
    t = {(int(r[0]), int(r[1])): [(int(r[2 + 2 * i]), int(r[3 + 2 * i])) for i in range(4)] for r in golden["crop_table"]}
    assert t[(240, 427)] == [(1, 1), (2, 2), (4, 6), (8, 10)]
    assert t[(480, 854)] == [(1, 1), (2, 3), (4, 5), (8, 13)]
    assert t[(1080, 1920)] == [(1, 1), (2, 2), (4, 4), (12, 8)]


# ---- KAT 3/4/5/8: the loss ---------------------------------------------------
def test_loss_known_answers(golden):
    z = torch.zeros(1, 1, 4, 5)
    lab = torch.zeros(1, 1, 4, 5)
    lab.view(-1)[:10] = 1
    v = float(oc.class_balanced_cross_entropy_loss(z, lab, size_average=False))
    assert abs(v - 2 * 10 * 10 * math.log(2) / 20) < 1e-5 and abs(v - 6.931472) < 1e-5
    assert abs(v - float(golden["loss.zero.ba"])) < 1e-5
    assert abs(float(oc.class_balanced_cross_entropy_loss(z, lab)) - 0.3465736) < 1e-6
    m = oc.class_balanced_cross_entropy_loss(torch.full((1, 1, 2, 2), -100.0),
                                             torch.tensor([1.0, 0, 0, 0]).view(1, 1, 2, 2), size_average=False)
    assert abs(float(m) - 75.0) < 1e-4 and abs(float(golden["loss.m100"]) - 75.0) < 1e-4
    p = oc.class_balanced_cross_entropy_loss(torch.full((1, 1, 2, 2), 100.0), torch.ones(1, 1, 2, 2), size_average=False)
    assert float(p) == 0.0 == float(golden["loss.p100"])
    assert float(golden["loss.nopos"]) == 0.0
    assert float(oc.class_balanced_cross_entropy_loss(torch.randn(1, 1, 3, 3), torch.zeros(1, 1, 3, 3),
                                                      size_average=False)) == 0.0


def test_loss_matches_reference_on_random(golden):
    g = torch.Generator().manual_seed(5)
    lo = torch.randn(2, 1, 9, 13, generator=g) * 4.0
    la = torch.rand(2, 1, 9, 13, generator=g)
    for key, kw in (("sa", {}), ("ba", dict(size_average=False)),
                    ("none", dict(size_average=False, batch_average=False))):
        got = float(oc.class_balanced_cross_entropy_loss(lo, la, **kw))
        assert abs(got - float(golden[f"loss.rand.{key}"])) <= 2e-6 * abs(float(golden[f"loss.rand.{key}"]))
    grad = oc.class_balanced_cross_entropy_grad(lo, la, size_average=False)
    assert maxrel(grad.numpy(), golden["loss.rand.grad"]) < 2e-6
    # closed-form gradient == autograd of the closed-form loss (fp64)
    lo64 = lo.double().requires_grad_(True)
    oc.class_balanced_cross_entropy_loss(lo64, la.double(), size_average=False).backward()
    assert maxrel(oc.class_balanced_cross_entropy_grad(lo.double(), la.double(), size_average=False), lo64.grad) < 1e-12


# ---- forward parity with the reference ---------------------------------------
@pytest.mark.parametrize("tag,n,h,w,seed", [("fwd_48x70", 1, 48, 70, 11), ("fwd_33x45_n2", 2, 33, 45, 12),
                                            ("fwd_240x427", 1, 240, 427, 1234)])
def test_forward_matches_reference(golden, params, tag, n, h, w, seed):
    x, _ = oc.synthetic_frame(n, h, w, seed)
    with torch.no_grad():
        outs = oc.osvos_forward(params, x)
    assert len(outs) == 5
    for i, o in enumerate(outs):
        assert tuple(o.shape) == (n, 1, h, w)
        got, ref, scale = golden_map(golden, tag, i, o)
        assert got.shape == ref.shape
        assert np.abs(got.astype(np.float64) - ref).max() / scale < 2e-5, (tag, i)
        # masks bit-exact except where |logit| is at the fp32 noise floor
        flips = ((got > 0) != (ref > 0)) & (np.abs(ref) > 1e-3 * scale)
        assert int(flips.sum()) == 0


def test_fusion_identity_vs_literal_route(params):
    """SURVEY.md 8a a8 / KAT 7: the linearity rewrite equals cat + 1x1 conv."""
    x, _ = oc.synthetic_frame(1, 40, 56, 21)
    p64 = {k: v.double() for k, v in params.items()}
    with torch.no_grad():
        a = oc.osvos_forward(p64, x.double())
        b = oc.osvos_forward_literal(p64, x.double())
    for u, v in zip(a, b):
        assert maxrel(u, v) < 1e-12


def test_config1_plumbing(golden):
    """BASELINE.json configs[0]: 240x427 frame, stock-scale init, CPU: shapes and a finite loss."""
    assert golden["cfg1.shapes"].tolist() == [[1, 1, 240, 427]] * 5
    assert np.isfinite(golden["cfg1.loss"]) and float(golden["cfg1.absmax"].max()) < 1e-6
    g = torch.Generator().manual_seed(7)
    p = {k: (torch.randn(v.shape, generator=g) * 0.001 if k.endswith("weight") else torch.zeros(v.shape))
         for k, v in oc.he_params(0).items()}
    x, gt = oc.synthetic_frame(1, 240, 427, 1234)
    with torch.no_grad():
        outs = oc.osvos_forward(p, x)
    assert [tuple(o.shape) for o in outs] == [(1, 1, 240, 427)] * 5
    loss = oc.class_balanced_cross_entropy_loss(outs[-1], gt, size_average=False)
    assert torch.isfinite(loss)
    # logits ~ 0  ->  loss == 2 P Nn ln2 / N, which is what the reference printed too
    assert abs(float(loss) - float(golden["cfg1.loss"])) < 1e-3 * float(golden["cfg1.loss"])


# ---- backward parity ----------------------------------------------------------
@pytest.mark.parametrize("tag", ["online", "parent"])
def test_backward_matches_reference(golden, params, tag):
    x, gt = oc.synthetic_frame(1, 40, 56, 21)
    loss, outs, grads = oc.forward_backward(params, x, gt, objective=tag, side_weight=0.75)
    assert abs(float(loss) - float(golden[f"bwd.{tag}.loss"])) < 2e-5 * abs(float(golden[f"bwd.{tag}.loss"]))
    none_ref = sorted(k.split("none.")[1] for k in golden if k.startswith(f"bwd.{tag}.none."))
    if tag == "online":   # KAT 9
        assert none_ref == sorted([f"score_dsn.{i}.{p}" for i in range(4) for p in ("weight", "bias")]
                                  + [f"upscale_.{i}.weight" for i in range(4)])
    else:
        assert none_ref == []
    for name in oc.param_shapes():
        if name.startswith("upscale"):
            continue
        if name in none_ref:
            assert name not in grads
            continue
        gsum = grads[name].double()
        ref_norm = float(golden[f"bwd.{tag}.norm.{name}"])
        assert abs(float(gsum.norm()) - ref_norm) < 1e-4 * ref_norm, name
        idx = golden[f"bwd.{tag}.idx.{name}"]
        val = golden[f"bwd.{tag}.val.{name}"]
        got = gsum.flatten()[torch.from_numpy(idx)].numpy()
        assert np.abs(got - val).max() < 2e-4 * max(np.abs(val).max(), ref_norm / math.sqrt(gsum.numel())), name


def test_batch_semantics(golden, params):
    """KAT 8: P / Nn are counted over the whole batch tensor (layers/osvos_layers.py:30-32)."""
    x, gt = oc.synthetic_frame(3, 24, 40, 31)
    with torch.no_grad():
        o = oc.osvos_forward(params, x)[-1]
    whole = float(oc.class_balanced_cross_entropy_loss(o, gt, size_average=False))
    per = [float(oc.class_balanced_cross_entropy_loss(o[i:i + 1], gt[i:i + 1], size_average=False)) for i in range(3)]
    assert abs(whole - float(golden["batch3.loss"])) < 1e-4 * abs(whole)
    np.testing.assert_allclose(per, golden["batch3.per_sample"], rtol=1e-4)
    assert abs(whole - float(np.mean(per))) > 1e-6 * abs(whole)      # NOT the mean of per-sample losses


def test_param_inventory():
    shapes = oc.param_shapes()
    assert len(shapes) == 52      # (SURVEY.md says 50; the reference state_dict has 52)
    total = sum(int(np.prod(s)) for s in shapes.values())
    assert total == 15267157
    frozen = sum(int(np.prod(s)) for k, s in shapes.items() if k.startswith("upscale"))
    assert frozen == 349520 and total - frozen == 14917637
    assert abs(oc.conv_flops(480, 854) / 1e9 - 258.23) < 0.01
    assert abs(oc.conv_flops(240, 427) / 1e9 - 64.77) < 0.01


# ---- 8(f) rows ------------------------------------------------------------------------------------------
def test_png_payload_known_answers():
    """bytescale of the sigmoid map (train_online.py:183-187 + scipy 1.0 pilutil.bytescale): extrema map to 0 / 255,
    a constant map to 0, and the mid value rounds half up."""
    x = np.array([[-50.0, 50.0], [0.0, 0.0]], dtype=np.float32)
    out = oc.png_payload(x)
    assert out.dtype == np.uint8 and out[0, 0] == 0 and out[0, 1] == 255
    assert out[1, 0] == 128                                     # (0.5 - ~0) * 255 = 127.5 -> +0.5 -> 128
    assert int(oc.png_payload(np.full((3, 4), 2.0, np.float32)).max()) == 0
    y = np.linspace(-4, 4, 97, dtype=np.float32).reshape(1, -1)
    o = oc.png_payload(y)
    assert o[0, 0] == 0 and o[0, -1] == 255 and np.all(np.diff(o[0].astype(int)) >= 0)


def test_sgd_oracle_matches_torch_optim_sgd():
    """The reference's optimizer IS torch.optim.SGD (train_online.py:79-88): pin the fp64 restatement to it."""
    g = torch.Generator().manual_seed(0)
    p = torch.nn.Parameter(torch.randn(257, generator=g))
    opt = torch.optim.SGD([{"params": [p], "weight_decay": 0.02}], lr=0.03, momentum=0.9)
    rp, rb = p.detach().clone(), None
    for _ in range(4):
        p.grad = torch.randn(257, generator=g)
        rp, rb = oc.sgd_momentum_step(rp, p.grad, rb, 0.03, 0.02, 0.9)
        opt.step()
        assert float((p.detach() - rp).abs().max()) < 1e-6


def test_scale_n_rotate_known_answers():
    """Analytic cases of the warp restatement (custom_transforms.py:7-54): identity, pure flip, 180 degrees about
    (w/2, h/2), and a 2x zoom sampling the half-pixel grid with the A = -0.75 cubic."""
    g = np.random.default_rng(0)
    img = g.standard_normal((3, 12, 17)).astype(np.float32)
    assert np.array_equal(oc.scale_n_rotate(img, 0.0, 1.0, False, False), img)           # X & 31 == 0 -> weights 0,1,0,0
    assert np.array_equal(oc.scale_n_rotate(img, 0.0, 1.0, True, False), img[:, :, ::-1])
    m = (g.random((1, 12, 17)) > 0.5).astype(np.float32)
    assert np.array_equal(oc.scale_n_rotate(m, 0.0, 1.0, False, True), m)
    r = oc.scale_n_rotate(img, 180.0, 1.0, False, True)                                    # dst(x,y) = src(w-x, h-y)
    assert np.array_equal(r[:, 1:, 1:], img[:, :0:-1, :0:-1]) and not r[:, 0].any() and not r[:, :, 0].any()
    ramp = np.tile(np.arange(17, dtype=np.float32), (1, 12, 1))                            # linear ramp along x
    z = oc.scale_n_rotate(ramp, 0.0, 2.0, False, False)                                    # src_x = 8.5 + (x - 8.5)/2
    xs = np.arange(4, 14)
    # OpenCV's A = -0.75 cubic does not reproduce linear ramps off the half-pixel: at fraction 1/4 the weights are
    # (-0.10546875, 0.87890625, 0.26171875, -0.03515625) -> first moment 0.296875 instead of 0.25 (and 0.703125 at 3/4)
    src = 8.5 + (xs - 8.5) / 2
    want = np.floor(src) + np.where(src - np.floor(src) < 0.5, 0.296875, 0.703125)
    assert np.allclose(z[0, 6, xs], want, atol=1e-5)
    const = np.full((1, 12, 17), 3.0, dtype=np.float32)
    assert np.allclose(oc.scale_n_rotate(const, 10.0, 1.2, False, False)[0, 3:9, 4:13], 3.0, atol=1e-5)   # weights sum to 1
    q = oc.scale_n_rotate(img, 17.0, 0.9, True, False)
    assert q.shape == img.shape and np.isfinite(q).all() and abs(q).max() <= abs(img).max() * 1.6


def _augment_fixture():
    import os
    path = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference_augment.npz")
    return np.load(path)


AUG_MEAN = np.array((104.00699, 116.66877, 122.67892), dtype=np.float32)


def test_scale_n_rotate_matches_the_reference_transforms():
    """PIN for 8(f) item 2: the restatement against outputs of the reference's own RandomHorizontalFlip + ScaleNRotate
    (dataloaders/custom_transforms.py:7-54, :87-100) run with the real cv2 by tests/golden/make_golden_augment.py.
    Nearest-neighbour masks must be bit-exact (integer coordinate pipeline); cubic pixels agree to fp32 summation
    order: 2e-4 on values of magnitude <= 255 * 1.4 (measured 9.2e-5)."""
    fx = _augment_fixture()
    for k in range(int(fx["n_cases"])):
        u8, gt_u8 = fx[f"c{k}.image_u8"], fx[f"c{k}.gt_u8"]
        flip, rot, sc = fx[f"c{k}.draws"]
        img = (u8.astype(np.float32) - AUG_MEAN).transpose(2, 0, 1)
        got_i = oc.scale_n_rotate(img, float(rot), float(sc), bool(flip), nearest=False)
        got_g = oc.scale_n_rotate(gt_u8.astype(np.float32)[None], float(rot), float(sc), bool(flip), nearest=True)
        assert np.array_equal(got_g[0], fx[f"c{k}.out_gt"]), k
        err = np.abs(got_i.transpose(1, 2, 0) - fx[f"c{k}.out_image"]).max()
        assert err <= 2e-4, (k, err)


def test_gated_forward_is_the_same_piecewise_linear_function():
    """oc.trunk_forward(gates=...) with the gates of the oracle's OWN forward reproduces outputs and gradients exactly
    (the gated form is the test aid of tests/test_gpu_backward.py::test_backward_with_injected_gates_*)."""
    import torch.nn.functional as F
    params = oc.he_params(seed=0)
    x, gt = oc.synthetic_frame(2, 33, 45, 5)
    names = oc.trunk_conv_names()
    outs, k, a = [], 0, x
    with torch.no_grad():
        for i, chans in enumerate(oc.STAGE_CHANNELS):
            if i > 0:
                a = F.max_pool2d(a, 2, 2, ceil_mode=True)
            for _ in chans:
                a = F.relu(F.conv2d(a, params[names[k] + ".weight"], params[names[k] + ".bias"], padding=1))
                outs.append(a)
                k += 1
    gates = oc.gates_from_activations(outs)
    l0, o0, g0 = oc.forward_backward(params, x, gt, objective="parent", side_weight=0.5)
    l1, o1, g1 = oc.forward_backward(params, x, gt, objective="parent", side_weight=0.5, gates=gates)
    assert float(l0) == float(l1)
    for a, b in zip(o0, o1):
        assert torch.equal(a, b)
    assert set(g0) == set(g1)
    for k in g0:
        assert torch.allclose(g0[k], g1[k], rtol=1e-6, atol=1e-9), k
