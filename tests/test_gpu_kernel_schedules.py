"""The persistent tensor-core kernels at shapes where each CTA runs more than one work item, against CPU fp64.

The per-kernel tests (test_gpu_kernels.py, test_gpu_backward.py, test_gpu_side_folded.py) launch at most one tile or
item per CTA and never reach the 128-wide halo instantiations.  Here every case is sized from the device's SM count so
that the launch plan (osvos_conv3x3_plan / osvos_conv3x3_wgrad_plan, the same choice function the launchers call)
reports at least 2 * grid + 1 items with a ragged last round: each CTA reaches its second tile (TMEM accumulator stage
1, the tempty hand-back, the next tile's halo prefetch, the epilogues of later tiles) and the first CTAs come back to
stage 0 with the phase flipped.  Shapes are 480x854 stage shapes where that holds at batch 1, otherwise the smallest
batch that gets there.  The fp64 references are computed once per module; comparisons are elementwise (maxrel).
Run on the B200 box:  pytest -m gpu tests/test_gpu_kernel_schedules.py -v -rP  (-rP prints the coverage table)."""
import math

import pytest
import torch
import torch.nn.functional as F

from gpu_util import maxrel, split_round

pytestmark = pytest.mark.gpu

EXACT_TOL = 3e-5    # split-bf16 three-pass products: ~2^-16 relative operand error
FAST_TOL = 3e-2     # single bf16 pass
KTILE_H, KTILE_W = 16, 8   # halo conv output tile (conv_common.cuh)


@pytest.fixture(scope="module")
def dev():
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    from osvos_pytorch_b200 import _native
    _native.load()
    return torch.device("cuda:0")


@pytest.fixture(scope="module")
def sms(dev):
    return torch.cuda.get_device_properties(0).multi_processor_count


def _tiles(h, w):
    return math.ceil(h / KTILE_H) * math.ceil(w / KTILE_W)


def _batch(n0, frame_items, sms, per_cta=2):
    """Smallest batch >= n0 whose launch has at least per_cta * SMs + 1 items (frame_items items per frame)."""
    return max(n0, math.ceil((per_cta * sms + 1) / frame_items))


def _assert_multi(plan, what, min_per_cta=2):
    items, grid = plan["items"], plan["grid"]
    assert items >= min_per_cta * grid + 1, (what, plan)
    assert items % grid != 0, (what, "last round not ragged", plan)


# ---------------------------------------------------------------- fp64 references on NHWC tensors
def conv3x3_f64(x, w, bias=None):
    """3x3 / pad 1 convolution, x [n,h,w,cin] and w [cout,cin,3,3] fp64 -> [n,h,w,cout]: nine fp64 GEMMs over the shifted
    input (the same sum as F.conv2d, whose fp64 CPU path is ~30x slower; test_fp64_references_match_conv2d)."""
    n, h, wd, cin = x.shape
    cout = w.shape[0]
    xp = F.pad(x, (0, 0, 1, 1, 1, 1))
    y = torch.zeros(n * h * wd, cout, dtype=torch.float64)
    for r in range(3):
        for s in range(3):
            y.addmm_(xp[:, r:r + h, s:s + wd, :].reshape(-1, cin), w[:, :, r, s].t())
    if bias is not None:
        y += bias
    return y.view(n, h, wd, cout)


def wgrad_f64(x, dz):
    """dW [cout,cin,3,3] of conv3x3_f64: dW[co][ci][r][s] = sum_px dz[px][co] x[px + (r-1, s-1)][ci]."""
    n, h, wd, cin = x.shape
    dz2 = dz.reshape(-1, dz.shape[3])
    xp = F.pad(x, (0, 0, 1, 1, 1, 1))
    dw = torch.empty(dz.shape[3], cin, 3, 3, dtype=torch.float64)
    for r in range(3):
        for s in range(3):
            dw[:, :, r, s] = dz2.t() @ xp[:, r:r + h, s:s + wd, :].reshape(-1, cin)
    return dw


def dgrad_weight(w):
    """The operand of the data gradient as a forward conv: w.flip(2, 3).transpose(0, 1) - what
    pack_conv3x3_weights(w, transpose_flip=True) packs."""
    return w.flip(2, 3).transpose(0, 1)


def test_fp64_references_match_conv2d():
    g = torch.Generator().manual_seed(0)
    x = torch.randn(2, 9, 13, 24, generator=g, dtype=torch.float64)
    w = torch.randn(40, 24, 3, 3, generator=g, dtype=torch.float64)
    b = torch.randn(40, generator=g, dtype=torch.float64)
    dz = torch.randn(2, 9, 13, 40, generator=g, dtype=torch.float64)
    want = F.conv2d(x.permute(0, 3, 1, 2), w, b, padding=1).permute(0, 2, 3, 1)
    assert float((conv3x3_f64(x, w, b) - want).abs().max()) < 1e-12
    wr = torch.zeros_like(w, requires_grad=True)
    F.conv2d(x.permute(0, 3, 1, 2), wr, None, padding=1).backward(dz.permute(0, 3, 1, 2))
    assert float((wgrad_f64(x, dz) - wr.grad).abs().max()) < 1e-11
    xr = x.permute(0, 3, 1, 2).clone().requires_grad_(True)
    F.conv2d(xr, w, None, padding=1).backward(dz.permute(0, 3, 1, 2))
    assert float((conv3x3_f64(dz, dgrad_weight(w)) - xr.grad.permute(0, 2, 3, 1)).abs().max()) < 1e-11


# ---------------------------------------------------------------- operands
def _act(ops, t, fast=False):
    """NHWC fp32 (device) -> Act, and the fp64 CPU copy of exactly what the exact-mode kernels read (hi + lo)."""
    a = ops.nchw_to_act(t.permute(0, 3, 1, 2), fast)
    return a, split_round(t).cpu().double()


def _randn(shape, seed, scale=1.0, dev="cuda"):
    g = torch.Generator(device=dev).manual_seed(seed)
    return torch.randn(shape, generator=g, device=dev) * scale


def _nhwc(ops, a):
    return ops.act_to_nchw(a).permute(0, 2, 3, 1).cpu()


# ---------------------------------------------------------------- forward halo conv
# name -> (frame (h, w), batch at least, cin, cout, relu, {variant: expected (block_n, planes, split_acc, lean)}).
# Tile counts at 148 SMs: stage2 304 (batch 1), conv1_2 494, stage3 432, stage4 448 (batch 2; the real batch-1 stage 4
# is 224 < 2 * 148 + 1), conv4_1 300 tiles of 256, side_prep 342 (batch 3).
FWD = {
    "stage2_64to128_250x150": ((250, 150), 1, 64, 128, True,
                               {"general": (128, 2, 1, 0), "lean": (128, 2, 1, 1), "lean_pool": (128, 2, 1, 1),
                                "threepass": (128, 2, 0, 0)}),
    "conv1_2_64to64_200x300": ((200, 300), 1, 64, 64, True,
                               {"general": (64, 2, 1, 0), "lean": (64, 2, 1, 1), "lean_pool": (64, 2, 1, 1),
                                "fast": (64, 1, 0, 0)}),
    "stage3_256to256_120x214": ((120, 214), 1, 256, 256, True,
                                {"general": (128, 2, 1, 0), "lean": (128, 2, 1, 1), "fast": (128, 1, 0, 0)}),
    "stage4_512to512_60x107": ((60, 107), 2, 512, 512, True,
                               {"general": (128, 2, 1, 0), "lean_pool": (128, 2, 1, 1)}),
    "conv4_1_256to512_155x117": ((155, 117), 1, 256, 512, True, {"fast": (256, 1, 0, 0)}),
    "side_prep_128to16_90x150": ((90, 150), 3, 128, 16, False, {"general": (16, 2, 1, 0), "fast": (16, 1, 0, 0)}),
}


def _fwd_shape(name, sms):
    (h, w), n0, cin, cout, relu, variants = FWD[name]
    block_n = min(bn for bn, *_ in variants.values())
    return _batch(n0, _tiles(h, w) * (cout // block_n), sms), h, w, cin, cout


def _fwd_kwargs(variant, relu, cout, dev):
    """ops.conv3x3 keyword arguments of a variant: general = act + fp32 outputs (+ column sums), lean = what the inference
    pass issues (bias, ReLU, act and / or pooled act only)."""
    fast = variant == "fast"
    if variant in ("general", "fast", "threepass"):
        colsum = torch.zeros(cout, device=dev) if cout >= 64 and variant == "general" else None
        return dict(relu=relu, fast=fast, out_act=True, out_f32=True, colsum=colsum)
    return dict(relu=relu, pool=variant == "lean_pool")


_FWD_CACHE = {}


def _fwd_case(name, sms, dev):
    """Operands and fp64 reference of a forward case, once per module."""
    if name not in _FWD_CACHE:
        from osvos_pytorch_b200 import ops
        n, h, w, cin, cout = _fwd_shape(name, sms)
        relu = FWD[name][4]
        seed = 1000 + cin + cout + h
        x = _randn((n, h, w, cin), seed, 3.0)
        wt = (_randn((cout, cin, 3, 3), seed + 1) * math.sqrt(2.0 / (9 * cin))).cpu()
        b = (_randn((cout,), seed + 2) * 0.1).cpu()
        xa, x64 = _act(ops, x)
        ref = conv3x3_f64(x64, split_round(wt).double(), b.double())
        if relu:
            ref = ref.relu()
        _FWD_CACHE[name] = dict(x=x, xa=xa, xa_fast=ops.nchw_to_act(x.permute(0, 3, 1, 2), True), w=wt.to(dev),
                                wp=ops.pack_conv3x3_weights(wt.to(dev)), b=b.to(dev), ref=ref, n=n)
    return _FWD_CACHE[name]


def _run_fwd(ops, c, variant, relu, cout, dev, expect):
    kw = _fwd_kwargs(variant, relu, cout, dev)
    xa = c["xa_fast"] if variant == "fast" else c["xa"]
    plan = ops.conv3x3_plan(xa, c["wp"], c["b"], cout, **kw)
    assert (plan["block_n"], plan["planes"], plan["split_acc"], plan["lean"]) == expect, (variant, plan)
    _assert_multi(plan, variant)
    out = ops.conv3x3(xa, c["wp"], c["b"], cout, **kw)
    torch.cuda.synchronize()
    return kw, out


@pytest.mark.parametrize("name", list(FWD))
def test_halo_forward_multi_tile(dev, sms, monkeypatch, name):
    from osvos_pytorch_b200 import ops
    (_, _, cin, cout, relu, variants) = FWD[name]
    c = _fwd_case(name, sms, dev)
    ref = c["ref"]
    general_act = None
    if "general" in variants:
        kw, (y, yf, _) = _run_fwd(ops, c, "general", relu, cout, dev, variants["general"])
        assert maxrel(yf.cpu(), ref) < EXACT_TOL, maxrel(yf.cpu(), ref)
        general_act = _nhwc(ops, y)
        assert torch.equal(general_act, split_round(yf.cpu()))            # act = split rounding of the fp32 result
        if kw["colsum"] is not None:
            assert maxrel(kw["colsum"].cpu(), ref.sum((0, 1, 2))) < EXACT_TOL
    for variant in ("lean", "lean_pool"):
        if variant not in variants:
            continue
        _, out = _run_fwd(ops, c, variant, relu, cout, dev, variants[variant])
        full = _nhwc(ops, out[0])
        assert maxrel(full, ref) < EXACT_TOL, (variant, maxrel(full, ref))
        if general_act is not None:
            assert torch.equal(full, general_act), variant                   # lean and general epilogues: same bits
        if variant == "lean_pool":
            want = F.max_pool2d(full.permute(0, 3, 1, 2), 2, 2, ceil_mode=True).permute(0, 2, 3, 1)
            assert torch.equal(_nhwc(ops, out[1]), want)                      # selection of the stored values
    if "fast" in variants:
        _, (y, yf, _) = _run_fwd(ops, c, "fast", relu, cout, dev, variants["fast"])
        assert maxrel(yf.cpu(), ref) < FAST_TOL, maxrel(yf.cpu(), ref)
        assert torch.equal(_nhwc(ops, y), yf.cpu().to(torch.bfloat16).float())
    if "threepass" in variants:
        monkeypatch.setenv("OSVOS_SPLITACC128", "0")                         # re-read per dispatch (conftest)
        _, (y, yf, _) = _run_fwd(ops, c, "threepass", relu, cout, dev, variants["threepass"])
        monkeypatch.delenv("OSVOS_SPLITACC128")
        assert maxrel(yf.cpu(), ref) < EXACT_TOL, maxrel(yf.cpu(), ref)
        assert torch.equal(_nhwc(ops, y), split_round(yf.cpu()))


# ---------------------------------------------------------------- dgrad, exactly as autograd.py issues it
# name -> (frame, batch at least, conv cin, conv cout, form, expected plan, tiles per CTA at least).  The dgrad conv maps
# dz [.., cout] to dx [.., cin] with the transpose-flipped packing.  "mask": a stage's inner conv (ReLU mask of the
# previous conv's output + the fused bias gradient of that conv); "dpool": a stage's first conv (no bias, no mask, no
# colsum: the lean path with bias == NULL).  Tiles at 148 SMs: 432, 432 (batch 2), 494.
DGRAD = {
    "conv3_2_mask_colsum_120x214": ((120, 214), 1, 256, 256, "mask", (128, 2, 1, 0), 2),
    "conv3_1_dpool_120x214": ((120, 214), 2, 128, 256, "dpool", (128, 2, 1, 1), 2),
    "conv1_2_mask_colsum_200x300": ((200, 300), 1, 64, 64, "mask", (64, 2, 1, 0), 3),
}


def _dgrad_shape(name, sms):
    (h, w), n0, cin, cout, form, expect, per_cta = DGRAD[name]
    return _batch(n0, _tiles(h, w) * (cin // expect[0]), sms, per_cta), h, w, cin, cout


def _dgrad_kwargs(form, cin, dev, mask_act):
    if form == "mask":
        return dict(mask=mask_act.hi, colsum=torch.zeros(cin, device=dev))
    return {}


@pytest.mark.parametrize("name", list(DGRAD))
def test_halo_dgrad_multi_tile(dev, sms, name):
    from osvos_pytorch_b200 import ops
    (_, _, cin, cout, form, expect, per_cta) = DGRAD[name]
    n, h, w, cin, cout = _dgrad_shape(name, sms)
    seed = 2000 + cin + cout
    dz = _randn((n, h, w, cout), seed, 0.5)
    wt = (_randn((cout, cin, 3, 3), seed + 1) * math.sqrt(2.0 / (9 * cin))).cpu()
    dza, dz64 = _act(ops, dz)
    wp = ops.pack_conv3x3_weights(wt.to(dev), transpose_flip=True)
    ref = conv3x3_f64(dz64, dgrad_weight(split_round(wt).double()))
    mask_act = None
    if form == "mask":
        xin = _randn((n, h, w, cin), seed + 2).clamp(min=0)                   # the forward output this gradient flows into
        mask_act, x64 = _act(ops, xin)
        ref = ref * (x64 > 0)
    kw = _dgrad_kwargs(form, cin, dev, mask_act)
    plan = ops.conv3x3_plan(dza, wp, None, cin, **kw)
    assert (plan["block_n"], plan["planes"], plan["split_acc"], plan["lean"]) == expect, plan
    _assert_multi(plan, name, per_cta)
    dx, _, _ = ops.conv3x3(dza, wp, None, cin, **kw)
    torch.cuda.synchronize()
    got = _nhwc(ops, dx)
    assert maxrel(got, ref) < EXACT_TOL, maxrel(got, ref)
    if form == "mask":
        assert maxrel(kw["colsum"].cpu(), ref.sum((0, 1, 2))) < EXACT_TOL


# ---------------------------------------------------------------- wgrad with several items per CTA
# name -> (frame, conv cin, conv cout, expected tap mode).  The batch is the smallest that the split rule
# (wgrad_tc.cu plan_wgrad) deals more than one item per CTA - at 148 SMs: conv1_2 at 480x854 needs 5 frames (444 items:
# three full rounds, the only multi-item schedule of tap rows), conv2_1 / conv2_2 at 240x427 need 4 (295 / 441 items).
# Nine-tap layers with Cin = Cout >= 256 never get a second item at 148 SMs (test_schedule_coverage).
WGRAD = {
    "conv1_2_rows_480x854": ((480, 854), 64, 64, 3),
    "conv2_1_pairs_240x427": ((240, 427), 64, 128, 5),
    "conv2_2_nine_240x427": ((240, 427), 128, 128, 9),
}


def _wgrad_plan_shape(n, h, w, cin, cout, dev):
    from osvos_pytorch_b200 import ops
    return ops.conv3x3_wgrad_plan(ops.Act.empty(n, h, w, cin, dev), ops.Act.empty(n, h, w, cout, dev), cout)


def _wgrad_batch(name, dev):
    (h, w), cin, cout, _ = WGRAD[name]
    for n in range(1, 17):
        plan = _wgrad_plan_shape(n, h, w, cin, cout, dev)
        if plan["items"] > plan["grid"]:
            return n
    raise AssertionError(f"{name}: no batch up to 16 gives more than one item per CTA on this device")


_WG_CACHE = {}


def _wgrad_case(name, dev):
    if name not in _WG_CACHE:
        from osvos_pytorch_b200 import ops
        (h, w), cin, cout, _ = WGRAD[name]
        n = _wgrad_batch(name, dev)
        seed = 3000 + cin + cout + h
        x = _randn((n, h, w, cin), seed).clamp(min=0)
        dz = _randn((n, h, w, cout), seed + 1, 0.1)
        xa, x64 = _act(ops, x)
        dza, dz64 = _act(ops, dz)
        del x, dz
        _WG_CACHE[name] = dict(xa=xa, dza=dza, ref=wgrad_f64(x64, dz64), cin=cin, cout=cout)
        del x64, dz64
    return _WG_CACHE[name]


@pytest.mark.parametrize("name", list(WGRAD))
def test_wgrad_multi_item(dev, name):
    from osvos_pytorch_b200 import ops
    c = _wgrad_case(name, dev)
    plan = ops.conv3x3_wgrad_plan(c["xa"], c["dza"], c["cout"])
    assert plan["tap_mode"] == WGRAD[name][3] and plan["planes"] == 2 and plan["split_acc"] == 1, plan
    assert plan["items"] > plan["grid"], plan
    dw = ops.conv3x3_wgrad(c["xa"], c["dza"], c["cout"])
    torch.cuda.synchronize()
    assert maxrel(dw, c["ref"]) < EXACT_TOL, maxrel(dw, c["ref"])


def test_wgrad_deferred_three_layers_one_finish(dev):
    """The training form (autograd.py): the three layers accumulate into slices of ONE zeroed arena, one wgrad_finish
    launch adds them onto existing gradients (accumulate=True, pre-filled with 0.5)."""
    from osvos_pytorch_b200 import ops
    cases = [_wgrad_case(name, dev) for name in WGRAD]
    sizes = [ops.wgrad_workspace_floats(c["cout"], c["cin"]) for c in cases]
    arena = torch.zeros(sum(sizes), device=dev)
    items, off = [], 0
    for c, sz in zip(cases, sizes):
        it = ops.conv3x3_wgrad(c["xa"], c["dza"], c["cout"], deferred_ws=arena[off:off + sz])
        off += sz
        it["dw"] = torch.full((c["cout"], c["cin"], 3, 3), 0.5, device=dev)
        it["accumulate"] = True
        items.append(it)
    ops.wgrad_finish(items)
    torch.cuda.synchronize()
    for name, c, it in zip(WGRAD, cases, items):
        assert maxrel(it["dw"], c["ref"] + 0.5) < EXACT_TOL, (name, maxrel(it["dw"], c["ref"] + 0.5))


# ---------------------------------------------------------------- stage-sized backward kernels
def _literal_branch(x, side_w, side_b, ws, bs, wf, dp, dq):
    """fp64 autograd of the literal branch: returns grads of (x, side_w, side_b, ws, bs, wf)."""
    xs = x.double().requires_grad_(True)
    p = [t.double().requires_grad_(True) for t in (side_w, side_b, ws, bs, wf)]
    feat = F.conv2d(xs, p[0], p[1], padding=1)
    pp = (feat * p[2].view(1, 16, 1, 1)).sum(1) + p[3]
    qq = (feat * p[4].view(1, 16, 1, 1)).sum(1)
    ((pp * dp.double()).sum() + (qq * dq.double()).sum()).backward()
    return [xs.grad] + [t.grad for t in p]


def _unpool_schedule(n, h, w, c, pooled, sms):
    """launch_unpool's tiles, grid and weight-table placement, restated from bwd_kernels.cu:459-465 (grid_cap(tiles, 2))."""
    oh, ow = ((h + 1) // 2, (w + 1) // 2) if pooled else (h, w)
    ppb = 256 // (c // 8)
    tiles = n * oh * math.ceil(ow / ppb)
    grid = max(1, min(tiles, 2 * sms))
    return tiles, grid, tiles >= 4 * grid


# c -> frame and batch: stage 2 at 480x854, and the 256 / 512 channel counts at frames where the weight table also goes
# to shared memory (1680 / 1680 / 1620 pooled tiles on 296 blocks at 148 SMs).
UNPOOL = {128: ((240, 427), 1), 256: ((120, 214), 2), 512: ((120, 214), 1)}


@pytest.mark.parametrize("c", list(UNPOOL))
def test_unpool_side_mask_stage_sized(dev, sms, c):
    from osvos_pytorch_b200 import ops
    (h, w), n = UNPOOL[c]
    g = torch.Generator().manual_seed(4000 + c)
    x = split_round(torch.randn(n, c, h, w, generator=g).clamp(min=0) * 2)       # a post-ReLU stage output
    side_w = torch.randn(16, c, 3, 3, generator=g) * 0.05
    side_b = torch.randn(16, generator=g) * 0.1
    ws, wf = torch.randn(16, generator=g), torch.randn(16, generator=g)
    bs = torch.randn(1, generator=g)
    dp, dq = torch.randn(n, h, w, generator=g), torch.randn(n, h, w, generator=g)
    dpool = split_round(torch.randn(n, c, (h + 1) // 2, (w + 1) // 2, generator=g))
    dx_ref = _literal_branch(x, side_w, side_b, ws, bs, wf, dp, dq)[0]
    xr = x.clone().double().requires_grad_(True)
    F.max_pool2d(xr, 2, 2, ceil_mode=True).backward(dpool.double())
    proj = torch.cat([ws, wf]).to(dev)
    (_, _, wfold), = ops.fold_side_weights_multi([(side_w.to(dev), side_b.to(dev), proj, bs.to(dev))])
    xa = ops.nchw_to_act(x.to(dev))
    dpq = torch.stack([dp, dq], dim=-1).contiguous().to(dev)
    for pooled in (True, False):
        tiles, grid, in_smem = _unpool_schedule(n, h, w, c, pooled, sms)
        assert in_smem and tiles >= 2 * grid + 1 and tiles % grid, (pooled, tiles, grid)
        want = ((xr.grad if pooled else 0) + dx_ref) * (x > 0)
        colsum = torch.zeros(c, device=dev)
        dz = ops.unpool_side_mask(ops.nchw_to_act(dpool.to(dev)) if pooled else None, xa, dpq, wfold, colsum=colsum)
        got = ops.act_to_nchw(dz).cpu()
        assert maxrel(got, want) < EXACT_TOL, (pooled, maxrel(got, want))
        assert maxrel(colsum.cpu(), want.sum((0, 2, 3))) < EXACT_TOL, pooled


SW_SLAB, SW_CHUNK, SW_STAGES = 128, 28, 4     # side_bwd_folded.cu: channels per block, pixels per chunk, ring depth


def _side_wgrad_blocks(shapes, sms):
    """Blocks per scale and chunks per block of osvos_side_folded_wgrad_multi, restated from side_bwd_folded.cu:366-377."""
    work = [n * h * math.ceil(w / SW_CHUNK) * (c // SW_SLAB) for n, h, w, c in shapes]
    total, budget, out = sum(work), 2 * sms, []
    for (n, h, w, c), wk in zip(shapes, work):
        slabs = c // SW_SLAB
        chunks = wk // slabs
        b = min(max((budget * wk + total // 2) // total // slabs, 1), chunks)
        out.append((b * slabs, chunks // b))          # (blocks, chunks of the block with the fewest)
    return out


def test_side_folded_wgrad_multi_480p_stages(dev, sms):
    """G (all nine taps) and S of the four 480x854 stage outputs in one launch; every block walks more chunks than the
    ring has stages, so the ring's phases wrap."""
    from osvos_pytorch_b200 import ops
    shapes = [(1, 240, 427, 128), (1, 120, 214, 256), (1, 60, 107, 512), (1, 30, 54, 512)]
    for (blocks, min_chunks), shape in zip(_side_wgrad_blocks(shapes, sms), shapes):
        assert min_chunks > SW_STAGES, (shape, blocks, min_chunks)
    xs, dpqs, refs = [], [], []
    for k, (n, h, w, c) in enumerate(shapes):
        x = _randn((n, h, w, c), 5000 + k, 2.0).clamp(min=0)
        dpq = _randn((n, h, w, 2), 5100 + k)
        xa, x64 = _act(ops, x)
        xs.append(xa)
        dpqs.append(dpq)
        d64 = dpq.cpu().double().reshape(-1, 2)
        xp = F.pad(x64, (0, 0, 1, 1, 1, 1))
        G = torch.stack([d64.t() @ xp[:, r:r + h, s:s + w, :].reshape(-1, c) for r in range(3) for s in range(3)])
        refs.append((G, d64.sum(0)))
    gs = [torch.zeros(ops.side_folded_wgrad_floats(c), device=dev) for *_, c in shapes]
    ops.side_folded_wgrad_multi(xs, dpqs, gs)
    torch.cuda.synchronize()
    for (n, h, w, c), gb, (G, S) in zip(shapes, gs, refs):
        got = gb.cpu()
        assert maxrel(got[:18 * c].view(9, 2, c), G) < EXACT_TOL, (c, maxrel(got[:18 * c].view(9, 2, c), G))
        assert maxrel(got[18 * c:], S) < EXACT_TOL, (c, got[18 * c:], S)


def test_conv_first_bwd_480p(dev):
    """conv1_1's weight and input gradients at 480x854 (the wgrad kernel's partial sums are replicated over kFwCopies
    slots and every block walks many 64-pixel tiles)."""
    from osvos_pytorch_b200 import ops
    h, w = 480, 854
    x = _randn((1, 3, h, w), 6000, 50.0)
    dz = _randn((1, h, w, 64), 6001, 0.1)
    wt = _randn((64, 3, 3, 3), 6002, 0.2)
    dza, dz64 = _act(ops, dz)
    dw, dx = ops.conv_first_bwd(x, dza, wt, True)
    torch.cuda.synchronize()
    x64 = x.cpu().double().permute(0, 2, 3, 1)
    assert maxrel(dw, wgrad_f64(x64, dz64)) < EXACT_TOL, maxrel(dw, wgrad_f64(x64, dz64))
    want_dx = conv3x3_f64(dz64, dgrad_weight(wt.cpu().double())).permute(0, 3, 1, 2)
    assert maxrel(dx, want_dx) < EXACT_TOL, maxrel(dx, want_dx)


# ---------------------------------------------------------------- coverage guard
def test_schedule_coverage(dev, sms, monkeypatch):
    """Every halo instantiation reachable under the default switches, and every wgrad tap mode, appears above with more
    items than CTAs.  Recorded rather than hidden: exact 256-wide halo tiles are never chosen (2200 waves256 <
    1000 waves128 cannot hold while waves128 <= 2 waves256), and nine-tap wgrad layers with Cin = Cout >= 256 never get a
    second item on this device.  Prints the table (-rP)."""
    from osvos_pytorch_b200 import ops
    rows = []
    for name, ((h, w), n0, cin, cout, relu, variants) in FWD.items():
        n = _fwd_shape(name, sms)[0]
        for variant, expect in variants.items():
            if variant == "threepass":
                monkeypatch.setenv("OSVOS_SPLITACC128", "0")
            x = ops.Act.empty(n, h, w, cin, dev, variant == "fast")
            plan = ops.conv3x3_plan(x, torch.empty(1, device=dev), torch.empty(cout, device=dev), cout,
                                    **_fwd_kwargs(variant, relu, cout, dev))
            monkeypatch.delenv("OSVOS_SPLITACC128", raising=False)
            rows.append(("conv3x3", (plan["block_n"], plan["planes"], plan["split_acc"], plan["lean"]), variant == "threepass",
                         f"{name} {variant} n={n}", plan))
    for name, ((h, w), n0, cin, cout, form, expect, per_cta) in DGRAD.items():
        n = _dgrad_shape(name, sms)[0]
        mask = ops.Act.empty(n, h, w, cin, dev)
        plan = ops.conv3x3_plan(ops.Act.empty(n, h, w, cout, dev), torch.empty(1, device=dev), None, cin,
                                **_dgrad_kwargs(form, cin, dev, mask))
        rows.append(("conv3x3", (plan["block_n"], plan["planes"], plan["split_acc"], plan["lean"]), False,
                     f"{name} n={n}", plan))
    for name, ((h, w), cin, cout, mode) in WGRAD.items():
        n = _wgrad_batch(name, dev)
        plan = _wgrad_plan_shape(n, h, w, cin, cout, dev)
        rows.append(("wgrad", plan["tap_mode"], False, f"{name} n={n}", plan))
    print(f"\nlaunch plans on {torch.cuda.get_device_name(0)} ({sms} SMs):")
    for kernel, key, _, what, p in rows:
        splits = f" pixel splits {p['pixel_splits']}" if kernel == "wgrad" else ""
        print(f"  {kernel:8s} {str(key):15s} {what:44s} items {p['items']:4d} grid {p['grid']:3d}{splits}")
    for kernel, key, _, what, p in rows:
        assert p["items"] > p["grid"], (what, p)
    # (block_n, planes, split_acc, lean) of every halo instantiation dispatch_halo can reach with default switches
    default_reachable = {(16, 1, 0, 0), (16, 2, 1, 0), (64, 1, 0, 0), (64, 2, 1, 0), (64, 2, 1, 1), (128, 1, 0, 0),
                         (128, 2, 1, 0), (128, 2, 1, 1), (256, 1, 0, 0)}
    seen = {key for kernel, key, switched, *_ in rows if kernel == "conv3x3" and not switched}
    assert seen == default_reachable, (sorted(seen), sorted(default_reachable))
    assert {key for kernel, key, *_ in rows if kernel == "wgrad"} == {3, 5, 9}
    # exact 256-wide tiles: no output size reaches them (one frame row of m tiles, cout 256 and 512, lean and general)
    chosen = set()
    for m in range(1, 6 * sms + 1):
        x = ops.Act.empty(1, KTILE_H, KTILE_W * m, 64, dev)
        for cout in (256, 512):
            for kw in (dict(relu=True), dict(out_act=True, out_f32=True)):
                p = ops.conv3x3_plan(x, torch.empty(1, device=dev), None, cout, **kw)
                chosen.add((p["block_n"], p["planes"]))
    assert (256, 1) not in chosen and (256, 2) not in chosen and chosen == {(64, 2), (128, 2)}, chosen
    print("  exact 256-wide halo tiles: never chosen for 1 .. 6 x SMs pixel tiles (cout 256 / 512)")
    # nine-tap wgrad at Cin = Cout >= 256: at most one item per CTA for the 480x854 stage shapes at any batch up to 16
    worst = 0.0
    for (h, w), c in (((120, 214), 256), ((60, 107), 512), ((30, 54), 512)):
        for n in range(1, 17):
            p = _wgrad_plan_shape(n, h, w, c, c, dev)
            worst = max(worst, p["items"] / p["grid"])
    assert worst <= 1.0, worst
    print("  nine-tap wgrad, Cin = Cout in {256, 512}: one item per CTA at every batch 1 .. 16 of the stage shapes")
