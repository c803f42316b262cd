"""Tensor-level wrappers over the C ABI: they allocate outputs with torch (device
memory + stream plumbing only) and enqueue the native kernels on the current
torch stream.  No arithmetic happens in Python / PyTorch here."""
from ctypes import byref

import torch

from . import _native as nat


# number of native kernels enqueued since import (bench.py reports the per-step delta)
KERNEL_LAUNCHES = [0]


def _stream():
    return torch.cuda.current_stream().cuda_stream


def _count(n=1):
    KERNEL_LAUNCHES[0] += n


class Act:
    """Split-bf16 NHWC activation tensor: value ~= hi + lo (lo is None in fast mode)."""
    __slots__ = ("hi", "lo")

    def __init__(self, hi, lo):
        self.hi = hi
        self.lo = lo

    @property
    def shape(self):
        return tuple(self.hi.shape)

    @staticmethod
    def empty(n, h, w, c, device, fast=False):
        hi = torch.empty((n, h, w, c), dtype=torch.bfloat16, device=device)
        lo = None if fast else torch.empty((n, h, w, c), dtype=torch.bfloat16, device=device)
        return Act(hi, lo)


def _require_cuda(t, name):
    if not t.is_cuda:
        raise RuntimeError(f"osvos_pytorch_b200: {name} must be a CUDA tensor; the OSVOS hot path has no CPU fallback "
                           "(the CPU restatement under oracle/ is test infrastructure only)")


def pack_conv3x3_weights(weight, transpose_flip=False, col_pad=64):
    """nn.Conv2d weight (OIHW fp32) -> packed split-bf16 GEMM operand (see include/osvos_b200.h)."""
    _require_cuda(weight, "weight")
    lib = nat.load()
    w = weight.detach().contiguous().float()
    cout, cin = int(w.shape[0]), int(w.shape[1])
    rows, cols = (cin, cout) if transpose_flip else (cout, cin)
    colp = (cols + col_pad - 1) // col_pad * col_pad
    nbytes = lib.osvos_packed_weight_bytes(rows, colp)
    packed = torch.empty(nbytes // 2, dtype=torch.bfloat16, device=w.device)
    _count()
    nat.check(lib.osvos_pack_conv3x3_weights(w.data_ptr(), packed.data_ptr(), cout, cin, int(transpose_flip), col_pad,
                                             _stream()), "osvos_pack_conv3x3_weights")
    return packed


def nchw_to_act(x, fast=False):
    _require_cuda(x, "x")
    lib = nat.load()
    x = x.contiguous().float()
    n, c, h, w = (int(v) for v in x.shape)
    a = Act.empty(n, h, w, c, x.device, fast)
    _count()
    nat.check(lib.osvos_nchw_to_act(x.data_ptr(), a.hi.data_ptr(), nat.ptr(a.lo), n, c, h, w, _stream()),
              "osvos_nchw_to_act")
    return a


def act_to_nchw(a):
    lib = nat.load()
    n, h, w, c = a.shape
    y = torch.empty((n, c, h, w), dtype=torch.float32, device=a.hi.device)
    _count()
    nat.check(lib.osvos_act_to_nchw(a.hi.data_ptr(), nat.ptr(a.lo), y.data_ptr(), n, c, h, w, _stream()),
              "osvos_act_to_nchw")
    return y


def conv_first(x, weight, bias, relu=True, fast=False):
    """conv1_1 (+ReLU) straight from the NCHW fp32 frame."""
    _require_cuda(x, "x")
    lib = nat.load()
    n, c, h, w = (int(v) for v in x.shape)
    assert c == 3 and tuple(weight.shape) == (64, 3, 3, 3)
    y = Act.empty(n, h, w, 64, x.device, fast)
    flags = (nat.FLAG_RELU if relu else 0) | (nat.FLAG_FAST if fast else 0)
    _count()
    nat.check(lib.osvos_conv_first_fwd(x.data_ptr(), weight.data_ptr(), nat.ptr(bias), y.hi.data_ptr(), nat.ptr(y.lo),
                                       n, h, w, flags, _stream()), "osvos_conv_first_fwd")
    return y


def fold_side_weights(side_w, side_b, proj_w, proj_b):
    """side_prep o {score_dsn, fuse slice} -> (packed [2, cin, 3, 3] operand, bias2 [2]); see include/osvos_b200.h."""
    lib = nat.load()
    side_w = side_w.detach().contiguous().float()
    cin = int(side_w.shape[1])
    packed = torch.empty(lib.osvos_packed_weight_bytes(2, cin) // 2, dtype=torch.bfloat16, device=side_w.device)
    bias2 = torch.empty(2, dtype=torch.float32, device=side_w.device)
    _count()
    nat.check(lib.osvos_fold_side_weights(side_w.data_ptr(), nat.ptr(side_b), proj_w.data_ptr(), nat.ptr(proj_b),
                                          packed.data_ptr(), bias2.data_ptr(), cin, _stream()), "osvos_fold_side_weights")
    return packed, bias2


def fold_side_weights_multi(entries, want_f32=True):
    """All side scales folded in ONE launch.  entries: [(side_w, side_b, proj_w [32], proj_b)] ->
    [(packed, bias2, folded_f32 [9, 2, cin] | None)]; see include/osvos_b200.h (osvos_fold_side_weights_multi)."""
    lib = nat.load()
    items = (nat.FoldItem * len(entries))()
    outs, keep = [], []
    for k, (side_w, side_b, proj_w, proj_b) in enumerate(entries):
        side_w = side_w.detach().contiguous().float()
        cin = int(side_w.shape[1])
        dev = side_w.device
        packed = torch.empty(lib.osvos_packed_weight_bytes(2, cin) // 2, dtype=torch.bfloat16, device=dev)
        bias2 = torch.empty(2, dtype=torch.float32, device=dev)
        f32 = torch.empty((9, 2, cin), dtype=torch.float32, device=dev) if want_f32 else None
        it = items[k]
        it.side_w, it.side_b = side_w.data_ptr(), nat.ptr(side_b)
        it.proj_w, it.proj_b = proj_w.data_ptr(), nat.ptr(proj_b)
        it.packed, it.bias2, it.folded_f32, it.cin = packed.data_ptr(), bias2.data_ptr(), nat.ptr(f32), cin
        keep.append(side_w)
        outs.append((packed, bias2, f32))
    _count()
    nat.check(lib.osvos_fold_side_weights_multi(items, len(entries), _stream()), "osvos_fold_side_weights_multi")
    return outs


def stage1_fused(x, w1, b1, w2_packed, b2, pool=True, out_act=False):
    """conv1_1 + ReLU + conv1_2 + ReLU (+ fused 2x2 ceil-mode max pool) of an fp32 NCHW frame in ONE kernel (exact
    mode, inference): -> (full-resolution Act | None, pooled Act | None).  See include/osvos_b200.h."""
    _require_cuda(x, "x")
    lib = nat.load()
    x = x.contiguous().float()
    n, _, h, w = (int(v) for v in x.shape)
    dev = x.device
    y = Act.empty(n, h, w, 64, dev) if out_act else None
    yp = Act.empty(n, (h + 1) // 2, (w + 1) // 2, 64, dev) if pool else None
    a = nat.Stage1Args()
    a.x, a.w1, a.b1 = x.data_ptr(), w1.data_ptr(), nat.ptr(b1)
    a.w2_packed, a.b2 = w2_packed.data_ptr(), nat.ptr(b2)
    a.y_hi, a.y_lo = (y.hi.data_ptr(), y.lo.data_ptr()) if y is not None else (None, None)
    a.pool_hi, a.pool_lo = (yp.hi.data_ptr(), yp.lo.data_ptr()) if yp is not None else (None, None)
    a.n, a.h, a.w = n, h, w
    _count()
    nat.check(lib.osvos_stage1_fused(byref(a), _stream()), "osvos_stage1_fused")
    return y, yp


def side_folded(x, packed, bias2, fast=False):
    """pq [n,h,w,2] of the folded side branch (cout == 2 call of osvos_conv3x3)."""
    lib = nat.load()
    n, h, w, cin = x.shape
    dev = x.hi.device
    pq = torch.empty((n, h, w, 2), dtype=torch.float32, device=dev)
    a = nat.Conv3x3Args()
    a.x_hi, a.x_lo = x.hi.data_ptr(), nat.ptr(x.lo)
    a.w_packed, a.bias, a.pq = packed.data_ptr(), bias2.data_ptr(), pq.data_ptr()
    a.n, a.h, a.w, a.cin, a.cout = n, h, w, cin, 2
    a.flags = nat.FLAG_FAST if fast else 0
    _count()
    nat.check(lib.osvos_conv3x3(byref(a), _stream()), "osvos_conv3x3 (folded side branch)")
    return pq


def side_folded_multi(xs, folded, fast=False):
    """The folded side branches of several scales in ONE launch: xs = stage outputs (Acts), folded = [(packed, bias2, ...)]
    per scale -> list of pq [n,h,w,2] in the same order (osvos_side_folded_multi)."""
    lib = nat.load()
    arr = (nat.Conv3x3Args * len(xs))()
    pqs = []
    for k, (x, f) in enumerate(zip(xs, folded)):
        n, h, w, cin = x.shape
        pq = torch.empty((n, h, w, 2), dtype=torch.float32, device=x.hi.device)
        a = arr[k]
        a.x_hi, a.x_lo = x.hi.data_ptr(), nat.ptr(x.lo)
        a.w_packed, a.bias, a.pq = f[0].data_ptr(), f[1].data_ptr(), pq.data_ptr()
        a.n, a.h, a.w, a.cin, a.cout = n, h, w, cin, 2
        a.flags = nat.FLAG_FAST if fast else 0
        pqs.append(pq)
    _count()
    nat.check(lib.osvos_side_folded_multi(arr, len(xs), _stream()), "osvos_side_folded_multi")
    return pqs


def _conv3x3_call(x, w_packed, bias, cout, relu, fast, out_act, out_f32, mask, proj_w, proj_b, pool, colsum, k_valid):
    """Outputs and the osvos_conv3x3_args block of one conv3x3 call -> (args, y, yf, pq, yp)."""
    n, h, w, cin = x.shape
    dev = x.hi.device
    y = Act.empty(n, h, w, cout, dev, fast) if out_act else None
    yf = torch.empty((n, h, w, cout), dtype=torch.float32, device=dev) if out_f32 else None
    pq = torch.empty((n, h, w, 2), dtype=torch.float32, device=dev) if proj_w is not None else None
    a = nat.Conv3x3Args()
    a.x_hi, a.x_lo = x.hi.data_ptr(), nat.ptr(x.lo)
    a.w_packed, a.bias = w_packed.data_ptr(), nat.ptr(bias)
    a.y_hi = nat.ptr(y.hi) if y is not None else None
    a.y_lo = nat.ptr(y.lo) if y is not None else None
    a.y_f32 = nat.ptr(yf)
    a.mask_hi = nat.ptr(mask)
    a.proj_w, a.proj_b, a.pq = nat.ptr(proj_w), nat.ptr(proj_b), nat.ptr(pq)
    yp = Act.empty(n, (h + 1) // 2, (w + 1) // 2, cout, dev, fast) if pool else None
    a.pool_hi = nat.ptr(yp.hi) if pool else None
    a.pool_lo = nat.ptr(yp.lo) if pool else None
    a.colsum = nat.ptr(colsum)
    a.k_valid = k_valid
    a.n, a.h, a.w, a.cin, a.cout = n, h, w, cin, cout
    a.flags = (nat.FLAG_RELU if relu else 0) | (nat.FLAG_FAST if fast else 0) | \
              (nat.FLAG_RELU_MASK if mask is not None else 0)
    return a, y, yf, pq, yp


def conv3x3(x, w_packed, bias, cout, relu=False, fast=False, out_act=True, out_f32=False, mask=None,
            proj_w=None, proj_b=None, simt=False, pool=False, colsum=None, k_valid=0):
    """3x3 / pad 1 conv of an Act through the tcgen05 kernel.  Returns (Act|None, f32|None, pq|None), or
    (Act, pooled Act) when pool=True (fused MaxPool2d(2,2,ceil_mode)).  `colsum` ([cout] fp32, pre-zeroed)
    receives the per-channel sum of the output (fused bias gradient)."""
    lib = nat.load()
    a, y, yf, pq, yp = _conv3x3_call(x, w_packed, bias, cout, relu, fast, out_act, out_f32, mask, proj_w, proj_b, pool,
                                     colsum, k_valid)
    fn = lib.osvos_conv3x3_simt if simt else lib.osvos_conv3x3
    _count()
    nat.check(fn(byref(a), _stream()), "osvos_conv3x3")
    if pool:
        return y, yp
    return y, yf, pq


def _plan_dict(plan):
    return {name: int(getattr(plan, name)) for name, _ in nat.LaunchPlan._fields_}


def conv3x3_plan(x, w_packed, bias, cout, relu=False, fast=False, out_act=True, out_f32=False, mask=None,
                 proj_w=None, proj_b=None, pool=False, colsum=None, k_valid=0):
    """The launch plan (osvos_conv3x3_plan) of the conv3x3 call with the same arguments, as a dict: block_n, planes,
    split_acc, lean, items, grid (tap_mode and pixel_splits are 0).  Nothing is launched."""
    lib = nat.load()
    a, *_ = _conv3x3_call(x, w_packed, bias, cout, relu, fast, out_act, out_f32, mask, proj_w, proj_b, pool, colsum,
                          k_valid)
    plan = nat.LaunchPlan()
    nat.check(lib.osvos_conv3x3_plan(byref(a), byref(plan)), "osvos_conv3x3_plan")
    return _plan_dict(plan)


def maxpool2x2(x):
    lib = nat.load()
    n, h, w, c = x.shape
    y = Act.empty(n, (h + 1) // 2, (w + 1) // 2, c, x.hi.device, x.lo is None)
    _count()
    nat.check(lib.osvos_maxpool2x2_fwd(x.hi.data_ptr(), nat.ptr(x.lo), y.hi.data_ptr(), nat.ptr(y.lo), n, h, w, c,
                                       _stream()), "osvos_maxpool2x2_fwd")
    return y


def side_project(feat, proj_w, proj_b):
    lib = nat.load()
    n, h, w, c = (int(v) for v in feat.shape)
    assert c == 16
    pq = torch.empty((n, h, w, 2), dtype=torch.float32, device=feat.device)
    _count()
    nat.check(lib.osvos_side_project(feat.data_ptr(), proj_w.data_ptr(), nat.ptr(proj_b), pq.data_ptr(), n, h, w,
                                     _stream()), "osvos_side_project")
    return pq


def tail_fwd(pqs, fuse_bias, n, h, w, label=None, out=None, loss_weights=None, divisor=None):
    """Upsample + crop + fuse (+ loss sums, + the five class-balanced BCE losses and their weighted total).
    Returns (out [5,n,1,h,w] fp32, sums [TAIL_SUMS] f64 | None) and, with `loss_weights` (5 floats) and `divisor`,
    additionally losses [6] fp32 = the five per-map losses and sum_k loss_weights[k] * loss_k."""
    lib = nat.load()
    dev = pqs[0].device
    if out is None:
        # each map starts on a 16-byte boundary so the kernel can use 128-bit stores
        per = (n * h * w + 3) // 4 * 4
        out = torch.empty((5, per), dtype=torch.float32, device=dev)[:, :n * h * w].view(5, n, 1, h, w)
    sums = torch.empty(nat.TAIL_SUMS, dtype=torch.float64, device=dev) if label is not None else None
    a = nat.TailFwdArgs()
    for k in range(4):
        a.pq[k] = pqs[k].data_ptr()
    for k in range(5):
        a.out[k] = out[k].data_ptr()
    a.fuse_bias = nat.ptr(fuse_bias)
    a.label = nat.ptr(label)
    a.sums = nat.ptr(sums)
    losses = None
    if loss_weights is not None:
        if label is None or divisor is None:
            raise ValueError("tail_fwd: loss_weights needs label and divisor")
        losses = torch.empty(6, dtype=torch.float32, device=dev)
        a.losses = losses.data_ptr()
        for k in range(5):
            a.loss_weights[k] = float(loss_weights[k])
        a.divisor = float(divisor)
    a.n, a.h, a.w = n, h, w
    _count()
    nat.check(lib.osvos_tail_fwd(byref(a), _stream()), "osvos_tail_fwd")
    if losses is not None:
        return out, sums, losses
    return out, sums


def tail_loss_bwd(out, label, sums, loss_weights, divisor, upstream, n, h, w, want_fuse_bias=True):
    """Backward of tail + the weighted class-balanced BCE objective in one launch (see include/osvos_b200.h):
    -> (list of 4 dpq tensors [n,hk,wk,2], fuse.bias gradient [1] | None)."""
    lib = nat.load()
    dev = out.device
    a = nat.TailLossBwdArgs()
    for k in range(5):
        a.logits[k] = out[k].data_ptr()
        a.loss_weights[k] = float(loss_weights[k])
    a.label, a.sums, a.upstream = label.data_ptr(), sums.data_ptr(), nat.ptr(upstream)
    a.divisor = float(divisor)
    dpq, hk, wk = [], h, w
    for k in range(4):
        hk, wk = (hk + 1) // 2, (wk + 1) // 2
        t = torch.empty((n, hk, wk, 2), dtype=torch.float32, device=dev)
        dpq.append(t)
        a.dpq[k] = t.data_ptr()
    fb = torch.empty(1, dtype=torch.float32, device=dev) if want_fuse_bias else None
    a.fuse_bias_grad = nat.ptr(fb)
    a.n, a.h, a.w = n, h, w
    _count(1)
    nat.check(lib.osvos_tail_loss_bwd(byref(a), _stream()), "osvos_tail_loss_bwd")
    return dpq, fb


# ------------------------------------------------------------------ backward ops
def wgrad_workspace_floats(dz_channels, cin):
    return nat.load().osvos_wgrad_workspace_bytes(dz_channels, cin) // 4


def _wgrad_args(x, dz, cout, fast):
    n, h, w, cin = x.shape
    a = nat.WgradArgs()
    a.x_hi, a.x_lo, a.dz_hi, a.dz_lo = x.hi.data_ptr(), nat.ptr(x.lo), dz.hi.data_ptr(), nat.ptr(dz.lo)
    a.n, a.h, a.w, a.cin, a.cout, a.dz_channels = n, h, w, cin, cout, dz.shape[3]
    a.flags = nat.FLAG_FAST if fast else 0
    return a


def conv3x3_wgrad(x, dz, cout, fast=False, deferred_ws=None):
    """dW [cout, cin, 3, 3] of a 3x3 conv from its input act `x` and output-gradient act `dz`.
    With `deferred_ws` (a ZEROED fp32 workspace of wgrad_workspace_floats(dz.channels, cin)) only the tensor-core
    accumulation is enqueued and a finish item for ops.wgrad_finish is returned instead of dW."""
    lib = nat.load()
    cin, dzc = x.shape[3], dz.shape[3]
    a = _wgrad_args(x, dz, cout, fast)
    if deferred_ws is not None:
        a.dw, a.workspace = None, deferred_ws.data_ptr()
        a.flags |= nat.FLAG_DEFER_FINISH
        _count(1)
        nat.check(lib.osvos_conv3x3_wgrad(byref(a), _stream()), "osvos_conv3x3_wgrad")
        return {"ws": deferred_ws, "cout": cout, "cin": cin, "dz_channels": dzc}
    dw = torch.empty((cout, cin, 3, 3), dtype=torch.float32, device=x.hi.device)
    ws = torch.empty(lib.osvos_wgrad_workspace_bytes(dzc, cin) // 4, dtype=torch.float32, device=x.hi.device)
    a.dw, a.workspace = dw.data_ptr(), ws.data_ptr()
    _count(3)
    nat.check(lib.osvos_conv3x3_wgrad(byref(a), _stream()), "osvos_conv3x3_wgrad")
    return dw


def conv3x3_wgrad_plan(x, dz, cout, fast=False):
    """The launch plan (osvos_conv3x3_wgrad_plan) of conv3x3_wgrad(x, dz, cout, fast) as a dict: block_n, planes,
    split_acc, lean, items, grid, tap_mode (nat.TAP_ROWS / TAP_PAIRS / TAP_NINE), pixel_splits.  Nothing is launched."""
    lib = nat.load()
    a = _wgrad_args(x, dz, cout, fast)
    a.dw = a.workspace = x.hi.data_ptr()     # required non-NULL by the argument check; never written by the query
    plan = nat.LaunchPlan()
    nat.check(lib.osvos_conv3x3_wgrad_plan(byref(a), byref(plan)), "osvos_conv3x3_wgrad_plan")
    return _plan_dict(plan)


def wgrad_finish(items):
    """One launch for the workspace -> OIHW step of many layers.  items: dicts from conv3x3_wgrad(deferred_ws=...)
    extended with 'dw' (destination tensor) and 'accumulate' (add into it, e.g. the parameter's .grad)."""
    lib = nat.load()
    for lo in range(0, len(items), nat.WGRAD_FINISH_MAX):
        part = items[lo:lo + nat.WGRAD_FINISH_MAX]
        arr = (nat.WgradFinishItem * len(part))()
        for f, it in zip(arr, part):
            f.workspace, f.dw = it["ws"].data_ptr(), it["dw"].data_ptr()
            f.cout, f.cin, f.dz_channels = it["cout"], it["cin"], it["dz_channels"]
            f.accumulate, f.scale = int(bool(it.get("accumulate"))), 1.0
        _count(1)
        nat.check(lib.osvos_wgrad_finish(arr, len(part), _stream()), "osvos_wgrad_finish")


def tail_bwd(grads, n, h, w):
    """grads: list of 5 tensors [n,1,h,w] or None -> list of 4 dpq tensors [n,hk,wk,2]."""
    lib = nat.load()
    dev = next(g for g in grads if g is not None).device
    a = nat.TailBwdArgs()
    keep = []
    for k in range(5):
        g = grads[k]
        if g is not None:
            g = g.contiguous().float()
            keep.append(g)
        a.grad_out[k] = nat.ptr(g)
    dpq, hk, wk = [], h, w
    for k in range(4):
        hk, wk = (hk + 1) // 2, (wk + 1) // 2
        t = torch.empty((n, hk, wk, 2), dtype=torch.float32, device=dev)
        dpq.append(t)
        a.dpq[k] = t.data_ptr()
    a.n, a.h, a.w = n, h, w
    _count(1)
    nat.check(lib.osvos_tail_bwd(byref(a), _stream()), "osvos_tail_bwd")
    return dpq


def sum_f32(x):
    lib = nat.load()
    x = x.contiguous().float()
    scratch = torch.empty(2, dtype=torch.float64, device=x.device)
    out = torch.empty(1, dtype=torch.float32, device=x.device)
    _count(1)
    nat.check(lib.osvos_sum_f32(x.data_ptr(), x.numel(), scratch.data_ptr(), out.data_ptr(), _stream()),
              "osvos_sum_f32")
    return out


def unpool_add_mask(dpool, x, dside, colsum=None):
    lib = nat.load()
    n, h, w, c = x.shape
    dz = Act.empty(n, h, w, c, x.hi.device, x.lo is None)
    _count()
    nat.check(lib.osvos_unpool_add_mask(dpool.hi.data_ptr(), nat.ptr(dpool.lo), x.hi.data_ptr(), nat.ptr(x.lo),
                                        nat.ptr(dside), dz.hi.data_ptr(), nat.ptr(dz.lo), nat.ptr(colsum), n, h, w, c,
                                        _stream()),
              "osvos_unpool_add_mask")
    return dz


def unpool_side_mask(dpool, x, dpq, wfold, colsum=None):
    """dz = ReLU'(x) * (unpool(dpool) + folded side gradient of dpq); dpool None: no pooling consumer."""
    lib = nat.load()
    n, h, w, c = x.shape
    dz = Act.empty(n, h, w, c, x.hi.device, x.lo is None)
    _count()
    nat.check(lib.osvos_unpool_side_mask(dpool.hi.data_ptr() if dpool is not None else None,
                                         nat.ptr(dpool.lo) if dpool is not None else None, x.hi.data_ptr(), nat.ptr(x.lo),
                                         dpq.data_ptr(), wfold.data_ptr(), dz.hi.data_ptr(), nat.ptr(dz.lo),
                                         nat.ptr(colsum), n, h, w, c, _stream()),
              "osvos_unpool_side_mask")
    return dz


def side_folded_wgrad_floats(c):
    return int(nat.load().osvos_side_folded_wgrad_floats(c))


def side_folded_wgrad(x, dpq, g):
    """g ([18 c + 2] fp32, PRE-ZEROED) += folded weight gradient of the side branch (include/osvos_b200.h)."""
    lib = nat.load()
    n, h, w, c = x.shape
    _count()
    nat.check(lib.osvos_side_folded_wgrad(x.hi.data_ptr(), nat.ptr(x.lo), dpq.data_ptr(), g.data_ptr(), n, h, w, c,
                                          _stream()), "osvos_side_folded_wgrad")
    return g


def side_folded_wgrad_multi(xs, dpqs, gs):
    """side_folded_wgrad of several scales in ONE launch (osvos_side_folded_wgrad_multi)."""
    lib = nat.load()
    arr = (nat.SideWgradItem * len(xs))()
    for it, x, dpq, g in zip(arr, xs, dpqs, gs):
        n, h, w, c = x.shape
        it.x_hi, it.x_lo, it.dpq, it.g = x.hi.data_ptr(), nat.ptr(x.lo), dpq.data_ptr(), g.data_ptr()
        it.n, it.h, it.w, it.c = n, h, w, c
    _count()
    nat.check(lib.osvos_side_folded_wgrad_multi(arr, len(xs), _stream()), "osvos_side_folded_wgrad_multi")


def side_grads_finish(entries, accumulate):
    """entries: dicts with g, side_w, side_b, proj_w, d_side_w, d_side_b, d_score_w, d_score_b, d_fuse_w (tensors or
    None), c.  One launch for all scales."""
    lib = nat.load()
    items = (nat.SideGradsItem * len(entries))()
    for k, e in enumerate(entries):
        it = items[k]
        it.g, it.side_w, it.side_b, it.proj_w = e["g"].data_ptr(), e["side_w"].data_ptr(), nat.ptr(e["side_b"]), \
            e["proj_w"].data_ptr()
        it.d_side_w, it.d_side_b = e["d_side_w"].data_ptr(), e["d_side_b"].data_ptr()
        it.d_score_w, it.d_score_b, it.d_fuse_w = nat.ptr(e.get("d_score_w")), nat.ptr(e.get("d_score_b")), \
            nat.ptr(e.get("d_fuse_w"))
        it.c, it.accumulate = int(e["c"]), 1 if accumulate else 0
    _count()
    nat.check(lib.osvos_side_grads_finish(items, len(entries), _stream()), "osvos_side_grads_finish")


def channel_sum(a):
    lib = nat.load()
    n, h, w, c = a.shape
    out = torch.empty(c, dtype=torch.float32, device=a.hi.device)
    _count()
    nat.check(lib.osvos_channel_sum(a.hi.data_ptr(), nat.ptr(a.lo), out.data_ptr(), n * h * w, c, _stream()),
              "osvos_channel_sum")
    return out


def conv_first_bwd(x, dz, weight, need_dx):
    lib = nat.load()
    n, _, h, w = (int(v) for v in x.shape)
    dw = torch.empty((64, 3, 3, 3), dtype=torch.float32, device=x.device)
    dx = torch.empty_like(x) if need_dx else None
    ws = torch.empty(lib.osvos_conv_first_bwd_workspace_bytes(), dtype=torch.uint8, device=x.device)
    _count(2 if need_dx else 1)
    nat.check(lib.osvos_conv_first_bwd(x.data_ptr(), dz.hi.data_ptr(), nat.ptr(dz.lo), weight.data_ptr(),
                                       dw.data_ptr(), nat.ptr(dx), ws.data_ptr(), n, h, w, _stream()),
              "osvos_conv_first_bwd")
    return dw, dx


_U8_MODES = {"prob": nat.U8_PROB, "bytescale": nat.U8_BYTESCALE, "mask": nat.U8_MASK}


def logits_to_u8(logits, mode="bytescale", out=None):
    """Test-time output path on the device (reference train_online.py:181-187): fused logits [N,1,H,W] fp32 ->
    uint8 [N,1,H,W].  mode 'bytescale' is the PNG payload the reference's sigmoid + scipy.misc.imsave writes,
    'prob' is round(255*sigmoid), 'mask' is 255*(logit > 0)."""
    lib = nat.load()
    _require_cuda(logits, "logits")
    x = logits.detach().contiguous().float()
    frames = int(x.shape[0])
    per = x.numel() // frames
    if out is None:
        out = torch.empty(x.shape, dtype=torch.uint8, device=x.device)
    ws = torch.empty(2 * frames, dtype=torch.int32, device=x.device) if mode == "bytescale" else None
    _count(3 if mode == "bytescale" else 1)
    nat.check(lib.osvos_logits_to_u8(x.data_ptr(), out.data_ptr(), nat.ptr(ws), frames, per, _U8_MODES[mode], _stream()),
              "osvos_logits_to_u8")
    return out
