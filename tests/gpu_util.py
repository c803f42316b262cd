import numpy as np
import torch


def maxrel(a, b, scale=None):
    """max |a - b| / max |b|, or over `scale` when b is a sample of a larger map whose max |.| is `scale`."""
    a = a.detach().double().cpu().numpy() if isinstance(a, torch.Tensor) else np.asarray(a, dtype=np.float64)
    b = b.detach().double().cpu().numpy() if isinstance(b, torch.Tensor) else np.asarray(b, dtype=np.float64)
    return float(np.abs(a - b).max() / max(np.abs(b).max() if scale is None else scale, 1e-30))


def golden_map(golden, tag, i, got):
    """Logit map i of the golden forward case `tag` -> (got, ref, max |ref|) on the pixels the fixture keeps: all of
    them, or for a large map the seeded sample `<tag>.idx` (flat indices), with the maximum over the whole map stored
    beside it (tests/golden/make_golden.py)."""
    got = got.detach().cpu().numpy() if isinstance(got, torch.Tensor) else np.asarray(got)
    ref = golden[f"{tag}.out{i}"]
    if f"{tag}.idx" not in golden:
        return got, ref, float(np.abs(ref).max())
    return got.reshape(-1)[golden[f"{tag}.idx"]], ref, float(golden[f"{tag}.absmax{i}"])


def rmsrel(a, b):
    a = a.detach().double().cpu().numpy() if isinstance(a, torch.Tensor) else np.asarray(a, dtype=np.float64)
    b = b.detach().double().cpu().numpy() if isinstance(b, torch.Tensor) else np.asarray(b, dtype=np.float64)
    return float(np.sqrt(((a - b) ** 2).mean()) / max(np.sqrt((b ** 2).mean()), 1e-30))


def split_round(t):
    """What the split-bf16 representation stores: bf16(v) + bf16(v - bf16(v)) (fp32 tensor in, fp32 out)."""
    hi = t.to(torch.bfloat16).float()
    lo = (t - hi).to(torch.bfloat16).float()
    return hi + lo
