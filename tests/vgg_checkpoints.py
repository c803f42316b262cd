"""Synthetic VGG-16 checkpoints in the two formats `OSVOS(pretrained=1|2)` reads, drawn from fixed seeds, so that the
loader fixture (tests/golden/reference_loaders.json, made by tests/golden/make_golden_loaders.py) and the tests that
check against it see the same files."""
import hashlib

import numpy as np
import scipy.io
import torch

from oracle import osvos_oracle as oc

# torchvision's VGG-16 `features`: conv widths, 'M' = max-pool; every conv is followed by a ReLU
VGG16 = [64, 64, 'M', 128, 128, 'M', 256, 256, 256, 'M', 512, 512, 512, 'M', 512, 512, 512, 'M']


def write_caffe_mat(path, seed=5):
    """vgg_caffe.mat in the Caffe export layout (weights[0][k] = (kw, kh, cin, cout), biases[0][k] = (cout, 1)), random
    values.  -> the weights object array as written."""
    rng = np.random.default_rng(seed)
    shapes = [oc.param_shapes()[n + ".weight"] for n in oc.trunk_conv_names()]
    weights = np.empty((1, len(shapes)), dtype=object)
    biases = np.empty((1, len(shapes)), dtype=object)
    for k, (co, ci, kh, kw) in enumerate(shapes):
        weights[0, k] = rng.standard_normal((kw, kh, ci, co)).astype(np.float32)
        biases[0, k] = rng.standard_normal((co, 1)).astype(np.float32)
    scipy.io.savemat(path, {"weights": weights, "biases": biases})
    return weights


def write_torchvision_pth(path, seed=11):
    """vgg_pytorch.pth with the keys of torchvision's VGG-16 state_dict: random `features.<i>` convs, and the three
    `classifier` Linear layers, which no OSVOS loader reads, as broadcast zeros (a few bytes on disk instead of 124 M
    floats).  -> [(weight, bias)] of the convs in order."""
    rng = np.random.default_rng(seed)
    sd, convs, i, cin = {}, [], 0, 3
    for v in VGG16:
        if v == 'M':
            i += 1
            continue
        w = torch.from_numpy((rng.standard_normal((v, cin, 3, 3)) * 0.05).astype(np.float32))
        b = torch.from_numpy((rng.standard_normal(v) * 0.1).astype(np.float32))
        sd[f"features.{i}.weight"], sd[f"features.{i}.bias"] = w, b
        convs.append((w, b))
        i, cin = i + 2, v
    for j, (cout, cin) in zip((0, 3, 6), ((4096, 512 * 7 * 7), (4096, 4096), (1000, 4096))):
        sd[f"classifier.{j}.weight"] = torch.zeros(()).expand(cout, cin)
        sd[f"classifier.{j}.bias"] = torch.zeros(()).expand(cout)
    torch.save(sd, path)
    return convs


def trunk_digests(state_dict):
    """SHA-256 of dtype, shape and C-order bytes of every `stages.*` tensor: a bit-exact fingerprint of the loaded trunk."""
    return {k: hashlib.sha256(f"{v.dtype}{tuple(v.shape)}".encode() + v.detach().contiguous().numpy().tobytes()).hexdigest()
            for k, v in state_dict.items() if k.startswith("stages.")}
