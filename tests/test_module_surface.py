"""Drop-in surface of the OSVOS module (SURVEY.md section 8b) - CPU only, no compute."""
import json
import os

import torch
import torch.nn as nn

from oracle import osvos_oracle as oc
from osvos_pytorch_b200.layers import osvos_layers as L
from osvos_pytorch_b200.networks.vgg_osvos import OSVOS

import numpy as np
import pytest
import vgg_checkpoints


@pytest.fixture(scope="module")
def net():
    return OSVOS(pretrained=0, verbose=False)


def test_state_dict_matches_reference_layout(net):
    sd = net.state_dict()
    shapes = oc.param_shapes()
    assert set(sd) == set(shapes)
    for k, v in sd.items():
        assert tuple(v.shape) == shapes[k], k
    # registration order of the reference: upscale, upscale_, stages, side_prep, score_dsn, fuse
    prefixes = [k.split(".")[0] for k in sd]
    order = [p for i, p in enumerate(prefixes) if i == 0 or prefixes[i - 1] != p]
    assert order == ["upscale", "upscale_", "stages", "side_prep", "score_dsn", "fuse"]


def test_containers_support_the_training_scripts(net):
    # optimizer construction of train_online.py:79-88 / train_parent.py:87-103
    groups = [[p for n_, p in net.stages.named_parameters() if "weight" in n_],
              [p for n_, p in net.stages.named_parameters() if "bias" in n_],
              [p for n_, p in net.side_prep.named_parameters() if "weight" in n_],
              [p for n_, p in net.score_dsn.named_parameters() if "bias" in n_],
              [p for n_, p in net.upscale.named_parameters() if "weight" in n_],
              [p for n_, p in net.upscale_.named_parameters() if "weight" in n_]]
    assert [len(g) for g in groups] == [13, 13, 4, 4, 4, 4]
    torch.optim.SGD([{"params": g} for g in groups] + [{"params": net.fuse.weight}, {"params": net.fuse.bias}],
                    lr=1e-8, momentum=0.9)
    # VGG loader walks stages[i][j] looking for nn.Conv2d (reference networks/vgg_osvos.py:104-109)
    idx = [[j for j, m in enumerate(s) if isinstance(m, nn.Conv2d)] for s in net.stages]
    assert idx == [[0, 2], [1, 3], [1, 3, 5], [1, 3, 5], [1, 3, 5]]
    assert isinstance(net.stages[1][0], nn.MaxPool2d) and net.stages[1][0].ceil_mode


def test_init_matches_reference_rules(net):
    for i in range(4):
        w = net.upscale[i].weight.detach()
        assert torch.equal(w, oc.interp_weight(16, 2 ** (i + 1)))
        assert torch.equal(net.upscale_[i].weight.detach(), oc.interp_weight(1, 2 ** (i + 1)))
    assert float(net.fuse.bias.abs().max()) == 0.0
    assert 5e-4 < float(net.stages[2][1].weight.std()) < 2e-3


def test_state_dict_round_trip(net):
    params = oc.he_params(seed=3, include_upscale=True)
    net2 = OSVOS(pretrained=0, verbose=False)
    net2.load_state_dict(params)
    for k, v in net2.state_dict().items():
        assert torch.equal(v, params[k])


def test_layer_helpers(golden):
    for s in (4, 8, 16, 32):
        np.testing.assert_array_equal(L.upsample_filt(s), golden[f"upsample_filt.{s}"])
    lay = nn.ConvTranspose2d(3, 3, 4, stride=2, bias=False)
    with torch.no_grad():
        lay.weight.zero_()
    w = L.interp_surgery(lay)
    assert torch.equal(w, oc.interp_weight(3, 2))
    with pytest.raises(ValueError):
        L.interp_surgery(nn.ConvTranspose2d(2, 3, 4, bias=False))
    with pytest.raises(ValueError):
        L.interp_surgery(nn.ConvTranspose2d(2, 2, (4, 6), bias=False))
    t = torch.arange(2 * 1 * 11 * 14).float().view(2, 1, 11, 14)
    assert torch.equal(L.center_crop(t, 8, 9), oc.center_crop(t, 8, 9))
    assert torch.equal(L.center_crop(t, 8, 9), t[:, :, 1:9, 2:11])
    assert abs(L.sigmoid_np(L.logit(np.array(0.3))) - 0.3) < 1e-6
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        L.class_balanced_cross_entropy_loss(torch.zeros(1, 1, 2, 2), torch.zeros(1, 1, 2, 2))


def _reference_loaders():
    with open(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference_loaders.json")) as f:
        return json.load(f)


def _assert_trunk_matches_reference(sd, ref):
    assert list(sd.keys()) == ref["keys"]
    got, want = vgg_checkpoints.trunk_digests(sd), ref["stages_sha256"]
    assert len(want) == 26 and got.keys() == want.keys()
    for name in want:
        assert got[name] == want[name], name


def test_caffe_vgg_loader_matches_the_reference_loader(tmp_path, monkeypatch):
    """`OSVOS(pretrained=2)` reads models/vgg_caffe.mat exactly like the reference's loader
    (networks/vgg_osvos.py:110-125): a synthetic .mat in the Caffe export layout (weights[0][k] = (kw, kh, cin, cout),
    biases[0][k] = (cout, 1)) goes through this package's loader, and every trunk tensor must come out bit-identical to
    what the reference's own loader (unmodified) made of the same file (tests/golden/reference_loaders.json)."""
    (tmp_path / "models").mkdir()
    weights = vgg_checkpoints.write_caffe_mat(str(tmp_path / "models" / "vgg_caffe.mat"))
    monkeypatch.chdir(tmp_path)                       # Path.models_dir() defaults to ./models, as in the reference
    monkeypatch.delenv("OSVOS_MODELS_DIR", raising=False)
    mine = OSVOS(pretrained=2, verbose=False)
    my_sd = mine.state_dict()
    _assert_trunk_matches_reference(my_sd, _reference_loaders()["caffe"])
    # the tensor the kernels will read is what Caffe stored: conv k, output channel o, input channel i, tap (r, s)
    k = 3
    w = my_sd[oc.trunk_conv_names()[k] + ".weight"]
    assert float(w[5, 7, 1, 2]) == float(weights[0, k][2, 1, 7, 5])


def test_torchvision_vgg_loader_matches_the_reference_loader(tmp_path, monkeypatch):
    """`OSVOS(pretrained=1)` reads models/vgg_pytorch.pth like the reference's loader (networks/vgg_osvos.py:93-109): a
    synthetic checkpoint with the keys of torchvision's VGG-16 (features + classifier, random conv weights) goes through
    this package's loader, and every trunk tensor must be bit-identical to what the reference's own loader (unmodified)
    made of the same file (tests/golden/reference_loaders.json)."""
    (tmp_path / "models").mkdir()
    want = vgg_checkpoints.write_torchvision_pth(str(tmp_path / "models" / "vgg_pytorch.pth"))
    monkeypatch.chdir(tmp_path)                       # Path.models_dir() defaults to ./models, as in the reference
    monkeypatch.delenv("OSVOS_MODELS_DIR", raising=False)
    mine = OSVOS(pretrained=1, verbose=False)
    _assert_trunk_matches_reference(mine.state_dict(), _reference_loaders()["torchvision"])
    convs = [m for stage in mine.stages for m in stage if isinstance(m, torch.nn.Conv2d)]
    assert len(convs) == len(want)
    for conv, (w, b) in zip(convs, want):
        assert torch.equal(conv.weight.detach(), w) and torch.equal(conv.bias.detach(), b)
