"""Golden fixture of the reference's VGG-16 weight loaders, produced by the UNMODIFIED reference.

    python tests/golden/make_golden_loaders.py <reference checkout>

It writes the synthetic checkpoints of tests/vgg_checkpoints.py into a temporary ./models, builds the reference's own
``OSVOS(pretrained=2)`` (models/vgg_caffe.mat) and ``OSVOS(pretrained=1)`` (models/vgg_pytorch.pth) from them, and
stores the state_dict key order and a SHA-256 of every trunk tensor it loaded.  tests/test_module_surface.py holds the
package's loaders to them bit for bit.
"""
import contextlib
import io
import json
import os
import sys
import tempfile

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))


def main(reference):
    sys.path.insert(0, ROOT)
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    sys.path.insert(0, os.path.abspath(reference))       # the reference's networks/, layers/, mypath.py come first
    import networks.vgg_osvos as ref_net                  # reference, unmodified
    assert os.path.abspath(ref_net.__file__).startswith(os.path.abspath(reference)), ref_net.__file__
    import vgg_checkpoints as ck
    fx = {}
    cwd = os.getcwd()
    with tempfile.TemporaryDirectory() as tmp:
        os.makedirs(os.path.join(tmp, "models"))
        ck.write_caffe_mat(os.path.join(tmp, "models", "vgg_caffe.mat"))
        ck.write_torchvision_pth(os.path.join(tmp, "models", "vgg_pytorch.pth"))
        os.chdir(tmp)                                     # the reference's Path.models_dir() is ./models
        try:
            for name, pretrained in (("caffe", 2), ("torchvision", 1)):
                with contextlib.redirect_stdout(io.StringIO()):
                    sd = ref_net.OSVOS(pretrained=pretrained).state_dict()
                fx[name] = {"keys": list(sd.keys()), "stages_sha256": ck.trunk_digests(sd)}
        finally:
            os.chdir(cwd)
    path = os.path.join(HERE, "reference_loaders.json")
    with open(path, "w") as f:
        json.dump(fx, f, indent=1)
        f.write("\n")
    print("wrote", path, os.path.getsize(path), "bytes")


if __name__ == "__main__":
    if len(sys.argv) != 2:
        sys.exit(__doc__)
    main(sys.argv[1])
