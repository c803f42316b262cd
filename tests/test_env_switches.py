"""The library reads every environment switch by one rule (csrc/runtime.cu): the first read of a switch is kept for the
process, and under OSVOS_ENV_RELOAD=1 every call re-reads it.  Checked without a GPU through the two launch-plan queries,
which read switches of two different files (conv3x3_halo.cu, wgrad_tc.cu).  Each case runs in a fresh process, because
the reload flag itself is read once."""
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

# Flips OSVOS_SPLITACC128 and OSVOS_WGRAD_ROWS between two queries and prints [split_acc, tap_mode] of both.  The
# pointers are never dereferenced by a plan query; they only have to pass the argument checks.
PROBE = r"""
import ctypes, json, os
from osvos_pytorch_b200 import _native as nat
lib = nat.load()
conv = nat.Conv3x3Args(x_hi=256, x_lo=256, w_packed=256, bias=256, y_hi=256, y_lo=256, n=1, h=480, w=854, cin=128,
                       cout=128, flags=nat.FLAG_RELU)
wgrad = nat.WgradArgs(x_hi=256, x_lo=256, dz_hi=256, dz_lo=256, dw=256, workspace=256, n=1, h=480, w=854, cin=64,
                      cout=64, dz_channels=64)
def plans():
    p, q = nat.LaunchPlan(), nat.LaunchPlan()
    nat.check(lib.osvos_conv3x3_plan(ctypes.byref(conv), ctypes.byref(p)), "osvos_conv3x3_plan")
    nat.check(lib.osvos_conv3x3_wgrad_plan(ctypes.byref(wgrad), ctypes.byref(q)), "osvos_conv3x3_wgrad_plan")
    return [p.split_acc, q.tap_mode]
first = plans()
os.environ["OSVOS_SPLITACC128"] = "0"
os.environ["OSVOS_WGRAD_ROWS"] = "0"
print(json.dumps([first, plans()]))
"""


@pytest.fixture(scope="module")
def lib_path():
    from osvos_pytorch_b200 import build
    return build.build()


@pytest.mark.parametrize("reload", [False, True])
def test_switches_share_one_caching_rule(lib_path, reload):
    from osvos_pytorch_b200 import _native as nat
    env = {k: v for k, v in os.environ.items() if k not in ("OSVOS_ENV_RELOAD", "OSVOS_SPLITACC128", "OSVOS_WGRAD_ROWS")}
    if reload:
        env["OSVOS_ENV_RELOAD"] = "1"
    r = subprocess.run([sys.executable, "-c", PROBE], cwd=ROOT, env=env, capture_output=True, text=True, timeout=120)
    assert r.returncode == 0, r.stderr
    first, second = json.loads(r.stdout.strip().splitlines()[-1])
    assert first == [1, nat.TAP_ROWS]
    assert second == ([0, nat.TAP_PAIRS] if reload else [1, nat.TAP_ROWS])
