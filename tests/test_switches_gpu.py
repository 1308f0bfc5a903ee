"""The engine's remaining A/B switches must still compute the same features: MADM_NO_SPLITK=1 (no split-K: the reference summation
order) and MADM_GEMM_TMA_EPI=0 (the coalesced-store GEMM epilogue everywhere) select another summation order or another store path, never
other arithmetic.  Each switch runs tools/check_switch.py in its own process (the switches are read when plans are built) on the seeded
synthetic product model; results are compared with the default run."""
import os
import subprocess
import sys

import pytest
import torch

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

SWITCHES = [("base", "MADM_NO_SPLITK=1"), ("base", "MADM_GEMM_TMA_EPI=0"), ("s0", "MADM_GEMM_TMA_EPI=0")]


def _run(tmp_path, variant, env_kv, tag):
    out = tmp_path / f"{tag}.pt"
    env = dict(os.environ)
    if env_kv:
        k, v = env_kv.split("=")
        env[k] = v
    r = subprocess.run([sys.executable, os.path.join(ROOT, "tools", "check_switch.py"), str(out), variant], env=env, capture_output=True, text=True,
                       timeout=600)
    assert r.returncode == 0, (env_kv, r.stdout[-500:], r.stderr[-1500:])
    return torch.load(out)


@pytest.fixture(scope="module")
def defaults(tmp_path_factory, cuda_device):
    d = tmp_path_factory.mktemp("switch_default")
    return {v: _run(d, v, None, "default_" + v) for v in ("base", "s0")}


@pytest.mark.parametrize("variant,env_kv", SWITCHES)
def test_switch_computes_the_same_features(tmp_path, defaults, variant, env_kv):
    got = _run(tmp_path, variant, env_kv, "sw")
    ref = defaults[variant]
    assert got.keys() == ref.keys()
    for k in ref:
        err = ((got[k] - ref[k]).abs().max() / ref[k].abs().max()).item()
        print(f"{variant} {env_kv} {k}: max_rel vs default {err:.2e}")
        assert err <= 1e-2, (variant, env_kv, k, err)  # 16-bit vs fp32 storage of a stream / another summation order, not other arithmetic
