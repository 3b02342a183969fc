import os
import sys
from pathlib import Path

import numpy as np
import pytest
import torch

ROOT = Path(__file__).resolve().parent.parent
if str(ROOT) not in sys.path:
    sys.path.insert(0, str(ROOT))

GOLDEN_DIR = Path(__file__).resolve().parent / "golden"
GOLDEN_CASES = ["small64", "llama128", "ties128", "half64"]


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box with -m gpu)")


REFERENCE_DIR = Path("/root/reference")      # build container only; absent on the GPU box


class Golden:
    """One tests/golden/<name>.npz produced by make_golden.py from the imported reference — or, `live`, the same
    arrays produced right now by the imported reference on THIS host (only where /root/reference exists). The stored
    files were written on one particular host; large bf16/fp16 GEMMs (the q_proj / covariance prologue) round
    differently under another CPU's GEMM kernels, so only a live case pins the prologue restatement bit for bit
    everywhere; every stage downstream of the stored intermediates is bit-exact on any host."""

    def __init__(self, name: str, live: bool = False):
        self.name = name
        self.live = live
        if live:
            from tests.golden import make_golden

            self.z = make_golden.build_case(**make_golden.CASES[name])
        else:
            self.z = np.load(GOLDEN_DIR / f"{name}.npz")
        self.B, self.Hq, self.Hkv, self.D, self.hidden, self.S, self.seed = (int(x) for x in self.z["meta"])
        self.dtype = torch.float16 if name.startswith("half") else torch.bfloat16
        self.ratios = [float(r) for r in self.z["ratios"]]

    def t(self, key: str) -> torch.Tensor:
        a = self.z[key]
        if a.dtype == np.uint16:
            return torch.from_numpy(a.copy()).view(self.dtype)
        return torch.from_numpy(a.copy())

    def __contains__(self, key):
        return key in self.z


@pytest.fixture(params=GOLDEN_CASES)
def golden(request) -> Golden:
    return Golden(request.param)


@pytest.fixture(params=GOLDEN_CASES + ["live:" + c for c in GOLDEN_CASES])
def golden_or_live(request) -> Golden:
    """The stored cases plus, where the reference is importable, the same cases generated live on this host."""
    name = request.param
    if name.startswith("live:"):
        if not os.path.isdir(REFERENCE_DIR):             # absent, or not readable by this user
            pytest.skip("no /root/reference here: live pinning runs in the build container only")
        return Golden(name[5:], live=True)
    return Golden(name)


def assert_gemm_prologue(got: torch.Tensor, want: torch.Tensor, exact: bool, what: str = ""):
    """Outputs of the big 16-bit prologue GEMMs (q_proj over the prompt, query mean / covariance): bit-exact against
    a live reference; against a STORED file bit-exact or within the rounding spread of another host's GEMM kernels
    (different summation order): |diff| <= 4 eps of max(|want|, max|want| / 16), and >= 96 % of the elements equal."""
    if torch.equal(got, want):
        return
    assert not exact, f"{what}: differs from the reference run live on this host"
    eps = torch.finfo(want.dtype).eps
    w = want.float().abs()
    tol = 4 * eps * w.clamp_min(w.max() / 16)
    diff = (got.float() - want.float()).abs()
    assert (diff <= tol).all(), f"{what}: beyond GEMM rounding spread (max {float((diff / tol).max()):.2f} tol)"
    assert (diff == 0).float().mean().item() >= 0.96, what


def ulp16_diff(a: torch.Tensor, b: torch.Tensor) -> torch.Tensor:
    """Distance in units-in-the-last-place between two 16-bit float tensors of the same dtype."""
    def ordered(x):
        bits = x.contiguous().view(torch.int16).to(torch.int32) & 0xFFFF
        neg = bits >= 0x8000
        return torch.where(neg, 0x8000 - (bits & 0x7FFF), bits + 0x8000)
    return (ordered(a) - ordered(b)).abs()
