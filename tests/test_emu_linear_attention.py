"""csrc/linear_attention.cu's KERNEL SOURCE executed on the CPU (tests/emu/host_emu.h) against the fp64 formula of the
performer's non-causal linear attention (reference ddsp/pcmer.py:220-229) and against the reference function itself."""
import ctypes
import os
import shutil
import subprocess

import numpy as np
import pytest
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
pytestmark = pytest.mark.skipif(shutil.which("g++") is None, reason="g++ not available")


@pytest.fixture(scope="module")
def emu(tmp_path_factory):
    so = str(tmp_path_factory.mktemp("emu") / "libemu_linattn.so")
    cmd = ["g++", "-std=c++20", "-O2", "-shared", "-fPIC", "-pthread", "-Wno-unknown-pragmas", "-o", so,
           os.path.join(HERE, "emu", "emu_linear_attention.cpp")]
    proc = subprocess.run(cmd, capture_output=True, text=True)
    assert proc.returncode == 0, proc.stderr
    lib = ctypes.CDLL(so)
    fp = ctypes.POINTER(ctypes.c_float)
    lib.emu_linear_attention.argtypes = [fp, fp, fp, fp, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_float]
    lib.emu_linear_attention.restype = ctypes.c_int

    def run(qf, kf, v, eps=1e-8):
        B, H, T, J = qf.shape
        arrs = [np.ascontiguousarray(a, np.float32) for a in (qf, kf, v)]
        out = np.full((B, T, H, 64), np.nan, np.float32)
        ptr = lambda a: ctypes.cast(a.ctypes.data, fp)
        assert lib.emu_linear_attention(ptr(arrs[0]), ptr(arrs[1]), ptr(arrs[2]), ptr(out), B, H, T, J, eps) == 0
        return out

    return run


def _features(rng, B, H, T, J):
    # positive random features like the softmax kernel produces (ratio * exp(...) + eps)
    return (np.exp(rng.standard_normal((B, H, T, J)) * 0.5) / np.sqrt(J)).astype(np.float32)


@pytest.mark.parametrize("B,H,T,J", [(1, 1, 1, 266), (1, 2, 16, 266), (2, 3, 37, 266), (1, 1, 50, 8), (1, 2, 33, 272), (1, 1, 17, 129)])
def test_matches_fp64_formula(emu, B, H, T, J):
    rng = np.random.default_rng(T * 7 + J)
    qf, kf = _features(rng, B, H, T, J), _features(rng, B, H, T, J)
    v = rng.standard_normal((B, H, T, 64)).astype(np.float32)
    out = emu(qf, kf, v)
    q64, k64, v64 = qf.astype(np.float64), kf.astype(np.float64), v.astype(np.float64)
    ksum = k64.sum(axis=2)                                           # [B, H, J]
    ctx = np.einsum("bhtj,bhtd->bhjd", k64, v64)
    want = np.einsum("bhtj,bhjd->bhtd", q64, ctx) / (np.einsum("bhtj,bhj->bht", q64, ksum) + 1e-8)[..., None]
    want = want.transpose(0, 2, 1, 3)                                # the kernel writes [B, T, H, D]
    assert not np.isnan(out).any()
    assert np.abs(out - want).max() < 2e-5 * max(1.0, np.abs(want).max())


def reference_inputs():
    g = torch.Generator().manual_seed(1)
    q = torch.rand(2, 3, 20, 266, generator=g, dtype=torch.float64)
    k = torch.rand(2, 3, 20, 266, generator=g, dtype=torch.float64)
    v = torch.randn(2, 3, 20, 64, generator=g, dtype=torch.float64)
    return q, k, v


def test_matches_the_reference_function():
    """the fp64 formula above IS the reference's linear_attention (pcmer.py:220-229): checked against its own outputs,
    stored in tests/golden/ref_oracle_fresh.npz by tests/golden/make_golden_models.py"""
    from tests import util
    q, k, v = (t.numpy() for t in reference_inputs())
    want = util.load_golden("ref_oracle_fresh")["linear_attention"]
    ctx = np.einsum("bhtj,bhtd->bhjd", k, v)
    mine = np.einsum("bhtj,bhjd->bhtd", q, ctx) / (np.einsum("bhtj,bhj->bht", q, k.sum(2)) + 1e-8)[..., None]
    assert want.dtype == np.float64
    assert np.abs(util.sampled(mine, want.size) - want).max() < 1e-12
