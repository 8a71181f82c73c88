"""The numpy restatement of the caller-side prologue / epilogue (oracle/frontend.py) against outputs of the live
reference: the committed fixtures tests/golden/frontend_*.npz (made by tests/golden/make_golden_frontend.py) and its
own code's outputs on fresh inputs (tests/golden/ref_oracle_fresh.npz, made by tests/golden/make_golden_models.py)."""
import glob
import os

import numpy as np
import pytest
import torch

from oracle import frontend as fe
from tests import util

HERE = os.path.dirname(os.path.abspath(__file__))
GOLD = sorted(glob.glob(os.path.join(HERE, "golden", "frontend_*.npz")))


@pytest.mark.parametrize("path", GOLD, ids=[os.path.basename(p)[:-4] for p in GOLD])
def test_restatement_reproduces_the_reference_fixtures(path):
    z = np.load(path)
    hop = int(z["hop"])
    vol = fe.volume_extract(z["audio"], hop)
    assert vol.dtype == z["volume"].dtype and np.array_equal(vol, z["volume"])
    mask = fe.volume_mask(vol, -40)
    assert np.array_equal(mask, z["mask"])
    up = fe.upsample(torch.from_numpy(mask).float().unsqueeze(-1).unsqueeze(0), hop).squeeze(-1).numpy()
    assert np.array_equal(up, z["mask_up"])
    out = fe.cross_fade(z["fade_a"], z["fade_b"], int(z["fade_idx"]))
    assert np.array_equal(out, z["fade_out"])


FRESH = ((11, 9000, 512), (12, 777, 256), (13, 30011, 441))       # (seed, samples, hop)
FADE_IDX = (0, 1, 250, 399)


def fade_inputs(seed):
    g = np.random.default_rng(seed)
    return g.standard_normal(400).astype(np.float32), g.standard_normal(500).astype(np.float32)


def test_restatement_equals_the_live_reference_on_fresh_inputs():
    from tests.golden.make_golden_frontend import inputs
    gold = util.load_golden("ref_oracle_fresh")
    for seed, T, hop in FRESH:
        audio = inputs(seed, T)
        want = gold["fe%d__volume" % seed]
        vol = fe.volume_extract(audio, hop)
        assert vol.dtype == want.dtype and np.array_equal(vol, want)
        assert np.array_equal(fe.volume_mask(want, -45), gold["fe%d__mask" % seed])
        a, b = fade_inputs(seed)
        for idx in FADE_IDX:
            got, want = fe.cross_fade(a, b, idx), gold["fe%d__fade%d" % (seed, idx)]
            assert got.size == gold["fe%d__fade%d_len" % (seed, idx)] and np.array_equal(util.sampled(got, want.size), want)


def test_interpolation_weight_arithmetic_of_the_mask_kernel_equals_torch():
    """csrc/frontend.cu::mask_weight restated in numpy (fp32 operation by operation: scale = f32(nF) / f32(nF P),
    src = scale * f32(t), lambda = src - floor(src), w = fma(1 - lambda, v0, lambda * v1)) against torch's
    upsample_linear1d(align_corners=True) on GENERAL frame values, power-of-two and other block sizes: bit-identical."""
    rng = np.random.default_rng(0)
    f32 = np.float32
    for P in (512, 441, 300, 256, 7):
        for nF in (1, 3, 46, 259):
            m = rng.standard_normal(nF).astype(f32)
            ref = fe.upsample(torch.from_numpy(m)[None, :, None], P)[0, :, 0].numpy()
            t = np.arange(nF * P, dtype=np.int64)
            src = (f32(nF) / f32(nF * P) * t.astype(f32)).astype(f32)
            i0 = np.minimum(np.floor(src).astype(np.int64), nF)
            lam = np.clip((src - i0.astype(f32)).astype(f32), 0, 1).astype(f32)
            i1 = i0 + (i0 < nF)
            v0, v1 = m[np.minimum(i0, nF - 1)], m[np.minimum(i1, nF - 1)]
            w0 = (f32(1) - lam).astype(f32)
            w = ((lam * v1).astype(f32).astype(np.float64) + w0.astype(np.float64) * v0.astype(np.float64)).astype(f32)   # fma
            assert np.array_equal(w, ref), (P, nF)
