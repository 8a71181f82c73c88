"""The restatement of the mel front end (oracle/mel.py) against the reference: fixtures produced by the reference's own
nvSTFT.py (tests/golden/mel_*.npz and, on fresh inputs, ref_oracle_fresh.npz), and torchaudio's independent implementation of the
librosa / Slaney mel filterbank (librosa itself is an absent third-party dependency)."""
import glob
import os

import numpy as np
import pytest
import torch

from oracle import mel as om
from tests import util

HERE = os.path.dirname(os.path.abspath(__file__))
GOLD = sorted(glob.glob(os.path.join(HERE, "golden", "mel_*.npz")))


# the reference's outputs were computed with this many intra-op threads: torch's CPU matmul splits its reduction by the
# thread count, so the last bit of a mel value depends on it
FIXTURE_THREADS = 8


@pytest.fixture
def fixture_threads():
    n = torch.get_num_threads()
    torch.set_num_threads(FIXTURE_THREADS)
    yield
    torch.set_num_threads(n)


@pytest.mark.parametrize("path", GOLD, ids=[os.path.basename(p)[:-4] for p in GOLD])
def test_restatement_reproduces_the_reference_fixtures(path, fixture_threads):
    z = np.load(path)
    with torch.no_grad():
        got = om.get_mel(torch.from_numpy(z["y"]), hop_length=int(z["hop"])).numpy()
    assert got.shape == z["mel"].shape
    assert np.array_equal(got, z["mel"])


def test_filterbank_agrees_with_torchaudio_and_with_the_product_host_code():
    import torchaudio.functional as TF
    from ddsp_svc_b200 import mel as pm
    for sr, n_fft, n_mels, fmin, fmax in ((44100, 2048, 128, 40, 16000), (22050, 1024, 80, 20, 11025), (44100, 2048, 128, 0, None)):
        ours = om.librosa_mel(sr, n_fft, n_mels, fmin, fmax)
        ta = TF.melscale_fbanks(n_fft // 2 + 1, float(fmin), float(fmax or sr / 2), n_mels, sr, norm="slaney", mel_scale="slaney").T.numpy()
        assert ours.dtype == np.float32 and ours.shape == ta.shape
        assert np.abs(ours - ta).max() < 1e-5 * ours.max()
        prod = pm.mel_filterbank(sr, n_fft, n_mels, fmin, fmax)
        assert np.abs(prod - ours).max() < 1e-6 * ours.max()
        lohi = pm._support(prod)
        for m in range(n_mels):                      # the sparse form the kernel uses covers every non-zero weight
            assert not prod[m, :lohi[m, 0]].any() and not prod[m, lohi[m, 1]:].any()
        assert (ours.sum(1) > 0).all()


def fresh_inputs():
    g = torch.Generator().manual_seed(9)
    for T, hop in ((512 * 9 + 17, 512), (900, 512), (256 * 30, 256)):
        yield 0.2 * torch.randn(2, T, generator=g), hop


def test_restatement_equals_the_live_reference_code(fixture_threads):
    gold = util.load_golden("ref_oracle_fresh")
    for i, (y, hop) in enumerate(fresh_inputs()):
        with torch.no_grad():
            got = om.get_mel(y, hop_length=hop)
        want = gold["mel%d__mel" % i]
        assert list(got.shape) == list(gold["mel%d__shape" % i])
        assert np.array_equal(util.sampled(got, want.size), want)
