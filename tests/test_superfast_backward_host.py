"""CPU-side checks of the CombSubSuperFast backward: the C ABI returns its argument errors before any CUDA call, and
patch_reference(training=True) rebinds only the reference's CombSubSuperFast, to a class built on the reference's own
Unit2Control (stand-in modules laid out like the reference's, as in test_dropin.py)."""
import sys
import types

import pytest
import torch

import ddsp_svc_b200 as pkg
from ddsp_svc_b200 import _lib


@pytest.fixture(scope="module")
def lib():
    _lib.build()
    return _lib.lib()


def test_backward_argument_errors_do_not_touch_the_device(lib):
    C = 1025
    ok = dict(ws=16, hm=16, hp=16, nm=16, np_=16, cs=4 * C, noise=0, seed=0, utt=0, g=16, B=1, nF=4, block=512,
              win=2048, ghm=16, ghp=16, gnm=16, gnp=16, gs=4 * C)

    def call(**kw):
        a = dict(ok, **kw)
        return lib.b2d_superfast_backward(a["ws"], a["hm"], a["hp"], a["nm"], a["np_"], a["cs"], a["noise"], a["seed"],
                                          a["utt"], a["g"], a["B"], a["nF"], a["block"], a["win"], a["ghm"], a["ghp"],
                                          a["gnm"], a["gnp"], a["gs"], 0)

    assert call(ws=0) == -1                       # B2D_ERR_NULL
    assert call(g=0) == -1
    assert call(gnp=0) == -1
    assert b"null" in lib.b2d_last_error()
    assert call(B=0) == -2                        # B2D_ERR_SHAPE
    assert call(nF=0) == -2
    assert call(cs=1024) == -2                    # control stride < 1025
    assert call(gs=1000) == -2                    # gradient stride < 1025
    assert call(win=1024, cs=C, gs=C) == -4       # B2D_ERR_UNSUPPORTED
    assert call(block=256) == -4
    assert call(B=70000) == -4
    assert call(ws=20) == -3                      # B2D_ERR_ALIGN
    assert call(noise=20) == -3


def test_training_patch_rebinds_only_combsubsuperfast(monkeypatch):
    names = ("Sins", "CombSub", "CombSubSuperFast", "CombSubFast", "Volume_Extractor")
    V = types.ModuleType("ddsp.vocoder")
    for n in names:
        setattr(V, n, type(n, (), {}))

    class Unit2Control(torch.nn.Module):           # stand-in for the reference's ddsp.unit2control.Unit2Control
        def __init__(self, n_unit, n_spk, split_map, **kw):
            super().__init__()
            self.args = (n_unit, n_spk, split_map, kw)
            self.dense_out = torch.nn.Linear(n_unit, sum(split_map.values()))

    U = types.ModuleType("ddsp.unit2control")
    U.Unit2Control = Unit2Control
    stft = types.ModuleType("nsf_hifigan.nvSTFT")
    stft.STFT = type("STFT", (), {})
    for pkgname in ("ddsp", "nsf_hifigan"):
        parent = types.ModuleType(pkgname)
        parent.__path__ = []
        monkeypatch.setitem(sys.modules, pkgname, parent)
    for modname, m in (("ddsp.vocoder", V), ("ddsp.unit2control", U), ("nsf_hifigan.nvSTFT", stft)):
        monkeypatch.setitem(sys.modules, modname, m)
        setattr(sys.modules[modname.split(".")[0]], modname.split(".")[1], m)
    originals = {n: getattr(V, n) for n in names}
    orig_stft = stft.STFT

    saved = pkg.patch_reference(training=True)
    try:
        assert set(saved) == {"CombSubSuperFast"}
        for n in names:
            assert (getattr(V, n) is originals[n]) == (n != "CombSubSuperFast"), n
        assert stft.STFT is orig_stft
        cls = V.CombSubSuperFast
        assert issubclass(cls, pkg.CombSubSuperFast)
        m = cls(44100, 512, 2048, n_unit=16, n_spk=2, use_pitch_aug=True)     # the reference's constructor arguments
        assert isinstance(m.unit2ctrl, Unit2Control)
        n_unit, n_spk, split_map, kw = m.unit2ctrl.args
        assert (n_unit, n_spk) == (16, 2) and split_map == pkg.CombSubSuperFast.split_map(2048)
        assert kw == {"use_pitch_aug": True, "use_naive_v2": True, "use_conv_stack": True}
        assert {"sampling_rate", "block_size", "win_length", "window", "unit2ctrl.dense_out.weight"} <= set(m.state_dict())
        with pytest.raises(ValueError, match="block_size"):
            cls(44100, 256, 2048)
    finally:
        pkg.unpatch_reference(saved)
    assert all(getattr(V, n) is c for n, c in originals.items())
