"""Drop-in contract: constructor arguments, buffers / state-dict keys and class dispatch match
the reference (SURVEY.md appendix D).  The reference's state-dict layouts (keys, shapes, buffers) are stored in
tests/golden/ref_state_dicts.npz (made by tests/golden/make_golden_models.py from its classes)."""
import sys
import types

import pytest
import torch

import ddsp_svc_b200 as pkg
from ddsp_svc_b200 import dropin
from tests import util

# name -> constructor, given the module holding the classes (this package, or the reference's ddsp.vocoder)
STATE_DICT_CASES = {
    "Sins": lambda V: V.Sins(44100, 512, 128, 256, 256, n_unit=768, n_spk=1),
    "CombSub": lambda V: V.CombSub(44100, 512, 256, 512, 256, n_unit=768, n_spk=2),
    "CombSubSuperFast": lambda V: V.CombSubSuperFast(44100, 512, 2048, n_unit=768, n_spk=1),
    "CombSubFast": lambda V: V.CombSubFast(44100, 512, n_unit=768, n_spk=1),
}


def test_buffers_and_forward_signature_without_reference():
    import inspect
    m = pkg.Sins(44100, 512, 128, 256, 256, unit2ctrl=pkg.FixedControls())
    assert set(m.state_dict()) == {"sampling_rate", "block_size"}
    assert m.sampling_rate.dtype == torch.int64 and m.sampling_rate.dim() == 0
    sig = inspect.signature(m.forward)
    for name in ("units_frames", "f0_frames", "volume_frames", "spk_id", "spk_mix_dict", "initial_phase", "infer",
                 "max_upsample_dim"):
        assert name in sig.parameters
    c = pkg.CombSub(44100, 512, 256, 512, 256, unit2ctrl=pkg.FixedControls())
    assert set(c.state_dict()) == {"sampling_rate", "block_size"}
    cf = pkg.CombSubFast(44100, 512, unit2ctrl=pkg.FixedControls())
    assert list(cf.state_dict()) == ["sampling_rate", "block_size", "window"] and cf.window.shape == (1024,)
    g = pkg.SineGen(44100, harmonic_num=8)
    assert g.dim == 9 and len(g.state_dict()) == 0
    sm = pkg.SourceModuleHnNSF(44100, harmonic_num=8)
    assert list(sm.state_dict()) == ["l_linear.weight", "l_linear.bias"]
    assert sm.l_linear.weight.shape == (1, 9) and sm.l_sin_gen.dim == 9
    assert "voiced_threshod" in inspect.signature(pkg.SourceModuleHnNSF.__init__).parameters   # reference spelling
    with pytest.raises(ValueError, match="Unknown Model"):
        dropin.build_model(dropin.DotDict({"model": {"type": "Nope"}, "data": {}}))
    # no unit2ctrl argument: the package's own Unit2Control (no dependency on the reference package), same head as the
    # reference's (SURVEY appendix D: dense_out -> 640 outputs for Sins 128/256/256)
    own = pkg.Sins(44100, 512, 128, 256, 256, n_unit=768)
    from ddsp_svc_b200.unit2control import Unit2Control
    assert isinstance(own.unit2ctrl, Unit2Control) and own.unit2ctrl.dense_out.weight_v.shape == (640, 256)
    assert {"unit2ctrl.dense_out.weight_g", "unit2ctrl.dense_out.weight_v", "unit2ctrl.dense_out.bias"} <= set(own.state_dict())
    with pytest.raises(ValueError, match="block_size"):
        pkg.Sins(44100, 441, 128, 256, 256, unit2ctrl=pkg.FixedControls())          # unsupported shapes fail at build time


def test_module_refuses_cpu_tensors():
    m = pkg.Sins(44100, 512, 4, 9, 9, unit2ctrl=pkg.FixedControls())
    with pytest.raises(ValueError, match="CUDA"):
        m(None, torch.zeros(1, 3, 1), None)


def _reference_state_dict(module, gold, prefix):
    """seeded weights in the reference's layout, with the reference's own buffers"""
    sd = util.seeded_state_dict(module, 0)
    for k in sd:
        if prefix + "buffer__" + k in gold:
            sd[k] = torch.from_numpy(gold[prefix + "buffer__" + k])
    return sd


def test_state_dict_round_trip_with_the_reference_classes(tmp_path):
    gold = util.load_golden("ref_state_dicts")
    for name, make in STATE_DICT_CASES.items():
        ours = make(pkg)                                # this package's Unit2Control
        util.check_state_dict_layout(ours, gold, name + "__")
        sd = _reference_state_dict(ours, gold, name + "__")
        ours.load_state_dict(sd)                        # strict, like ddsp/vocoder.py:527
        for k, v in ours.state_dict().items():
            assert torch.equal(v, sd[k]), k
    # load_model: config.yaml next to the checkpoint -> class dispatch -> strict load
    import yaml
    cfg = {"data": {"sampling_rate": 44100, "block_size": 512, "encoder_out_channels": 768},
           "model": {"type": "CombSubSuperFast", "win_length": 2048, "n_spk": 1}}
    (tmp_path / "config.yaml").write_text(yaml.safe_dump(cfg))
    sd = _reference_state_dict(STATE_DICT_CASES["CombSubSuperFast"](pkg), gold, "CombSubSuperFast__")
    torch.save({"global_step": 1, "model": sd}, tmp_path / "model_1.pt")
    model, args = dropin.load_model(str(tmp_path / "model_1.pt"), device="cpu")
    assert isinstance(model, pkg.CombSubSuperFast) and args.model.win_length == 2048
    ours_sm = pkg.SourceModuleHnNSF(44100, harmonic_num=8)      # state dict of the reference class loads strictly
    util.check_state_dict_layout(ours_sm, gold, "SourceModuleHnNSF__")
    ours_sm.load_state_dict(util.seeded_state_dict(ours_sm, 0))


def test_patch_reference_rebinds_and_restores_the_reference_names(monkeypatch):
    """patch_reference() on modules laid out like the reference's ddsp.vocoder / nsf_hifigan.models / nsf_hifigan.nvSTFT:
    the reference's entry points resolve these names at call time, so after patching they build this package's
    classes; unpatch_reference() restores the originals."""
    mods = {}
    for modname, names in (("ddsp.vocoder", ("Sins", "CombSub", "CombSubSuperFast", "CombSubFast", "Volume_Extractor")),
                           ("nsf_hifigan.models", ("SineGen", "SourceModuleHnNSF")), ("nsf_hifigan.nvSTFT", ("STFT",))):
        m = mods[modname] = types.ModuleType(modname)
        for n in names:
            setattr(m, n, type(n, (), {}))
    for pkgname in ("ddsp", "nsf_hifigan"):
        parent = types.ModuleType(pkgname)
        parent.__path__ = []
        monkeypatch.setitem(sys.modules, pkgname, parent)
    for modname, m in mods.items():
        monkeypatch.setitem(sys.modules, modname, m)
        setattr(sys.modules[modname.split(".")[0]], modname.split(".")[1], m)
    V, nsf, stft = mods["ddsp.vocoder"], mods["nsf_hifigan.models"], mods["nsf_hifigan.nvSTFT"]
    originals = {n: getattr(V, n) for n in ("Sins", "CombSub", "CombSubSuperFast", "CombSubFast", "Volume_Extractor")}
    originals.update(SineGen=nsf.SineGen, SourceModuleHnNSF=nsf.SourceModuleHnNSF)
    orig_stft = stft.STFT
    from ddsp_svc_b200 import frontend, mel
    saved = pkg.patch_reference()
    try:
        assert "_not_patched" not in saved
        assert V.Sins is pkg.Sins and V.CombSub is pkg.CombSub and V.CombSubSuperFast is pkg.CombSubSuperFast
        assert V.CombSubFast is pkg.CombSubFast and V.Volume_Extractor is frontend.Volume_Extractor
        assert nsf.SineGen is pkg.SineGen and nsf.SourceModuleHnNSF is pkg.SourceModuleHnNSF and stft.STFT is mel.STFT
    finally:
        pkg.unpatch_reference(saved)
    assert all(getattr(V if hasattr(V, n) else nsf, n) is c for n, c in originals.items())
    assert stft.STFT is orig_stft
