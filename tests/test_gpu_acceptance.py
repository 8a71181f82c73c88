"""Acceptance run on the GPU: the reference's call (main.py:259, `model(seg_units, seg_f0, seg_volume, spk_id=...,
spk_mix_dict=...)` under torch.no_grad, then `seg_output *= mask` in place, main.py:260) on this package's synthesizers,
built through `load_model` (config.yaml next to the checkpoint -> class dispatch -> strict load of a checkpoint in the
reference's layout, this package's Unit2Control included) -- real torch.split views of dense_out, real spk_id embedding
/ spk_mix_dict -- and the waveforms compared with the reference's classes run on the same seeded weights and inputs.

The reference's outputs are stored in tests/golden/ref_acceptance.npz (a seeded sample of each waveform plus its full
RMS; made by tests/golden/make_golden_models.py on the CPU).  Its white noise (rand_like / randn_like) was replaced by
seeded draws there (tests.util.seeded_draw); the test feeds the same samples to the B200 module (`noise=`), so the full
signal is comparable; the exact main.py call without `noise=` (in-kernel Philox) is checked on its deterministic part
and on the noise level."""
import numpy as np
import pytest
import torch
import yaml

import ddsp_svc_b200 as pkg
from tests import report, util

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
SR, P, NU = 44100, 512, 768
SEED = 1
# The reference's DSP runs on the CPU (the oracle path, SURVEY A.10) and so do the kernels' formulas; reference-on-GPU
# differs from reference-on-CPU by a few 1e-6 absolute at this signal level (RMS 0.06-0.08, i.e. <= 1e-4 relative:
# torch's fp32 cumsum accumulates in fp32 on CUDA and in fp64 on the CPU).  The bound is the north star's 1e-4 RMS;
# parity at the 1e-8 level is pinned on identical controls by the golden tests.
GATE_RMS = 1e-4


# `make` takes the module holding the classes: ddsp_svc_b200 here, the reference's ddsp.vocoder for the stored outputs
CASES = {
    "Sins": dict(model={"type": "Sins", "n_harmonics": 128, "n_mag_allpass": 256, "n_mag_noise": 256, "n_spk": 2},
                 make=lambda V: V.Sins(SR, P, 128, 256, 256, n_unit=NU, n_spk=2), uniform=True, parts=True),
    "CombSub": dict(model={"type": "CombSub", "n_mag_allpass": 256, "n_mag_harmonic": 512, "n_mag_noise": 256, "n_spk": 2},
                    make=lambda V: V.CombSub(SR, P, 256, 512, 256, n_unit=NU, n_spk=2), uniform=True, parts=True),
    "CombSubSuperFast": dict(model={"type": "CombSubSuperFast", "win_length": 2048, "n_spk": 2},
                             make=lambda V: V.CombSubSuperFast(SR, P, 2048, n_unit=NU, n_spk=2), uniform=False, parts=False,
                             ),
    "CombSubFast": dict(model={"type": "CombSubFast", "n_spk": 2},
                        make=lambda V: V.CombSubFast(SR, P, n_unit=NU, n_spk=2), uniform=True, parts=False),
}


def inputs():
    """one main.py segment (~1.5 s), B = 1, on the CPU: units, f0, volume and the caller's silence mask"""
    nF = 130
    g = torch.Generator().manual_seed(2)
    units = torch.randn(1, nF, NU, generator=g)
    f0 = 220.0 * 2 ** (torch.rand(1, nF, 1, generator=g) * 0.3)
    f0[:, 40:48] = 0.0                              # an unvoiced stretch, as f0 extractors produce
    volume = 0.1 * torch.rand(1, nF, 1, generator=g)
    mask = (torch.rand(1, nF * P, generator=g) > 0.1).float()
    return units, f0, volume, mask


def calls():
    spk_id = torch.LongTensor([[2]])
    return [dict(spk_id=spk_id, spk_mix_dict=None), dict(spk_id=spk_id, spk_mix_dict={1: 0.3, 2: 0.7})]


def source_module_f0():
    f0 = 200.0 + 50.0 * torch.rand(2, 40, generator=torch.Generator().manual_seed(3))
    f0[:, 10:14] = 0.0
    return f0


@pytest.mark.parametrize("kind", list(CASES))
def test_main_py_call_reference_vs_patched(kind, tmp_path):
    case = CASES[kind]
    gold = util.load_golden("ref_acceptance")
    cfg = {"data": {"sampling_rate": SR, "block_size": P, "encoder_out_channels": NU}, "model": case["model"]}
    (tmp_path / "config.yaml").write_text(yaml.safe_dump(cfg))
    torch.save({"global_step": 1, "model": util.seeded_state_dict(case["make"](pkg), SEED)}, tmp_path / "model_1.pt")
    model, args = pkg.load_model(str(tmp_path / "model_1.pt"), device=DEV)
    assert type(model) is getattr(pkg, kind)
    units, f0, volume, mask = (t.to(DEV) for t in inputs())
    tol = case.get("tol", GATE_RMS)
    with torch.no_grad():
        for i, kw in enumerate(calls()):
            p = "%s__c%d__" % (kind, i)
            kw = {k: (v.to(DEV) if torch.is_tensor(v) else v) for k, v in kw.items()}
            drawn = util.stored_draws(gold, p)
            assert len(drawn) == 1 and (drawn[0][0] == "rand") == case["uniform"]
            noise = (drawn[0][1] * 2 - 1 if case["uniform"] else drawn[0][1]).reshape(1, -1).to(DEV)
            r_sig, r_hid, r_h, r_n = (gold.get(p + k) for k in ("signal", "hidden", "harmonic", "noise"))
            # (1) same noise samples -> the whole signal is comparable
            sig, hidden, (s_h, s_n) = model(units, f0, volume, noise=noise, **kw)
            # this package's Unit2Control (fused kernels + fp32 library GEMMs) against the reference's class in fp32
            assert util.rms(util.sampled(hidden, r_hid.size) - r_hid) < 1e-4 * max(util.rms(r_hid), 1e-6)
            d = util.sampled(sig, r_sig.size) - r_sig
            e = util.rms(d)
            report.record("acceptance/%s/%s" % (kind, "mix" if kw["spk_mix_dict"] else "spk"), err=e,
                          max=np.abs(d).max(), signal_rms=float(gold[p + "signal_rms"]))
            assert e < tol
            if case["parts"]:
                assert util.rms(util.sampled(s_h, r_h.size) - r_h) < tol and util.rms(util.sampled(s_n, r_n.size) - r_n) < tol
            # (2) the exact main.py lines: no `noise=`, then the in-place mask multiply on the returned tensor
            seg_output, _, (s_h2, s_n2) = model(units, f0, volume, **kw)
            if case["parts"]:
                assert util.rms(util.sampled(s_h2, r_h.size) - r_h) < tol                    # deterministic part
                lvl = util.rms(s_n2.cpu()) / max(float(gold[p + "noise_rms"]), 1e-12)
                assert 0.9 < lvl < 1.1                                                     # same noise level, other samples
                keep_h = s_h2.clone()
            else:
                lvl = util.rms(seg_output.cpu()) / max(float(gold[p + "signal_rms"]), 1e-12)
                assert 0.8 < lvl < 1.25
            before = seg_output.clone()
            seg_output *= mask                                                              # main.py:260
            assert torch.equal(seg_output, before * mask)
            if case["parts"]:
                assert torch.equal(s_h2, keep_h)                                           # outputs are not aliased


def test_enhancer_source_module_through_patch_reference():
    """enhancer.py's generator builds `SourceModuleHnNSF(...)` from nsf_hifigan.models, which patch_reference() rebinds to
    the fused B200 module (tests/test_dropin.py): same state dict, and with the reference's random phases / noise fed in,
    the same output as the reference's class."""
    gold = util.load_golden("ref_acceptance")
    ours = pkg.SourceModuleHnNSF(SR, harmonic_num=8).to(DEV).eval()
    ours.load_state_dict(util.seeded_state_dict(ours, SEED))
    drawn = util.stored_draws(gold, "source_module__")
    assert [k for k, _ in drawn] == ["rand", "randn"]          # SineGen's initial phases, then its additive noise
    rand_ini = drawn[0][1].clone(); rand_ini[..., 0] = 0
    with torch.no_grad():
        out = ours(source_module_f0().to(DEV), 512, rand_ini=rand_ini.to(DEV), noise=drawn[1][1].to(DEV))
    want = gold["source_module__out"]
    e = util.rms(util.sampled(out, want.size) - want)
    report.record("acceptance/source_module", err=e, rms=util.rms(want))
    assert list(out.shape) == list(gold["source_module__shape"]) and e < 1e-4
