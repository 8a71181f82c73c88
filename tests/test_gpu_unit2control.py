"""GPU parity of this package's Unit2Control (fused kernels of csrc/unit2control.cu + library GEMMs) against the reference's
own class (ddsp/unit2control.py with PCmer / ConformerNaiveEncoder) evaluated on the CPU in fp32, on the same seeded
weights (tests.util.seeded_state_dict, strict load) and inputs.  The reference's outputs are stored in
tests/golden/ref_u2c_gpu.npz (a seeded sample of each output; made by tests/golden/make_golden_models.py)."""
import numpy as np
import pytest
import torch

import ddsp_svc_b200 as pkg
from ddsp_svc_b200.unit2control import Unit2Control
from tests import report, util

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
SEED = 3

VARIANTS = {
    "pcmer_sins": (dict(), {"amplitudes": 128, "group_delay": 256, "noise_magnitude": 256}),
    "pcmer_sins_fused_attention": (dict(), {"amplitudes": 128, "group_delay": 256, "noise_magnitude": 256}),
    "naive_superfast": (dict(use_naive_v2=True, use_conv_stack=True, use_pitch_aug=True),
                        {"harmonic_magnitude": 1025, "harmonic_phase": 1025, "noise_magnitude": 1025, "noise_phase": 1025}),
    "pcmer_norm_plainconv": (dict(pcmer_norm=True, use_conv_stack=False), {"a": 33, "b": 7}),
}
# variant -> the stored reference outputs it is compared with (the fused attention computes the same function)
REF_OUTPUTS = {n: n for n in VARIANTS}
REF_OUTPUTS["pcmer_sins_fused_attention"] = "pcmer_sins"


def calls(kw):
    c = [dict(spk_id=torch.LongTensor([[2], [3]])), dict(spk_id=torch.LongTensor([[1]]), spk_mix_dict={1: 0.25, 3: 0.75})]
    if kw.get("use_pitch_aug"):
        c.append(dict(spk_id=torch.LongTensor([[1], [1]]), aug_shift=torch.tensor([[[2.0]], [[-3.0]]])))
    return c


def _inputs(B, T, n_unit, seed):
    g = torch.Generator().manual_seed(seed)
    units = torch.randn(B, T, n_unit, generator=g)
    f0 = 220.0 * 2 ** (torch.rand(B, T, 1, generator=g) * 2 - 1)
    f0[:, 5:9] = 0.0
    phase = (torch.rand(B, T, 1, generator=g) * 2 - 1) * 3.14159
    volume = 0.2 * torch.rand(B, T, 1, generator=g)
    return units, f0, phase, volume


@pytest.mark.parametrize("name", list(VARIANTS))
def test_unit2control_matches_the_reference_class(name):
    kw, splits = VARIANTS[name]
    gold, ref_name = util.load_golden("ref_u2c_gpu"), REF_OUTPUTS[name]
    torch.manual_seed(SEED)
    ours = Unit2Control(768, 3, splits, **kw)
    util.check_state_dict_layout(ours, gold, ref_name + "__")
    ours.load_state_dict(util.seeded_state_dict(ours, SEED))                # strict
    ours = ours.to(DEV).eval()
    ours.fused_attention = name.endswith("fused_attention")      # the opt-in one-kernel linear attention (csrc/linear_attention.cu)
    B, T = 2, 150
    units, f0, phase, volume = _inputs(B, T, 768, 4)
    for i, c in enumerate(calls(kw)):
        cg = {k: (v.to(DEV) if torch.is_tensor(v) else v) for k, v in c.items()}
        got_c, got_h = ours(units.to(DEV), f0.to(DEV), phase.to(DEV), volume.to(DEV), **cg)
        assert list(got_c.keys()) == [str(k) for k in gold[ref_name + "__ctrl_names"]]
        dense_w, want_h = gold["%s__c%d__controls" % (ref_name, i)], gold["%s__c%d__hidden" % (ref_name, i)]
        dense_g = util.sampled(torch.cat([got_c[k] for k in got_c], -1), dense_w.size)
        first = next(iter(got_c.values()))
        assert first.stride(1) == sum(splits.values())                      # views of one dense tensor, like torch.split
        e_c = util.rms(dense_g - dense_w) / max(util.rms(dense_w), 1e-12)
        e_h = util.rms(util.sampled(got_h, want_h.size) - want_h) / max(util.rms(want_h), 1e-12)
        report.record("unit2control/%s/%d" % (name, i), controls_rel_rms=e_c, hidden_rel_rms=e_h,
                      controls_max=np.abs(dense_g - dense_w).max())
        assert e_c < 2e-5 and e_h < 2e-5


def test_sins_forward_end_to_end_without_the_reference_unit2ctrl():
    """Sins built WITHOUT a unit2ctrl argument now owns this package's Unit2Control: a reference checkpoint loads strictly
    and the whole forward (control network + DSP) matches the reference's CPU forward within the north-star bound."""
    gold = util.load_golden("ref_u2c_gpu")
    torch.manual_seed(5)
    ours = pkg.Sins(44100, 512, 128, 256, 256, n_unit=768, n_spk=2)
    assert isinstance(ours.unit2ctrl, Unit2Control)
    ours.load_state_dict(util.seeded_state_dict(ours, SEED))
    ours = ours.to(DEV).eval()
    units, f0, _, volume = _inputs(1, 90, 768, 6)
    spk = torch.LongTensor([[2]])
    drawn = util.stored_draws(gold, "e2e__")          # the reference's one rand_like
    assert [k for k, _ in drawn] == ["rand"]
    noise = (drawn[0][1] * 2 - 1).reshape(1, -1)
    with torch.no_grad():
        got, got_h, (gh, gn) = ours(units.to(DEV), f0.to(DEV), volume.to(DEV), spk_id=spk.to(DEV), noise=noise.to(DEV))
    want, wh, wn = gold["e2e__signal"], gold["e2e__harmonic"], gold["e2e__noise"]
    e = util.rms(util.sampled(got, want.size) - want)
    report.record("unit2control/sins_e2e", err=e, signal_rms=util.rms(want), harmonic=util.rms(util.sampled(gh, wh.size) - wh),
                  noise=util.rms(util.sampled(gn, wn.size) - wn))
    assert e < 1e-4 and e < 2e-3 * util.rms(want)
