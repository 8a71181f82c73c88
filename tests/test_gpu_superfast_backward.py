"""GPU checks of the CombSubSuperFast backward (fused kernel b2d_superfast_backward, through the module's autograd
Function): gradients against the live reference's fp32 gradients and the float64 truth, full-size determinism and
shard invariance, in-kernel noise regenerated consistently with the forward, and training a small control network."""
import math

import numpy as np
import pytest
import torch

from ddsp_svc_b200 import CombSubSuperFast, FixedControls, ops, synthetic as syn
from oracle import torch_port as tp
from tests import report
from tests import superfast_grad as SG
from tests.golden import cases as G

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
SR, P, WIN, C = G.SR, G.P, 2048, 1025
OFFICIAL_REL = 1e-4
TRUTH_REL = 1e-5


def _grads(f0, dense, noise, g, seed=None, utterance_offset=0):
    """control gradients of sum(g * signal) through the module (leaf controls: views of one dense leaf)"""
    B, nF = dense.shape[0], dense.shape[1]
    leaf = dense.detach().to(DEV).clone().requires_grad_()
    ctrls = syn.split_views(leaf, syn.superfast_split_map(WIN))
    model = CombSubSuperFast(SR, P, WIN, unit2ctrl=FixedControls(ctrls, torch.zeros(B, nF, 256, device=DEV))).to(DEV)
    if seed is not None:
        torch.manual_seed(seed)
    signal, _, _ = model(None, f0.to(DEV), None, noise=None if noise is None else noise.to(DEV),
                         utterance_offset=utterance_offset)
    signal.backward(g.to(DEV))
    return signal.detach(), {k: v for k, v in zip(SG.KEYS, torch.split(leaf.grad, C, dim=-1))}


@pytest.mark.parametrize("name", SG.CASES)
def test_gradients_match_reference_and_float64_truth(name):
    inp = G.build_inputs(name)
    B, nF = inp["case"]["B"], inp["case"]["nF"]
    g = SG.upstream(name, (B, nF * P))
    _, got = _grads(inp["f0"], inp["dense"], inp["noise"], g)
    gold = np.load(SG.golden_path(name))
    comb = tp.superfast_source(inp["f0"], SR, P)[0]                 # the reference's fp32 comb
    tru = SG.truth(comb, inp["noise"], inp["ctrls"], g)
    rec = {}
    for k in SG.KEYS:
        mine, ref, t = got[k].cpu().numpy(), gold["grad_" + k], tru[k].numpy()
        rec[k + "_vs_ref"], rec[k + "_vs_truth"], rec[k + "_ref_vs_truth"] = (
            SG.rel_rms(mine, ref), SG.rel_rms(mine, t), SG.rel_rms(ref, t))
    report.record("superfast_backward/" + name, **rec)
    for k in SG.KEYS:
        assert rec[k + "_vs_ref"] < OFFICIAL_REL, (k, rec)
        assert rec[k + "_vs_truth"] < TRUTH_REL, (k, rec)


def test_full_size_deterministic_shard_invariant_and_true():
    """B = 32 x 10 s (BASELINE config 3)"""
    B, nF = 32, syn.n_frames_for(10.0)
    T = nF * P
    f0 = syn.make_f0(B, nF, SR, P, seed=11, unvoiced_fraction=0.05).to(DEV)
    dense, _ = syn.make_ctrl(B, nF, syn.superfast_split_map(WIN), seed=12)
    dense = dense.to(DEV)
    views = syn.split_views(dense, syn.superfast_split_map(WIN))
    gen = torch.Generator(device=DEV).manual_seed(13)
    g = torch.randn(B, T, device=DEV, generator=gen)
    noise = torch.randn(B, T, device=DEV, generator=gen)
    ws, _ = ops.superfast_scan(f0, P, SR)
    c = [views[k] for k in SG.KEYS]
    run = lambda **kw: torch.cat(ops.superfast_backward(ws, *c, g, P, WIN, **kw), dim=-1)
    a, b = run(noise_in=noise), run(noise_in=noise)
    assert torch.isfinite(a).all() and torch.equal(a, b)
    full = run(seed=5)                                              # in-kernel noise
    assert torch.isfinite(full).all() and torch.equal(full, run(seed=5))
    ws8, _ = ops.superfast_scan(f0[8:], P, SR)
    part = torch.cat(ops.superfast_backward(ws8, *[v[8:] for v in c], g[8:], P, WIN, seed=5, utterance_offset=8), -1)
    assert torch.equal(full[8:], part)
    # two sampled utterances against the float64 truth (whole utterance, rows compared in full)
    errs = {}
    for u in (3, 27):
        comb = tp.superfast_source(f0[u:u + 1].cpu(), SR, P)[0]
        tru = SG.truth(comb, noise[u:u + 1].cpu(), {k: views[k][u:u + 1].cpu() for k in SG.KEYS}, g[u:u + 1].cpu())
        for i, k in enumerate(SG.KEYS):
            errs["u%d_%s" % (u, k)] = SG.rel_rms(a[u, :, i * C:(i + 1) * C].cpu().numpy(), tru[k][0].numpy())
    report.record("superfast_backward/full_size_b32_10s", **errs)
    assert max(errs.values()) < TRUTH_REL, errs


def test_in_kernel_noise_matches_a_central_difference_of_the_forward():
    """Without noise_in the backward regenerates the forward's Philox noise: <grad, d> equals the central difference of
    sum(g * signal) along a seeded direction d.  Checked as is, and with the harmonic part muted (exp(-30)), where the
    signal is the filtered noise alone and a wrong noise stream would show in full."""
    B, nF = 2, 24
    f0 = syn.make_f0(B, nF, SR, P, seed=21).to(DEV)
    dense, _ = syn.make_ctrl(B, nF, syn.superfast_split_map(WIN), seed=22)
    dense = dense.to(DEV)
    muted = dense.clone()
    muted[..., :C] = -30.0
    gen = torch.Generator(device=DEV).manual_seed(23)
    g = torch.randn(B, nF * P, device=DEV, generator=gen)
    d = torch.randn(B, nF, 4 * C, device=DEV, generator=gen)
    ws, _ = ops.superfast_scan(f0, P, SR)
    views = lambda x: [x[..., i * C:(i + 1) * C] for i in range(4)]
    loss = lambda x: (ops.superfast_synth(ws, *views(x), P, WIN, seed=9).double() * g.double()).sum().item()
    res = {}
    for what, c in (("all", dense), ("noise_only", muted)):
        grad = torch.cat(ops.superfast_backward(ws, *views(c), g, P, WIN, seed=9), dim=-1)
        eps = 1e-3
        fd = (loss(c + eps * d) - loss(c - eps * d)) / (2 * eps)
        an = (grad.double() * d.double()).sum().item()
        res[what] = abs(fd - an) / abs(an)
    report.record("superfast_backward/in_kernel_noise_central_difference", **res)
    assert res["all"] < 1e-3 and res["noise_only"] < 1e-3, res


def _rss(x, y, n_ffts=(256, 512, 1024, 2047), eps=1e-7):
    """the reference's RSSLoss (ddsp/loss.py) restated with fixed n_ffts: normalised magnitude spectrogram without
    centring, spectral convergence + L1 of the log magnitudes, averaged over the scales"""
    total = 0.
    for n in n_ffts:
        w = torch.hann_window(n, device=x.device)
        spec = lambda z: torch.stft(z, n, hop_length=n, window=w, center=False, normalized=True,
                                    return_complex=True).abs() + eps
        st, sp = spec(y), spec(x)
        total = total + torch.mean(torch.linalg.norm(st - sp, dim=(1, 2)) / torch.linalg.norm(st + sp, dim=(1, 2))) \
            + torch.nn.functional.l1_loss(st.log(), sp.log())
    return total / len(n_ffts)


class _LinearCtrl(torch.nn.Module):
    """seeded Linear(n_unit -> 4100) + split_to_dict: a small differentiable unit2ctrl"""

    def __init__(self, n_unit, seed):
        super().__init__()
        torch.manual_seed(seed)
        self.dense_out = torch.nn.Linear(n_unit, 4 * C)
        with torch.no_grad():
            self.dense_out.weight.mul_(0.2)
            self.dense_out.bias.fill_(-1.0)

    def forward(self, units, f0, phase, volume, **kw):
        out = self.dense_out(units)
        return dict(zip(SG.KEYS, torch.split(out, C, dim=-1))), out


def _eager(unit2ctrl, units, comb, noise):
    """the same pipeline in eager torch on the GPU (the reference's stft -> filter -> istft)"""
    ctrls, _ = unit2ctrl(units, None, None, None)
    window = torch.hann_window(WIN, device=DEV)
    hold_last = lambda z: torch.cat((z, z[:, -1:, :]), dim=1)
    hs = hold_last(torch.exp(ctrls["harmonic_magnitude"] + 1.j * math.pi * ctrls["harmonic_phase"]))
    hn = hold_last(torch.exp(ctrls["noise_magnitude"] + 1.j * math.pi * ctrls["noise_phase"]) / 128)
    stft = lambda z: torch.stft(z, WIN, P, WIN, window=window, center=True, return_complex=True, pad_mode="reflect")
    spec = stft(comb) * hs.permute(0, 2, 1) + stft(noise) * hn.permute(0, 2, 1)
    return torch.istft(spec, WIN, P, WIN, window=window, center=True)


def test_module_trains_a_control_network():
    B, nF, n_unit = 2, 40, 16
    f0 = syn.make_f0(B, nF, SR, P, seed=31)
    gen = torch.Generator().manual_seed(32)
    units = torch.randn(B, nF, n_unit, generator=gen).to(DEV)
    noise = torch.randn(B, nF * P, generator=gen).to(DEV)
    comb = tp.superfast_source(f0, SR, P)[0].to(DEV)
    f0 = f0.to(DEV)
    teacher = _LinearCtrl(n_unit, 1).to(DEV)
    with torch.no_grad():
        target = _eager(teacher, units, comb, noise)
    student = _LinearCtrl(n_unit, 2).to(DEV)
    model = CombSubSuperFast(SR, P, WIN, unit2ctrl=student).to(DEV)

    # under grad the forward is the inference kernel, bit for bit
    signal, _, _ = model(units, f0, None, noise=noise)
    assert signal.requires_grad
    with torch.no_grad():
        plain, _, _ = model(units, f0, None, noise=noise)
    assert torch.equal(signal.detach(), plain)

    # weight gradient against the same pipeline in eager torch.  Both are driven by the same dL/dsignal (the loss's
    # gradient at the kernel's signal): the L1 term on log magnitudes turns the ~1e-7 difference between the two
    # forwards into a larger difference of dL/dsignal (its sign and 1/|S| at near-zero bins), which is the loss's
    # conditioning, not the backward's error; that end-to-end figure is recorded and loosely bounded.
    W = student.dense_out.weight
    signal_e = _eager(student, units, comb, noise)
    s_k, s_e = signal.detach().requires_grad_(), signal_e.detach().requires_grad_()
    loss, loss_e = _rss(s_k, target), _rss(s_e, target)
    (gs,) = torch.autograd.grad(loss, [s_k])
    (gs_e,) = torch.autograd.grad(loss_e, [s_e])
    (gw,) = torch.autograd.grad(signal, [W], grad_outputs=gs, retain_graph=True)
    (gw_e,) = torch.autograd.grad(signal_e, [W], grad_outputs=gs, retain_graph=True)
    (gw_e2e,) = torch.autograd.grad(signal_e, [W], grad_outputs=gs_e)
    rel = lambda a, b: ((a - b).norm() / b.norm()).item()
    res = dict(weight_grad_same_upstream=rel(gw, gw_e), weight_grad_end_to_end=rel(gw, gw_e2e),
               loss_grad=rel(gs, gs_e), signal=rel(signal.detach(), signal_e.detach()), loss=loss.item(),
               loss_eager=loss_e.item())
    report.record("superfast_backward/module_weight_grad_vs_eager", **res)
    assert res["weight_grad_same_upstream"] < 1e-4, res
    assert res["weight_grad_end_to_end"] < 1e-2, res

    # 20 Adam steps lower the loss
    opt = torch.optim.Adam(student.parameters(), lr=1e-2)
    losses = []
    for _ in range(21):
        opt.zero_grad()
        l = _rss(model(units, f0, None, noise=noise)[0], target)
        l.backward()
        opt.step()
        losses.append(l.item())
    report.record("superfast_backward/module_adam", first=losses[0], after_20_steps=losses[-1])
    assert losses[-1] < losses[0], losses

    # what the backward does not provide
    with pytest.raises(NotImplementedError, match="f0"):
        model(units, f0.clone().requires_grad_(), None, noise=noise)
    with pytest.raises(NotImplementedError, match="noise"):
        model(units, f0, None, noise=noise.clone().requires_grad_())
    with pytest.raises(ValueError, match="signal_out"):
        model(units, f0, None, noise=noise, signal_out=torch.empty(B, nF * P, device=DEV))
