"""Host logic of ddsp_svc_b200.unit2control.Unit2Control on the CPU: parameter tree (state-dict keys / shapes), weight
packing (k = 3 convolution as one GEMM over shifted inputs, fused q/k/v weights, weight-norm) and the order of operations,
with the five fused CUDA kernels replaced by their torch definitions, against the reference's class: its state-dict
layout and its outputs on seeded weights and inputs, stored in tests/golden/ref_u2c_host.npz by
tests/golden/make_golden_models.py.  (The kernels themselves are checked on the GPU in tests/test_gpu_unit2control.py.)"""
import math

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from ddsp_svc_b200 import unit2control as U
from tests import util

SEED = 3
VARIANTS = {"pcmer": (dict(), {"a": 33, "b": 7}),
            "naive_conformer": (dict(use_naive_v2=True, use_conv_stack=True, use_pitch_aug=True), {"a": 33, "b": 7}),
            "pcmer_norm_plainconv": (dict(pcmer_norm=True, use_conv_stack=False), {"a": 33, "b": 7})}


def inputs():
    g = torch.Generator().manual_seed(1)
    units, f0 = torch.randn(2, 50, 64, generator=g), 200 + 100 * torch.rand(2, 50, 1, generator=g)
    ph, vo = torch.rand(2, 50, 1, generator=g), torch.rand(2, 50, 1, generator=g)
    return units, f0, ph, vo


def calls(kw):
    c = [dict(spk_id=torch.LongTensor([[2], [3]])), dict(spk_id=torch.LongTensor([[1]]), spk_mix_dict={1: 0.3, 2: 0.7})]
    if kw.get("use_pitch_aug"):
        c.append(dict(spk_id=torch.LongTensor([[1], [1]]), aug_shift=torch.tensor([[[2.0]], [[-3.0]]])))
    return c


def _layernorm(x, w, b):
    return F.layer_norm(x, (x.shape[-1],), w, b, 1e-5)


def _conv_module(self, x, Ly, pre_norm):
    B, T, C = x.shape
    h = _layernorm(x, Ly["cln_w"], Ly["cln_b"]) if pre_norm else x
    h = torch.addmm(Ly["pw1_b"], h.reshape(-1, C), Ly["pw1_w"].t()).reshape(B, T, -1)
    inner = Ly["dw_w"].shape[0]
    g = h[..., :inner] * torch.sigmoid(h[..., inner:])
    g = F.conv1d(F.pad(g.transpose(1, 2), (15, 15)), Ly["dw_w"].unsqueeze(1), Ly["dw_b"], groups=inner).transpose(1, 2)
    g = g * torch.sigmoid(g)
    return torch.addmm(Ly["pw2_b"], g.reshape(-1, inner), Ly["pw2_w"].t()).reshape(B, T, C)


def _attention(self, x, Ly):
    B, T, C = x.shape
    a = self.decoder._layers[0].attn
    H, d = a.heads, a.dim_head
    h = _layernorm(x, Ly["ln_w"], Ly["ln_b"])
    qkv = torch.addmm(Ly["qkv_b"], h.reshape(-1, C), Ly["qkv_w"].t()).reshape(B, T, 3, H, d)
    q, k, v = (qkv[:, :, i].permute(0, 2, 1, 3).contiguous() for i in range(3))
    if self.pcmer_norm:
        q = q / (q.norm(dim=-1, keepdim=True) + 1e-8)
        k = k / (k.norm(dim=-1, keepdim=True) + 1e-8)
    J = Ly["proj_t"].shape[1]
    feats = []
    for data, is_q in ((q, 1), (k, 0)):
        dd = torch.mm(data.reshape(-1, d), Ly["proj_t"])                  # the d^-1/4 normaliser is folded into proj_t
        diag = (data.reshape(-1, d) ** 2).sum(-1, keepdim=True) / 2 * (d ** -0.5)
        dd = (J ** -0.5) * (torch.exp(dd - diag - dd.max(-1, keepdim=True).values) + 1e-4) if is_q else (J ** -0.5) * torch.exp(dd - diag + 1e-4)
        feats.append(dd.reshape(B, H, T, J))
    qf, kf = feats
    d_inv = 1.0 / (torch.einsum("bhnj,bhj->bhn", qf, kf.sum(dim=-2)) + 1e-8)
    out = torch.matmul(qf, torch.matmul(kf.transpose(-1, -2), v)) * d_inv.unsqueeze(-1)
    return torch.addmm(Ly["out_b"], out.permute(0, 2, 1, 3).reshape(B * T, H * d), Ly["out_w"].t()).reshape(B, T, C)


class _Fp32:
    mode = "fp32"

    @staticmethod
    def linear(x2d, w, bias):
        return torch.addmm(bias, x2d, w.t())


def _forward(self, units, f0, phase, volume, spk_id=None, spk_mix_dict=None, aug_shift=None):
    B, T, _ = units.shape
    P = self._pack()
    x = self._conv3(_Fp32, units, P["c1_w"], P["c1_b"])
    if self.use_conv_stack:
        x = F.leaky_relu(F.group_norm(x.transpose(1, 2), 4, P["gn_w"], P["gn_b"], 1e-5), 0.01).transpose(1, 2)
        x = self._conv3(_Fp32, x, P["c2_w"], P["c2_b"])
    e = P["emb"]
    x = x + (e[0] * torch.log(1 + f0 / 700) + e[1]) + (e[2] * (phase / math.pi) + e[3]) + (e[4] * volume + e[5])
    if self.n_spk and self.n_spk > 1:
        if spk_mix_dict is not None:
            x = x + sum(float(v) * self.spk_embed.weight[int(k) - 1] for k, v in spk_mix_dict.items())
        else:
            x = x + self.spk_embed(spk_id - 1)
    if self.aug_shift_embed is not None and aug_shift is not None:
        x = x + e[6] * (aug_shift / 5)
    for Ly in P["layers"]:
        if not self.use_naive_v2:
            x = x + self._attention(x, Ly)
        x = x + self._conv_module(x, Ly, pre_norm=not self.use_naive_v2)
    x = _layernorm(x, P["n_w"], P["n_b"])
    e = torch.addmm(P["do_b"], x.reshape(-1, 256), P["do_w"].t()).reshape(B, T, self.n_out)
    return U.split_to_dict(e, self.output_splits), x


@pytest.fixture
def torch_kernels(monkeypatch):
    monkeypatch.setattr(U.Unit2Control, "_layernorm", staticmethod(_layernorm))
    monkeypatch.setattr(U.Unit2Control, "_conv_module", _conv_module)
    monkeypatch.setattr(U.Unit2Control, "_attention", _attention)
    monkeypatch.setattr(U.Unit2Control, "forward", _forward)
    monkeypatch.setattr(U.Unit2Control, "gemm_precision", "fp32")       # plain [O, K] weights in the packed dict


@pytest.mark.parametrize("name", list(VARIANTS))
def test_parameter_tree_and_host_logic_match_the_reference(name, torch_kernels):
    kw, splits = VARIANTS[name]
    gold = util.load_golden("ref_u2c_host")
    torch.manual_seed(SEED)
    ours = U.Unit2Control(64, 3, splits, **kw).eval()
    util.check_state_dict_layout(ours, gold, name + "__")
    ours.load_state_dict(util.seeded_state_dict(ours, SEED))     # strict
    units, f0, ph, vo = inputs()
    for i, c in enumerate(calls(kw)):
        with torch.no_grad():
            gc, gh = ours(units, f0, ph, vo, **c)
        assert list(gc) == [str(k) for k in gold[name + "__ctrl_names"]]
        dw, wh = gold["%s__c%d__controls" % (name, i)], gold["%s__c%d__hidden" % (name, i)]
        dg = util.sampled(torch.cat(list(gc.values()), -1), dw.size)
        assert np.abs(dw - dg).max() < 2e-5 * max(1.0, np.abs(dw).max())
        assert np.abs(wh - util.sampled(gh, wh.size)).max() < 2e-5 * max(1.0, np.abs(wh).max())
