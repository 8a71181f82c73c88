"""The closed form of the CombSubSuperFast backward (DESIGN.md section 4.6b), restated in numpy (tests/superfast_grad.py),
against torch autograd in float64 of the oracle port's stft -> filter -> istft, on the three golden shapes: reflect
padding (nF = 24, 5) and constant padding (nF = 2)."""
import numpy as np
import pytest
import torch

from oracle import torch_port
from tests import superfast_grad as SG
from tests.golden import cases as G


@pytest.mark.parametrize("name", SG.CASES)
def test_closed_form_matches_float64_autograd_of_the_oracle(name):
    inp = G.build_inputs(name)
    leaves = {k: inp["ctrls"][k].detach().double().requires_grad_() for k in SG.KEYS}
    old = torch.get_default_dtype()
    torch.set_default_dtype(torch.float64)          # the port's hann_window follows the default dtype
    try:
        out = torch_port.superfast_forward(inp["f0"].double(), leaves, G.SR, G.P, 2048, noise=inp["noise"].double())
    finally:
        torch.set_default_dtype(old)
    g = SG.upstream(name, out["signal"].shape).double()
    (out["signal"] * g).sum().backward()
    comb, noise = out["comb"].detach(), out["noise_in"].detach()
    got = SG.model(comb.numpy(), noise.numpy(), {k: v.detach().numpy() for k, v in leaves.items()}, g.numpy())
    tru = SG.truth(comb, noise, leaves, g)          # the restated float64 truth the GPU tests use
    for k in SG.KEYS:
        want = leaves[k].grad.numpy()
        assert SG.rel_rms(got[k], want) <= 1e-10, (name, k, SG.rel_rms(got[k], want))
        assert SG.rel_rms(tru[k].numpy(), want) <= 1e-12, (name, k)
