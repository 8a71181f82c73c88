"""Generate tests/golden/ref_grad_superfast_*.npz: the LIVE reference's CombSubSuperFast gradients with respect to its
four controls.  Run where the reference is available, like make_golden.py:

    python tests/golden/make_golden_grad.py

For each superfast case of cases.CASES, the reference's Unit2Control is replaced by a module returning leaf controls
(regenerated with cases.build_inputs), the noise is pinned by torch.manual_seed right before forward() (as in
make_golden.py), and the loss sum(g * signal) with the seeded N(0, 1) upstream gradient of tests/superfast_grad.py is
back-propagated through the reference's fp32 stft / istft on the CPU.
"""
import contextlib
import io
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)

from oracle import ref_loader  # noqa: E402
from tests import superfast_grad as SG  # noqa: E402
from tests.golden import cases as G  # noqa: E402


def run_reference(name):
    V, _, _ = ref_loader.load()
    inp = G.build_inputs(name)
    case, sd = inp["case"], G.seeds(name)
    B, nF = case["B"], case["nF"]
    leaves = {k: inp["ctrls"][k].detach().clone().contiguous().requires_grad_() for k in SG.KEYS}

    class Ctrl(torch.nn.Module):
        def forward(self, units, f0, phase, volume, **kw):
            return leaves, torch.zeros(B, nF, 256)

    with contextlib.redirect_stdout(io.StringIO()):
        m = V.CombSubSuperFast(G.SR, G.P, case["win"], n_unit=8)
    m.unit2ctrl = Ctrl()
    torch.manual_seed(sd["noise"])
    signal, _, _ = m(None, inp["f0"], None)
    g = SG.upstream(name, signal.shape)
    (signal * g).sum().backward()
    return inp, g, {k: leaves[k].grad for k in SG.KEYS}


def main():
    if not ref_loader.available():
        raise SystemExit("live reference not found; goldens can only be regenerated where it is available")
    for name in SG.CASES:
        inp, g, grads = run_reference(name)
        payload = {"grad_" + k: v.numpy().astype(np.float32) for k, v in grads.items()}
        payload.update({k: np.float64(v) for k, v in G.input_checksums(inp).items()})
        payload["cs_upstream"] = np.float64(G.input_checksums({"f0": g})["cs_f0"])
        payload["torch_version"] = np.array(torch.__version__)
        np.savez_compressed(SG.golden_path(name), **payload)
        print("%-28s %s" % (name, {k: tuple(v.shape) for k, v in payload.items() if getattr(v, "ndim", 0) > 0}))


if __name__ == "__main__":
    main()
