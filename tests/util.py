"""Shared helpers for the tests (oracle access lives here: tests are allowed to use it)."""
import math

import numpy as np
import torch

from tests.golden import cases as G


def rms(a):
    a = np.asarray(a, np.float64)
    return float(np.sqrt(np.mean(np.square(a)))) if a.size else 0.0


def load_golden(name):
    z = np.load(G.path(name), allow_pickle=False)
    return {k: z[k] for k in z.files}


# float buffers a module computes deterministically at construction (kept as built, never replaced by seeded values)
_FIXED_BUFFERS = ("window",)


def seeded_state_dict(module, seed):
    """Deterministic weights for `module`'s state dict, so that a test can rebuild exactly the weights a stored reference
    output (tests/golden/) was computed with.  Depends only on the keys, shapes and dtypes in state-dict order: the
    reference's classes and this package's produce the same values.  Scales follow torch's default initialisation:
    U(-1, 1) / sqrt(fan_in) for matrices and kernels, 1 + U(-0.1, 0.1) for 1-D norm weights, U(-1, 1) / 16 for biases,
    N(0, 1) for the random-feature projection of the linear attention."""
    g = torch.Generator().manual_seed(seed)
    out = {}
    for k, v in module.state_dict().items():
        if not v.is_floating_point() or k.endswith(_FIXED_BUFFERS):
            out[k] = v.clone()
            continue
        if k.endswith("projection_matrix"):
            w = torch.empty(v.shape, dtype=torch.float64).normal_(generator=g)
        else:
            u = torch.empty(v.shape, dtype=torch.float64).uniform_(-1, 1, generator=g)
            if v.dim() == 1:
                w = 1 + 0.1 * u if k.endswith("weight") else u / 16
            else:
                w = u / math.sqrt(v[0].numel())
        out[k] = w.to(v.dtype)
    return out


def seeded_draw(kind, shape, seed):
    """The stand-in for one torch.rand / torch.rand_like ("rand") or torch.randn_like ("randn") draw of the reference:
    when the stored reference outputs were made, each such draw returned this tensor (float32, CPU)."""
    g = torch.Generator().manual_seed(int(seed))
    t = torch.empty(tuple(int(s) for s in shape), dtype=torch.float32)
    return t.uniform_(0, 1, generator=g) if str(kind) == "rand" else t.normal_(generator=g)


def stored_draws(gold, prefix):
    """The random draws a stored reference call made, regenerated: [(kind, tensor)] in call order."""
    return [(str(k), seeded_draw(k, [int(x) for x in s.split(",")], seed))
            for k, s, seed in zip(gold[prefix + "draw_kind"], gold[prefix + "draw_shape"], gold[prefix + "draw_seed"])]


def check_state_dict_layout(module, gold, prefix):
    """`module`'s state dict has the reference's keys, in the reference's order, with the reference's shapes."""
    sd = module.state_dict()
    assert list(sd) == [str(k) for k in gold[prefix + "keys"]]
    assert [",".join(map(str, v.shape)) for v in sd.values()] == [str(s) for s in gold[prefix + "shapes"]]


def sample_index(n, k, seed=0):
    """Sorted positions of a fixed, seeded sample of k of n elements (all n when k >= n): stored reference outputs keep
    only these elements of a flattened output."""
    if k >= n:
        return np.arange(n)
    return np.sort(np.random.default_rng(seed).choice(n, size=k, replace=False))


def sampled(t, k, seed=0):
    """The elements of `t` (torch tensor or array, flattened) at sample_index(t.size, k, seed), as numpy."""
    a = t.detach().cpu().numpy() if torch.is_tensor(t) else np.asarray(t)
    a = a.reshape(-1)
    return a[sample_index(a.size, k, seed)]


def check_inputs_match_golden(name, inp, gold):
    """The goldens were produced from seeded inputs; make sure this torch build regenerates
    the same inputs (otherwise the comparison is meaningless)."""
    for k, v in G.input_checksums(inp).items():
        assert k in gold, k
        assert abs(float(gold[k]) - v) <= 1e-9 * max(1.0, abs(v)), \
            "input %s of %s differs from the one the golden was made with" % (k, name)


def port_outputs(name, inp):
    """Run the oracle's torch port on a golden case."""
    from oracle import torch_port as tp
    case = inp["case"]
    with torch.no_grad():
        if case["kind"] == "sins":
            return tp.sins_forward(inp["f0"], inp["ctrls"], G.SR, G.P, noise=inp["noise"],
                                   initial_phase=inp.get("initial_phase"))
        if case["kind"] == "combsub":
            return tp.combsub_forward(inp["f0"], inp["ctrls"], G.SR, G.P, noise=inp["noise"])
        if case["kind"] == "superfast":
            return tp.superfast_forward(inp["f0"], inp["ctrls"], G.SR, G.P, case["win"], noise=inp["noise"])
        if case["kind"] == "combsubfast":
            return tp.combsubfast_forward(inp["f0"], inp["ctrls"], G.SR, G.P, noise=inp["noise"],
                                          initial_phase=inp.get("initial_phase"))
        if case["kind"] == "source_module":
            gold = load_golden(name)          # the seeded Linear(9 -> 1) parameters travel with the golden
            return tp.source_module_forward(inp["f0"], case["upp"], G.SR, torch.from_numpy(gold["weight"]),
                                            torch.from_numpy(gold["bias"]), case["harmonic_num"],
                                            rand_ini=inp["rand_ini"], noise=inp["noise"])
        return tp.sinegen_forward(inp["f0"], case["upp"], G.SR, case["harmonic_num"],
                                  rand_ini=inp["rand_ini"], noise=inp["noise"])


def closed_form_outputs(name, inp):
    from oracle import closed_form as cf
    case = inp["case"]
    npc = lambda d: {k: v.numpy() for k, v in d.items()}
    if case["kind"] == "sins":
        ip = inp.get("initial_phase")
        return cf.sins(inp["f0"].numpy(), npc(inp["ctrls"]), G.SR, G.P, inp["noise"].numpy(),
                       None if ip is None else ip.numpy())
    if case["kind"] == "combsub":
        return cf.combsub(inp["f0"].numpy(), npc(inp["ctrls"]), G.SR, G.P, inp["noise"].numpy())
    if case["kind"] == "combsubfast":
        ip = inp.get("initial_phase")
        return cf.combsubfast(inp["f0"].numpy(), npc(inp["ctrls"]), G.SR, G.P, inp["noise"].numpy(),
                              None if ip is None else ip.numpy())
    if case["kind"] == "superfast":
        return cf.superfast(inp["f0"].numpy(), npc(inp["ctrls"]), G.SR, G.P, case["win"], inp["noise"].numpy())
    sines = cf.sinegen(inp["f0"].numpy(), case["upp"], G.SR, inp["rand_ini"].numpy().reshape(-1), inp["noise"].numpy())
    if case["kind"] == "source_module":
        gold = load_golden(name)
        return {"out": np.tanh(sines @ gold["weight"].astype(np.float64).T + gold["bias"].astype(np.float64))}
    return {"out": sines}
