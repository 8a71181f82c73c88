"""Shared pieces of the CombSubSuperFast backward tests and of tests/golden/make_golden_grad.py: the cases, the seeded
upstream gradient, the float64 truth (torch autograd of stft -> filter -> istft) and a numpy model of the backward's
closed form (DESIGN.md section 4.6b)."""
import math

import numpy as np
import torch

from tests.golden import cases as G

P, N = G.P, 2048
KEYS = ("harmonic_magnitude", "harmonic_phase", "noise_magnitude", "noise_phase")
# the superfast golden cases: reflect padding (nF = 24, 5) and constant padding (nF = 2)
CASES = [n for n, c in G.CASES.items() if c["kind"] == "superfast"]


def golden_path(name):
    return G.path("ref_grad_" + name)


def upstream(name, shape):
    """The seeded N(0, 1) dL/dsignal of a case (loss = sum(g * signal))."""
    gen = torch.Generator().manual_seed(5000 + sum(ord(c) for c in name))
    return torch.empty(tuple(shape), dtype=torch.float32).normal_(generator=gen)


def truth(comb, noise, ctrls, g):
    """dL/dcontrols by torch autograd in float64 of the reference's stft -> filter -> istft, on the given (fp32)
    comb and noise.  ctrls: dict of [B, nF, 1025]; returns a dict of float64 tensors."""
    leaves = {k: ctrls[k].detach().double().requires_grad_() for k in KEYS}
    window = torch.hann_window(N, dtype=torch.float64)
    hold_last = lambda z: torch.cat((z, z[:, -1:, :]), dim=1)
    h_src = hold_last(torch.exp(leaves["harmonic_magnitude"] + 1.j * math.pi * leaves["harmonic_phase"]))
    h_noise = hold_last(torch.exp(leaves["noise_magnitude"] + 1.j * math.pi * leaves["noise_phase"]) / 128)
    pad_mode = "reflect" if comb.shape[-1] > N // 2 else "constant"
    stft = lambda z: torch.stft(z.double(), n_fft=N, win_length=N, hop_length=P, window=window, center=True,
                                return_complex=True, pad_mode=pad_mode)
    spec = stft(comb) * h_src.permute(0, 2, 1) + stft(noise) * h_noise.permute(0, 2, 1)
    signal = torch.istft(spec, n_fft=N, win_length=N, hop_length=P, window=window, center=True)
    (signal * g.double()).sum().backward()
    return {k: leaves[k].grad for k in KEYS}


def model(comb, noise, ctrls, g):
    """The backward's closed form in numpy float64: u_q = w g / env, G_q = (c_k / N) rfft(u_q), X_q / Z_q = rfft of the
    windowed source frames, dL/dm = Re(conj(G) Y), dL/dp = pi Im(G conj(Y)); frame nF folds into row nF-1."""
    comb, noise, g = (np.asarray(a, np.float64) for a in (comb, noise, g))
    B, T = g.shape
    nF = T // P
    w = 0.5 - 0.5 * np.cos(2 * np.pi * np.arange(N) / N)
    env = np.zeros(T + N)
    for q in range(nF + 1):
        env[q * P:q * P + N] += w * w
    gp = np.zeros((B, T + N))
    gp[:, N // 2:N // 2 + T] = g / env[N // 2:N // 2 + T]
    frames = lambda x: np.stack([x[:, q * P:q * P + N] for q in range(nF + 1)], axis=1) * w
    c = np.full(N // 2 + 1, 2.0 / N)
    c[0] = c[-1] = 1.0 / N
    Gs = np.fft.rfft(frames(gp), axis=-1) * c
    mode = "reflect" if T > N // 2 else "constant"
    pad = lambda x: np.pad(x, ((0, 0), (N // 2, N // 2)), mode=mode)
    X, Z = np.fft.rfft(frames(pad(comb)), axis=-1), np.fft.rfft(frames(pad(noise)), axis=-1)
    c64 = {k: np.asarray(ctrls[k], np.float64) for k in KEYS}
    hold = lambda z: np.concatenate([z, z[:, -1:]], axis=1)
    Yh = X * hold(np.exp(c64["harmonic_magnitude"] + 1j * np.pi * c64["harmonic_phase"]))
    Yn = Z * hold(np.exp(c64["noise_magnitude"] + 1j * np.pi * c64["noise_phase"]) / 128)
    out = {}
    for (km, kp), Y in ((("harmonic_magnitude", "harmonic_phase"), Yh), (("noise_magnitude", "noise_phase"), Yn)):
        for k, full in ((km, np.real(np.conj(Gs) * Y)), (kp, np.pi * np.imag(Gs * np.conj(Y)))):
            r = full[:, :nF].copy()
            r[:, -1] += full[:, nF]
            out[k] = r
    return out


def rel_rms(got, want):
    got, want = np.asarray(got, np.float64), np.asarray(want, np.float64)
    return float(np.sqrt(np.mean((got - want) ** 2)) / np.sqrt(np.mean(want ** 2)))
