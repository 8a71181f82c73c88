"""Timing of the CombSubSuperFast backward on one GPU; prints one JSON line (and writes it to --out FILE if given).

    python tools/bench_superfast_backward.py [--out FILE] [--reps 20]

Shapes: the training shape of configs/combsub.yaml (B = 24 x 2 s, nF = 172) and B = 32 x 10 s.  Every timing is the
median over --reps passes of CUDA events around the work, each pass after a 256 MiB memset that evicts the L2, after
warm-up.  Timed per shape:
  * backward_kernel_ms: b2d_superfast_backward alone (ops.superfast_backward);
  * forward_kernel_ms: b2d_superfast_synth alone;
  * module_fwd_bwd_ms: CombSubSuperFast forward + backward with leaf controls (views of one dense [B, nF, 4100] leaf,
    as Unit2Control's split produces them): scan, forward kernel, backward kernel and torch's SplitBackward
    concatenation of the four gradients into the leaf's gradient;
  * split_backward_cat_ms: that concatenation alone (torch.cat of four [B, nF, 1025] tensors into [B, nF, 4100]);
  * eager_fwd_bwd_ms: the reference's stft -> filter -> istft forward + autograd backward in torch on the same GPU;
  * peak allocated memory above the inputs for the last two.
The algorithmic bytes of the backward (g 4 B per sample, the four controls and the frame parameters read, the four
gradients written) over backward_kernel_ms give its achieved bandwidth; HBM floor at the 7.7 TB/s of the data sheet.
"""
import argparse
import json
import math
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

from ddsp_svc_b200 import CombSubSuperFast, FixedControls, ops, synthetic as syn  # noqa: E402
from oracle import torch_port as tp  # noqa: E402

SR, P, WIN, C = 44100, 512, 2048, 1025
HBM_BYTES_PER_S = 7.7e12


def gpu_info():
    q = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    name, power, clk = (s.strip() for s in q.stdout.strip().split(",")) if q.returncode == 0 else ("?", "?", "?")
    return {"torch_name": torch.cuda.get_device_name(0), "nvidia_smi_name": name, "power_limit": power,
            "max_sm_clock": clk}


def timed(fn, flush, reps, warmup=3):
    for _ in range(warmup):
        fn()
    ts = []
    for _ in range(reps):
        flush.zero_()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        torch.cuda.synchronize()
        ts.append(a.elapsed_time(b))
    ts.sort()
    return ts[len(ts) // 2]


def peak_mib(fn):
    fn()
    torch.cuda.synchronize()
    base = torch.cuda.memory_allocated()
    torch.cuda.reset_peak_memory_stats()
    fn()
    torch.cuda.synchronize()
    return (torch.cuda.max_memory_allocated() - base) / 2 ** 20


def bench_shape(B, seconds, flush, reps):
    dev = "cuda:0"
    nF = syn.n_frames_for(seconds)
    T = nF * P
    f0 = syn.make_f0(B, nF, SR, P, seed=1).to(dev)
    dense, _ = syn.make_ctrl(B, nF, syn.superfast_split_map(WIN), seed=2)
    dense = dense.to(dev)
    views = syn.split_views(dense, syn.superfast_split_map(WIN))
    c = [views[k] for k in views]
    g = torch.randn(B, T, device=dev)
    ws, _ = ops.superfast_scan(f0, P, SR)
    out = {"B": B, "seconds": seconds, "n_frames": nF, "samples": B * T}

    out["backward_kernel_ms"] = timed(lambda: ops.superfast_backward(ws, *c, g, P, WIN, seed=3), flush, reps)
    out["forward_kernel_ms"] = timed(lambda: ops.superfast_synth(ws, *c, P, WIN, seed=3), flush, reps)
    grads = ops.superfast_backward(ws, *c, g, P, WIN, seed=3)
    conts = [t.contiguous() for t in grads]
    out["split_backward_cat_ms"] = timed(lambda: torch.cat(conts, dim=-1), flush, reps)

    leaf = dense.clone().requires_grad_()
    model = CombSubSuperFast(SR, P, WIN, unit2ctrl=FixedControls(None, None)).to(dev)

    def module_step():
        leaf.grad = None
        model.unit2ctrl.ctrls = syn.split_views(leaf, syn.superfast_split_map(WIN))
        signal, _, _ = model(None, f0, None)
        signal.backward(g)

    out["module_fwd_bwd_ms"] = timed(module_step, flush, reps)
    out["module_fwd_bwd_peak_mib"] = peak_mib(module_step)

    comb = tp.superfast_source(f0.cpu(), SR, P)[0].to(dev)          # the source is not part of the timed eager step
    noise = torch.randn(B, T, device=dev)
    window = torch.hann_window(WIN, device=dev)

    def eager_step():
        leaf.grad = None
        ct = syn.split_views(leaf, syn.superfast_split_map(WIN))
        hold_last = lambda z: torch.cat((z, z[:, -1:, :]), dim=1)
        hs = hold_last(torch.exp(ct["harmonic_magnitude"] + 1.j * math.pi * ct["harmonic_phase"]))
        hn = hold_last(torch.exp(ct["noise_magnitude"] + 1.j * math.pi * ct["noise_phase"]) / 128)
        stft = lambda z: torch.stft(z, WIN, P, WIN, window=window, center=True, return_complex=True, pad_mode="reflect")
        spec = stft(comb) * hs.permute(0, 2, 1) + stft(noise) * hn.permute(0, 2, 1)
        torch.istft(spec, WIN, P, WIN, window=window, center=True).backward(g)

    out["eager_fwd_bwd_ms"] = timed(eager_step, flush, max(3, reps // 4), warmup=2)
    out["eager_fwd_bwd_peak_mib"] = peak_mib(eager_step)

    # algorithmic bytes of the backward: g, four controls + frame parameters read, four gradients written
    nbytes = B * T * 4 + 2 * B * nF * 4 * C * 4 + B * nF * 16
    out["backward_bytes"] = nbytes
    out["backward_bytes_per_sample"] = nbytes / (B * T)
    out["backward_achieved_TBps"] = nbytes / (out["backward_kernel_ms"] * 1e-3) / 1e12
    out["backward_hbm_floor_ms"] = nbytes / HBM_BYTES_PER_S * 1e3
    out["eager_over_module"] = out["eager_fwd_bwd_ms"] / out["module_fwd_bwd_ms"]
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None, help="also write the JSON to this file")
    ap.add_argument("--reps", type=int, default=20)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device")
    torch.manual_seed(0)
    flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device="cuda:0")     # > 126 MB L2
    res = {"gpu": gpu_info(), "timing": "median of %d passes, CUDA events, L2 flushed before each, after warm-up"
           % args.reps, "shapes": [bench_shape(24, 2.0, flush, args.reps), bench_shape(32, 10.0, flush, args.reps)]}
    res["gpu_after"] = gpu_info()
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(res, f, indent=1)
    print(json.dumps(res))


if __name__ == "__main__":
    main()
