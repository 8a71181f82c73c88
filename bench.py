#!/usr/bin/env python
"""Benchmark of the DDSP synthesis hot path (BASELINE.json metric: audio Msamples/s at 44.1 kHz,
128 harmonics; % of the HBM roofline).

    python bench.py --gpus N --steps K --warmup W [--impl reference] [--workload sins|...] [--dump-outputs DIR]

One process per GPU (torchrun sets RANK/LOCAL_RANK/WORLD_SIZE).  A "step" is one pass of the
Sins synthesis path (frame phase scan -> sinusoid bank -> impulse responses -> two time-varying
FIRs + mix, in-kernel Philox noise) over one batch of B=32 utterances x 10 s per GPU
(BASELINE configs[1]; configs[3] at N=8 = 256 utterances); at N>1 the step also gathers every
rank's `signal` to rank 0 over NCCL (the path's only collective).  Prints ONE JSON line on rank 0.

--dump-outputs DIR (one GPU) writes what the last timed step returned as DIR/<name>.npy in float32, so that two builds
can be compared output for output: inputs are seeded and the in-kernel noise seeds come from torch's CPU generator,
seeded before the first step, so the same arguments give the same inputs on every run.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

SR, P = 44100, 512
DUMP_BYTES = 64 * 10 ** 6          # --dump-outputs: at most this many bytes of .npy files in all
OTHER_WORKLOADS = ("sins_cfg1", "combsub", "superfast", "combsubfast", "sinegen", "srcmod", "mel", "maskmul")

# N -> (gather mode, chunks, compute streams) chosen by `--gather auto` (measured on B200, see DESIGN.md section 5)
# round 2, ms/step at N=8 with 0.84 ms of kernels (profiles/r2_scale_m8_*.json): peer stores 1.077 | per-chunk peer stores
# 4 chunks x 2 streams 1.069 | copy-engine push 2.42-2.49 | NCCL gather 1.425 | no gather 0.848.  The 7 x 56.4 MB
# arrive while the FIR kernel (0.375 ms) runs: 395 MB / (0.375 + 0.23 ms exposed) = 653 GB/s into rank 0.
AUTO_GATHER = {2: ("peer", 1, 1), 4: ("peer", 1, 1), 8: ("peer", 1, 1)}

WORKLOADS = {
    # name: (kind, batch per GPU, seconds, params, algorithmic bytes per output sample (SURVEY 8d))
    "sins": dict(kind="sins", B=32, sec=10, H=128, Ma=256, Mn=256,
                 label="Sins forward DSP, B=32 x 10 s x 128 harmonics, 44.1 kHz, n_mag 256/256 (BASELINE configs[1])"),
    "sins_cfg1": dict(kind="sins", B=1, sec=2, H=64, Ma=256, Mn=256,
                      label="Sins forward DSP, B=1 x 2 s x 64 harmonics (BASELINE configs[0])"),
    "combsub": dict(kind="combsub", B=32, sec=10, Ma=256, Mh=512, Mn=256,
                    label="CombSub (old) forward DSP, B=32 x 10 s, n_mag 256/512/256 (BASELINE configs[2], class CombSub)"),
    "superfast": dict(kind="superfast", B=32, sec=10, win=2048,
                      label="CombSubSuperFast forward DSP (configs/combsub.yaml), B=32 x 10 s, win 2048 (BASELINE configs[2])"),
    "combsubfast": dict(kind="combsubfast", B=32, sec=10,
                        label="CombSubFast forward DSP (the variant diffusion / reflow embed), B=32 x 10 s, 1024-point sqrt-Hann frames"),
    "sinegen": dict(kind="sinegen", B=64, sec=10, dim=9,
                    label="nsf_hifigan SineGen, B=64 x 10 s, 9 harmonics (BASELINE configs[4])"),
    "srcmod": dict(kind="srcmod", B=64, sec=10, dim=9,
                   label="nsf_hifigan SourceModuleHnNSF = SineGen + tanh(Linear(9->1)) fused, B=64 x 10 s (SURVEY 8f)"),
    "mel": dict(kind="mel", B=32, sec=10, n_mels=128,
                label="nsf_hifigan STFT.get_mel log-mel front end, B=32 x 10 s, n_fft 2048 / hop 512 / 128 mels (SURVEY 8f)"),
    "maskmul": dict(kind="maskmul", B=32, sec=10,
                    label="caller epilogue `seg_output *= upsample(mask, block)` (main.py:215,260), B=32 x 10 s (SURVEY 8f)"),
}


def algorithmic_bytes(w, nF):
    """bytes the path must move per launch of the whole path: controls + f0 read once, every
    returned tensor written once (SURVEY.md section 8d)."""
    B, T = w["B"], nF * P
    if w["kind"] == "sins":
        c = w["H"] + w["Ma"] + w["Mn"]
        return 4 * B * nF * (1 + c) + 4 * B * T * 3
    if w["kind"] == "combsub":
        c = w["Ma"] + w["Mh"] + w["Mn"]
        return 4 * B * nF * (1 + c) + 4 * B * T * 3
    if w["kind"] == "superfast":
        return 4 * B * nF * (1 + 4 * (w["win"] // 2 + 1)) + 4 * B * T
    if w["kind"] == "combsubfast":
        return 4 * B * nF * (1 + 3 * (P + 1)) + 4 * B * T
    if w["kind"] == "sinegen":
        return 4 * B * nF + 4 * B * T * w["dim"]
    if w["kind"] == "srcmod":
        return 4 * B * nF + 4 * B * T
    if w["kind"] == "mel":
        return 4 * B * T + 4 * B * nF * w["n_mels"]
    if w["kind"] == "maskmul":
        return 4 * B * nF + 2 * 4 * B * T
    raise ValueError(w["kind"])


def split_map_of(w):
    from ddsp_svc_b200 import synthetic as syn
    k = w["kind"]
    if k == "sins":
        return syn.sins_split_map(w["H"], w["Ma"], w["Mn"])
    if k == "combsub":
        return syn.combsub_split_map(w["Ma"], w["Mh"], w["Mn"])
    if k == "superfast":
        return syn.superfast_split_map(w["win"])
    if k == "combsubfast":
        return syn.combsubfast_split_map(P)
    return None


def oracle_forward(w, f0, ctrls):
    """The reference's CPU algorithm (oracle port) for one workload kind."""
    from oracle import torch_port as tp
    k = w["kind"]
    if k == "sins":
        return tp.sins_forward(f0, ctrls, SR, P)
    if k == "combsub":
        return tp.combsub_forward(f0, ctrls, SR, P)
    if k == "superfast":
        return tp.superfast_forward(f0, ctrls, SR, P, w["win"])
    if k == "combsubfast":
        return tp.combsubfast_forward(f0, ctrls, SR, P)
    if k == "mel":
        from oracle import mel as om
        return {"out": om.get_mel(f0)}             # `f0` carries the audio for this kind
    if k == "maskmul":
        from oracle import frontend as fe
        import torch
        return {"out": torch.cat([fe.mask_apply(f0[i:i + 1], ctrls[0].numpy(), P) for i in range(f0.shape[0])])}
    if k == "srcmod":
        import torch
        g = torch.Generator().manual_seed(5)
        return tp.source_module_forward(f0[..., 0], P, SR, torch.randn(1, w["dim"], generator=g) / 3, torch.zeros(1), w["dim"] - 1)
    return tp.sinegen_forward(f0[..., 0], P, SR, w["dim"] - 1)


def oracle_inputs(w, batch, nF):
    """seeded CPU inputs of the oracle for `batch` utterances: (f0 or waveform, controls or mask)"""
    import torch
    from ddsp_svc_b200 import synthetic as syn
    if w["kind"] in ("mel", "maskmul"):
        g = torch.Generator().manual_seed(99)
        audio = 0.1 * torch.randn(batch, nF * P, generator=g)
        return audio, ([(torch.rand(nF, generator=g) > 0.2).float()] if w["kind"] == "maskmul" else None)
    sm = split_map_of(w)
    return syn.make_f0(batch, nF, SR, P), (syn.make_ctrl(batch, nF, sm)[1] if sm else None)


def _first(ctrls, n):
    if ctrls is None:
        return None
    return {k: v[:n] for k, v in ctrls.items()} if isinstance(ctrls, dict) else ctrls


# ------------------------------------------------------------------------------------------
class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.idx, self.rows, self.proc = gpu_index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.idx), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "20"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, smax, reasons = [], [], set()
        for r in self.rows:
            try:
                sm.append(float(r[1])); smax.append(float(r[2]))
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[5:9]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
            except Exception:
                continue
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        return {"sm_mhz": statistics.median(sm), "sm_max_mhz": max(smax), "reasons": sorted(reasons), "samples": len(sm)}


def ncu_traffic(workload, kernel_label):
    """dram__bytes_read.sum + dram__bytes_write.sum per launch of the dominant kernel, from the committed
    ncu --set full capture (profiles/r2_traffic.json); None when no capture is recorded for it."""
    try:
        with open(os.path.join(ROOT, "profiles", "r2_traffic.json")) as f:
            ent = json.load(f).get(workload, {})
        return ent.get("dram_bytes_per_launch") if ent.get("bench_kernel") == kernel_label else None
    except Exception:
        return None


def measured_peak_hbm():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "MEASURED_PEAKS.json hbm_gbs (measured copy bandwidth)"
    except Exception:
        return 6650.0, "fallback 6.65 TB/s (B200_PROFILING.md; MEASURED_PEAKS.json absent)"


# ------------------------------------------------------------------------------------------
def cpu_reference_run(w, batch, reps, threads=None):
    """Time the reference's CPU algorithm (oracle port on the same ATen CPU operators) on
    `batch` utterances of the workload.  Returns (Msamples/s, seconds per rep, cores)."""
    import torch
    from ddsp_svc_b200 import synthetic as syn
    from oracle import torch_port as tp
    cores = threads or best_thread_count(w)
    torch.set_num_threads(cores)
    nF = syn.n_frames_for(w["sec"], SR, P)
    f0, ctrls = oracle_inputs(w, batch, nF)
    best = None
    with torch.no_grad():
        oracle_forward(w, f0[:1], _first(ctrls, 1))  # warm-up (small)
        for _ in range(reps):
            t0 = time.perf_counter()
            oracle_forward(w, f0, ctrls)
            dt = time.perf_counter() - t0
            best = dt if best is None else min(best, dt)
    return batch * nF * P / best / 1e6, best, cores


_best_threads = {}


def best_thread_count(w):
    """The reference runs PyTorch with its default intra-op pool (all cores).  On many-core hosts
    that is slower than a smaller pool for these medium-sized ops, so give the CPU arm its best
    setting: try a few pool sizes on one utterance and keep the fastest."""
    import torch
    from ddsp_svc_b200 import synthetic as syn
    from oracle import torch_port as tp
    key = w["label"]
    if key in _best_threads:
        return _best_threads[key]
    ncpu = os.cpu_count() or 1
    nF = syn.n_frames_for(min(w["sec"], 2), SR, P)
    f0, ctrls = oracle_inputs(w, 2, nF)
    best, best_t = ncpu, None
    for n in sorted({c for c in (4, 8, 16, 32, 64, ncpu) if c <= ncpu}):
        torch.set_num_threads(n)
        dt = None
        with torch.no_grad():
            oracle_forward(w, f0, ctrls)
            for _ in range(2):                     # best of two: one noisy pass must not flip the choice between runs
                t0 = time.perf_counter()
                oracle_forward(w, f0, ctrls)
                d = time.perf_counter() - t0
                dt = d if dt is None else min(dt, d)
        if best_t is None or dt < 0.95 * best_t:    # a larger pool must win by 5 % (ascending order: the smaller one stays on ties)
            best, best_t = n, dt
    _best_threads[key] = best
    return best


def metric_name(w):
    return "audio Msamples/s (44.1 kHz, %s)" % ("%d harmonics" % w["H"] if "H" in w else w["kind"])


def run_reference_arm(args, w):
    """--impl reference: the reference's own CPU implementation of the path on this box's host
    cores.  /root/reference (Python) cannot travel to the GPU box, so this times the oracle port,
    which is bit-identical to it on CPU (tests/test_oracle_vs_reference.py)."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from ddsp_svc_b200 import synthetic as syn
    nF = syn.n_frames_for(w["sec"], SR, P)
    sample_b = min(w["B"], 4)
    vals = []
    for _ in range(args.warmup):
        cpu_reference_run(w, sample_b, 1)
    t_total = 0.0
    for _ in range(args.steps):
        v, dt, cores = cpu_reference_run(w, sample_b, 1)
        vals.append(v); t_total += dt
    value = sample_b * nF * P * args.steps / t_total / 1e6
    sample = "%d of %d utterances x %d s per step (bounded sample of the same workload)" % (sample_b, w["B"], w["sec"])
    line = {"impl": "reference", "metric": metric_name(w), "value": value,
            "unit": "Msamples/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": 1e3 * t_total / args.steps, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": w["label"], "sample": sample, "l2": "n/a (CPU)"},
            "cpu_baseline": {"value": value, "unit": "Msamples/s", "cores": cores, "kind": "port", "sample": sample},
            "e2e": {"value": value, "unit": "Msamples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line))


# ------------------------------------------------------------------------------------------
class Runner:
    """Per-workload device state: how to run one step and how to time each kernel alone."""

    def __init__(self, w, dev, rank, torch):
        from ddsp_svc_b200 import (CombSub, CombSubFast, CombSubSuperFast, FixedControls, SineGen, SourceModuleHnNSF,
                                   Sins, ops, synthetic as syn)
        self.w, self.dev, self.rank, self.torch, self.ops, self.syn = w, dev, rank, torch, ops, syn
        B = self.B = w["B"]
        nF = self.nF = syn.n_frames_for(w["sec"], SR, P)
        self.T = nF * P
        self.sm = split_map_of(w)
        if w["kind"] in ("mel", "maskmul"):            # waveform-in workloads on either side of the synthesizer
            from ddsp_svc_b200 import frontend, mel
            g = torch.Generator().manual_seed(99 + rank)
            self.audio_h = (0.1 * torch.randn(B, self.T, generator=g)).pin_memory()
            self.audio_d = self.audio_h.to(dev)
            self.h2d = self.audio_h.numel() * 4
            self.sg, self.width = False, 1
            if w["kind"] == "mel":
                self.stft = mel.STFT(SR, w["n_mels"], 2048, 2048, P, 40, 16000)
                self.out_h = torch.empty(B, w["n_mels"], nF, dtype=torch.float32).pin_memory()
            else:
                self.frontend = frontend
                self.mask_d = (torch.rand(B, nF, generator=g) > 0.2).float().to(dev)
                self.out_h = torch.empty(B, self.T, dtype=torch.float32).pin_memory()
            return
        self.f0_h = syn.make_f0(B, nF, SR, P, seed=1234 + rank).pin_memory()
        self.f0_d = self.f0_h.to(dev)
        self.h2d = self.f0_h.numel() * 4
        k = w["kind"]
        self.sg = k in ("sinegen", "srcmod")           # f0-only excitation generators
        self.width = w["dim"] if k == "sinegen" else 1
        if self.sg:
            self.rand_ini = torch.rand(w["dim"]); self.rand_ini[0] = 0
            if k == "sinegen":
                self.model = SineGen(SR, harmonic_num=w["dim"] - 1)
            else:
                self.model = SourceModuleHnNSF(SR, harmonic_num=w["dim"] - 1).to(dev).eval()
            self.out_h = torch.empty(B, self.T, self.width, dtype=torch.float32).pin_memory()
            return
        self.dense_h = syn.make_ctrl(B, nF, self.sm, seed=7 + rank)[0].pin_memory()
        self.dense_d = self.dense_h.to(dev)
        self.ctrl_d = syn.split_views(self.dense_d, self.sm)
        self.h2d += self.dense_h.numel() * 4
        self.fixed = FixedControls(self.ctrl_d, torch.zeros(B, nF, 256, device=dev))
        if k == "sins":
            self.model = Sins(SR, P, w["H"], w["Ma"], w["Mn"], unit2ctrl=self.fixed).to(dev)
        elif k == "combsub":
            self.model = CombSub(SR, P, w["Ma"], w["Mh"], w["Mn"], unit2ctrl=self.fixed).to(dev)
        elif k == "combsubfast":
            self.model = CombSubFast(SR, P, unit2ctrl=self.fixed).to(dev)
        else:
            self.model = CombSubSuperFast(SR, P, w["win"], unit2ctrl=self.fixed).to(dev)
        self.out_h = torch.empty(B, self.T, dtype=torch.float32).pin_memory()

    # one pass of the hot path with inputs resident in HBM; returns the waveform to gather
    def _wave_op(self, audio, lo=0):
        if self.w["kind"] == "mel":
            return self.stft.get_mel(audio)
        return self.frontend.mask_apply_(audio, self.mask_d[lo:lo + audio.shape[0]], P)

    keep_outputs = False               # step() keeps what the caller receives in self.outputs (--dump-outputs)

    def step(self, f0=None):
        if self.w["kind"] in ("mel", "maskmul"):
            out = self._wave_op(self.audio_d)
        else:
            f0 = self.f0_d if f0 is None else f0
            if self.sg:
                out = self.model(f0[..., 0], P, rand_ini=self.rand_ini, utterance_offset=self.rank * self.B)
            else:
                signal, _, (harmonic, noise) = self.model(None, f0, None, utterance_offset=self.rank * self.B)
                if self.keep_outputs:  # CombSubFast / CombSubSuperFast return the signal three times
                    self.outputs = ({"signal": signal, "harmonic": harmonic, "noise": noise}
                                    if self.w["kind"] in ("sins", "combsub") else {"signal": signal})
                return signal
        if self.keep_outputs:
            self.outputs = {"out": out}
        return out

    # rows [lo, hi) of the local batch (for the chunked synth+gather pipeline) -> [hi-lo, row_len]
    @property
    def row_len(self):
        return self.T * self.width

    def step_rows(self, lo, hi, signal_out=None):
        f0 = self.f0_d[lo:hi]
        if self.sg:
            out = self.model(f0[..., 0], P, rand_ini=self.rand_ini, utterance_offset=self.rank * self.B + lo)
            return out.reshape(hi - lo, -1)
        full = self.fixed.ctrls
        self.fixed.ctrls = self.syn.split_views(self.dense_d[lo:hi], self.sm)
        kw = {"signal_out": signal_out} if signal_out is not None else {}
        try:
            return self.model(None, f0, None, utterance_offset=self.rank * self.B + lo, **kw)[0]
        finally:
            self.fixed.ctrls = full

    # the same through HOST buffers: pinned inputs -> H2D -> public module API -> D2H of the result
    e2e_streams = 1

    def step_e2e(self, chunks=4):
        """public API with host buffers: HostPipeline (chunked upload | kernels | download) around the module's
        forward; returns the event to synchronise on."""
        from ddsp_svc_b200 import HostPipeline
        if getattr(self, "_pipe", None) is None or self._pipe.chunks != chunks:
            self._pipe = HostPipeline(self.dev, chunks=chunks, compute_streams=self.e2e_streams)
        if self.w["kind"] in ("mel", "maskmul"):
            return self._pipe.run({"audio": self.audio_h}, lambda d, lo, hi: self._wave_op(d["audio"], lo), self.out_h)
        host = {"f0": self.f0_h}
        if not self.sg:
            host["dense"] = self.dense_h

        def fwd(d, lo, hi):
            if self.sg:
                return self.model(d["f0"][..., 0], P, rand_ini=self.rand_ini, utterance_offset=self.rank * self.B + lo)
            self.fixed.ctrls = self.syn.split_views(d["dense"], self.sm)
            try:
                return self.model(None, d["f0"], None, utterance_offset=self.rank * self.B + lo)[0]
            finally:
                self.fixed.ctrls = self.ctrl_d

        return self._pipe.run(host, fwd, self.out_h)

    def kernels(self):
        """name -> callable launching exactly that kernel (inputs prepared beforehand)."""
        k = self.w["kind"]
        if k in ("mel", "maskmul"):
            return {("mel_kernel" if k == "mel" else "mask_apply_kernel"): lambda: self._wave_op(self.audio_d)}
        ops, w, c, f0, B, nF, T = self.ops, self.w, getattr(self, "ctrl_d", None), self.f0_d, self.B, self.nF, self.T
        torch, dev = self.torch, self.dev
        L = ops._lib.lib()
        st = torch.cuda.current_stream().cuda_stream
        if k == "sinegen":
            return {"sinegen(scan+stream)": lambda: ops.sinegen(f0[..., 0], P, SR, w["dim"], self.rand_ini, seed=1)}
        if k == "srcmod":
            lw, lb = self.model.l_linear.weight, float(self.model.l_linear.bias)
            return {"source_module(scan+stream)": lambda: ops.source_module(f0[..., 0], P, SR, w["dim"], self.rand_ini,
                                                                            lw, lb, seed=1)}
        if k == "combsubfast":
            fp, _ = ops.phase_scan(f0, P, SR)
            comb = ops.comb_source(f0, fp, P, SR)
            return {"phase_scan": lambda: ops.phase_scan(f0, P, SR),
                    "comb_source": lambda: ops.comb_source(f0, fp, P, SR),
                    "combsubfast_kernel": lambda: ops.combsubfast_filter(comb, c["harmonic_magnitude"], c["harmonic_phase"],
                                                                         c["noise_magnitude"], P, seed=1)}
        if k == "superfast":
            ws, _ = ops.superfast_scan(f0, P, SR)
            return {"superfast_scan": lambda: ops.superfast_scan(f0, P, SR),
                    "superfast_kernel": lambda: ops.superfast_synth(ws, c["harmonic_magnitude"], c["harmonic_phase"],
                                                                    c["noise_magnitude"], c["noise_phase"], P, w["win"], seed=1)}
        fp, _ = ops.phase_scan(f0, P, SR)
        buf = [torch.empty(B, T, device=dev) for _ in range(3)]
        if k == "sins":
            sinus = ops.sins_bank(f0, fp, c["amplitudes"], P, SR)
            ir_a = ops.ir_build(c["group_delay"], ops.IR_ALLPASS, SR)
            ir_n = ops.ir_build(c["noise_magnitude"], ops.IR_MAG_HANN, SR)
            La, Ln = ir_a.shape[2], ir_n.shape[2]
            return {"phase_scan": lambda: ops.phase_scan(f0, P, SR),
                    "sins_bank": lambda: ops.sins_bank(f0, fp, c["amplitudes"], P, SR),
                    "ir_build_allpass": lambda: ops.ir_build(c["group_delay"], ops.IR_ALLPASS, SR),
                    "ir_build_noise": lambda: ops.ir_build(c["noise_magnitude"], ops.IR_MAG_HANN, SR),
                    "ltv_fir_x2_mix": lambda: L.b2d_ltv_fir(sinus.data_ptr(), ir_a.data_ptr(), La, buf[0].data_ptr(), 0,
                                                            ir_n.data_ptr(), Ln, buf[1].data_ptr(), buf[2].data_ptr(),
                                                            1, 0, B, nF, P, st)}
        comb = ops.comb_source(f0, fp, P, SR)
        ir_a = ops.ir_build(c["group_delay"], ops.IR_ALLPASS, SR)
        ir_h = ops.ir_build(c["harmonic_magnitude"], ops.IR_MAG_DYNAMIC, SR, f0_frames=f0)
        ir_n = ops.ir_build(c["noise_magnitude"], ops.IR_MAG_HANN, SR)
        return {"phase_scan": lambda: ops.phase_scan(f0, P, SR),
                "comb_source": lambda: ops.comb_source(f0, fp, P, SR),
                "ir_build_allpass": lambda: ops.ir_build(c["group_delay"], ops.IR_ALLPASS, SR),
                "ir_build_dynamic": lambda: ops.ir_build(c["harmonic_magnitude"], ops.IR_MAG_DYNAMIC, SR, f0_frames=f0),
                "ir_build_noise": lambda: ops.ir_build(c["noise_magnitude"], ops.IR_MAG_HANN, SR),
                "ltv_fir_allpass+noise": lambda: L.b2d_ltv_fir(comb.data_ptr(), ir_a.data_ptr(), ir_a.shape[2],
                                                               buf[0].data_ptr(), 0, ir_n.data_ptr(), ir_n.shape[2],
                                                               buf[1].data_ptr(), 0, 1, 0, B, nF, P, st),
                "ltv_fir_harmonic_1022": lambda: ops.ltv_fir(comb, ir_h, P)}


def dump_outputs(outputs, out_dir, torch):
    """Write each output tensor as out_dir/<name>.npy in float32.  When all of them together exceed DUMP_BYTES, each is
    replaced by the same fixed, seeded sample of its flattened elements (sorted positions, an equal share of the
    budget per tensor)."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    total = sum(4 * t.numel() for t in outputs.values())
    cap = (DUMP_BYTES - 4096) // (4 * len(outputs))
    for name, t in outputs.items():
        t = t.detach()
        if total > DUMP_BYTES and t.numel() > cap:
            idx = np.sort(np.random.default_rng(0).choice(t.numel(), size=cap, replace=False))
            t = t.reshape(-1)[torch.from_numpy(idx).to(t.device)]
        np.save(os.path.join(out_dir, name + ".npy"), t.float().cpu().numpy())


def time_e2e(run, chunks, flush, reps, torch):
    ee = []
    for i in range(reps + 1):
        flush.zero_()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        run.step_e2e(chunks).synchronize()
        b.record()                     # recorded on the main stream, which waits for the download stream
        b.synchronize()
        if i > 0:
            ee.append(a.elapsed_time(b))
    return statistics.median(ee)        # robust to a pass in which the host thread was descheduled while enqueueing


def time_kernels(run, flush, reps, torch):
    kt = {}
    for name, fn in run.kernels().items():
        ts = []
        fn()                               # untimed: first use of this call path
        for _ in range(reps):
            flush.zero_()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record(); fn(); b.record(); b.synchronize()
            ts.append(a.elapsed_time(b))
        kt[name] = statistics.median(ts)   # average launch duration, robust to a stray slow launch
    return kt


def time_other_workload(name, dev, flush, torch, steps=10, warmup=3):
    """One more workload of the path, device-timed like the headline (L2 flushed, CUDA events per step): the numbers the
    single BENCH line carries under `other_workloads` so every default kernel has a driver-visible timing."""
    w = WORKLOADS[name]
    run = Runner(w, dev, 0, torch)
    for _ in range(warmup):
        run.step()
    torch.cuda.synchronize()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
    for a, b in ev:
        flush.zero_()
        a.record(); run.step(); b.record()
    torch.cuda.synchronize()
    # median of the per-step times: these auxiliary lines share one process with the headline run, and a step that has to
    # grow the caching allocator (SineGen's 1 GB output) would otherwise dominate a 10-step mean
    ms = statistics.median(a.elapsed_time(b) for a, b in ev)
    e2e_ms = time_e2e(run, (6, 10, 10, 6) if w["B"] >= 16 else 1, flush, 5, torch)
    kt = time_kernels(run, flush, 5, torch)
    peak, _ = measured_peak_hbm()
    dom = max(kt, key=kt.get)
    alg = algorithmic_bytes(w, run.nF)
    n = w["B"] * run.T
    out = {"workload": w["label"], "value": n / (ms * 1e-3) / 1e6, "unit": "Msamples/s", "ms_per_step": ms,
           "e2e_value": n / (e2e_ms * 1e-3) / 1e6, "e2e_ms_per_step": e2e_ms,
           "roofline": {"kernel": dom, "frac": alg / (kt[dom] * 1e-3) / 1e9 / peak,
                        "whole_path_frac": alg / (ms * 1e-3) / 1e9 / peak, "algorithmic_bytes_per_launch": alg,
                        "traffic": ncu_traffic(name, dom), "kernel_ms": kt}}
    del run
    torch.cuda.empty_cache()
    return out


def eager_gpu_baseline(w, run, flush, torch, reps=3):
    """The secondary bar of SURVEY 8(d): the reference's own algorithm under eager PyTorch on THIS GPU (oracle port =
    the same ATen operators as ddsp/vocoder.py:556-611, here on device='cuda'), full batch, CUDA-event timed.  A
    baseline only -- nothing of it is on the product path."""
    if run.sg or run.sm is None:
        f0, ctrls = run.f0_d, None
    else:
        f0, ctrls = run.f0_d, run.ctrl_d
    kind, what = "port", "oracle port of the reference (same ATen operators)"
    fwd = lambda f, c: oracle_forward(w, f, c)
    if w["kind"] == "sins":
        try:                                   # the unmodified reference class when its sources travelled (baseline/_ref)
            import contextlib, io
            from oracle import ref_loader
            if ref_loader.available():
                with contextlib.redirect_stdout(io.StringIO()):
                    V = ref_loader.load()[0]
                    ref = V.Sins(SR, P, w["H"], w["Ma"], w["Mn"], n_unit=8, n_spk=1).to(run.dev).eval()

                class Fixed(torch.nn.Module):
                    def forward(self, *a, **k):
                        return self.c, None
                ref.unit2ctrl = Fixed()

                def fwd(f, c):                 # noqa: F811 -- Sins.forward of the reference, DSP only (controls preset)
                    ref.unit2ctrl.c = c
                    return ref(None, f, None)
                kind, what = "reference", "the reference's own ddsp.vocoder.Sins.forward (unmodified sources staged under baseline/_ref, Unit2Control replaced by preset controls)"
        except Exception as e:                 # fall back to the port, say why
            what += " [reference classes unavailable: %s]" % (str(e).splitlines()[0][:80] if str(e) else type(e).__name__)
    fwd(f0[:2], {k: v[:2] for k, v in ctrls.items()} if ctrls else None)     # cuFFT plans, allocator
    ts = []
    for _ in range(reps):
        flush.zero_()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record(); fwd(f0, ctrls); b.record(); b.synchronize()
        ts.append(a.elapsed_time(b))
    torch.cuda.empty_cache()
    ms = min(ts)
    return {"value": w["B"] * run.T / (ms * 1e-3) / 1e6, "unit": "Msamples/s", "ms_per_step": ms, "kind": kind,
            "what": what + " run eagerly on this GPU, full batch, inputs resident in HBM, best of %d" % reps}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="sins", choices=sorted(WORKLOADS))
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-gather", action="store_true", help="N>1: skip the NCCL gather of the waveform")
    ap.add_argument("--gather", default="auto", choices=["auto", "peer", "peer-chunks", "peer-copy", "nccl"],
                    help="N>1: 'peer' = the FIR kernel stores the waveform into rank 0's peer-mapped buffer; "
                         "'peer-chunks' = the same per chunk of utterances; 'peer-copy' = chunked synthesis + copy-engine "
                         "DMA into that buffer; 'nccl' = gather; 'auto' = the measured best per N (AUTO_GATHER)")
    ap.add_argument("--gather-chunks", type=int, default=1,
                    help="N>1: split the local batch into this many chunks and overlap their gather with synthesis")
    ap.add_argument("--gather-streams", type=int, default=1,
                    help="N>1, chunked peer modes: compute streams the chunks alternate between")
    ap.add_argument("--no-others", action="store_true",
                    help="skip the eager-PyTorch-on-GPU baseline and the `other_workloads` timings of the default run")
    ap.add_argument("--e2e-only", action="store_true",
                    help="host-buffer pipeline timing only (sweeps of --e2e-chunks / --e2e-streams): prints {e2e_ms}")
    ap.add_argument("--quick", action="store_true",
                    help="device-timed step only: skip the host-buffer e2e, per-kernel and CPU legs (sweeps)")
    ap.add_argument("--e2e-chunks", default="6,10,10,6",
                    help="utterance chunks of the host-buffer pipeline: a count (1 = serial) or comma-separated "
                         "relative sizes (default tapered: short fill and drain; round-2 sweep on the Sins workload, "
                         "gpurun_out/e2e_sweep.txt: 6,10,10,6 -> 2.02 ms, 4,8,12,6,2 -> 2.10, 16,16 -> 2.35)")
    ap.add_argument("--e2e-streams", type=int, default=1,
                    help="compute streams of the host-buffer pipeline (HostPipeline(compute_streams=...); >1 not yet measured)")
    ap.add_argument("--fir-impl", default="auto", choices=["auto", "cuda", "tc", "cuda8", "fft"],
                    help="A/B switch for the time-varying FIR kernel (ops.set_fir_impl)")
    ap.add_argument("--fft-arith", default="packed", choices=["scalar", "packed"],
                    help="A/B switch: packed f32x2 complex additions in the FFT kernels (ops.set_fft_arith)")
    ap.add_argument("--sins-impl", default="auto", choices=["auto", "split", "fused", "spectrum"],
                    help="A/B switch (ops.set_sins_impl): bank fused into the FFT-domain FIR kernel, or separate kernels")
    ap.add_argument("--overlap", type=int, default=None,
                    help="A/B switch (ops.set_overlap): 0 in order, 1 impulse responses beside the bank, k >= 2 "
                         "additionally k staggered sub-batches on two streams")
    ap.add_argument("--sinegen-impl", default="auto", choices=["auto", "v1", "v2", "v2p", "v2r7"],
                    help="A/B switch for the SineGen / source-module kernel (ops.set_sinegen_impl)")
    ap.add_argument("--breakdown", action="store_true", help="also print per-kernel times to stderr")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last one returned as DIR/<name>.npy (float32; a fixed, "
                         "seeded sample of each output when all of them exceed 64 MB); one GPU only")
    args = ap.parse_args()
    w = WORKLOADS[args.workload]
    if args.dump_outputs and (args.impl == "reference" or args.e2e_only or args.gpus > 1
                              or int(os.environ.get("WORLD_SIZE", "1")) > 1):
        ap.error("--dump-outputs needs the device-timed steps of a single-GPU run")
    if args.impl == "reference":
        return run_reference_arm(args, w)
    args.warmup = max(args.warmup, 3)

    import torch
    import torch.distributed as dist
    from ddsp_svc_b200 import ops, sharding

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (no CPU fallback for the product path)")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)

    torch.manual_seed(0)                       # in-kernel noise seeds and SineGen phases: the same on every run
    run = Runner(w, dev, rank, torch)
    run.keep_outputs = bool(args.dump_outputs)
    e2e_chunks = int(args.e2e_chunks) if args.e2e_chunks.isdigit() else tuple(int(x) for x in args.e2e_chunks.split(","))
    run.e2e_streams = args.e2e_streams
    if args.sinegen_impl != "auto":
        run.ops.set_sinegen_impl(args.sinegen_impl)
    if args.fir_impl != "auto":
        run.ops.set_fir_impl(args.fir_impl)
    if args.overlap is not None:
        run.ops.set_overlap(args.overlap)
    if args.sins_impl != "auto":
        run.ops.set_sins_impl(args.sins_impl)
    if args.fft_arith != "packed":
        run.ops.set_fft_arith(args.fft_arith)
    B, nF, T = run.B, run.nF, run.T
    do_gather = world > 1 and not args.no_gather
    flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device=dev)  # > 126 MB L2

    n_chunks, n_streams = args.gather_chunks, args.gather_streams
    peer = None
    mode = args.gather
    if mode == "auto":
        mode, n_chunks, n_streams = AUTO_GATHER.get(world, AUTO_GATHER[8])
    if do_gather and mode.startswith("peer") and w["kind"] == "sins":
        try:                                   # rank 0's buffer peer-mapped on every rank (NVLink)
            peer = sharding.PeerGather(B, T, dev, dst=0)
        except Exception as e:                 # symmetric memory unavailable: use the NCCL gather
            if rank == 0:
                print("peer gather unavailable (%s); using NCCL" % (str(e).splitlines()[0][:120],), file=sys.stderr)
            peer = None
    if peer is None and mode.startswith("peer"):
        mode = "nccl"
    gather_mode = {"peer": "peer-mapped stores over NVLink from the FIR kernel + device barrier",
                   "peer-chunks": "%d chunks on %d compute stream(s), each chunk's FIR kernel stores into rank 0's "
                                  "peer-mapped buffer" % (n_chunks, n_streams),
                   "peer-copy": "%d chunks on %d compute stream(s), copy-engine DMA of finished chunks into rank 0's "
                                "peer-mapped buffer" % (n_chunks, n_streams),
                   "nccl": "NCCL gather, %d chunk(s)" % n_chunks}[mode] if do_gather else "none"

    def step():
        if not do_gather:
            return run.step()
        if mode == "peer":
            run.model(None, run.f0_d, None, utterance_offset=rank * B, signal_out=peer.my_rows)
            return peer.finish()
        if mode in ("peer-copy", "peer-chunks"):
            return sharding.synthesize_and_push(run.step_rows, peer, B, dev, chunks=n_chunks, streams=n_streams,
                                                direct=mode == "peer-chunks")
        if n_chunks <= 1:
            sig = run.step()
            return sharding.gather_waveform(sig.reshape(B, -1), world * B, dst=0)
        # chunked: the NCCL transfer of finished utterances overlaps the synthesis of the rest
        return sharding.synthesize_and_gather(run.step_rows, B, world * B, run.row_len, dev, dst=0, chunks=n_chunks)

    def check_gather():
        """Untimed: one more step with the same host seed on every rank, then rank 0 re-synthesizes every rank's
        utterances locally (that rank's seeded inputs, utterance_offset = r*B, same chunking -> same seed draws) and
        compares them bit for bit with the rows that arrived."""
        torch.manual_seed(4242)
        got = step()
        sync_all()
        if rank != 0:
            return None
        bad = 0
        for r in range(world):
            other = Runner(w, dev, r, torch) if r else run
            torch.manual_seed(4242)
            if mode in ("peer-copy", "peer-chunks") or (mode == "nccl" and n_chunks > 1):
                want = torch.cat([other.step_rows(lo, hi) for lo, hi in sharding._chunk_bounds(B, n_chunks)])
            else:
                want = other.step()
            bad += int(not torch.equal(got[r * B:(r + 1) * B], want.reshape(B, -1)))
            del other, want
        return bad == 0

    def sync_all():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    if args.e2e_only:
        with torch.no_grad():
            for _ in range(args.warmup):
                step()
            ms = time_e2e(run, e2e_chunks, flush, max(5, min(args.steps, 20)), torch)
        print(json.dumps({"e2e_only": True, "e2e_ms": ms, "chunks": args.e2e_chunks, "streams": args.e2e_streams,
                          "value": B * T / (ms * 1e-3) / 1e6}))
        return
    with torch.no_grad():
        for _ in range(args.warmup):
            step()
        sync_all()
        clocks = ClockSampler(local)
        if rank == 0:
            clocks.start()
        ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
        n0 = ops.launches()
        sync_all()
        wall0 = time.perf_counter()
        for a, b in ev:
            flush.zero_()                      # evict L2 between steps (untimed)
            a.record()
            step()
            b.record()
        sync_all()
        wall = time.perf_counter() - wall0
        launches = ops.launches() - n0
        dev_ms = sum(a.elapsed_time(b) for a, b in ev)
        if args.dump_outputs:
            dump_outputs(run.outputs, args.dump_outputs, torch)
            run.keep_outputs, run.outputs = False, None
        gather_checked = check_gather() if do_gather else None

        # ---- end to end through the public module API with HOST buffers ----
        e2e_ms = float("nan")
        if not args.quick:
            e2e_ms = time_e2e(run, e2e_chunks, flush, max(10, min(args.steps, 20)), torch)
        clk = clocks.stop() if rank == 0 else None

        # ---- per-kernel durations (CUDA events on the launching stream), for the roofline ----
        kt = time_kernels(run, flush, max(5, min(args.steps, 20)), torch) if not args.quick else {}

    # ---- reduce over ranks: max device time ----
    if world > 1:
        t = torch.tensor([dev_ms, e2e_ms], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dev_ms, e2e_ms = t[0].item(), t[1].item()
    ms_per_step = dev_ms / args.steps
    samples_step = world * B * T
    value = samples_step / (ms_per_step * 1e-3) / 1e6

    if rank == 0:
        peak, peak_src = measured_peak_hbm()
        alg_bytes = algorithmic_bytes(w, nF)
        if args.quick:
            print(json.dumps({"quick": True, "n_gpus": world, "ms_per_step": ms_per_step, "value": value,
                              "gather": gather_mode, "gather_checked": gather_checked,
                              "sm_mhz": clk and clk.get("sm_mhz")}))
            if world > 1:
                dist.destroy_process_group()
            return
        dom = max(kt, key=kt.get)
        achieved = alg_bytes / (kt[dom] * 1e-3) / 1e9
        line = {
            "metric": metric_name(w),
            "value": value, "unit": "Msamples/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic",
            "config": {"workload": w["label"], "per_gpu_batch": B, "global_batch": world * B, "n_frames": nF,
                       "samples_per_utterance": T, "noise": "in-kernel Philox4x32-10",
                       "outputs": "signal+harmonic+noise" if w["kind"] in ("sins", "combsub") else "signal",
                       "parallelism": "batch-sharded x%d%s" % (
                           world, (", waveform gathered on rank 0 inside the step: " + gather_mode) if do_gather else ""),
                       "l2": "flushed between steps (256 MiB memset, untimed); per-step CUDA events summed",
                       "wall_ms_per_step_incl_flush": 1e3 * wall / args.steps},
            "roofline": {"bound": "hbm", "kernel": dom, "achieved": achieved, "peak": peak, "unit": "GB/s",
                         "frac": achieved / peak, "traffic": ncu_traffic(args.workload, dom), "peak_source": peak_src,
                         "algorithmic_bytes_per_launch": alg_bytes, "kernel_ms": kt,
                         "whole_path_frac": alg_bytes / (ms_per_step * 1e-3) / 1e9 / peak if world == 1 else None,
                         "note": "achieved = algorithmic bytes of the whole path / duration of the dominant kernel; "
                                 "Sins/CombSub are FP32/SFU-issue bound by construction (see DESIGN.md)"},
            "e2e": {"value": samples_step / (e2e_ms * 1e-3) / 1e6, "unit": "Msamples/s", "ms_per_step": e2e_ms,
                    "h2d_bytes_per_step": run.h2d, "d2h_bytes_per_step": run.out_h.numel() * 4,
                    "what": "pinned host f0+controls -> H2D -> module forward -> D2H of the waveform, through "
                            "ddsp_svc_b200.HostPipeline (utterance chunks %s; upload, kernels and download overlap); "
                            "median of %d passes, each timed separately with the L2 flushed before it"
                            % (args.e2e_chunks, max(10, min(args.steps, 20)))},
            "gpu_launches": launches,
            "clocks": clk,
        }
        if do_gather:
            line["gather_checked"] = gather_checked
        if world == 1 and args.workload == "sins" and not args.no_others:
            with torch.no_grad():
                line["eager_gpu_baseline"] = eager_gpu_baseline(w, run, flush, torch)
                line["other_workloads"] = {n: time_other_workload(n, dev, flush, torch) for n in OTHER_WORKLOADS}
        if world == 1 and not args.no_cpu_baseline:
            sample_b = 4 if w["B"] >= 4 else w["B"]
            v, dt, cores = cpu_reference_run(w, sample_b, 3)
            line["cpu_baseline"] = {"value": v, "unit": "Msamples/s", "cores": cores, "kind": "port",
                                    "sample": "%d of %d utterances x %d s, best of 3 (%.2f s per pass)" % (
                                        sample_b, B, w["sec"], dt)}
        if args.breakdown:
            print(json.dumps(kt), file=sys.stderr)
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
