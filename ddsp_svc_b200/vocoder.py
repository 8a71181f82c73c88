"""Drop-in synthesizer modules: same constructor arguments, buffers (state-dict keys) and
forward() contract as the reference's ddsp/vocoder.py classes, with the DSP executed by the
sm_100a kernels of libb200ddsp.so.

    signal, hidden, (harmonic, noise) = model(units_frames, f0_frames, volume_frames,
                                              spk_id=..., spk_mix_dict=..., initial_phase=..., infer=True)

``unit2ctrl`` (the small network that predicts the frame-rate controls, reference
ddsp/unit2control.py) is outside the accelerated path: pass your own module, or leave it None
to use the reference's Unit2Control when the reference package is importable (the
``patch_reference()`` drop-in scenario).

Two noise modes: by default white noise is generated inside the FIR kernel (Philox, seeded
from torch's CPU generator so ``torch.manual_seed`` makes runs reproducible); pass
``noise=tensor [B, T]`` to feed explicit samples (parity tests feed what the reference's
``rand_like`` drew).
"""
import torch

from . import ops


def _reference_unit2ctrl(n_unit, n_spk, split_map, **kw):
    """The control network: this package's own Unit2Control (same parameter tree as the reference's
    ddsp/unit2control.py, so its checkpoints load strictly; fused B200 kernels + library GEMMs, inference only)."""
    from .unit2control import Unit2Control
    return Unit2Control(n_unit, n_spk, split_map, **kw)


def _host_seed():
    # consumes torch's CPU generator (reproducible under torch.manual_seed), no device sync
    return int(torch.randint(0, 2 ** 62, (1,), dtype=torch.int64).item())


def _check_shape(cls, ok, what):
    """Shapes the kernels do not cover fail when the model is BUILT (load_model / patch_reference time), not at the
    first forward after some kernels have already been launched."""
    if not ok:
        raise ValueError("%s on B200: %s (every config the reference ships uses block_size 512)" % (cls, what))


class _SynthBase(torch.nn.Module):
    def _scalars(self):
        """sampling_rate / block_size live in 0-dim buffers (state-dict compatible with the
        reference, ddsp/vocoder.py:546-547); read them once, not on every call."""
        c = self.__dict__.get("_scalar_cache")
        if c is None:
            c = (int(self.sampling_rate.item()), int(self.block_size.item()))
            self.__dict__["_scalar_cache"] = c
        return c

    def _load_from_state_dict(self, *a, **k):
        super()._load_from_state_dict(*a, **k)
        self.__dict__["_scalar_cache"] = None

    @staticmethod
    def _forward_only(ctrls):
        if torch.is_grad_enabled() and any(v.requires_grad for v in ctrls.values()):
            raise NotImplementedError(
                "the B200 synthesis kernels are forward-only; call under torch.no_grad() "
                "(every inference caller of the reference does, e.g. main.py:250)")


class Sins(_SynthBase):
    """Sinusoids additive synthesiser -- reference ddsp/vocoder.py:532-611."""

    def __init__(self, sampling_rate, block_size, n_harmonics, n_mag_allpass, n_mag_noise, n_unit=256, n_spk=1,
                 unit2ctrl=None):
        super().__init__()
        _check_shape("Sins", int(block_size) % 256 == 0 and 0 < int(block_size) <= 2048, "block_size %s must be a "
                     "multiple of 256 up to 2048" % (block_size,))
        _check_shape("Sins", 0 < int(n_harmonics) <= 512 and min(int(n_mag_allpass), int(n_mag_noise)) >= 2 and
                     max(int(n_mag_allpass), int(n_mag_noise)) <= 1025, "n_harmonics <= 512 and 2 <= n_mag <= 1025")
        self.register_buffer("sampling_rate", torch.tensor(sampling_rate))
        self.register_buffer("block_size", torch.tensor(block_size))
        split_map = {
            "amplitudes": n_harmonics,
            "group_delay": n_mag_allpass,
            "noise_magnitude": n_mag_noise,
        }
        self.unit2ctrl = unit2ctrl if unit2ctrl is not None else _reference_unit2ctrl(n_unit, n_spk, split_map)

    def forward(self, units_frames, f0_frames, volume_frames, spk_id=None, spk_mix_dict=None, initial_phase=None,
                infer=True, max_upsample_dim=32, noise=None, utterance_offset=0, signal_out=None):
        """units_frames B x n_frames x n_unit; f0_frames B x n_frames x 1; volume_frames B x n_frames x 1.
        ``max_upsample_dim`` only chunks the reference's temporaries and has no effect here.
        ``signal_out``: optional preallocated [B, T] destination of ``signal`` (may be peer-mapped memory)."""
        sr, block = self._scalars()
        frame_phase, phase_frames = ops.phase_scan(f0_frames, block, sr, initial_phase, infer)
        ctrls, hidden = self.unit2ctrl(units_frames, f0_frames, phase_frames, volume_frames, spk_id=spk_id,
                                       spk_mix_dict=spk_mix_dict)
        self._forward_only(ctrls)
        signal, harmonic, noise_out = ops.sins_synth(
            f0_frames, frame_phase, ctrls["amplitudes"], ctrls["group_delay"], ctrls["noise_magnitude"], block, sr,
            noise_in=noise, seed=0 if noise is not None else _host_seed(), utterance_offset=utterance_offset,
            infer=infer, signal_out=signal_out)
        return signal, hidden, (harmonic, noise_out)


class CombSub(_SynthBase):
    """Combtooth subtractive synthesiser (old version) -- reference ddsp/vocoder.py:788-862."""

    def __init__(self, sampling_rate, block_size, n_mag_allpass, n_mag_harmonic, n_mag_noise, n_unit=256, n_spk=1,
                 unit2ctrl=None):
        super().__init__()
        _check_shape("CombSub", int(block_size) % 256 == 0 and 0 < int(block_size) <= 2048, "block_size %s must be a "
                     "multiple of 256 up to 2048" % (block_size,))
        _check_shape("CombSub", min(int(n_mag_allpass), int(n_mag_harmonic), int(n_mag_noise)) >= 2 and
                     max(int(n_mag_allpass), int(n_mag_harmonic), int(n_mag_noise)) <= 1025, "2 <= n_mag <= 1025")
        self.register_buffer("sampling_rate", torch.tensor(sampling_rate))
        self.register_buffer("block_size", torch.tensor(block_size))
        split_map = {
            "group_delay": n_mag_allpass,
            "harmonic_magnitude": n_mag_harmonic,
            "noise_magnitude": n_mag_noise,
        }
        self.unit2ctrl = unit2ctrl if unit2ctrl is not None else _reference_unit2ctrl(n_unit, n_spk, split_map)

    def forward(self, units_frames, f0_frames, volume_frames, spk_id=None, spk_mix_dict=None, initial_phase=None,
                infer=True, noise=None, utterance_offset=0, signal_out=None, **kwargs):
        sr, block = self._scalars()
        frame_phase, phase_frames = ops.phase_scan(f0_frames, block, sr, initial_phase, infer)
        ctrls, hidden = self.unit2ctrl(units_frames, f0_frames, phase_frames, volume_frames, spk_id=spk_id,
                                       spk_mix_dict=spk_mix_dict)
        self._forward_only(ctrls)
        signal, harmonic, noise_out = ops.combsub_synth(
            f0_frames, frame_phase, ctrls["group_delay"], ctrls["harmonic_magnitude"], ctrls["noise_magnitude"],
            block, sr, noise_in=noise, seed=0 if noise is not None else _host_seed(),
            utterance_offset=utterance_offset, infer=infer, signal_out=signal_out)
        return signal, hidden, (harmonic, noise_out)


class _SuperFastSynth(torch.autograd.Function):
    """superfast_synth with a backward for the four controls (the fused kernel of b2d_superfast_backward).  The
    forward is the inference kernel unchanged; the backward recomputes the source from the scan workspace and the
    noise from noise_in or (seed, utterance_offset), so nothing but the controls is kept alive."""

    @staticmethod
    def forward(ctx, ws, hm, hp, nm, np_, block, win, noise, seed, utterance_offset):
        signal = ops.superfast_synth(ws, hm, hp, nm, np_, block, win, noise_in=noise, seed=seed,
                                     utterance_offset=utterance_offset)
        ctx.save_for_backward(ws, hm, hp, nm, np_, noise)
        ctx.args = (block, win, seed, utterance_offset)
        return signal

    @staticmethod
    @torch.autograd.function.once_differentiable
    def backward(ctx, grad_signal):
        ws, hm, hp, nm, np_, noise = ctx.saved_tensors
        block, win, seed, utterance_offset = ctx.args
        grads = ops.superfast_backward(ws, hm, hp, nm, np_, grad_signal, block, win, noise_in=noise, seed=seed,
                                       utterance_offset=utterance_offset)
        return (None,) + tuple(grads) + (None,) * 5


class CombSubSuperFast(_SynthBase):
    """Combtooth subtractive synthesiser (STFT-domain filtering; what configs/combsub.yaml
    selects) -- reference ddsp/vocoder.py:613-710.  Returns (signal, hidden, (signal, signal))
    with the same tensor three times, like the reference.

    Trainable: when grad is enabled and a control requires grad, the signal is differentiable with respect to the
    four controls (fused backward kernel); gradients to f0 and to explicit noise are not provided."""

    def __init__(self, sampling_rate, block_size, win_length, n_unit=256, n_spk=1, use_pitch_aug=False,
                 pcmer_norm=False, unit2ctrl=None):
        super().__init__()
        _check_shape("CombSubSuperFast", int(block_size) == 512 and int(win_length) == 2048,
                     "only block_size 512 / win_length 2048 (configs/combsub.yaml) is built, got %s / %s" % (block_size, win_length))
        self.register_buffer("sampling_rate", torch.tensor(sampling_rate))
        self.register_buffer("block_size", torch.tensor(block_size))
        self.register_buffer("win_length", torch.tensor(win_length))
        self.register_buffer("window", torch.hann_window(win_length))
        self.unit2ctrl = unit2ctrl if unit2ctrl is not None else _reference_unit2ctrl(
            n_unit, n_spk, self.split_map(win_length), use_pitch_aug=use_pitch_aug, use_naive_v2=True,
            use_conv_stack=True)

    @staticmethod
    def split_map(win_length):
        n = int(win_length) // 2 + 1
        return {"harmonic_magnitude": n, "harmonic_phase": n, "noise_magnitude": n, "noise_phase": n}

    def _scalars(self):
        c = self.__dict__.get("_scalar_cache")
        if c is None:
            c = (int(self.sampling_rate.item()), int(self.block_size.item()), int(self.win_length.item()))
            self.__dict__["_scalar_cache"] = c
        return c

    def forward(self, units_frames, f0_frames, volume_frames, spk_id=None, spk_mix_dict=None, aug_shift=None,
                initial_phase=None, infer=True, noise=None, utterance_offset=0, signal_out=None, **kwargs):
        """``initial_phase`` is accepted and ignored, like the reference (ddsp/vocoder.py:653-661)."""
        sr, block, win = self._scalars()
        ws, phase_frames = ops.superfast_scan(f0_frames, block, sr)
        ctrls, hidden = self.unit2ctrl(units_frames, f0_frames, phase_frames, volume_frames, spk_id=spk_id,
                                       spk_mix_dict=spk_mix_dict, aug_shift=aug_shift)
        c = [ctrls[k] for k in ("harmonic_magnitude", "harmonic_phase", "noise_magnitude", "noise_phase")]
        seed = 0 if noise is not None else _host_seed()
        if torch.is_grad_enabled() and any(v.requires_grad for v in c):
            if f0_frames.requires_grad or (noise is not None and noise.requires_grad):
                raise NotImplementedError("CombSubSuperFast on B200 differentiates with respect to the four controls "
                                          "only; detach f0_frames and noise")
            if signal_out is not None:
                raise ValueError("signal_out cannot be combined with a differentiable forward")
            signal = _SuperFastSynth.apply(ws, *c, block, win, noise, seed, utterance_offset)
        else:
            signal = ops.superfast_synth(ws, *c, block, win, noise_in=noise, seed=seed,
                                         utterance_offset=utterance_offset, signal_out=signal_out)
        return signal, hidden, (signal, signal)


class CombSubFast(_SynthBase):
    """Combtooth subtractive synthesiser with 2*block sqrt-Hann frames (the variant the diffusion / reflow vocoders
    embed) -- reference ddsp/vocoder.py:712-786.  Returns (signal, hidden, (signal, signal)) like the reference.

    Parity on B200: 2e-8 RMS against the live-reference goldens (tests/test_gpu_combsubfast.py)."""

    def __init__(self, sampling_rate, block_size, n_unit=256, n_spk=1, use_pitch_aug=False, pcmer_norm=False,
                 unit2ctrl=None):
        super().__init__()
        _check_shape("CombSubFast", int(block_size) == 512, "only block_size 512 is built, got %s" % (block_size,))
        self.register_buffer("sampling_rate", torch.tensor(sampling_rate))
        self.register_buffer("block_size", torch.tensor(block_size))
        self.register_buffer("window", torch.sqrt(torch.hann_window(2 * block_size)))
        split_map = {
            "harmonic_magnitude": block_size + 1,
            "harmonic_phase": block_size + 1,
            "noise_magnitude": block_size + 1,
        }
        self.unit2ctrl = unit2ctrl if unit2ctrl is not None else _reference_unit2ctrl(
            n_unit, n_spk, split_map, use_pitch_aug=use_pitch_aug, pcmer_norm=pcmer_norm)

    def forward(self, units_frames, f0_frames, volume_frames, spk_id=None, spk_mix_dict=None, aug_shift=None,
                initial_phase=None, infer=True, noise=None, utterance_offset=0, **kwargs):
        sr, block = self._scalars()
        frame_phase, phase_frames = ops.phase_scan(f0_frames, block, sr, initial_phase, infer)
        ctrls, hidden = self.unit2ctrl(units_frames, f0_frames, phase_frames, volume_frames, spk_id=spk_id,
                                       spk_mix_dict=spk_mix_dict, aug_shift=aug_shift)
        self._forward_only(ctrls)
        comb = ops.comb_source(f0_frames, frame_phase, block, sr, infer)
        signal = ops.combsubfast_filter(comb, ctrls["harmonic_magnitude"], ctrls["harmonic_phase"],
                                        ctrls["noise_magnitude"], block, noise_in=noise,
                                        seed=0 if noise is not None else _host_seed(),
                                        utterance_offset=utterance_offset)
        return signal, hidden, (signal, signal)


class FixedControls(torch.nn.Module):
    """Stand-in for Unit2Control that returns preset raw controls: isolates the DSP path (the
    seam the parity tests and the benchmark use; reference ddsp/vocoder.py:578)."""

    def __init__(self, ctrls=None, hidden=None):
        super().__init__()
        self.ctrls, self.hidden = ctrls, hidden

    def forward(self, units, f0, phase, volume, **kw):
        self.last_phase_frames = phase
        return self.ctrls, self.hidden
