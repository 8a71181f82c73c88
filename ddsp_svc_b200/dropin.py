"""Drop-in wiring for an existing DDSP-SVC checkout.

``patch_reference()`` rebinds the reference's synthesizer classes to the B200 ones so that its
unmodified entry points (main.py, flask_api.py, gui.py, enhancer.py, ...) run on the CUDA
kernels:

    import ddsp_svc_b200
    ddsp_svc_b200.patch_reference()      # before `from ddsp.vocoder import load_model`
    # ... the rest of main.py unchanged

``load_model`` mirrors the reference's ``ddsp/vocoder.py:475-529`` (config.yaml next to the
checkpoint -> class dispatch -> strict load_state_dict) for use without patching.
"""
import os

import torch
import yaml

from . import sinegen, vocoder


class DotDict(dict):
    """Attribute access to nested config dicts (same behaviour as the reference's DotDict,
    ddsp/vocoder.py:467-473 / logger/utils.py:49-56)."""

    def __getattr__(self, key):
        val = self.get(key)
        return DotDict(val) if type(val) is dict else val

    __setattr__ = dict.__setitem__
    __delattr__ = dict.__delitem__


_MODEL_TYPES = {
    "Sins": lambda a: vocoder.Sins(
        sampling_rate=a.data.sampling_rate, block_size=a.data.block_size, n_harmonics=a.model.n_harmonics,
        n_mag_allpass=a.model.n_mag_allpass, n_mag_noise=a.model.n_mag_noise,
        n_unit=a.data.encoder_out_channels, n_spk=a.model.n_spk),
    "CombSub": lambda a: vocoder.CombSub(
        sampling_rate=a.data.sampling_rate, block_size=a.data.block_size, n_mag_allpass=a.model.n_mag_allpass,
        n_mag_harmonic=a.model.n_mag_harmonic, n_mag_noise=a.model.n_mag_noise,
        n_unit=a.data.encoder_out_channels, n_spk=a.model.n_spk),
    "CombSubFast": lambda a: vocoder.CombSubFast(
        sampling_rate=a.data.sampling_rate, block_size=a.data.block_size,
        n_unit=a.data.encoder_out_channels, n_spk=a.model.n_spk),
    "CombSubSuperFast": lambda a: vocoder.CombSubSuperFast(
        sampling_rate=a.data.sampling_rate, block_size=a.data.block_size, win_length=a.model.win_length,
        n_unit=a.data.encoder_out_channels, n_spk=a.model.n_spk),
}


def build_model(args):
    """Config (DotDict) -> synthesizer module; unknown types raise like the reference (:522)."""
    make = _MODEL_TYPES.get(args.model.type)
    if make is None:
        raise ValueError(f" [x] Unknown Model: {args.model.type}")
    return make(args)


def load_model(model_path, device="cuda"):
    config_file = os.path.join(os.path.split(model_path)[0], "config.yaml")
    with open(config_file, "r") as config:
        args = DotDict(yaml.safe_load(config))
    model = build_model(args)
    print(" [Loading] " + model_path)
    ckpt = torch.load(model_path, map_location=torch.device(device))
    model.to(device)
    model.load_state_dict(ckpt["model"])
    model.eval()
    return model, args


def _trainable_superfast(unit2ctrl_cls):
    """CombSubSuperFast whose control network is the reference's own Unit2Control (eager torch, differentiable, the
    same parameter tree, so checkpoints stay interchangeable); the synthesis runs on the B200 kernels with their
    fused backward."""

    class CombSubSuperFast(vocoder.CombSubSuperFast):
        def __init__(self, sampling_rate, block_size, win_length, n_unit=256, n_spk=1, use_pitch_aug=False,
                     pcmer_norm=False):
            u2c = unit2ctrl_cls(n_unit, n_spk, vocoder.CombSubSuperFast.split_map(win_length),
                                use_pitch_aug=use_pitch_aug, use_naive_v2=True, use_conv_stack=True)
            super().__init__(sampling_rate, block_size, win_length, n_unit=n_unit, n_spk=n_spk,
                             use_pitch_aug=use_pitch_aug, pcmer_norm=pcmer_norm, unit2ctrl=u2c)

    return CombSubSuperFast


def patch_reference(training=False):
    """Swap the synthesizer classes inside the (importable) reference package.  Returns the dict
    of original classes so a caller can restore them; its keys say what was patched.  If the enhancer stack
    (nsf_hifigan.models) cannot be imported, only the synthesizers are patched and the reason is returned under
    ``"_not_patched"`` -- any other failure propagates.

    ``training=True`` (for the reference's train.py and the reflow / diffusion training that calls it through
    ``ddsp_loss``): rebinds only ``ddsp.vocoder.CombSubSuperFast``, to a class that builds the reference's own
    ``ddsp.unit2control.Unit2Control``; every other class keeps the reference's (they have no backward here)."""
    import ddsp.vocoder as ref_vocoder          # the reference checkout must be on sys.path
    if training:
        import ddsp.unit2control as ref_u2c
        saved = {"CombSubSuperFast": ref_vocoder.CombSubSuperFast}
        ref_vocoder.CombSubSuperFast = _trainable_superfast(ref_u2c.Unit2Control)
        return saved
    names = ("Sins", "CombSub", "CombSubSuperFast", "CombSubFast")
    saved = {name: getattr(ref_vocoder, name) for name in names}
    for name in names:
        setattr(ref_vocoder, name, getattr(vocoder, name))
    from . import frontend                      # Volume_Extractor (numpy in -> numpy out like the reference, computed on the GPU)
    saved["Volume_Extractor"] = ref_vocoder.Volume_Extractor
    ref_vocoder.Volume_Extractor = frontend.Volume_Extractor
    try:                                        # mel front end of the enhancer / diffusion vocoders (needs librosa to import)
        import nsf_hifigan.nvSTFT as ref_stft
        from . import mel
        saved["STFT"] = ref_stft.STFT
        ref_stft.STFT = mel.STFT
    except ImportError as e:
        saved.setdefault("_not_patched", {})["nsf_hifigan.nvSTFT"] = "%s: %s" % (type(e).__name__, e)
    try:
        import nsf_hifigan.models as ref_nsf
    except ImportError as e:                    # enhancer stack not importable: synthesizers only (reported below)
        saved.setdefault("_not_patched", {})["nsf_hifigan.models"] = "%s: %s" % (type(e).__name__, e)
        return saved
    saved["SineGen"] = ref_nsf.SineGen
    saved["SourceModuleHnNSF"] = ref_nsf.SourceModuleHnNSF
    ref_nsf.SineGen = sinegen.SineGen
    ref_nsf.SourceModuleHnNSF = sinegen.SourceModuleHnNSF
    return saved


def unpatch_reference(saved):
    import ddsp.vocoder as ref_vocoder
    for name in ("Sins", "CombSub", "CombSubSuperFast", "CombSubFast", "Volume_Extractor"):
        if name in saved:
            setattr(ref_vocoder, name, saved[name])
    if "STFT" in saved:
        import nsf_hifigan.nvSTFT as ref_stft
        ref_stft.STFT = saved["STFT"]
    if "SineGen" in saved:
        import nsf_hifigan.models as ref_nsf
        ref_nsf.SineGen = saved["SineGen"]
        if "SourceModuleHnNSF" in saved:
            ref_nsf.SourceModuleHnNSF = saved["SourceModuleHnNSF"]
