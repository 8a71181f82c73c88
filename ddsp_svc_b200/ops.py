"""Thin tensor-level wrappers over the C ABI: PyTorch CUDA tensors in, PyTorch CUDA tensors out.

PyTorch is only the plumbing here (device memory from its caching allocator, the current
stream); all arithmetic happens in libb200ddsp.so.  Every function requires CUDA fp32 inputs
and raises otherwise -- there is no CPU path.
"""
import threading

import torch

from . import _lib

IR_ALLPASS, IR_MAG_HANN, IR_MAG_DYNAMIC = 0, 1, 2

# kernel launches issued through this module (bench.py reports it as gpu_launches)
_launches = 0
_tables = {}
_overlap_mode = 1   # mirrors the library's default (b2d_set_overlap)
_sins_impl = "auto"
_fir_impl = "auto"
_tables_lock = threading.Lock()


def set_fir_impl(impl):
    """'auto' (FFT-domain kernel for block size 512 and <= 1024 taps, else CUDA cores), 'cuda' (CUDA-core direct
    form), 'tc' (tcgen05 3xTF32 kernel, block size 512), 'cuda8' (older scalar CUDA-core kernel) or 'fft'."""
    global _fir_impl
    _lib.check(_lib.lib().b2d_set_fir_impl({"auto": 0, "cuda": 1, "tc": 2, "cuda8": 3, "fft": 4}[impl]), "b2d_set_fir_impl")
    _fir_impl = impl


def set_ir_impl(impl):
    """'auto' (tcgen05 when supported), 'cuda' (CUDA-core kernel) or 'tc' (tcgen05 3xTF32 kernel)."""
    _lib.check(_lib.lib().b2d_set_ir_impl({"auto": 0, "cuda": 1, "tc": 2}[impl]), "b2d_set_ir_impl")


def launches():
    return _launches


def _count(n):
    global _launches
    _launches += n


def _stream():
    return torch.cuda.current_stream().cuda_stream


def _ptr(t):
    return 0 if t is None else t.data_ptr()


def _need_cuda_f32(name, t, dtype=torch.float32, local=True):
    if not isinstance(t, torch.Tensor) or not t.is_cuda:
        raise ValueError("%s must be a CUDA tensor (the B200 kernels have no CPU fallback)" % name)
    if t.dtype != dtype:
        raise ValueError("%s must be %s, got %s" % (name, dtype, t.dtype))
    if local and t.device.index != torch.cuda.current_device():
        # the library launches on the calling thread's current device and on torch's current stream of it
        raise ValueError("%s lives on %s but the current CUDA device is %d; call torch.cuda.set_device(%d) "
                         "(one process per GPU) or wrap the call in torch.cuda.device(...)"
                         % (name, t.device, torch.cuda.current_device(), t.device.index))


def _need_frame_phase(frame_phase, B, nF):
    _need_cuda_f32("frame_phase", frame_phase, torch.float64)
    if tuple(frame_phase.shape) != (B, nF) or not frame_phase.is_contiguous():
        raise ValueError("frame_phase must be a contiguous [%d, %d] tensor (phase_scan of the same f0), got %s"
                         % (B, nF, tuple(frame_phase.shape)))


def _noise_rows(noise_in, B, T):
    """explicit noise samples for B utterances of T samples -> contiguous [B, T]"""
    _need_cuda_f32("noise_in", noise_in)
    if noise_in.numel() != B * T:
        raise ValueError("noise must hold B*T = %d*%d samples, got %s" % (B, T, tuple(noise_in.shape)))
    return noise_in.reshape(B, T).contiguous()


def _frames_2d(f0_frames):
    """[B, nF, 1] or [B, nF] -> contiguous [B, nF]."""
    _need_cuda_f32("f0_frames", f0_frames)
    f0 = f0_frames.squeeze(-1) if f0_frames.dim() == 3 else f0_frames
    if f0.dim() != 2:
        raise ValueError("f0_frames must be [B, n_frames, 1] or [B, n_frames]")
    return f0.contiguous()


def _ctrl_view(name, c, B, nF):
    """A raw control tensor [B, nF, C] that is a strided view of the dense Unit2Control output
    (torch.split, reference ddsp/unit2control.py:22): returns (tensor, frame stride)."""
    _need_cuda_f32(name, c)
    if c.dim() != 3 or c.shape[0] != B or c.shape[1] != nF:
        raise ValueError("Batch/frame size of %s %s does not match f0 (%d, %d)" % (name, tuple(c.shape), B, nF))
    if c.stride(2) != 1 or (B > 1 and c.stride(0) != nF * c.stride(1)) or c.stride(1) < c.shape[2]:
        c = c.contiguous()
    return c, c.stride(1)


def dft_tables(n_mag, device):
    """Constant cos/sin matrices of the 2(n_mag-1)-point inverse real DFT, cached per device."""
    key = (int(n_mag), torch.device(device).index)
    with _tables_lock:
        t = _tables.get(key)
        if t is None:
            L = _lib.lib()
            nbytes = L.b2d_dft_tables_bytes(int(n_mag))
            if nbytes == 0:
                raise ValueError("n_mag=%d out of range" % n_mag)
            t = torch.empty(nbytes // 4, dtype=torch.float32, device=device)
            _lib.check(L.b2d_dft_tables(int(n_mag), t.data_ptr(), _stream()), "b2d_dft_tables")
            _count(2)
            # built once per device and then read from whatever stream the caller is on: make it visible to all of them
            torch.cuda.current_stream().synchronize()
            _tables[key] = t
    return t


def phase_scan(f0_frames, block, sampling_rate, initial_phase=None, infer=True):
    """-> (frame_phase fp64 [B, nF] unwrapped cycles, phase_frames fp32 [B, nF, 1] radians)."""
    f0 = _frames_2d(f0_frames)
    B, nF = f0.shape
    ip = None
    if initial_phase is not None:
        ip = initial_phase.to(device=f0.device, dtype=torch.float32).reshape(-1).contiguous()
        if ip.numel() == 1 and B > 1:
            ip = ip.expand(B).contiguous()
        if ip.numel() != B:
            raise ValueError("initial_phase must have one value per utterance")
    frame_phase = torch.empty(B, nF, dtype=torch.float64, device=f0.device)
    phase_frames = torch.empty(B, nF, 1, dtype=torch.float32, device=f0.device)
    rc = _lib.lib().b2d_phase_scan(f0.data_ptr(), _ptr(ip), B, nF, int(block), float(sampling_rate),
                                   0 if infer else 1, frame_phase.data_ptr(), phase_frames.data_ptr(), _stream())
    _lib.check(rc, "b2d_phase_scan")
    _count(1)
    return frame_phase, phase_frames


def sins_bank(f0_frames, frame_phase, c_amp, block, sampling_rate, infer=True):
    f0 = _frames_2d(f0_frames)
    B, nF = f0.shape
    _need_frame_phase(frame_phase, B, nF)
    c, stride = _ctrl_view("amplitudes", c_amp, B, nF)
    out = torch.empty(B, nF * block, dtype=torch.float32, device=f0.device)
    rc = _lib.lib().b2d_sins_bank(f0.data_ptr(), frame_phase.data_ptr(), c.data_ptr(), stride, B, nF, int(block),
                                  c.shape[2], float(sampling_rate), 0 if infer else 1, out.data_ptr(), _stream())
    _lib.check(rc, "b2d_sins_bank")
    _count(1)
    return out


def ir_build(c_raw, mode, sampling_rate, f0_frames=None):
    """raw control [B, nF, M] -> impulse responses [B, nF, 2(M-1)]."""
    _need_cuda_f32("control", c_raw)
    B, nF, M = c_raw.shape
    c, stride = _ctrl_view("control", c_raw, B, nF)
    f0 = _frames_2d(f0_frames) if f0_frames is not None else None
    ir = torch.empty(B, nF, 2 * (M - 1), dtype=torch.float32, device=c.device)
    tab = dft_tables(M, c.device)
    rc = _lib.lib().b2d_ir_build(c.data_ptr(), stride, int(mode), _ptr(f0), tab.data_ptr(), B, nF, M,
                                 float(sampling_rate), ir.data_ptr(), _stream())
    _lib.check(rc, "b2d_ir_build")
    _count(1)
    return ir


def ltv_fir(x, ir, block, seed=0, utterance_offset=0, generic=False):
    """Time-varying FIR of x [B, T] (or None = in-kernel uniform noise) with ir [B, nF, L]."""
    _need_cuda_f32("ir", ir)
    ir = ir.contiguous()
    B, nF, L = ir.shape
    if x is not None:
        _need_cuda_f32("x", x)
        if x.shape[0] != B:
            raise ValueError("Batch size of audio ({}) and impulse response ({}) must be the same."
                             .format(x.shape[0], B))
        if x.dim() != 2 or x.shape[1] != nF * int(block):
            raise ValueError("audio must be [B, n_frames*block] = [%d, %d], got %s (the reference derives the hop "
                             "from the lengths, ddsp/core.py:156; here block is explicit)" % (B, nF * int(block), tuple(x.shape)))
        x = x.contiguous()
    y = torch.empty(B, nF * block, dtype=torch.float32, device=ir.device)
    Lh = _lib.lib()
    if generic:
        rc = Lh.b2d_ltv_fir_generic(_ptr(x), ir.data_ptr(), L, y.data_ptr(), B, nF, int(block), _stream())
    else:
        rc = Lh.b2d_ltv_fir(_ptr(x), ir.data_ptr(), L, y.data_ptr(), 0, 0, 0, 0, 0, int(seed),
                            int(utterance_offset), B, nF, int(block), _stream())
    _lib.check(rc, "b2d_ltv_fir")
    _count(1)
    return y


def sins_synth(f0_frames, frame_phase, c_amp, c_group_delay, c_noise, block, sampling_rate, noise_in=None,
               seed=0, utterance_offset=0, infer=True, want_parts=True, signal_out=None):
    """Whole Sins DSP after Unit2Control -> (signal, harmonic, noise) [B, T] each.
    ``signal_out``: optional preallocated [B, T] fp32 CUDA tensor for the mixed signal; it may live in
    another GPU's memory (peer-mapped, see sharding.PeerGather): the FIR kernel then writes the
    waveform straight over NVLink."""
    f0 = _frames_2d(f0_frames)
    B, nF = f0.shape
    _need_frame_phase(frame_phase, B, nF)
    ca, s0 = _ctrl_view("amplitudes", c_amp, B, nF)
    cg, s1 = _ctrl_view("group_delay", c_group_delay, B, nF)
    cn, s2 = _ctrl_view("noise_magnitude", c_noise, B, nF)
    if not (s0 == s1 == s2):  # views of different tensors: densify so one stride describes all
        ca, cg, cn = ca.contiguous(), cg.contiguous(), cn.contiguous()
        dense = torch.cat((ca, cg, cn), dim=-1)
        ca, cg, cn = torch.split(dense, [ca.shape[2], cg.shape[2], cn.shape[2]], dim=-1)
        s0 = dense.stride(1)
    H, Ma, Mn = ca.shape[2], cg.shape[2], cn.shape[2]
    dev = f0.device
    T = nF * block
    if noise_in is not None:
        noise_in = _noise_rows(noise_in, B, T)
    L = _lib.lib()
    ws_bytes = L.b2d_sins_workspace_bytes(B, nF, int(block), Ma, Mn)
    ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)
    if signal_out is not None:
        _need_cuda_f32("signal_out", signal_out, local=False)        # may be peer-mapped memory of another GPU
        if tuple(signal_out.shape) != (B, T) or not signal_out.is_contiguous():
            raise ValueError("signal_out must be a contiguous [B, T] tensor")
        signal = signal_out
    else:
        signal = torch.empty(B, T, dtype=torch.float32, device=dev)
    harmonic = torch.empty(B, T, dtype=torch.float32, device=dev) if want_parts else None
    noise = torch.empty(B, T, dtype=torch.float32, device=dev) if (want_parts or Ma != Mn) else None
    ta, tn = dft_tables(Ma, dev), dft_tables(Mn, dev)
    rc = L.b2d_sins_synth(f0.data_ptr(), frame_phase.data_ptr(), ca.data_ptr(), cg.data_ptr(), cn.data_ptr(), s0,
                          _ptr(noise_in), int(seed), int(utterance_offset), ta.data_ptr(), tn.data_ptr(), B, nF,
                          int(block), H, Ma, Mn, float(sampling_rate), 0 if infer else 1, signal.data_ptr(),
                          _ptr(harmonic), _ptr(noise), ws.data_ptr(), ws_bytes, _stream())
    _lib.check(rc, "b2d_sins_synth")
    fft_ok = int(block) == 512 and max(Ma, Mn) <= 257 and _fir_impl in ("auto", "fft")
    fused = _sins_impl == "fused" and Ma == Mn and fft_ok and H <= 128
    spectrum = _sins_impl == "spectrum" and fft_ok
    nsplit = max(1, min(abs(_overlap_mode), B)) if abs(_overlap_mode) >= 2 else 1
    _count(3 if fused else 5 if spectrum else 2 + nsplit * (2 if Ma == Mn else 3))
    return signal, harmonic, noise


def sinegen(f0, upp, sampling_rate, dim, rand_ini, sine_amp=0.1, noise_std=0.003, voiced_threshold=0.0,
            noise_in=None, seed=0, utterance_offset=0):
    """f0 [B, nF] -> [B, nF*upp, dim]  (reference nsf_hifigan/models.py:150-165)."""
    _need_cuda_f32("f0", f0)
    if f0.dim() != 2:
        raise ValueError("f0 must be [B, n_frames]")
    f0 = f0.contiguous()
    B, nF = f0.shape
    rand_ini = rand_ini.to(device=f0.device, dtype=torch.float32).reshape(-1).contiguous()
    if rand_ini.numel() != dim:
        raise ValueError("rand_ini must have %d elements" % dim)
    if noise_in is not None:
        _need_cuda_f32("noise_in", noise_in)
        if tuple(noise_in.shape) != (B, nF * upp, dim):
            raise ValueError("noise_in must be [B, n_frames*upp, dim]")
        noise_in = noise_in.contiguous()
    out = torch.empty(B, nF * upp, dim, dtype=torch.float32, device=f0.device)
    ws = torch.empty(B, nF, dtype=torch.float32, device=f0.device)
    rc = _lib.lib().b2d_sinegen(f0.data_ptr(), rand_ini.data_ptr(), _ptr(noise_in), int(seed), int(utterance_offset),
                                B, nF, int(upp), int(dim), float(sampling_rate), float(sine_amp), float(noise_std),
                                float(voiced_threshold), ws.data_ptr(), out.data_ptr(), _stream())
    _lib.check(rc, "b2d_sinegen")
    _count(2)
    return out


def comb_source(f0_frames, frame_phase, block, sampling_rate, infer=True):
    f0 = _frames_2d(f0_frames)
    B, nF = f0.shape
    _need_frame_phase(frame_phase, B, nF)
    out = torch.empty(B, nF * block, dtype=torch.float32, device=f0.device)
    rc = _lib.lib().b2d_comb_source(f0.data_ptr(), frame_phase.data_ptr(), B, nF, int(block), float(sampling_rate),
                                    0 if infer else 1, out.data_ptr(), _stream())
    _lib.check(rc, "b2d_comb_source")
    _count(1)
    return out


def _same_stride(named, B, nF):
    """Views of one dense control tensor share a frame stride; otherwise densify."""
    views = [_ctrl_view(n, c, B, nF) for n, c in named]
    if len({s for _, s in views}) == 1:
        return [c for c, _ in views], views[0][1]
    dense = torch.cat([c.contiguous() for c, _ in views], dim=-1)
    parts = torch.split(dense, [c.shape[2] for c, _ in views], dim=-1)
    return list(parts), dense.stride(1)


def combsub_synth(f0_frames, frame_phase, c_group_delay, c_harmonic, c_noise, block, sampling_rate, noise_in=None,
                  seed=0, utterance_offset=0, infer=True, signal_out=None):
    """Whole old-CombSub DSP after Unit2Control -> (signal, harmonic, noise) [B, T] each."""
    f0 = _frames_2d(f0_frames)
    B, nF = f0.shape
    _need_frame_phase(frame_phase, B, nF)
    (cg, ch, cn), stride = _same_stride([("group_delay", c_group_delay), ("harmonic_magnitude", c_harmonic),
                                         ("noise_magnitude", c_noise)], B, nF)
    Ma, Mh, Mn = cg.shape[2], ch.shape[2], cn.shape[2]
    dev, T = f0.device, nF * block
    if noise_in is not None:
        noise_in = _noise_rows(noise_in, B, T)
    L = _lib.lib()
    ws_bytes = L.b2d_combsub_workspace_bytes(B, nF, int(block), Ma, Mh, Mn)
    ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)
    signal, harmonic, noise = (torch.empty(B, T, dtype=torch.float32, device=dev) for _ in range(3))
    if signal_out is not None:
        _need_cuda_f32("signal_out", signal_out, local=False)        # may be peer-mapped memory of another GPU
        if tuple(signal_out.shape) != (B, T) or not signal_out.is_contiguous():
            raise ValueError("signal_out must be a contiguous [B, T] tensor")
        signal = signal_out
    rc = L.b2d_combsub_synth(f0.data_ptr(), frame_phase.data_ptr(), cg.data_ptr(), ch.data_ptr(), cn.data_ptr(),
                             stride, _ptr(noise_in), int(seed), int(utterance_offset), dft_tables(Ma, dev).data_ptr(),
                             dft_tables(Mh, dev).data_ptr(), dft_tables(Mn, dev).data_ptr(), B, nF, int(block), Ma,
                             Mh, Mn, float(sampling_rate), 0 if infer else 1, signal.data_ptr(), harmonic.data_ptr(),
                             noise.data_ptr(), ws.data_ptr(), ws_bytes, _stream())
    _lib.check(rc, "b2d_combsub_synth")
    _count(6 if Ma == Mn else 7)
    return signal, harmonic, noise


def superfast_scan(f0_frames, block, sampling_rate):
    """-> (workspace tensor holding per-frame source parameters, phase_frames [B, nF, 1])."""
    f0 = _frames_2d(f0_frames)
    B, nF = f0.shape
    L = _lib.lib()
    ws = torch.empty(L.b2d_superfast_workspace_bytes(B, nF), dtype=torch.uint8, device=f0.device)
    phase_frames = torch.empty(B, nF, 1, dtype=torch.float32, device=f0.device)
    rc = L.b2d_superfast_scan(f0.data_ptr(), B, nF, int(block), float(sampling_rate), ws.data_ptr(),
                              phase_frames.data_ptr(), _stream())
    _lib.check(rc, "b2d_superfast_scan")
    _count(1)
    return ws, phase_frames


def superfast_synth(ws, c_hm, c_hp, c_nm, c_np, block, win_length, noise_in=None, seed=0, utterance_offset=0,
                    signal_out=None):
    if c_hm.dim() != 3:
        raise ValueError("controls must be [B, n_frames, win_length/2+1]")
    B, nF = c_hm.shape[0], c_hm.shape[1]
    if not isinstance(ws, torch.Tensor) or not ws.is_cuda or ws.dtype != torch.uint8 or \
            ws.numel() < _lib.lib().b2d_superfast_workspace_bytes(B, nF):
        raise ValueError("ws must be the workspace superfast_scan returned for the same (B, n_frames) = (%d, %d)" % (B, nF))
    (hm, hp, nm, npz), stride = _same_stride([("harmonic_magnitude", c_hm), ("harmonic_phase", c_hp),
                                              ("noise_magnitude", c_nm), ("noise_phase", c_np)], B, nF)
    if hm.shape[2] != win_length // 2 + 1:
        raise ValueError("controls must have win_length/2+1 = %d bins" % (win_length // 2 + 1))
    T = nF * block
    if noise_in is not None:
        noise_in = _noise_rows(noise_in, B, T)
    if signal_out is not None:
        _need_cuda_f32("signal_out", signal_out, local=False)        # may be peer-mapped memory of another GPU
        if tuple(signal_out.shape) != (B, T) or not signal_out.is_contiguous():
            raise ValueError("signal_out must be a contiguous [B, T] tensor")
        signal = signal_out
    else:
        signal = torch.empty(B, T, dtype=torch.float32, device=hm.device)
    rc = _lib.lib().b2d_superfast_synth(ws.data_ptr(), hm.data_ptr(), hp.data_ptr(), nm.data_ptr(), npz.data_ptr(),
                                        stride, _ptr(noise_in), int(seed), int(utterance_offset), B, nF, int(block),
                                        int(win_length), signal.data_ptr(), _stream())
    _lib.check(rc, "b2d_superfast_synth")
    _count(1)
    return signal


def superfast_backward(ws, c_hm, c_hp, c_nm, c_np, grad_signal, block, win_length, noise_in=None, seed=0,
                       utterance_offset=0):
    """dL/dcontrols of superfast_synth given grad_signal = dL/dsignal [B, T]; the other arguments are those of the
    forward call (same noise_in, or the same seed and utterance_offset).  Returns the four gradients
    [B, n_frames, win_length/2+1], views of one dense [B, n_frames, 4 (win_length/2+1)] tensor."""
    if c_hm.dim() != 3:
        raise ValueError("controls must be [B, n_frames, win_length/2+1]")
    B, nF = c_hm.shape[0], c_hm.shape[1]
    if not isinstance(ws, torch.Tensor) or not ws.is_cuda or ws.dtype != torch.uint8 or \
            ws.numel() < _lib.lib().b2d_superfast_workspace_bytes(B, nF):
        raise ValueError("ws must be the workspace superfast_scan returned for the same (B, n_frames) = (%d, %d)" % (B, nF))
    (hm, hp, nm, npz), stride = _same_stride([("harmonic_magnitude", c_hm), ("harmonic_phase", c_hp),
                                              ("noise_magnitude", c_nm), ("noise_phase", c_np)], B, nF)
    C = win_length // 2 + 1
    if hm.shape[2] != C:
        raise ValueError("controls must have win_length/2+1 = %d bins" % C)
    T = nF * block
    _need_cuda_f32("grad_signal", grad_signal)
    if tuple(grad_signal.shape) != (B, T):
        raise ValueError("grad_signal must be [B, n_frames*block] = [%d, %d], got %s" % (B, T, tuple(grad_signal.shape)))
    grad_signal = grad_signal.contiguous()
    if noise_in is not None:
        noise_in = _noise_rows(noise_in, B, T)
    dense = torch.empty(B, nF, 4 * C, dtype=torch.float32, device=hm.device)
    grads = torch.split(dense, C, dim=-1)
    rc = _lib.lib().b2d_superfast_backward(ws.data_ptr(), hm.data_ptr(), hp.data_ptr(), nm.data_ptr(), npz.data_ptr(),
                                           stride, _ptr(noise_in), int(seed), int(utterance_offset),
                                           grad_signal.data_ptr(), B, nF, int(block), int(win_length),
                                           *(g.data_ptr() for g in grads), dense.stride(1), _stream())
    _lib.check(rc, "b2d_superfast_backward")
    _count(1)
    return grads


def source_module(f0, upp, sampling_rate, dim, rand_ini, linear_weight, linear_bias, sine_amp=0.1, noise_std=0.003,
                  voiced_threshold=0.0, noise_in=None, seed=0, utterance_offset=0):
    """SineGen + tanh(Linear(dim -> 1)) fused: f0 [B, nF] -> [B, nF*upp, 1]  (nsf_hifigan/models.py:201-204)."""
    _need_cuda_f32("f0", f0)
    f0 = f0.contiguous()
    B, nF = f0.shape
    rand_ini = rand_ini.to(device=f0.device, dtype=torch.float32).reshape(-1).contiguous()
    w = linear_weight.detach().to(device=f0.device, dtype=torch.float32).reshape(-1).contiguous()
    if rand_ini.numel() != dim or w.numel() != dim:
        raise ValueError("rand_ini and linear_weight must have %d elements" % dim)
    if noise_in is not None:
        _need_cuda_f32("noise_in", noise_in)
        if tuple(noise_in.shape) != (B, nF * upp, dim):
            raise ValueError("noise_in must be [B, n_frames*upp, dim]")
        noise_in = noise_in.contiguous()
    out = torch.empty(B, nF * upp, 1, dtype=torch.float32, device=f0.device)
    ws = torch.empty(B, nF, dtype=torch.float32, device=f0.device)
    rc = _lib.lib().b2d_source_module(f0.data_ptr(), rand_ini.data_ptr(), _ptr(noise_in), int(seed), int(utterance_offset),
                                      B, nF, int(upp), int(dim), float(sampling_rate), float(sine_amp), float(noise_std),
                                      float(voiced_threshold), w.data_ptr(), float(linear_bias), ws.data_ptr(),
                                      out.data_ptr(), _stream())
    _lib.check(rc, "b2d_source_module")
    _count(2)
    return out


def set_sinegen_impl(name):
    """'auto' | 'v1' (one sample per thread) | 'v2' (four per thread) | 'v2p' (four per thread, packed f32x2) | 'v2r7' (v2
    with Philox4x32-7 instead of -10 for the in-kernel noise)."""
    impl = {"auto": 0, "v1": 1, "v2": 2, "v2p": 3, "v2r7": 4}[name]
    _lib.check(_lib.lib().b2d_set_sinegen_impl(impl), "b2d_set_sinegen_impl")


def combsubfast_filter(comb, c_hm, c_hp, c_nm, block, noise_in=None, seed=0, utterance_offset=0):
    """CombSubFast after the source: comb [B, T] + raw controls [B, nF, block+1] -> signal [B, T]
    (reference ddsp/vocoder.py:758-784)."""
    _need_cuda_f32("comb", comb)
    if comb.dim() != 2 or comb.shape[1] % int(block) != 0:
        raise ValueError("comb must be [B, n_frames*block] with block=%d, got %s" % (block, tuple(comb.shape)))
    B, T = comb.shape
    nF = T // block
    (hm, hp, nm), stride = _same_stride([("harmonic_magnitude", c_hm), ("harmonic_phase", c_hp),
                                         ("noise_magnitude", c_nm)], B, nF)
    if hm.shape[2] != block + 1:
        raise ValueError("controls must have block_size+1 = %d bins" % (block + 1))
    comb = comb.contiguous()
    if noise_in is not None:
        noise_in = _noise_rows(noise_in, B, T)
    signal = torch.empty(B, T, dtype=torch.float32, device=comb.device)
    rc = _lib.lib().b2d_combsubfast_filter(comb.data_ptr(), hm.data_ptr(), hp.data_ptr(), nm.data_ptr(), stride,
                                           _ptr(noise_in), int(seed), int(utterance_offset), B, nF, int(block),
                                           signal.data_ptr(), _stream())
    _lib.check(rc, "b2d_combsubfast_filter")
    _count(1)
    return signal


def set_fft_arith(name):
    """'packed' (default: f32x2 complex additions in the FFT kernels) | 'scalar'."""
    _lib.check(_lib.lib().b2d_set_fft_arith({"scalar": 0, "packed": 1}[name]), "b2d_set_fft_arith")


def set_overlap(mode):
    """0 / False: every kernel of a synthesizer call in order on the current stream; 1 / True: impulse responses next to
    the bank on an internal side stream; k >= 2: additionally k staggered sub-batches on two streams (b200ddsp.h)."""
    global _overlap_mode
    _lib.check(_lib.lib().b2d_set_overlap(int(mode)), "b2d_set_overlap")
    _overlap_mode = int(mode)


def set_sins_impl(name):
    """'auto' (= 'split': separate bank kernel, measured fastest) | 'split' | 'fused' (bank inside the FFT-domain FIR kernel)
    | 'spectrum' (impulse-response spectra from their own kernel, read by the FIR kernel)."""
    global _sins_impl
    _lib.check(_lib.lib().b2d_set_sins_impl({"auto": 0, "split": 1, "fused": 2, "spectrum": 3}[name]), "b2d_set_sins_impl")
    _sins_impl = name
