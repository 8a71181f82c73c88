"""ctypes binding of libb200ddsp.so (the C ABI declared in include/b200ddsp.h).

The library is built in-tree by ``build()`` (nvcc, sm_100a only) and travels with the repo.
There is NO fallback: if the shared library is missing or fails to load, importing the ops
raises -- the product path never degrades to PyTorch or to the oracle.
"""
import ctypes
import os
import subprocess
import threading

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
CSRC = os.path.join(HERE, "csrc")
# B2D_LIB_PATH: load another build of the same library (A/B runs of compile-time variants; development only)
LIB_PATH = os.environ.get("B2D_LIB_PATH") or os.path.join(HERE, "libb200ddsp.so")
HEADER = os.path.join(ROOT, "include", "b200ddsp.h")

NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
              "-Xcompiler", "-fPIC", "-shared"]

c_f32p = ctypes.c_void_p   # device pointers travel as integers
c_f64p = ctypes.c_void_p
c_stream = ctypes.c_void_p

# name -> (restype, argtypes); must list every symbol include/b200ddsp.h declares
SIGNATURES = {
    "b2d_version": (ctypes.c_int, []),
    "b2d_last_error": (ctypes.c_char_p, []),
    "b2d_phase_scan": (ctypes.c_int, [c_f32p, c_f32p, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_double,
                                      ctypes.c_int, c_f64p, c_f32p, c_stream]),
    "b2d_sins_bank": (ctypes.c_int, [c_f32p, c_f64p, c_f32p, ctypes.c_int64, ctypes.c_int, ctypes.c_int,
                                     ctypes.c_int, ctypes.c_int, ctypes.c_double, ctypes.c_int, c_f32p, c_stream]),
    "b2d_set_ir_impl": (ctypes.c_int, [ctypes.c_int]),
    "b2d_dft_tables_bytes": (ctypes.c_size_t, [ctypes.c_int]),
    "b2d_dft_tables": (ctypes.c_int, [ctypes.c_int, c_f32p, c_stream]),
    "b2d_ir_build": (ctypes.c_int, [c_f32p, ctypes.c_int64, ctypes.c_int, c_f32p, c_f32p, ctypes.c_int,
                                    ctypes.c_int, ctypes.c_int, ctypes.c_double, c_f32p, c_stream]),
    "b2d_ltv_fir": (ctypes.c_int, [c_f32p, c_f32p, ctypes.c_int, c_f32p, c_f32p, c_f32p, ctypes.c_int, c_f32p,
                                   c_f32p, ctypes.c_uint64, ctypes.c_int64, ctypes.c_int, ctypes.c_int,
                                   ctypes.c_int, c_stream]),
    "b2d_set_fir_impl": (ctypes.c_int, [ctypes.c_int]),
    "b2d_ltv_fir_generic": (ctypes.c_int, [c_f32p, c_f32p, ctypes.c_int, c_f32p, ctypes.c_int, ctypes.c_int,
                                           ctypes.c_int, c_stream]),
    "b2d_sins_workspace_bytes": (ctypes.c_size_t, [ctypes.c_int] * 5),
    "b2d_sins_synth": (ctypes.c_int, [c_f32p, c_f64p, c_f32p, c_f32p, c_f32p, ctypes.c_int64, c_f32p,
                                      ctypes.c_uint64, ctypes.c_int64, c_f32p, c_f32p, ctypes.c_int, ctypes.c_int,
                                      ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_double,
                                      ctypes.c_int, c_f32p, c_f32p, c_f32p, ctypes.c_void_p, ctypes.c_size_t,
                                      c_stream]),
    "b2d_sinegen": (ctypes.c_int, [c_f32p, c_f32p, c_f32p, ctypes.c_uint64, ctypes.c_int64, ctypes.c_int,
                                   ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_double, ctypes.c_float,
                                   ctypes.c_float, ctypes.c_float, c_f32p, c_f32p, c_stream]),
    "b2d_source_module": (ctypes.c_int, [c_f32p, c_f32p, c_f32p, ctypes.c_uint64, ctypes.c_int64, ctypes.c_int,
                                         ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_double, ctypes.c_float,
                                         ctypes.c_float, ctypes.c_float, c_f32p, ctypes.c_float, c_f32p, c_f32p,
                                         c_stream]),
    "b2d_set_sinegen_impl": (ctypes.c_int, [ctypes.c_int]),
    "b2d_set_fft_arith": (ctypes.c_int, [ctypes.c_int]),
    "b2d_set_overlap": (ctypes.c_int, [ctypes.c_int]),
    "b2d_split_tf32": (ctypes.c_int, [c_f32p, c_f32p, c_f32p, ctypes.c_size_t, c_stream]),
    "b2d_u2c_embed": (ctypes.c_int, [c_f32p, c_f32p, c_f32p, c_f32p, c_f32p, c_f32p, ctypes.c_int, c_f32p, ctypes.c_int,
                                     ctypes.c_int, c_stream]),
    "b2d_u2c_groupnorm_lrelu": (ctypes.c_int, [c_f32p, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_int, c_f32p, c_f32p,
                                               ctypes.c_float, ctypes.c_float, c_f64p, c_stream]),
    "b2d_u2c_layernorm": (ctypes.c_int, [c_f32p, c_f32p, ctypes.c_int, ctypes.c_int, c_f32p, c_f32p, ctypes.c_float, c_stream]),
    "b2d_u2c_glu_dwconv_silu": (ctypes.c_int, [c_f32p, c_f32p, c_f32p, c_f32p, ctypes.c_int, ctypes.c_int, ctypes.c_int,
                                               ctypes.c_int, c_stream]),
    "b2d_u2c_softmax_features": (ctypes.c_int, [c_f32p, c_f32p, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_int,
                                                ctypes.c_float, c_stream]),
    "b2d_u2c_linear_attention": (ctypes.c_int, [c_f32p, c_f32p, c_f32p, c_f32p, ctypes.c_int, ctypes.c_int, ctypes.c_int,
                                                ctypes.c_int, ctypes.c_int, ctypes.c_float, c_stream]),
    "b2d_mel_frames": (ctypes.c_int, [ctypes.c_int] * 4),
    "b2d_mel_spectrogram": (ctypes.c_int, [c_f32p, c_f32p, c_f32p, ctypes.c_void_p, ctypes.c_int, ctypes.c_int, ctypes.c_int,
                                           ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_float, c_f32p, c_stream]),
    "b2d_volume_extract": (ctypes.c_int, [c_f32p, ctypes.c_int, ctypes.c_int, ctypes.c_int, c_f32p, c_stream]),
    "b2d_volume_mask": (ctypes.c_int, [c_f32p, ctypes.c_int, ctypes.c_int, ctypes.c_float, c_f32p, c_stream]),
    "b2d_mask_apply": (ctypes.c_int, [c_f32p, c_f32p, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_int,
                                      c_stream]),
    "b2d_cross_fade": (ctypes.c_int, [c_f32p, ctypes.c_int64, c_f32p, ctypes.c_int64, ctypes.c_int64, c_f32p, c_stream]),
    "b2d_set_sins_impl": (ctypes.c_int, [ctypes.c_int]),
    "b2d_combsubfast_filter": (ctypes.c_int, [c_f32p, c_f32p, c_f32p, c_f32p, ctypes.c_int64, c_f32p, ctypes.c_uint64,
                                              ctypes.c_int64, ctypes.c_int, ctypes.c_int, ctypes.c_int, c_f32p, c_stream]),
    "b2d_comb_source": (ctypes.c_int, [c_f32p, c_f64p, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_double,
                                       ctypes.c_int, c_f32p, c_stream]),
    "b2d_combsub_workspace_bytes": (ctypes.c_size_t, [ctypes.c_int] * 6),
    "b2d_combsub_synth": (ctypes.c_int, [c_f32p, c_f64p, c_f32p, c_f32p, c_f32p, ctypes.c_int64, c_f32p,
                                         ctypes.c_uint64, ctypes.c_int64, c_f32p, c_f32p, c_f32p, ctypes.c_int,
                                         ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_int,
                                         ctypes.c_double, ctypes.c_int, c_f32p, c_f32p, c_f32p, ctypes.c_void_p,
                                         ctypes.c_size_t, c_stream]),
    "b2d_superfast_workspace_bytes": (ctypes.c_size_t, [ctypes.c_int, ctypes.c_int]),
    "b2d_superfast_scan": (ctypes.c_int, [c_f32p, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_double,
                                          ctypes.c_void_p, c_f32p, c_stream]),
    "b2d_superfast_synth": (ctypes.c_int, [ctypes.c_void_p, c_f32p, c_f32p, c_f32p, c_f32p, ctypes.c_int64, c_f32p,
                                           ctypes.c_uint64, ctypes.c_int64, ctypes.c_int, ctypes.c_int, ctypes.c_int,
                                           ctypes.c_int, c_f32p, c_stream]),
    "b2d_superfast_backward": (ctypes.c_int, [ctypes.c_void_p, c_f32p, c_f32p, c_f32p, c_f32p, ctypes.c_int64, c_f32p,
                                              ctypes.c_uint64, ctypes.c_int64, c_f32p, ctypes.c_int, ctypes.c_int,
                                              ctypes.c_int, ctypes.c_int, c_f32p, c_f32p, c_f32p, c_f32p,
                                              ctypes.c_int64, c_stream]),
}

_lock = threading.Lock()
_lib = None


def sources():
    return sorted(os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith(".cu"))


def _stale():
    path = os.path.join(HERE, "libb200ddsp.so")
    if not os.path.isfile(path):
        return True
    t = os.path.getmtime(path)
    deps = sources() + [os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith(".cuh")] + [HEADER]
    return any(os.path.getmtime(d) > t for d in deps)


def build(force=False, verbose=False, out=None, defines=()):
    """Compile every CUDA source for sm_100a into ddsp_svc_b200/libb200ddsp.so (in-tree).
    ``out`` / ``defines``: build a compile-time variant (-DNAME=VALUE ...) into another file for A/B runs
    (loaded with B2D_LIB_PATH=<file>)."""
    default = os.path.join(HERE, "libb200ddsp.so")
    target = out or default
    if out is None and not force and not _stale():
        return target
    nvcc = os.environ.get("NVCC", "nvcc")
    cmd = ([nvcc] + NVCC_FLAGS + ["-D" + d for d in defines] + (["-Xptxas", "-v"] if verbose else []) +
           ["-o", target] + sources())
    proc = subprocess.run(cmd, capture_output=True, text=True)
    if proc.returncode != 0:
        raise RuntimeError("nvcc failed:\n%s\n%s" % (" ".join(cmd), proc.stderr))
    if verbose:
        print(proc.stderr)
    return target


def lib():
    """Load (once) and return the ctypes handle.  Raises if the library is unavailable."""
    global _lib
    if _lib is not None:
        return _lib
    with _lock:
        if _lib is None:
            if not os.path.isfile(LIB_PATH):
                raise RuntimeError(
                    "libb200ddsp.so is missing (%s). Run `python -c 'import __graft_entry__ as g; g.build()'`; "
                    "there is no CPU or PyTorch fallback for the synthesis kernels." % LIB_PATH)
            handle = ctypes.CDLL(LIB_PATH)
            for name, (res, args) in SIGNATURES.items():
                fn = getattr(handle, name)   # AttributeError if the symbol is not exported
                fn.restype = res
                fn.argtypes = args
            _lib = handle
    return _lib


class B2DError(RuntimeError):
    pass


def check(rc, what):
    """0 ok; <0 argument error -> ValueError (the reference raises ValueError for shape
    mismatches, ddsp/core.py:151-153); >0 CUDA error -> RuntimeError."""
    if rc == 0:
        return
    msg = lib().b2d_last_error()
    msg = msg.decode("utf-8", "replace") if msg else ""
    if rc < 0:
        raise ValueError("%s failed (%d): %s" % (what, rc, msg))
    raise B2DError("%s failed (cudaError %d): %s" % (what, rc, msg))
