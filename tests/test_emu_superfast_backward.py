"""The backward kernel SOURCE of csrc/superfast.cu executed on the CPU (tests/emu/host_emu.h): its control gradients
against the live reference's (tests/golden/ref_grad_superfast_*.npz), their independence of the chunking and of an
utterance_offset shard, and a ThreadSanitizer run of the same source (a missing or misplaced __syncthreads around
shared memory is a data race between the emulated threads)."""
import ctypes
import os
import shutil
import subprocess

import numpy as np
import pytest

from tests import superfast_grad as SG
from tests.golden import cases as G
from tests.test_emu_superfast import frame_par

HERE = os.path.dirname(os.path.abspath(__file__))
SRC = os.path.join(HERE, "emu", "emu_superfast_backward.cpp")
C = 1025
f32 = np.float32

pytestmark = pytest.mark.skipif(shutil.which("g++") is None, reason="g++ not available")


@pytest.fixture(scope="module")
def emu(tmp_path_factory):
    so = str(tmp_path_factory.mktemp("emu") / "libemu_sf_bwd.so")
    cmd = ["g++", "-std=c++20", "-O2", "-ffp-contract=off", "-shared", "-fPIC", "-pthread", "-Wno-unknown-pragmas",
           "-o", so, SRC]
    proc = subprocess.run(cmd, capture_output=True, text=True)
    assert proc.returncode == 0, proc.stderr
    lib = ctypes.CDLL(so)
    fp = ctypes.POINTER(ctypes.c_float)
    lib.emu_superfast_backward.argtypes = [fp, fp, fp, fp, fp, ctypes.c_longlong, fp, ctypes.c_ulonglong,
                                           ctypes.c_longlong, fp, ctypes.c_int, ctypes.c_int, ctypes.c_int,
                                           fp, fp, fp, fp, ctypes.c_longlong]

    def run(f0, dense, noise, g, pairs=16, seed=0, utt_off=0):
        B, nF = f0.shape[0], f0.shape[1]
        par = frame_par(np.asarray(f0).reshape(B, nF))
        dense = np.ascontiguousarray(dense, f32)
        g = np.ascontiguousarray(g, f32)
        nz = None if noise is None else np.ascontiguousarray(noise, f32)
        out = np.full((B, nF, 4 * C), np.nan, f32)          # one dense buffer holds the four gradients
        ptr = lambda a, off=0: ctypes.cast(a.ctypes.data + 4 * off, fp)
        rc = lib.emu_superfast_backward(ptr(par), ptr(dense, 0), ptr(dense, C), ptr(dense, 2 * C), ptr(dense, 3 * C),
                                        dense.shape[2], ptr(nz) if nz is not None else None, seed, utt_off, ptr(g),
                                        B, nF, pairs, ptr(out, 0), ptr(out, C), ptr(out, 2 * C), ptr(out, 3 * C),
                                        out.shape[2])
        assert rc == 0
        return {k: out[..., i * C:(i + 1) * C] for i, k in enumerate(SG.KEYS)}

    return run


def _inputs(name):
    inp = G.build_inputs(name)
    B, nF = inp["case"]["B"], inp["case"]["nF"]
    return inp["f0"].numpy(), inp["dense"].numpy(), inp["noise"].numpy(), SG.upstream(name, (B, nF * G.P)).numpy()


@pytest.mark.parametrize("name", SG.CASES)
def test_kernel_source_matches_reference_gradients(emu, name):
    f0, dense, noise, g = _inputs(name)
    gold = np.load(SG.golden_path(name))
    got = emu(f0, dense, noise, g)
    for k in SG.KEYS:
        assert not np.isnan(got[k]).any(), k
        e = SG.rel_rms(got[k], gold["grad_" + k])
        assert e < 1e-5, (name, k, e)


def test_gradients_do_not_depend_on_chunking_or_sharding(emu):
    f0, dense, noise, g = _inputs("superfast_b2_f24")
    ref = emu(f0, dense, noise, g, pairs=16)
    for pairs in (1, 3, 5):
        got = emu(f0, dense, noise, g, pairs=pairs)
        assert all(np.array_equal(got[k], ref[k]) for k in SG.KEYS), pairs
    # in-kernel noise: utterance 1 alone with utterance_offset=1 is the same as within the batch
    full = emu(f0, dense, None, g, pairs=2, seed=7)
    part = emu(f0[1:], dense[1:], None, g[1:], pairs=5, seed=7, utt_off=1)
    assert all(np.array_equal(full[k][1:], part[k]) and np.isfinite(full[k]).all() for k in SG.KEYS)


def test_kernel_source_has_no_shared_memory_race(tmp_path):
    exe = str(tmp_path / "tsan_superfast_backward")
    cmd = ["g++", "-std=c++20", "-O1", "-g", "-fsanitize=thread", "-pthread", "-Wno-unknown-pragmas", "-DTSAN_MAIN",
           "-o", exe, SRC]
    proc = subprocess.run(cmd, capture_output=True, text=True)
    if proc.returncode != 0 and "tsan" in proc.stderr.lower():
        pytest.skip("ThreadSanitizer runtime not available: " + proc.stderr.strip().splitlines()[-1])
    assert proc.returncode == 0, proc.stderr
    env = dict(os.environ, TSAN_OPTIONS="halt_on_error=0 exitcode=66")
    res = subprocess.run([exe], capture_output=True, text=True, timeout=600, env=env)
    assert "ThreadSanitizer" not in res.stderr, res.stderr[-4000:]
    assert res.returncode == 0 and "done" in res.stdout
