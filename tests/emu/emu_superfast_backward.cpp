// CPU execution of the backward kernel source in csrc/superfast.cu (see host_emu.h).  Built by
// tests/test_emu_superfast_backward.py, as a shared library and, with -DTSAN_MAIN, as a ThreadSanitizer executable.
// The frame scan (warp shuffles) is not emulated: the caller passes frame_par = (s, ds, acc_prev, 0) per frame.
#define B2D_HOST_EMU 1
#include "host_emu.h"
#include "../../ddsp_svc_b200/csrc/superfast.cu"

namespace { alignas(16) unsigned char smem_raw[1 << 17]; }   // the kernel's `extern __shared__` array

extern "C" int emu_superfast_backward(const float* frame_par, const float* hm, const float* hp, const float* nm,
                                      const float* np_, long long stride, const float* noise_in, unsigned long long seed,
                                      long long utt_off, const float* grad, int B, int nF, int pairs_per_cta,
                                      float* ghm, float* ghp, float* gnm, float* gnp, long long grad_stride) {
    static_assert(kBwdSmemBytes <= sizeof(smem_raw), "shared-memory emulation buffer too small");
    SfBwdParams p;
    p.frame_par = reinterpret_cast<const float4*>(frame_par);
    p.c_hm = hm; p.c_hp = hp; p.c_nm = nm; p.c_np = np_; p.ctrl_stride = stride; p.noise_in = noise_in; p.grad = grad;
    p.g_hm = ghm; p.g_hp = ghp; p.g_nm = gnm; p.g_np = gnp; p.grad_stride = grad_stride;
    p.nF = nF; p.P = 512; p.GP = pairs_per_cta; p.seed = seed; p.utt_off = utt_off;
    const int n_pairs = (nF + 1) / 2;
    emu::launch((unsigned)((n_pairs + pairs_per_cta - 1) / pairs_per_cta), (unsigned)B, kThreads,
                [&] { superfast_backward_kernel<false>(p); });
    return 0;
}

#ifdef TSAN_MAIN
#include <cstdio>
#include <random>
#include <vector>

int main() {
    std::mt19937 rng(1);
    std::normal_distribution<float> nd(0.f, 1.f);
    auto fill = [&](std::vector<float>& v, float scale, float shift = 0.f) { for (auto& e : v) e = nd(rng) * scale + shift; };
    double s = 0;
    for (int nF : {4, 5}) {   // even nF: frame nF is a pair of its own; odd: it completes the last pair
        const int B = 1, T = nF * 512, C = 4 * 1025;
        std::vector<float> par(B * nF * 4), noise(B * T), dense(B * nF * C), g(B * T), grads(B * nF * C);
        for (int k = 0; k < nF; ++k) {
            par[4 * k] = 0.005f + 0.0001f * k; par[4 * k + 1] = k + 1 < nF ? 0.0001f : 0.f;
            par[4 * k + 2] = 0.1f * k - (int)(0.1f * k); par[4 * k + 3] = 0.f;
        }
        fill(noise, 1.f); fill(dense, 0.3f, -1.f); fill(g, 1.f);
        const float* d = dense.data();
        float* o = grads.data();
        emu_superfast_backward(par.data(), d, d + 1025, d + 2050, d + 3075, C, noise.data(), 1, 0, g.data(), B, nF, 1,
                               o, o + 1025, o + 2050, o + 3075, C);
        emu_superfast_backward(par.data(), d, d + 1025, d + 2050, d + 3075, C, nullptr, 1, 0, g.data(), B, nF, 16,
                               o, o + 1025, o + 2050, o + 3075, C);
        for (float v : grads) s += v;
    }
    std::printf("done %g\n", s);
    return 0;
}
#endif
