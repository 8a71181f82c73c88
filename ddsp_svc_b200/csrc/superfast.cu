// K5: CombSubSuperFast -- comb-tooth source + STFT-domain filtering + iSTFT, fused.
// Replaces ddsp/vocoder.py:639-710 (fast_source_gen, torch.stft x2, complex filters, torch.istft).
//
//   comb  = sinc(rad / (s + 1e-5)), rad = closed-form in-frame phase + wrapped frame advance (fp32)
//   X_q   = STFT(comb), N_q = STFT(noise)     (n_fft = win = 2048, hop = P = 512, periodic Hann,
//                                               center=True, reflect padding)
//   Y_q   = X_q exp(m_h + j pi p_h) + N_q exp(m_n + j pi p_n) / 128        (frame nF reuses nF-1)
//   out   = iSTFT(Y) = OLA(irfft(Y_q) * win) / OLA(win^2), trimmed by n_fft/2
//
// Design (B200).  HBM traffic is dominated by the 4 x 1025 control values per frame (36 B per
// output sample); everything else stays on chip:
//  * one CTA owns a chunk of G consecutive hops of one utterance and walks the G+3 frames that
//    touch them in order, two frames per iteration;
//  * per frame ONE complex 2048-point FFT carries comb + j*noise (both real), split afterwards by
//    conjugate symmetry; per PAIR of frames one inverse FFT returns both real frames
//    (spectrum Ya + j Yb) -> 1.5 FFTs per frame instead of 3;
//  * the FFT is a shared-memory Stockham autosort with radix 16 x 16 x 8 passes (128 threads x 16
//    points in registers), data padded by one slot per 16 so every pass is bank-conflict free,
//    pass twiddles read from per-pass tables laid out along the lane index;
//  * overlap-add happens in a 4096-sample shared-memory ring; a hop is divided by the window
//    envelope and written with 128-bit stores as soon as its 4th frame has been added, so the
//    output is written exactly once and deterministically (no atomics, no workspace round trip).
// The 3 extra frames per chunk are recomputed by the neighbouring CTAs (G = 29 -> 10 %).
// The un-windowed source (comb, noise) of the current frame is kept in shared memory and shifted
// by one hop per frame, so every source sample is evaluated once per CTA (not once per
// overlapping frame); the frame's four control rows are prefetched into registers before the
// forward FFT so their DRAM latency hides behind it.
//
// The reference's fp32 operation order is kept for the source (its in-frame phase is fp32 and the
// sinc argument amplifies rounding by 1/s), the frame scan accumulates in fp64 like torch's CPU
// cumsum.  Noise: explicit N(0,1) samples (parity) or in-kernel Philox + Box-Muller.
#ifndef B2D_HOST_EMU               // tests/emu/ runs the main kernel's source on the CPU (host_emu.h provides the shims)
#include "b2d_common.cuh"
#endif
#include "fft_regs.cuh"

namespace {

constexpr int kN = 2048, kHalf = 1024, kThreads = 128;
constexpr int kPadN = kN + kN / 16;  // padded complex buffer length
constexpr int kRingHops = 6;            // OLA ring: 6 hops of 512 (5 are live at any time)
constexpr int kHop = 512;
constexpr int kScanThreads = 256;

__device__ __forceinline__ int padi(int i) { return i + (i >> 4); }

#ifndef B2D_HOST_EMU               // warp shuffles: not emulated (the test computes its output with numpy)
// ---- frame scan: per-frame (s, ds, acc_prev) and phase_frames  (vocoder.py:641-650) ----------
__global__ void __launch_bounds__(kScanThreads)
superfast_scan_kernel(const float* __restrict__ f0, int nF, int P, float sr, float4* __restrict__ frame_par,
                      float* __restrict__ phase_frames) {
    const int b = blockIdx.x;
    const float* f = f0 + (size_t)b * nF;
    const int per = (nF + kScanThreads - 1) / kScanThreads;
    const int k0 = min(nF, (int)threadIdx.x * per), k1 = min(nF, k0 + per);
    const float fP = (float)P, fPm1 = (float)(P - 1);
    auto s_of = [&](int k) { return __fdiv_rn(f[k], sr); };
    auto ds_of = [&](int k) { return (k + 1 < nF) ? __fsub_rn(s_of(k + 1), s_of(k)) : 0.0f; };
    auto adv = [&](int k) {
        // rad[k, P-1] = s*P + ((0.5*ds)*(P-1))*P / P
        const float t1 = __fmul_rn(s_of(k), fP);
        float t2 = __fmul_rn(__fmul_rn(__fmul_rn(0.5f, ds_of(k)), fPm1), fP);
        t2 = __fdiv_rn(t2, fP);
        const float last = __fadd_rn(t1, t2);
        return __fsub_rn(fmodf(__fadd_rn(last, 0.5f), 1.0f), 0.5f);
    };
    double local = 0.0;
    for (int k = k0; k < k1; ++k) local += (double)adv(k);
    __shared__ double warp_tot[kScanThreads / 32];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    double incl = local;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        double up = __shfl_up_sync(0xffffffffu, incl, d);
        if (lane >= d) incl += up;
    }
    if (lane == 31) warp_tot[warp] = incl;
    __syncthreads();
    double run = incl - local;
    for (int w = 0; w < warp; ++w) run += warp_tot[w];
    for (int k = k0; k < k1; ++k) {
        const float accp = (k == 0) ? 0.0f : fmodf((float)run, 1.0f);
        const float s = s_of(k);
        frame_par[(size_t)b * nF + k] = make_float4(s, ds_of(k), accp, 0.f);
        float rad0 = __fadd_rn(s, accp);   // rad[k,0] = s*1 + 0 + acc_prev
        rad0 = __fsub_rn(rad0, rintf(rad0));
        phase_frames[(size_t)b * nF + k] = __fmul_rn(B2D_TWO_PI_F, rad0);
        run += (double)adv(k);
    }
}

#endif

using namespace b2d_fft;   // cadd / csub / cmul / Dft<R>: register DFTs shared with combsubfast.cu

// One Stockham pass of radix R over the padded buffer (in place: all reads, barrier, all writes).
//   butterfly j: v[r] = buf[j + r N/R] * tw[r][j % Ns];  DFT_R;  buf[(j/Ns) Ns R + j%Ns + r Ns] = v[r]
// Padded positions are affine in r for all three passes (padi(i) = i + i/16):
//   reads : padi(j + r N/R)           = padi(j) + r (N/R + N/R/16)
//   writes: NS = 1   -> 17 j + r ;  NS = 16 -> (j/16) 272 + j%16 + 17 r ;  NS = 256 -> padi(j) + 272 r
// TW: 0 none (first pass), 1 full table [R-1][NS], 2 powers of tw[k] (= exp(-2 pi i k / (NS R)))
template <int R, int NS, int TW, bool PK>
__device__ __forceinline__ void fft_pass(float2* buf, const float2* __restrict__ tw, int tid) {
    constexpr int NB = kN / R;               // butterflies
    constexpr int PER = NB / kThreads;       // per thread (1 for R=16, 2 for R=8)
    constexpr int RS = NB + NB / 16;         // read stride in padded slots
    float2 v[PER][R];
#pragma unroll
    for (int u = 0; u < PER; ++u) {
        const int j = tid + u * kThreads;
        const int k = j % NS;
        const float2* src = buf + padi(j);
#pragma unroll
        for (int r = 0; r < R; ++r) v[u][r] = src[r * RS];
        if (TW == 1) {
#pragma unroll
            for (int r = 1; r < R; ++r) v[u][r] = cmul(v[u][r], tw[(r - 1) * NS + k]);
        } else if (TW == 2) {
            const float2 w1 = tw[k];
            const float2 w2 = cmul(w1, w1), w3 = cmul(w2, w1), w4 = cmul(w2, w2);
            v[u][1] = cmul(v[u][1], w1); v[u][2] = cmul(v[u][2], w2);
            v[u][3] = cmul(v[u][3], w3); v[u][4] = cmul(v[u][4], w4);
            if (R > 5) {
                const float2 w5 = cmul(w4, w1), w6 = cmul(w4, w2), w7 = cmul(w4, w3);
                v[u][5] = cmul(v[u][5], w5); v[u][6] = cmul(v[u][6], w6); v[u][7] = cmul(v[u][7], w7);
            }
        }
        Dft<R, PK>::run(v[u]);
    }
    __syncthreads();
#pragma unroll
    for (int u = 0; u < PER; ++u) {
        const int j = tid + u * kThreads;
        float2* dst;
        int ws;
        if (NS == 1) { dst = buf + 17 * j; ws = 1; }
        else if (NS == 16) { dst = buf + (j >> 4) * 272 + (j & 15); ws = 17; }
        else { dst = buf + padi(j); ws = 272; }
#pragma unroll
        for (int r = 0; r < R; ++r) dst[r * ws] = v[u][r];
    }
    __syncthreads();
}

template <bool PK>
__device__ __forceinline__ void fft2048(float2* buf, const float2* tw2, const float2* tw3, int tid) {
    fft_pass<16, 1, 0, PK>(buf, nullptr, tid);
    fft_pass<16, 16, 1, PK>(buf, tw2, tid);
    fft_pass<8, 256, 2, PK>(buf, tw3, tid);
}

struct SfParams {
    const float* f0;           // unused in the main kernel (frame_par carries s, ds, acc)
    const float4* frame_par;   // [B, nF]
    const float* c_hm; const float* c_hp; const float* c_nm; const float* c_np;
    long long ctrl_stride;
    const float* noise_in;     // [B, T] or nullptr
    float* out;                // [B, T]
    int nF, P, G;
    unsigned long long seed;
    long long utt_off;
};

// sinc(z) = sin(pi z)/(pi z).  |pi z| reaches ~1e3 rad, so the argument is reduced in turns
// (exactly: z - 2 rint(z/2)) and the SFU evaluates sin(pi r); for |pi z| < 1 an even polynomial
// avoids the SFU's absolute error being divided by a small number.
__device__ __forceinline__ float sinc_f32(float z) {
    const float pz = __fmul_rn(B2D_PI_F, z);
    const float p2 = pz * pz;
    // 1 - x^2/6 + x^4/120 - x^6/5040 + x^8/362880 - x^10/39916800
    float poly = fmaf(p2, -2.5052108e-8f, 2.7557319e-6f);
    poly = fmaf(p2, poly, -1.9841270e-4f);
    poly = fmaf(p2, poly, 8.3333333e-3f);
    poly = fmaf(p2, poly, -1.6666667e-1f);
    poly = fmaf(p2, poly, 1.0f);
    const float r = fmaf(-2.0f, rintf(0.5f * z), z);          // z mod 2 in [-1, 1], exact
    const float big = __fdividef(__sinf(B2D_PI_F * r), pz);
    return (p2 < 1.0f) ? poly : big;
}

__device__ __forceinline__ float comb_at(const float4* __restrict__ fp, int P, float fP, int m) {
    const int k = m >> 9, j = m & (kHop - 1);            // P = 512 (checked on the host)
    const float4 q = __ldg(fp + k);                      // (s, ds, acc_prev)
    const float fj = (float)j, fj1 = (float)(j + 1);
    const float t1 = __fmul_rn(q.x, fj1);
    float t2 = __fmul_rn(__fmul_rn(__fmul_rn(0.5f, q.y), fj), fj1);
    t2 = __fmul_rn(t2, 1.0f / 512.0f);                   // == t2 / P exactly (power of two)
    float rad = __fadd_rn(__fadd_rn(t1, t2), q.z);       // (:643,647)
    rad = __fsub_rn(rad, rintf(rad));                     // (:648)
    const float sup = __fadd_rn(q.x, __fmul_rn(__fmul_rn(q.y, fj), 1.0f / 512.0f));   // (:644)
    return sinc_f32(__fdiv_rn(rad, __fadd_rn(sup, 1e-5f)));                // (:649)
}

__device__ __forceinline__ float4 normals4(unsigned long long seed, unsigned long long utt, uint32_t quad) {
    uint4 r = b2d::philox4x32_10(make_uint4(quad, 0x5f5f5f5fu, (uint32_t)utt, (uint32_t)(utt >> 32)),
                                 make_uint2((uint32_t)seed, (uint32_t)(seed >> 32)));
    const float u1 = ((float)(r.x >> 8) + 1.0f) * (1.0f / 16777216.0f);
    const float u2 = (float)(r.y >> 8) * (1.0f / 16777216.0f);
    const float u3 = ((float)(r.z >> 8) + 1.0f) * (1.0f / 16777216.0f);
    const float u4 = (float)(r.w >> 8) * (1.0f / 16777216.0f);
    const float m1 = sqrtf(-2.0f * __logf(u1)), m2 = sqrtf(-2.0f * __logf(u3));
    float s1, c1, s2, c2;
    __sincosf(B2D_TWO_PI_F * u2, &s1, &c1);
    __sincosf(B2D_TWO_PI_F * u4, &s2, &c2);
    return make_float4(m1 * c1, m1 * s1, m2 * c2, m2 * s2);
}

// periodic Hann (first half, win[i] = win[2048 - i]) and the pass twiddles of fft2048
__device__ __forceinline__ void init_tables(float* winh, float2* tw2, float2* tw3, int tid) {
    for (int i = tid; i <= kHalf; i += kThreads) winh[i] = 0.5f - 0.5f * cospif((float)i * (2.0f / kN));
    for (int i = tid; i < 15 * 16; i += kThreads) {
        const int r = i / 16 + 1, k = i % 16;
        float sn, cs; sincospif(-2.0f * (float)(r * k) / 256.0f, &sn, &cs);
        tw2[i] = make_float2(cs, sn);
    }
    for (int i = tid; i < 256; i += kThreads) {
        float sn, cs; sincospif(-2.0f * (float)i / 2048.0f, &sn, &cs);
        tw3[i] = make_float2(cs, sn);
    }
}

__device__ __forceinline__ float win_of(const float* winh, int i) { return winh[i <= kHalf ? i : kN - i]; }

// iSTFT envelope OLA(win^2) over the frames q = 0..nF that exist, at sample i (0 <= i < 512) of hop h
__device__ __forceinline__ float ola_env(const float* winh, int h, int i, int nF) {
    float env = 0.f;
#pragma unroll
    for (int d = -1; d <= 2; ++d) {
        const int qq = h + d;
        if (qq >= 0 && qq <= nF) { const float w = win_of(winh, i - d * kHop + kHalf); env = fmaf(w, w, env); }
    }
    return env;
}

// un-windowed source (comb, noise) of absolute positions [mstart + i_lo, mstart + i_hi) -> src ring slots
// (i + off) & 2047; positions outside [0, T) follow the STFT's padding (reflect, or zeros when T <= 1024)
__device__ __forceinline__ void fill_source(float2* src, const float4* __restrict__ fpar, const float* noise_row,
                                            unsigned long long seed, unsigned long long utt, int T, int P,
                                            int mstart, int off, int i_lo, int i_hi, int tid) {
    const float fP = (float)P;
    const bool reflect = T > kHalf;                              // pad_mode (:672-675)
#pragma unroll 1
    for (int i0 = i_lo + (tid << 2); i0 < i_hi; i0 += kThreads << 2) {
        const int m0 = mstart + i0;
        float cv[4], nv[4];
        if (m0 >= 0 && m0 + 3 < T) {
            float4 nz;
            if (noise_row) nz = __ldg(reinterpret_cast<const float4*>(noise_row + m0));   // m0 % 4 == 0
            else nz = normals4(seed, utt, (uint32_t)(m0 >> 2));
            nv[0] = nz.x; nv[1] = nz.y; nv[2] = nz.z; nv[3] = nz.w;
#pragma unroll
            for (int e = 0; e < 4; ++e) cv[e] = comb_at(fpar, P, fP, m0 + e);
        } else {
#pragma unroll 1
            for (int e = 0; e < 4; ++e) {
                int m = m0 + e;
                bool valid = true;
                if (m < 0 || m >= T) {
                    if (reflect) m = (m < 0) ? -m : 2 * (T - 1) - m;
                    else valid = false;
                }
                cv[e] = 0.f; nv[e] = 0.f;
                if (valid) {
                    cv[e] = comb_at(fpar, P, fP, m);
                    if (noise_row) nv[e] = noise_row[m];
                    else {
                        const float4 g = normals4(seed, utt, (uint32_t)(m >> 2));
                        const int l = m & 3;
                        nv[e] = l == 0 ? g.x : l == 1 ? g.y : l == 2 ? g.z : g.w;
                    }
                }
            }
        }
#pragma unroll
        for (int e = 0; e < 4; ++e) src[(i0 + e + off) & (kN - 1)] = make_float2(cv[e], nv[e]);
    }
}

// shared-memory footprint (bytes): 2 x 17408 (bufA, bufS) + 16384 (src) + 12288 (ring) + 4112 (win)
// + 1920 (tw2) + 2048 (tw3) = 71568  -> 3 CTAs per SM
constexpr int kWinLen = kHalf + 4;   // window stored for i in [0, 1024]; win[i] = win[2048 - i]
constexpr size_t kSmemBytes = (size_t)2 * kPadN * sizeof(float2) + (size_t)kN * sizeof(float2) +
                              (size_t)kRingHops * kHop * sizeof(float) + (size_t)kWinLen * sizeof(float) +
                              (size_t)(15 * 16 + 256) * sizeof(float2);

// PK: complex additions of the FFT butterflies as packed f32x2 instructions (fft_regs.cuh Ar<true>)
template <bool PK>
__global__ void __launch_bounds__(kThreads, 3) superfast_kernel(SfParams p) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    float2* bufA = reinterpret_cast<float2*>(smem_raw);          // [kPadN] frame time/frequency data
    float2* bufS = bufA + kPadN;                                 // [kPadN] pair spectrum / pair output
    float2* src = bufS + kPadN;                                  // [kN]   un-windowed (comb, noise), ring-indexed
    float2* tw2 = src + kN;                                      // [15][16]  exp(-2 pi i r k / 256)
    float2* tw3 = tw2 + 15 * 16;                                 // [256]     exp(-2 pi i k / 2048)
    float* ring = reinterpret_cast<float*>(tw3 + 256);           // [6][512]  overlap-add
    float* winh = ring + kRingHops * kHop;                       // [1025]    periodic Hann, first half

    const int tid = threadIdx.x;
    const int b = blockIdx.y;
    const int nF = p.nF, P = p.P, T = nF * P;
    const int h0 = blockIdx.x * p.G, h1 = min(h0 + p.G, nF);
    const float4* fpar = p.frame_par + (size_t)b * nF;
    const float* noise_row = p.noise_in ? p.noise_in + (size_t)b * T : nullptr;
    const unsigned long long utt = (unsigned long long)(p.utt_off + b);

    // ---- one-time tables ----
    init_tables(winh, tw2, tw3, tid);
    for (int i = tid; i < kRingHops * kHop; i += kThreads) ring[i] = 0.f;
    __syncthreads();
    auto win_at = [&](int i) { return win_of(winh, i); };
    auto fill_src = [&](int mstart, int off, int i_lo, int i_hi) {
        fill_source(src, fpar, noise_row, p.seed, utt, T, P, mstart, off, i_lo, i_hi, tid);
    };

    const int qs = max(h0 - 1, 0), qe = min(h1 + 1, nF);
    int off = 0;            // src ring offset of the current frame's sample 0
    bool primed = false;

    for (int qa = qs; qa <= qe; qa += 2) {
        const int qb = qa + 1;
        const bool has_b = qb <= qe;
#pragma unroll 1
        for (int which = 0; which < 2; ++which) {
            if (which == 1 && !has_b) break;
            const int q = which ? qb : qa;
            const int mstart = q * P - kHalf;
            // ---- source: first frame of the CTA evaluates 2048 samples, later frames only the new hop ----
            if (!primed) { fill_src(mstart, off, 0, kN); primed = true; }
            else { off = (off + kHop) & (kN - 1); fill_src(mstart, off, kN - kHop, kN); }
            __syncthreads();
            // ---- windowed complex frame z[i] = win[i] * (comb + j noise) ----
#pragma unroll 4
            for (int i = tid; i < kN; i += kThreads) {
                const float2 v = src[(i + off) & (kN - 1)];
                const float w = win_at(i);
                bufA[padi(i)] = make_float2(w * v.x, w * v.y);
            }
            // ---- prefetch this frame's controls (bins tid + 128 it, and bin 1024 on thread 0) ----
            const int qc = min(q, nF - 1);
            const size_t crow = ((size_t)b * nF + qc) * p.ctrl_stride;
            float chm[9], chp[9], cnm[9], cnp[9];
#pragma unroll
            for (int it = 0; it < 8; ++it) {
                const size_t o = crow + tid + it * kThreads;
                chm[it] = __ldg(p.c_hm + o); chp[it] = __ldg(p.c_hp + o);
                cnm[it] = __ldg(p.c_nm + o); cnp[it] = __ldg(p.c_np + o);
            }
            chm[8] = chp[8] = cnm[8] = cnp[8] = 0.f;
            if (tid == 0) {
                chm[8] = __ldg(p.c_hm + crow + kHalf); chp[8] = __ldg(p.c_hp + crow + kHalf);
                cnm[8] = __ldg(p.c_nm + crow + kHalf); cnp[8] = __ldg(p.c_np + crow + kHalf);
            }
            __syncthreads();
            fft2048<PK>(bufA, tw2, tw3, tid);
            // ---- split comb/noise spectra, apply the filters, accumulate the pair spectrum ----
#pragma unroll
            for (int it = 0; it < 9; ++it) {
                const int bin = (it < 8) ? tid + it * kThreads : kHalf;
                if (it == 8 && tid != 0) break;
                const float2 za = bufA[padi(bin)];
                float2 zb = bufA[padi((kN - bin) & (kN - 1))];
                zb.y = -zb.y;                                                   // conj
                const float2 X = make_float2(0.5f * (za.x + zb.x), 0.5f * (za.y + zb.y));
                const float2 d = csub(za, zb);
                const float2 Nz = make_float2(0.5f * d.y, -0.5f * d.x);
                float sh, ch, sn, cn;
                __sincosf(B2D_PI_F * chp[it], &sh, &ch);
                __sincosf(B2D_PI_F * cnp[it], &sn, &cn);
                const float eh = __expf(chm[it]), en = __expf(cnm[it]) * 0.0078125f;   // /128 (:668)
                const float2 Hs = make_float2(eh * ch, eh * sh);                 // exp(m + j pi p)  (:666)
                const float2 Hn = make_float2(en * cn, en * sn);
                float2 Y = cadd(cmul(X, Hs), cmul(Nz, Hn));                      // (:699)
                if (bin == 0 || bin == kHalf) Y.y = 0.f;                         // irfft ignores Im of DC / Nyquist
                // pair spectrum S = Ya + j Yb with Hermitian extension, stored re/im SWAPPED so that a
                // forward FFT of the buffer yields the (swapped) inverse transform
                const int mir = (kN - bin) & (kN - 1);
                if (which == 0) {
                    bufS[padi(bin)] = make_float2(Y.y, Y.x);
                    if (bin != 0 && bin != kHalf) bufS[padi(mir)] = make_float2(-Y.y, Y.x);
                } else {
                    float2 s0 = bufS[padi(bin)];
                    s0.x += Y.x; s0.y -= Y.y;                                    // += j*Y       (swapped)
                    bufS[padi(bin)] = s0;
                    if (bin != 0 && bin != kHalf) {
                        float2 s1 = bufS[padi(mir)];
                        s1.x += Y.x; s1.y += Y.y;                                // += j*conj(Y) (swapped)
                        bufS[padi(mir)] = s1;
                    }
                }
            }
            __syncthreads();
        }
        // ---- inverse transform of the pair, windowed overlap-add into the ring ----
        fft2048<PK>(bufS, tw2, tw3, tid);
        const float inv_n = 1.0f / (float)kN;
        int hslot[5];       // ring slot (x512) of hops qa-2 .. qa+2
#pragma unroll
        for (int t = 0; t < 5; ++t) hslot[t] = ((qa - 2 + t + 6 * 1024) % kRingHops) * kHop;
#pragma unroll 4
        for (int i = tid; i < kN; i += kThreads) {
            const float2 sv = bufS[padi(i)];       // swapped: (im, re)
            const float w = win_at(i) * inv_n;
            const int hi = i >> 9, lo = i & (kHop - 1);
            ring[hslot[hi] + lo] += sv.y * w;
            if (has_b) ring[hslot[hi + 1] + lo] += sv.x * w;
        }
        __syncthreads();
        // ---- hops whose 4 frames are in: qa-2, qa-1; at the last pair everything up to h1-1 ----
        const int last = has_b ? qb : qa;
        const int h_hi = (last >= qe) ? max(h1 - 1, qa - 1) : qa - 1;
        for (int h = qa - 2; h <= h_hi; ++h) {
            const bool owned = h >= h0 && h < h1;
            float* rrow = ring + ((h + 6 * 1024) % kRingHops) * kHop;
            const int i4 = tid << 2;               // 128 threads x 4 samples = one hop
            const float4 acc = *reinterpret_cast<const float4*>(rrow + i4);
            *reinterpret_cast<float4*>(rrow + i4) = make_float4(0.f, 0.f, 0.f, 0.f);
            if (owned) {
                const int n = h * P + i4;
                float v[4] = {acc.x, acc.y, acc.z, acc.w};
#pragma unroll
                for (int e = 0; e < 4; ++e) v[e] = __fdiv_rn(v[e], ola_env(winh, h, i4 + e, nF));
                b2d::st_global_v4(p.out + (size_t)b * T + n, make_float4(v[0], v[1], v[2], v[3]));
            }
        }
        __syncthreads();
    }
}

// ---- backward: gradients of the four controls from g = dL/dsignal ---------------------------------------
// Adjoint of trim, envelope division, OLA and synthesis window:  u_q[i] = w[i] g[n] / env(n), n = qP - 1024 + i
// (0 outside [0, T));  adjoint of irfft:  G_q[k] = (c_k / N) FFT(u_q)[k], c_0 = c_1024 = 1, else 2.
// With the recomputed filtered spectra Yh = X exp(m_h + j pi p_h), Yn = Z exp(m_n + j pi p_n) / 128 of frame q:
//   dL/dm = Re(conj(G) Y),   dL/dp = pi Im(G conj(Y))          (row min(q, nF-1); frame nF folds into row nF-1)
// Frames are independent (no overlap-add), so a CTA walks a run of frame PAIRS (2m, 2m+1) with no halo:
//  * per pair ONE complex FFT of u_2m + j u_2m+1, split by conjugate symmetry into both frames' G;
//  * per frame ONE complex FFT of w (comb + j noise), split the same way (the forward's source, recomputed from
//    the frame parameters and the noise stream, so nothing but the controls is kept for the backward);
//  * g / env is kept in a ring indexed by sample position, like the source; each pair adds 1024 new samples.
// The pairing does not depend on the chunking, and every gradient row is written once by the CTA that owns it,
// so the result is bit-identical for every chunk size, batch split and utterance_offset shard.
struct SfBwdParams {
    const float4* frame_par;   // [B, nF]
    const float* c_hm; const float* c_hp; const float* c_nm; const float* c_np;
    long long ctrl_stride;
    const float* noise_in;     // [B, T] or nullptr
    const float* grad;         // [B, T]
    float* g_hm; float* g_hp; float* g_nm; float* g_np;
    long long grad_stride;
    int nF, P, GP;             // GP: frame pairs per CTA
    unsigned long long seed;
    long long utt_off;
};

constexpr int kGRing = 4096;   // g / env ring (a pair reads 2560 consecutive samples)
// 2 x 17408 (bufA, bufS) + 16384 (src) + 16384 (g ring) + 4112 (win) + 1920 (tw2) + 2048 (tw3) = 75664 -> 3 CTAs/SM
constexpr size_t kBwdSmemBytes = (size_t)2 * kPadN * sizeof(float2) + (size_t)kN * sizeof(float2) +
                                 (size_t)kGRing * sizeof(float) + (size_t)kWinLen * sizeof(float) +
                                 (size_t)(15 * 16 + 256) * sizeof(float2);

template <bool PK>
__global__ void __launch_bounds__(kThreads, 3) superfast_backward_kernel(SfBwdParams p) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    float2* bufA = reinterpret_cast<float2*>(smem_raw);          // [kPadN] source frame / its spectrum
    float2* bufS = bufA + kPadN;                                 // [kPadN] u pair / its spectrum
    float2* src = bufS + kPadN;                                  // [kN]   un-windowed (comb, noise), ring-indexed
    float2* tw2 = src + kN;
    float2* tw3 = tw2 + 15 * 16;
    float* gring = reinterpret_cast<float*>(tw3 + 256);          // [4096] g / env by sample position
    float* winh = gring + kGRing;                                // [1025]

    const int tid = threadIdx.x;
    const int b = blockIdx.y;
    const int nF = p.nF, P = p.P, T = nF * P;
    const int n_pairs = (nF + 1) / 2;                            // pairs of gradient rows 0..nF-1
    const int m0 = blockIdx.x * p.GP, m1 = min(m0 + p.GP, n_pairs);
    const int qe = (m1 == n_pairs) ? nF + 1 : 2 * m1;            // frames [2 m0, qe): the last CTA adds frame nF
    const float4* fpar = p.frame_par + (size_t)b * nF;
    const float* noise_row = p.noise_in ? p.noise_in + (size_t)b * T : nullptr;
    const float* grow = p.grad + (size_t)b * T;
    const unsigned long long utt = (unsigned long long)(p.utt_off + b);

    init_tables(winh, tw2, tw3, tid);
    __syncthreads();

    float keep[4][9];      // row nF-1 of frame nF-1, added to frame nF's in registers before the one store
    int off = 0;
    bool primed = false;
    for (int qa = 2 * m0; qa < qe; qa += 2) {
        const int qb = qa + 1;
        const bool has_b = qb < qe;
        const int n0 = qa * P - kHalf;                           // first sample of frame qa
        // ---- g / env of samples [n0, n0 + 2560): the first pair fills all, later pairs the 1024 new ones ----
        for (int n = (qa == 2 * m0 ? n0 : n0 + 3 * kHop) + tid; n < n0 + 5 * kHop; n += kThreads) {
            float v = 0.f;
            if (n >= 0 && n < T) v = __fdiv_rn(__ldg(grow + n), ola_env(winh, n >> 9, n & (kHop - 1), nF));
            gring[n & (kGRing - 1)] = v;
        }
        __syncthreads();
        // ---- u pair = w (g/env)[frame qa] + j w (g/env)[frame qb] ----
#pragma unroll 4
        for (int i = tid; i < kN; i += kThreads) {
            const float w = win_of(winh, i);
            const float ua = w * gring[(n0 + i) & (kGRing - 1)];
            const float ub = has_b ? w * gring[(n0 + kHop + i) & (kGRing - 1)] : 0.f;
            bufS[padi(i)] = make_float2(ua, ub);
        }
        __syncthreads();
        fft2048<PK>(bufS, tw2, tw3, tid);
#pragma unroll 1
        for (int which = 0; which < 2; ++which) {
            if (which == 1 && !has_b) break;
            const int q = which ? qb : qa;
            const int mstart = q * P - kHalf;
            if (!primed) { fill_source(src, fpar, noise_row, p.seed, utt, T, P, mstart, off, 0, kN, tid); primed = true; }
            else { off = (off + kHop) & (kN - 1); fill_source(src, fpar, noise_row, p.seed, utt, T, P, mstart, off, kN - kHop, kN, tid); }
            __syncthreads();
#pragma unroll 4
            for (int i = tid; i < kN; i += kThreads) {
                const float2 v = src[(i + off) & (kN - 1)];
                const float w = win_of(winh, i);
                bufA[padi(i)] = make_float2(w * v.x, w * v.y);
            }
            const int qc = min(q, nF - 1);
            const size_t crow = ((size_t)b * nF + qc) * p.ctrl_stride;
            float chm[9], chp[9], cnm[9], cnp[9];
#pragma unroll
            for (int it = 0; it < 8; ++it) {
                const size_t o = crow + tid + it * kThreads;
                chm[it] = __ldg(p.c_hm + o); chp[it] = __ldg(p.c_hp + o);
                cnm[it] = __ldg(p.c_nm + o); cnp[it] = __ldg(p.c_np + o);
            }
            chm[8] = chp[8] = cnm[8] = cnp[8] = 0.f;
            if (tid == 0) {
                chm[8] = __ldg(p.c_hm + crow + kHalf); chp[8] = __ldg(p.c_hp + crow + kHalf);
                cnm[8] = __ldg(p.c_nm + crow + kHalf); cnp[8] = __ldg(p.c_np + crow + kHalf);
            }
            __syncthreads();
            fft2048<PK>(bufA, tw2, tw3, tid);
            const size_t grow_out = ((size_t)b * nF + qc) * p.grad_stride;
#pragma unroll
            for (int it = 0; it < 9; ++it) {
                const int bin = (it < 8) ? tid + it * kThreads : kHalf;
                if (it == 8 && tid != 0) break;
                const int mir = (kN - bin) & (kN - 1);
                // comb / noise spectra of this frame
                const float2 za = bufA[padi(bin)];
                float2 zb = bufA[padi(mir)];
                zb.y = -zb.y;
                const float2 X = make_float2(0.5f * (za.x + zb.x), 0.5f * (za.y + zb.y));
                const float2 d = csub(za, zb);
                const float2 Nz = make_float2(0.5f * d.y, -0.5f * d.x);
                // this frame's half of the u-pair spectrum, scaled by c_k / N
                const float2 sa = bufS[padi(bin)];
                float2 sb = bufS[padi(mir)];
                sb.y = -sb.y;
                const float c = (bin == 0 || bin == kHalf) ? (1.0f / kN) : (2.0f / kN);
                float2 G;
                if (which == 0) G = make_float2(0.5f * c * (sa.x + sb.x), 0.5f * c * (sa.y + sb.y));
                else G = make_float2(0.5f * c * (sa.y - sb.y), -0.5f * c * (sa.x - sb.x));
                float sh, ch, sn, cn;
                __sincosf(B2D_PI_F * chp[it], &sh, &ch);
                __sincosf(B2D_PI_F * cnp[it], &sn, &cn);
                const float eh = __expf(chm[it]), en = __expf(cnm[it]) * 0.0078125f;
                const float2 Yh = cmul(X, make_float2(eh * ch, eh * sh));
                const float2 Yn = cmul(Nz, make_float2(en * cn, en * sn));
                float gr[4] = {G.x * Yh.x + G.y * Yh.y, B2D_PI_F * (G.y * Yh.x - G.x * Yh.y),
                               G.x * Yn.x + G.y * Yn.y, B2D_PI_F * (G.y * Yn.x - G.x * Yn.y)};
                if (q == nF - 1) {
#pragma unroll
                    for (int t = 0; t < 4; ++t) keep[t][it] = gr[t];
                    continue;
                }
                if (q == nF) {
#pragma unroll
                    for (int t = 0; t < 4; ++t) gr[t] = keep[t][it] + gr[t];
                }
                const size_t o = grow_out + bin;
                p.g_hm[o] = gr[0]; p.g_hp[o] = gr[1]; p.g_nm[o] = gr[2]; p.g_np[o] = gr[3];
            }
            __syncthreads();
        }
    }
}

}  // namespace

#ifndef B2D_HOST_EMU
extern "C" size_t b2d_superfast_workspace_bytes(int B, int n_frames) {
    if (B <= 0 || n_frames <= 0) return 0;
    return (size_t)B * n_frames * sizeof(float4);
}

extern "C" int b2d_superfast_scan(const float* f0_frames, int B, int n_frames, int block, double sampling_rate,
                                  void* workspace, float* phase_frames, void* stream) {
    if (!f0_frames || !workspace || !phase_frames) return b2d::fail(B2D_ERR_NULL, "superfast_scan: null pointer");
    if (B <= 0 || n_frames <= 0 || block <= 0) return b2d::fail(B2D_ERR_SHAPE, "superfast_scan: bad shape");
    if (!b2d::aligned16(workspace)) return b2d::fail(B2D_ERR_ALIGN, "superfast_scan: workspace must be 16-byte aligned");
    superfast_scan_kernel<<<B, kScanThreads, 0, (cudaStream_t)stream>>>(
        f0_frames, n_frames, block, (float)sampling_rate, static_cast<float4*>(workspace), phase_frames);
    return b2d::check_launch("superfast_scan");
}

extern "C" int b2d_superfast_synth(const void* workspace, const float* c_harmonic_magnitude,
                                   const float* c_harmonic_phase, const float* c_noise_magnitude,
                                   const float* c_noise_phase, int64_t ctrl_stride, const float* noise_in,
                                   uint64_t seed, int64_t utterance_offset, int B, int n_frames, int block,
                                   int win_length, float* signal, void* stream) {
    if (!workspace || !c_harmonic_magnitude || !c_harmonic_phase || !c_noise_magnitude || !c_noise_phase || !signal)
        return b2d::fail(B2D_ERR_NULL, "superfast_synth: null pointer");
    if (B <= 0 || n_frames <= 0 || block <= 0 || ctrl_stride < win_length / 2 + 1)
        return b2d::fail(B2D_ERR_SHAPE, "superfast_synth: bad shape");
    if (win_length != kN || block != 512)
        return b2d::fail(B2D_ERR_UNSUPPORTED, "superfast_synth: only win_length=2048 / block_size=512 (configs/combsub.yaml) "
                         "is implemented (got %d / %d)", win_length, block);
    if (B > 65535) return b2d::fail(B2D_ERR_UNSUPPORTED, "superfast_synth: batch %d > 65535", B);
    if (!b2d::aligned16(signal) || !b2d::aligned16(workspace) || (noise_in && !b2d::aligned16(noise_in)))
        return b2d::fail(B2D_ERR_ALIGN, "superfast_synth: signal / noise_in / workspace must be 16-byte aligned");
    SfParams p;
    p.f0 = nullptr; p.frame_par = static_cast<const float4*>(workspace);
    p.c_hm = c_harmonic_magnitude; p.c_hp = c_harmonic_phase; p.c_nm = c_noise_magnitude; p.c_np = c_noise_phase;
    p.ctrl_stride = ctrl_stride; p.noise_in = noise_in; p.out = signal;
    p.nF = n_frames; p.P = block;
    // chunk length: G+3 frames are transformed for G hops; keep >= ~4 CTAs per SM when the work allows
    int G = 29;
    while (G > 5 && (long long)B * ((n_frames + G - 1) / G) < 4 * 148) G -= 4;
    p.G = G;
    p.seed = seed; p.utt_off = utterance_offset;
    const size_t smem = kSmemBytes;
    auto go = [&](auto kern) -> int {
        cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) return b2d::fail((int)e, "superfast_synth: smem attr: %s", cudaGetErrorString(e));
        cudaFuncSetAttribute(kern, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared);
        kern<<<dim3((n_frames + G - 1) / G, B), kThreads, smem, (cudaStream_t)stream>>>(p);
        return 0;
    };
    const int rc = b2d::g_fft_packed.load(std::memory_order_relaxed) ? go(superfast_kernel<true>) : go(superfast_kernel<false>);
    if (rc) return rc;
    return b2d::check_launch("superfast_synth");
}

extern "C" int b2d_superfast_backward(const void* workspace, const float* c_harmonic_magnitude,
                                      const float* c_harmonic_phase, const float* c_noise_magnitude,
                                      const float* c_noise_phase, int64_t ctrl_stride, const float* noise_in,
                                      uint64_t seed, int64_t utterance_offset, const float* grad_signal, int B,
                                      int n_frames, int block, int win_length, float* g_harmonic_magnitude,
                                      float* g_harmonic_phase, float* g_noise_magnitude, float* g_noise_phase,
                                      int64_t grad_stride, void* stream) {
    if (!workspace || !c_harmonic_magnitude || !c_harmonic_phase || !c_noise_magnitude || !c_noise_phase ||
        !grad_signal || !g_harmonic_magnitude || !g_harmonic_phase || !g_noise_magnitude || !g_noise_phase)
        return b2d::fail(B2D_ERR_NULL, "superfast_backward: null pointer");
    if (B <= 0 || n_frames <= 0 || block <= 0 || ctrl_stride < win_length / 2 + 1 || grad_stride < win_length / 2 + 1)
        return b2d::fail(B2D_ERR_SHAPE, "superfast_backward: bad shape");
    if (win_length != kN || block != 512)
        return b2d::fail(B2D_ERR_UNSUPPORTED, "superfast_backward: only win_length=2048 / block_size=512 is implemented "
                         "(got %d / %d)", win_length, block);
    if (B > 65535) return b2d::fail(B2D_ERR_UNSUPPORTED, "superfast_backward: batch %d > 65535", B);
    if (!b2d::aligned16(workspace) || (noise_in && !b2d::aligned16(noise_in)))
        return b2d::fail(B2D_ERR_ALIGN, "superfast_backward: noise_in / workspace must be 16-byte aligned");
    SfBwdParams p;
    p.frame_par = static_cast<const float4*>(workspace);
    p.c_hm = c_harmonic_magnitude; p.c_hp = c_harmonic_phase; p.c_nm = c_noise_magnitude; p.c_np = c_noise_phase;
    p.ctrl_stride = ctrl_stride; p.noise_in = noise_in; p.grad = grad_signal;
    p.g_hm = g_harmonic_magnitude; p.g_hp = g_harmonic_phase; p.g_nm = g_noise_magnitude; p.g_np = g_noise_phase;
    p.grad_stride = grad_stride;
    p.nF = n_frames; p.P = block;
    // frame pairs per CTA: no halo to amortise, so shrink the chunk until there are >= ~4 CTAs per SM
    const int n_pairs = (n_frames + 1) / 2;
    int GP = 16;
    while (GP > 2 && (long long)B * ((n_pairs + GP - 1) / GP) < 4 * 148) GP -= 2;
    p.GP = GP;
    p.seed = seed; p.utt_off = utterance_offset;
    auto go = [&](auto kern) -> int {
        cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kBwdSmemBytes);
        if (e != cudaSuccess) return b2d::fail((int)e, "superfast_backward: smem attr: %s", cudaGetErrorString(e));
        cudaFuncSetAttribute(kern, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared);
        kern<<<dim3((n_pairs + GP - 1) / GP, B), kThreads, kBwdSmemBytes, (cudaStream_t)stream>>>(p);
        return 0;
    };
    const int rc = b2d::g_fft_packed.load(std::memory_order_relaxed) ? go(superfast_backward_kernel<true>)
                                                                      : go(superfast_backward_kernel<false>);
    if (rc) return rc;
    return b2d::check_launch("superfast_backward");
}
#endif  // B2D_HOST_EMU
