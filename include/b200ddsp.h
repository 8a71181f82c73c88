/*
 * b200ddsp.h -- C ABI of libb200ddsp.so: the B200 (sm_100a) DDSP harmonic-plus-noise
 * synthesis kernels behind the reference's Sins / CombSub / CombSubSuperFast / SineGen
 * forward() calls (yxlllc/DDSP-SVC).
 *
 * The reference has no FFI of its own: its "operator API" for this path is the Python
 * module call (ddsp/vocoder.py:556,653,811; nsf_hifigan/models.py:150).  This header is
 * what a maintainer binds (ctypes, see INTEGRATION.md) to replace the tensor code inside
 * those forward() methods.  Each entry point cites the reference lines it replaces.
 *
 * Conventions
 *  - plain C types only; every pointer is a DEVICE pointer to contiguous fp32 data unless
 *    stated otherwise; `stream` is a cudaStream_t passed as void*.
 *  - the library never allocates or frees device memory and never synchronises the stream.
 *    Its entry points are re-entrant from any host thread (the reference is called from the
 *    audio-callback thread of gui.py:376-414 and from Flask): the last-error string is
 *    thread-local, and the only process-wide state is (i) a mutex-protected, per-device
 *    cache of internal fork/join streams and events (b2d_sins_synth runs independent
 *    kernels side by side and joins them on the caller's stream before returning) and
 *    (ii) the b2d_set_* implementation selectors: atomics, each read ONCE at the top of a
 *    call.  The selectors exist for A/B measurements and tests; every setting computes the
 *    same function, so flipping one from another thread changes which kernel a later call
 *    uses, never a result.
 *  - return value: 0 = ok, <0 = argument error (B2D_ERR_*), >0 = cudaError_t of the failed
 *    launch.  No exceptions or aborts cross the ABI.  b2d_last_error() describes the last
 *    failure on the calling thread.
 *  - "ctrl_stride": raw control tensors arrive as strided views of ONE dense
 *    [B, n_frames, n_out] tensor (torch.split in ddsp/unit2control.py:12-23); every control
 *    pointer therefore comes with the element stride between consecutive frames.
 *  - T = n_frames * block.  Utterances (batch rows) are independent.
 */
#ifndef B200DDSP_H
#define B200DDSP_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define B2D_VERSION 100

#define B2D_ERR_NULL        (-1)  /* required pointer is NULL                         */
#define B2D_ERR_SHAPE       (-2)  /* non-positive or inconsistent dimension           */
#define B2D_ERR_ALIGN       (-3)  /* pointer / stride not aligned as required         */
#define B2D_ERR_UNSUPPORTED (-4)  /* configuration outside what the kernels implement */
#define B2D_ERR_WORKSPACE   (-5)  /* workspace too small                              */

/* impulse-response construction modes (b2d_ir_build) */
#define B2D_IR_ALLPASS      0  /* H = exp(j*cumsum(pi*tanh(c))), no window   (ddsp/vocoder.py:581,599) */
#define B2D_IR_MAG_HANN     1  /* H = exp(c)/128, periodic Hann window        (ddsp/vocoder.py:582,606) */
#define B2D_IR_MAG_DYNAMIC  2  /* H = exp(c), per-frame raised-cosine window  (ddsp/vocoder.py:835,849-851) */

int         b2d_version(void);
const char* b2d_last_error(void);

/* ---------------------------------------------------------------------------------------
 * Exciter phase at frame rate.                       replaces ddsp/vocoder.py:564-575
 * (same code at :743-753 and :819-829).
 *   frame_phase[b,k] = sum_{i<k} (P f_i + (f_{i+1}-f_i)(P-1)/2)/sr  (+ initial_phase/2pi),
 *                      unwrapped cycles, fp64  -- the closed form of the reference's
 *                      per-sample fp64 cumsum of the linearly upsampled f0.
 *   phase_frames[b,k] = 2*pi*fp32(wrap(x[k*P]))  -- the tensor handed to Unit2Control.
 * f0_frames [B, n_frames] Hz.  initial_phase: NULL or [B] radians.
 * round_fp32: 0 = infer=True (fp64 phase), 1 = infer=False (phase rounded to fp32 before
 * wrapping, ddsp/vocoder.py:568).
 */
int b2d_phase_scan(const float* f0_frames, const float* initial_phase, int B, int n_frames,
                   int block, double sampling_rate, int round_fp32,
                   double* frame_phase, float* phase_frames, void* stream);

/* ---------------------------------------------------------------------------------------
 * Additive sinusoid bank.                            replaces ddsp/vocoder.py:580,585-594
 * and ddsp/core.py:66-77 (upsample, remove_above_fmax).
 *   sinusoids[b,t] = sum_{h=1..H} sin(h * phase[t]) * up(A)[t,h],
 *   A[k,h] = exp(c_amp[k,h])/128 * (1[f0[k]*h < sr/2] + 1e-7).
 * c_amp: raw 'amplitudes' control, [B, n_frames, H] with frame stride ctrl_stride.
 */
int b2d_sins_bank(const float* f0_frames, const double* frame_phase, const float* c_amp,
                  int64_t ctrl_stride, int B, int n_frames, int block, int n_harmonics,
                  double sampling_rate, int round_fp32, float* sinusoids, void* stream);

/* ---------------------------------------------------------------------------------------
 * Frame-wise impulse responses from raw controls.    replaces ddsp/core.py:254-270
 * (frequency_impulse_response) + :185-237 / :240-251 (windows) and the activations at
 * ddsp/vocoder.py:581-582,599,606,835-836,845,849-851.
 *   ir[b,k,:] has L = 2*(n_mag-1) taps in causal form.
 * dft_tables: device buffer of b2d_dft_tables_bytes(n_mag) bytes filled once by
 * b2d_dft_tables() (constant cos/sin matrices of the L-point inverse real DFT).
 * f0_frames is only read in mode B2D_IR_MAG_DYNAMIC (window half-width 1.5*sr/(f0+1e-3)).
 */
/* Two implementations: tcgen05 tensor cores (3xTF32; default when the accumulators fit TMEM)
 * and CUDA cores.  b2d_set_ir_impl: 0 = automatic, 1 = CUDA cores, 2 = tensor cores (test knob).
 * The table buffer (256-byte aligned) holds the constant matrices for both. */
int    b2d_set_ir_impl(int impl);
size_t b2d_dft_tables_bytes(int n_mag);
int    b2d_dft_tables(int n_mag, float* dft_tables, void* stream);
int    b2d_ir_build(const float* c, int64_t ctrl_stride, int mode, const float* f0_frames,
                    const float* dft_tables, int B, int n_frames, int n_mag,
                    double sampling_rate, float* ir, void* stream);

/* ---------------------------------------------------------------------------------------
 * Linear time-varying FIR (frequency_filter's convolution).   replaces ddsp/core.py:120-182
 * (fft_convolve: Bartlett-windowed 50%-overlap frames, per-frame IR, overlap-add, crop
 * with delay L/2).  The linear convolution it defines is
 *   y[n] = sum_tau ((1-phi_m) h_f[tau] + phi_m h_{f+1}[tau]) x[m],  m = n + L/2 - tau,
 *   f = floor(m/P), phi_m = (m mod P)/P, h_{nF} := h_{nF-1}, x = 0 outside [0,T).
 * Up to two independent filters ("jobs") run in one launch and their outputs can be
 * summed into `mix` (signal = harmonic + noise, ddsp/vocoder.py:609).
 * x1 / x2: input [B, T]; NULL means "white noise U(-1,1) generated in-kernel" from
 * Philox4x32-10 keyed by (seed, utterance index + utterance_offset, sample index)
 * (replaces torch.rand_like(...)*2-1, ddsp/vocoder.py:603).
 * y1 / y2 / mix may be NULL when that output is not wanted; job 2 is skipped when ir2 is
 * NULL.
 */
int b2d_ltv_fir(const float* x1, const float* ir1, int taps1, float* y1,
                const float* x2, const float* ir2, int taps2, float* y2,
                float* mix, uint64_t seed, int64_t utterance_offset,
                int B, int n_frames, int block, void* stream);

/* Kernel selection for b2d_ltv_fir and the synthesizer drivers.  0 = automatic: the FFT-domain kernel
 * (ltv_fir_fft.cu: per input hop one N-point FFT per signal, the impulse responses' spectra and one inverse FFT per
 * pair of hops; N = 1024 up to 512 taps, 2048 up to 1024 taps; ~4x fewer instructions than the direct form,
 * 0.37 ms against 1.18 ms on B200 for Sins' two 510-tap filters) when the block size is 512 and no filter has more than
 * 1024 taps, otherwise the CUDA-core direct form (block size multiple of 256).  1 = CUDA-core direct form
 * (16 outputs per thread, packed fma.rn.f32x2), 2 = tcgen05 tensor cores (3xTF32, block size 512; correct but
 * operand-bandwidth bound and ~3x slower, see DESIGN.md), 3 = the older 8-outputs-per-thread scalar-FFMA direct form,
 * 4 = FFT-domain kernel wherever it applies.  B2D_FIR_AUTO=cuda in the environment makes 0 mean 1.
 * Process-wide test/diagnostic knob. */
int b2d_set_fir_impl(int impl);

/* Same result by the plain one-thread-per-sample formula (any block size / tap count);
 * used as the fallback for configurations the tiled kernel does not cover and as an
 * on-device cross-check. One job only. */
int b2d_ltv_fir_generic(const float* x, const float* ir, int taps, float* y,
                        int B, int n_frames, int block, void* stream);

/* ---------------------------------------------------------------------------------------
 * Whole Sins synthesizer after Unit2Control.         replaces ddsp/vocoder.py:580-611
 * Raw controls in, three waveforms out (any of signal/harmonic/noise_out may be NULL).
 * noise_in: [B, T] uniform(-1,1) samples (parity mode) or NULL (in-kernel Philox).
 * workspace: b2d_sins_workspace_bytes(...) bytes, 256-byte aligned.
 */
size_t b2d_sins_workspace_bytes(int B, int n_frames, int block, int n_mag_allpass, int n_mag_noise);
int    b2d_sins_synth(const float* f0_frames, const double* frame_phase,
                      const float* c_amp, const float* c_group_delay, const float* c_noise,
                      int64_t ctrl_stride, const float* noise_in, uint64_t seed,
                      int64_t utterance_offset, const float* dft_tables_allpass,
                      const float* dft_tables_noise, int B, int n_frames, int block,
                      int n_harmonics, int n_mag_allpass, int n_mag_noise,
                      double sampling_rate, int round_fp32,
                      float* signal, float* harmonic, float* noise_out,
                      void* workspace, size_t workspace_bytes, void* stream);

/* ---------------------------------------------------------------------------------------
 * NSF-HiFiGAN SineGen f0 excitation.                 replaces nsf_hifigan/models.py:134-165
 * (SineGen._f02sine + forward).  f0 [B, n_frames] (Hz, 0 = unvoiced), piecewise constant per
 * frame of `upp` samples; out [B, n_frames*upp, dim], dim = harmonic_num + 1 <= 16.
 * rand_ini [dim]: the random initial phases in cycles (element 0 = 0), drawn by the caller
 * (reference: torch.rand(1,1,dim), models.py:144-145).
 * noise_in [B, T, dim]: N(0,1) samples (parity mode) or NULL = in-kernel Philox + Box-Muller
 * (replaces torch.randn_like, models.py:163).
 * acc_workspace: B*n_frames floats (per-frame wrapped phase advance, models.py:139-141).
 */
int b2d_sinegen(const float* f0, const float* rand_ini, const float* noise_in, uint64_t seed,
                int64_t utterance_offset, int B, int n_frames, int upp, int dim,
                double sampling_rate, float sine_amp, float noise_std, float voiced_threshold,
                float* acc_workspace, float* out, void* stream);

/* ---------------------------------------------------------------------------------------
 * CombSub (old version): comb-tooth source.          replaces ddsp/vocoder.py:819-829,839-840
 *   comb[b,t] = sinc(sr * x[t] / (f0_up[t] + 1e-3)), x = wrapped phase (cycles, fp32).
 */
int b2d_comb_source(const float* f0_frames, const double* frame_phase, int B, int n_frames,
                    int block, double sampling_rate, int round_fp32, float* comb, void* stream);

/* Whole old-CombSub synthesizer after Unit2Control.  replaces ddsp/vocoder.py:834-862
 * comb -> all-pass (group delay) -> harmonic magnitude filter with the per-frame dynamic
 * window (half width 1.5*sr/(f0+1e-3)); noise -> Hann-windowed noise filter; signal = sum.
 * signal/harmonic/noise_out may be NULL.  workspace: b2d_combsub_workspace_bytes bytes.
 */
size_t b2d_combsub_workspace_bytes(int B, int n_frames, int block, int n_mag_allpass,
                                   int n_mag_harmonic, int n_mag_noise);
int    b2d_combsub_synth(const float* f0_frames, const double* frame_phase,
                         const float* c_group_delay, const float* c_harmonic, const float* c_noise,
                         int64_t ctrl_stride, const float* noise_in, uint64_t seed,
                         int64_t utterance_offset, const float* dft_tables_allpass,
                         const float* dft_tables_harmonic, const float* dft_tables_noise,
                         int B, int n_frames, int block, int n_mag_allpass, int n_mag_harmonic,
                         int n_mag_noise, double sampling_rate, int round_fp32,
                         float* signal, float* harmonic, float* noise_out,
                         void* workspace, size_t workspace_bytes, void* stream);

/* ---------------------------------------------------------------------------------------
 * CombSubSuperFast (what configs/combsub.yaml selects).   replaces ddsp/vocoder.py:639-710
 * Two steps around Unit2Control, like the reference:
 *  b2d_superfast_scan : per-frame source parameters (s, ds, wrapped phase advance) into
 *                       `workspace` (b2d_superfast_workspace_bytes) and phase_frames [B,nF]
 *                       = 2*pi*rad[:, :, 0]                      (fast_source_gen, :639-651)
 *  b2d_superfast_synth: comb source -> STFT (2048/512, Hann, reflect) of comb and of N(0,1)
 *                       noise -> Y = X exp(m_h + j pi p_h) + N exp(m_n + j pi p_n)/128 (last
 *                       frame repeated) -> iSTFT -> signal [B, n_frames*block]   (:666-708)
 * The four raw controls [B, n_frames, win_length/2+1] share ctrl_stride.
 * noise_in [B,T] N(0,1) (parity) or NULL (in-kernel Philox + Box-Muller).
 * Only win_length = 2048, block = 512 is implemented (B2D_ERR_UNSUPPORTED otherwise).
 */
size_t b2d_superfast_workspace_bytes(int B, int n_frames);
int    b2d_superfast_scan(const float* f0_frames, int B, int n_frames, int block,
                          double sampling_rate, void* workspace, float* phase_frames, void* stream);
int    b2d_superfast_synth(const void* workspace, const float* c_harmonic_magnitude,
                           const float* c_harmonic_phase, const float* c_noise_magnitude,
                           const float* c_noise_phase, int64_t ctrl_stride, const float* noise_in,
                           uint64_t seed, int64_t utterance_offset, int B, int n_frames, int block,
                           int win_length, float* signal, void* stream);
/* Backward of b2d_superfast_synth with respect to its four controls.  grad_signal [B, n_frames*block]
 * = dL/dsignal (contiguous); the same workspace, controls, noise_in / seed / utterance_offset as the
 * forward call (the source and the in-kernel noise are recomputed, not stored).  Writes
 * dL/dcontrol [B, n_frames, win_length/2+1] for each control with frame stride grad_stride (one dense
 * [B, n_frames, 4 (win_length/2+1)] buffer can hold all four); row n_frames-1 includes the repeated
 * last frame.  Every element is written once; the result does not depend on how the batch is split. */
int    b2d_superfast_backward(const void* workspace, const float* c_harmonic_magnitude,
                              const float* c_harmonic_phase, const float* c_noise_magnitude,
                              const float* c_noise_phase, int64_t ctrl_stride, const float* noise_in,
                              uint64_t seed, int64_t utterance_offset, const float* grad_signal, int B,
                              int n_frames, int block, int win_length, float* g_harmonic_magnitude,
                              float* g_harmonic_phase, float* g_noise_magnitude, float* g_noise_phase,
                              int64_t grad_stride, void* stream);

/* SineGen fused with the tail of SourceModuleHnNSF.   replaces nsf_hifigan/models.py:201-204
 * (sine_merge = tanh(l_linear(sine_wavs))) on top of b2d_sinegen: merged [B, n_frames*upp] =
 * tanh(linear_bias + sum_h linear_weight[h] * sine_wavs[..., h]); the [B, T, dim] tensor is never
 * materialised (4 instead of 36 bytes per sample).  SURVEY 8(f) rank 2 ("next") fusion. */
int b2d_source_module(const float* f0, const float* rand_ini, const float* noise_in, uint64_t seed,
                      int64_t utterance_offset, int B, int n_frames, int upp, int dim,
                      double sampling_rate, float sine_amp, float noise_std, float voiced_threshold,
                      const float* linear_weight, float linear_bias, float* acc_workspace,
                      float* merged, void* stream);

/* CombSubFast STFT-domain filter.   replaces ddsp/vocoder.py:758-784
 * comb [B, T] is the comb-tooth source of b2d_comb_source (the same expression as :764 on the same phase,
 * :743-751 = b2d_phase_scan); controls are raw Unit2Control outputs [B, n_frames, block+1] with a common frame
 * stride; noise_in [B, T] uniform(-1,1) or NULL = in-kernel Philox (same stream as b2d_ltv_fir).
 * Frames of 2*block at hop block, sqrt-Hann analysis and synthesis windows, filter row min(q, n_frames-1),
 * overlap-add cropped by block on both sides.  block must be 512. */
int b2d_combsubfast_filter(const float* comb, const float* c_harmonic_magnitude, const float* c_harmonic_phase,
                           const float* c_noise_magnitude, int64_t ctrl_stride, const float* noise_in,
                           uint64_t seed, int64_t utterance_offset, int B, int n_frames, int block,
                           float* signal, void* stream);

/* Arithmetic of the shared-memory FFT kernels (ltv_fir_fft, superfast, combsubfast): 1 (default) = packed
 * add/sub.rn.f32x2 (one FADD2 per complex addition; 15 % / 7 % fewer instructions in the FIR / SuperFast main loops by SASS
 * count, measured 2.5 % / 1.2 % faster on B200; outputs within 5e-8 of the scalar instantiation), 0 = scalar complex
 * additions.  B2D_FFT_ARITH=scalar in the environment selects 0 as the initial value.  Process-wide test/diagnostic knob
 * (atomic, read once per call). */
int b2d_set_fft_arith(int packed);

/* ---- caller-side prologue / epilogue (SURVEY 8f rank 2) -------------------------------------------------------------
 * Volume_Extractor.extract (ddsp/vocoder.py:147-157): audio [B, n_samples] -> volume [B, n_samples / hop + 1],
 * volume[n] = sqrt(mean(pad_reflect(audio^2, hop/2, (hop+1)/2)[n hop : (n+1) hop])). */
int b2d_volume_extract(const float* audio, int B, int n_samples, int hop, float* volume, void* stream);

/* Silence mask at frame rate (main.py:211-213): mask[n] = max over frames n-4..n+4 (clamped) of (volume > threshold). */
int b2d_volume_mask(const float* volume, int B, int n_frames, float threshold, float* mask_frames, void* stream);

/* `seg_output *= upsample(mask, block)[frame_offset*block : (frame_offset+n_frames)*block]` in place (main.py:215,260;
 * upsample = ddsp/core.py:66-70: linear, last frame held).  signal [B, n_frames*block], mask_frames [B, n_mask_frames]. */
int b2d_mask_apply(float* signal, const float* mask_frames, int B, int n_mask_frames, int frame_offset, int n_frames,
                   int block, void* stream);

/* Segment cross-fade (main.py:142-149): out[0 : idx + len_b] = a[:idx] | (1-k) a[idx:] + k b[:len_a-idx] | b[len_a-idx:],
 * k = linspace(0, 1, len_a - idx) evaluated in fp64.  Requires 0 <= idx < len_a and len_a - idx <= len_b. */
int b2d_cross_fade(const float* a, int64_t len_a, const float* b, int64_t len_b, int64_t idx, float* out, void* stream);

/* ---- fused frame-rate kernels of the control network (Unit2Control inference, ddsp/unit2control.py:84-109 with
 * ddsp/pcmer.py / diffusion/model_conformer_naive.py): everything that is not a plain GEMM.  Activations are token-major
 * [B, T, C] fp32; the model width is 256 as in the reference.
 * u2c_embed (:93-102): x [B*T, 256] += f0_embed(log(1 + f0/700)) + phase_embed(phase/pi) + volume_embed(volume) + spk
 *   (+ aug_embed(aug_shift/5)); embed_table [7, 256] = f0 w, f0 b, phase w, phase b, volume w, volume b, aug w;
 *   spk [spk_rows, 256] (spk_rows 1 or B) or NULL; aug_shift [B] or NULL.
 * u2c_groupnorm_lrelu (:50-52): GroupNorm(groups, C = 256) with statistics over (C/groups channels x T) of each utterance,
 *   then LeakyReLU(slope), in place; stats_ws: B * groups * 2 doubles of scratch.
 * u2c_layernorm: LayerNorm over the last dimension C (multiple of 32, <= 1024) of n_tokens rows.
 * u2c_glu_dwconv_silu (pcmer.py:211-215): in [B, T, 2 Ci] -> GLU -> depthwise Conv1d(k = 31, zero padding 15/15,
 *   weight [Ci, 31], bias [Ci]) -> SiLU -> out [B, T, Ci]; Ci multiple of 128.
 * u2c_softmax_features (pcmer.py:13-48): performer softmax-kernel feature map, in place on projected = (d^-1/4 data) proj^T
 *   [rows, n_features] with data [rows, dim_head]: query rows ratio (exp(p - diag - rowmax) + eps), key rows
 *   ratio exp(p - diag + eps), diag = |data|^2 / (2 sqrt(d)), ratio = n_features^-1/2. */
/* x [n] -> hi, lo [n]: x = hi + lo up to 2^-22 |x| with both parts exactly representable in TF32 (round to nearest even);
 * the operand preparation of 3xTF32 GEMMs (hi hi + lo hi + hi lo on the tensor cores = fp32-grade products). */
int b2d_split_tf32(const float* x, float* hi, float* lo, size_t n, void* stream);
int b2d_u2c_embed(float* x, const float* f0, const float* phase, const float* volume, const float* embed_table,
                  const float* spk, int spk_rows, const float* aug_shift, int B, int T, void* stream);
int b2d_u2c_groupnorm_lrelu(float* x, int B, int T, int C, int groups, const float* gamma, const float* beta, float eps,
                            float slope, double* stats_ws, void* stream);
int b2d_u2c_layernorm(const float* x, float* y, int n_tokens, int C, const float* gamma, const float* beta, float eps,
                      void* stream);
int b2d_u2c_glu_dwconv_silu(const float* in, const float* weight, const float* bias, float* out, int B, int T,
                            int inner_channels, int kernel_size, void* stream);
int b2d_u2c_softmax_features(float* projected, const float* data, int rows, int n_features, int dim_head, int is_query,
                             float eps, void* stream);
/* Fused non-causal linear attention of the performer layers (ddsp/pcmer.py:220-229), one CTA per (utterance, head):
 * q_features, k_features [B*H, T, n_features] (the feature maps above), v [B*H, T, dim_head] ->
 * out [B, T, H, dim_head] = (q' . (k'^T v)) / (q' . sum_t k' + eps).  dim_head must be 64, n_features <= 272. */
int b2d_u2c_linear_attention(const float* q_features, const float* k_features, const float* v, float* out, int B, int H,
                             int T, int n_features, int dim_head, float eps, void* stream);

/* ---- log-mel front end of the NSF-HiFiGAN vocoder: STFT.get_mel, nsf_hifigan/nvSTFT.py:73-117 (keyshift 0, speed 1) ----
 * audio [B, n_samples] -> mel [B, n_mels, n_frames], n_frames = b2d_mel_frames(...) (0 = signal too short):
 * reflect / constant padding by (win - hop)/2, frames of win_size = n_fft = 2048 at `hop`, periodic Hann `window` [2048],
 * magnitude sqrt(re^2 + im^2 + 1e-9), mel_basis [n_mels, n_fft/2 + 1] (librosa.filters.mel layout, n_mels <= 128),
 * log(max(., clip_val)).  filter_lohi [n_mels, 2] (int32, device): first and one-past-last non-zero bin of each filter. */
int b2d_mel_frames(int n_samples, int n_fft, int win_size, int hop);
int b2d_mel_spectrogram(const float* audio, const float* window, const float* mel_basis, const int* filter_lohi, int B,
                        int n_samples, int n_fft, int win_size, int hop, int n_mels, float clip_val, float* mel, void* stream);

/* b2d_sins_synth variants.  0 (default) = 1 = oscillator-bank kernel next to the impulse-response builds, then the FIR
 * kernel transforms the impulse responses itself.  2 = the bank is evaluated inside the FFT-domain FIR kernel (additionally <= 128 harmonics):
 * no [B, T] sinusoid tensor, one launch less -- measured 1.4 % slower on B200 (see api.cu), kept as a tested alternative.
 * 3 = spectrum path: a small kernel turns the impulse responses into packed 1024-point spectra once per frame (beside the
 * bank), the FIR kernel reads them: a quarter fewer transforms, 53 instead of 70 KB of shared memory (4 CTAs per SM); needs
 * block 512, both filters <= 512 taps, FIR selection 0/4; measured 4 % slower (the transform is only moved) -- the consumer
 * side of a future impulse-response GEMM that emits spectra.  Set it BEFORE querying b2d_sins_workspace_bytes (the spectra
 * live in the workspace).  All variants agree to round-off.  Process-wide test/diagnostic knob (atomic, read once per call). */
int b2d_set_sins_impl(int impl);

/* How b2d_sins_synth / b2d_combsub_synth overlap their independent kernels on an internal side stream that is joined on
 * the caller's stream before the call returns (event record/wait only; legal under stream capture).  0: every kernel on
 * the caller's stream, in order.  1: Sins: impulse-response builds next to the oscillator bank; CombSub: the dynamic-window
 * impulse response (needed by the last filter only) next to the comb source / all-pass / noise stage.  k >= 2: additionally the batch is cut into
 * k sub-batches that alternate between the two streams, staggered, so the FIR of one shares the SMs with the bank of the
 * next (-k: the same with a high-priority side stream).  Same results in every mode (the noise is keyed by the global
 * utterance index, the FFT-domain FIR is bit-identical for any batch split).  Process-wide test/diagnostic knob (atomic,
 * read once per call). */
int b2d_set_overlap(int mode);

/* Kernel selection for b2d_sinegen / b2d_source_module (measurement and A/B tests): 0 auto (= 4), 1 one sample per
 * thread (first kernel of round 1; also the only one for dim other than 1 or 9), 2 four samples per thread,
 * 3 four samples per thread with packed f32x2 arithmetic (3-5 % faster, but ptxas fuses its packed mul+add pairs, so
 * the sine argument is rounded once instead of twice: max error 3e-6 instead of 3e-8).  Impl 1 and 2/3 draw DIFFERENT in-kernel
 * noise streams (both Philox4x32-10 keyed by seed / global utterance / position).
 * 4 = variant 2 with Philox4x32-7 instead of -10 for the in-kernel normals (7 rounds: the smallest count reported to
 * pass BigCrush; 11 % faster; Kolmogorov-Smirnov / correlation tests in tests/test_gpu_combsub_sinegen.py). */
int b2d_set_sinegen_impl(int impl);

#ifdef __cplusplus
}
#endif
#endif /* B200DDSP_H */
