// C ABI of libddsp_b200.so - argument validation + kernel launches.
// See include/ddsp_b200.h for the contract and the reference file:line each
// entry point replaces.
#include <stdarg.h>
#include <string.h>

#include <algorithm>

#include "common.cuh"
#include "controls.cuh"
#include "harmonic.cuh"
#include "harmonic_common.cuh"
#include "harmonic_v4.cuh"
#include "noise.cuh"
#include "noise_fused.cuh"
#include "noise_ring.cuh"
#include "host_pipeline.cuh"
#include "backward.cuh"
#include "harmonic_bwd2.cuh"
#include "controls_bwd.cuh"
#include "oscbank.cuh"
#include "sinusoidal.cuh"
#include "wavetable.cuh"
#include "mod_delay.cuh"
#include "longconv.cuh"
#include "spectral.cuh"

namespace ddsp {

static thread_local char g_err[512] = "";
static thread_local uint64_t g_launches = 0;

void count_launch() { ++g_launches; }

void set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}

static inline int grid_for(int64_t n, int threads, int cap_per_sm = 8) {
  int64_t blocks = (n + threads - 1) / threads;
  int64_t cap = (int64_t)kNumSMs * cap_per_sm;
  return (int)std::max<int64_t>(1, std::min(blocks, cap));
}

static constexpr size_t kMaxDynSmem = 200 * 1024;  // of 227 KB usable per CTA

template <typename K>
static int set_smem(K kernel, size_t bytes, const char* name) {
  if (bytes > 48 * 1024) {
    cudaError_t e = cudaFuncSetAttribute(
        kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes);
    if (e != cudaSuccess) {
      set_error("%s: cannot reserve %zu B of shared memory: %s", name, bytes,
                cudaGetErrorString(e));
      return DDSP_B200_E_CUDA;
    }
  }
  return 0;
}

}  // namespace ddsp

using namespace ddsp;

namespace ddsp {
static inline int launch_harmonic_best(const HarmonicParams& p, cudaStream_t st) {
  return launch_harmonic_v4(p, st);
}
}  // namespace ddsp

extern "C" {

int ddsp_b200_version(void) { return DDSP_B200_VERSION; }

const char* ddsp_b200_last_error(void) { return g_err; }

uint64_t ddsp_b200_launch_count(void) { return g_launches; }

int ddsp_b200_harmonic_controls(const float* amps_in, const float* hd_in,
                                const float* f0_hz, float* amps_out,
                                float* hd_out, int B, int F, int K,
                                float sample_rate, int flags, void* stream) {
  DDSP_REQUIRE(amps_in && hd_in && f0_hz && amps_out && hd_out,
               DDSP_B200_E_INVALID, "harmonic_controls: null pointer");
  DDSP_REQUIRE(B >= 0 && F >= 0 && K >= 1, DDSP_B200_E_INVALID,
               "harmonic_controls: bad shape B=%d F=%d K=%d", B, F, K);
  const int64_t rows = (int64_t)B * F;
  if (rows == 0) return 0;
  DDSP_REQUIRE(rows < (1ll << 31) / 32, DDSP_B200_E_INVALID,
               "harmonic_controls: B*F too large");
  const int threads = 256;
  const int blocks = (int)((rows * 32 + threads - 1) / threads);
  harmonic_controls_kernel<<<blocks, threads, 0, (cudaStream_t)stream>>>(
      amps_in, hd_in, f0_hz, amps_out, hd_out, (int)rows, K,
      sample_rate * 0.5f, flags);
  DDSP_CHECK_LAUNCH("harmonic_controls");
  return 0;
}

int ddsp_b200_harmonic_forward(const float* f0_hz, const float* amps,
                               const float* hd, float* audio, int B, int F,
                               int K, int N, float sample_rate, int amp_method,
                               int phase_mode, int accumulate, void* stream) {
  DDSP_REQUIRE(f0_hz && amps && audio, DDSP_B200_E_INVALID,
               "harmonic_forward: null pointer");
  DDSP_REQUIRE(B >= 0 && F >= 1 && K >= 1 && N >= 1, DDSP_B200_E_INVALID,
               "harmonic_forward: bad shape B=%d F=%d K=%d N=%d", B, F, K, N);
  DDSP_REQUIRE(hd != nullptr || K == 1, DDSP_B200_E_INVALID,
               "harmonic_forward: harmonic_distribution is NULL but K=%d", K);
  DDSP_REQUIRE(amp_method == DDSP_B200_AMP_WINDOW ||
                   amp_method == DDSP_B200_AMP_LINEAR,
               DDSP_B200_E_INVALID, "harmonic_forward: bad amp_method %d",
               amp_method);
  DDSP_REQUIRE(phase_mode == DDSP_B200_PHASE_RECURRENCE ||
                   phase_mode == DDSP_B200_PHASE_DIRECT,
               DDSP_B200_E_INVALID, "harmonic_forward: bad phase_mode %d",
               phase_mode);
  // upsample_with_windows raises unless N % F == 0 and F < N (core.py:682-693);
  // the closed-form phase also needs an integer hop.
  DDSP_REQUIRE(N % F == 0, DDSP_B200_E_INVALID,
               "harmonic_forward: n_samples (%d) must be divisible by the "
               "number of frames (%d)", N, F);
  DDSP_REQUIRE(amp_method != DDSP_B200_AMP_WINDOW || F < N,
               DDSP_B200_E_INVALID,
               "harmonic_forward: window upsampling cannot downsample "
               "(frames %d >= timesteps %d)", F, N);
  DDSP_REQUIRE(sample_rate > 0.f, DDSP_B200_E_INVALID,
               "harmonic_forward: sample_rate must be positive");
  if (B == 0) return 0;
  DDSP_REQUIRE(B <= 65535, DDSP_B200_E_INVALID,
               "harmonic_forward: B=%d exceeds the 65535 grid limit", B);

  HarmonicParams p;
  p.f0 = f0_hz; p.amps = amps; p.hd = hd; p.audio = audio;
  p.B = B; p.F = F; p.K = K; p.N = N; p.hop = N / F;
  p.sample_rate = sample_rate;
  p.nyquist = sample_rate * 0.5f;
  p.inv_sr = 1.0 / (double)sample_rate;
  p.amp_method = amp_method;
  p.accumulate = accumulate;
  p.ctl_flags = 0;
  p.init_phase = nullptr; p.final_phase = nullptr; p.mask_nyquist = 1;
  cudaStream_t st = (cudaStream_t)stream;

  if (phase_mode == DDSP_B200_PHASE_RECURRENCE && harmonic_fused_supported(p)) {
    int rc = launch_harmonic_best(p, st);
    if (rc != 1) return rc;   // 1 = declined, fall through to the generic path
  }

  p.Kp = (K + 3) & ~3;
  // frames per tile: ~2048 samples, enough CTAs to fill the chip, bounded smem
  int FT = std::max(1, 2048 / p.hop);
  const int64_t want_ctas = 4ll * kNumSMs;
  int ft_fill = (int)std::max<int64_t>(1, ((int64_t)B * F + want_ctas - 1) / want_ctas);
  FT = std::min(FT, std::max(ft_fill, std::min(4, F)));
  FT = std::min(FT, F);
  while (FT > 1 && harm_smem_bytes(FT, p.Kp) > kMaxDynSmem) FT = (FT + 1) / 2;
  DDSP_REQUIRE(harm_smem_bytes(FT, p.Kp) <= kMaxDynSmem, DDSP_B200_E_UNSUPPORTED,
               "harmonic_forward: K=%d needs more shared memory than one CTA has",
               K);
  p.FT = FT;
  const size_t smem = harm_smem_bytes(FT, p.Kp);
  dim3 grid((F + FT - 1) / FT, B);
  if (phase_mode == DDSP_B200_PHASE_DIRECT) {
    int rc = set_smem(harmonic_generic_kernel<1>, smem, "harmonic_forward");
    if (rc) return rc;
    harmonic_generic_kernel<1><<<grid, kHarmThreads, smem, st>>>(p);
  } else {
    int rc = set_smem(harmonic_generic_kernel<0>, smem, "harmonic_forward");
    if (rc) return rc;
    harmonic_generic_kernel<0><<<grid, kHarmThreads, smem, st>>>(p);
  }
  DDSP_CHECK_LAUNCH("harmonic_forward");
  return 0;
}

int ddsp_b200_streaming_harmonic_forward(const float* f0_hz, const float* amps,
                                         const float* hd, const float* initial_phase,
                                         float* audio, float* final_phase, int B,
                                         int F, int K, int N, float sample_rate,
                                         int amp_method, void* stream) {
  DDSP_REQUIRE(f0_hz && amps && audio, DDSP_B200_E_INVALID,
               "streaming_harmonic_forward: null pointer");
  DDSP_REQUIRE(B >= 0 && F >= 1 && K >= 1 && N >= 1, DDSP_B200_E_INVALID,
               "streaming_harmonic_forward: bad shape B=%d F=%d K=%d N=%d", B, F, K, N);
  DDSP_REQUIRE(hd != nullptr || K == 1, DDSP_B200_E_INVALID,
               "streaming_harmonic_forward: harmonic_distribution is NULL but K=%d", K);
  DDSP_REQUIRE(amp_method == DDSP_B200_AMP_WINDOW ||
                   amp_method == DDSP_B200_AMP_LINEAR,
               DDSP_B200_E_INVALID, "streaming_harmonic_forward: bad amp_method %d",
               amp_method);
  DDSP_REQUIRE(N % F == 0, DDSP_B200_E_INVALID,
               "streaming_harmonic_forward: n_samples (%d) must be divisible by "
               "the number of frames (%d)", N, F);
  DDSP_REQUIRE(sample_rate > 0.f, DDSP_B200_E_INVALID,
               "streaming_harmonic_forward: sample_rate must be positive");
  if (B == 0) return 0;
  DDSP_REQUIRE(B <= 65535, DDSP_B200_E_INVALID,
               "streaming_harmonic_forward: B=%d exceeds the 65535 grid limit", B);
  HarmonicParams p;
  p.f0 = f0_hz; p.amps = amps; p.hd = hd; p.audio = audio;
  p.B = B; p.F = F; p.K = K; p.N = N; p.hop = N / F;
  p.sample_rate = sample_rate; p.nyquist = sample_rate * 0.5f;
  p.inv_sr = 1.0 / (double)sample_rate;
  p.amp_method = amp_method; p.accumulate = 0; p.ctl_flags = 0;
  p.init_phase = initial_phase; p.final_phase = final_phase; p.mask_nyquist = 0;
  p.Kp = (K + 3) & ~3;
  int FT = std::max(1, std::min(F, 2048 / p.hop));
  while (FT > 1 && harm_smem_bytes(FT, p.Kp) > kMaxDynSmem) FT = (FT + 1) / 2;
  DDSP_REQUIRE(harm_smem_bytes(FT, p.Kp) <= kMaxDynSmem, DDSP_B200_E_UNSUPPORTED,
               "streaming_harmonic_forward: K=%d needs too much shared memory", K);
  p.FT = FT;
  const size_t smem = harm_smem_bytes(FT, p.Kp);
  int rc = set_smem(harmonic_generic_kernel<0>, smem, "streaming_harmonic_forward");
  if (rc) return rc;
  dim3 grid((F + FT - 1) / FT, B);
  harmonic_generic_kernel<0><<<grid, kHarmThreads, smem, (cudaStream_t)stream>>>(p);
  DDSP_CHECK_LAUNCH("streaming_harmonic_forward");
  return 0;
}

int ddsp_b200_noise_controls(const float* mag_in, float* mag_out, int64_t n,
                             float initial_bias, int apply_scale, void* stream) {
  DDSP_REQUIRE(mag_in && mag_out, DDSP_B200_E_INVALID,
               "noise_controls: null pointer");
  DDSP_REQUIRE(n >= 0, DDSP_B200_E_INVALID, "noise_controls: n < 0");
  if (n == 0) return 0;
  noise_controls_kernel<<<grid_for(n, 256), 256, 0, (cudaStream_t)stream>>>(
      mag_in, mag_out, n, initial_bias, apply_scale);
  DDSP_CHECK_LAUNCH("noise_controls");
  return 0;
}

int ddsp_b200_ir_size(int nb, int window_size) {
  if (nb < 2) return DDSP_B200_E_INVALID;
  return make_ir_geom(nb, window_size).S;
}

int ddsp_b200_frequency_impulse_response(const float* mags, float* ir,
                                         int64_t BF, int nb, int window_size,
                                         void* stream) {
  DDSP_REQUIRE(mags && ir, DDSP_B200_E_INVALID,
               "frequency_impulse_response: null pointer");
  DDSP_REQUIRE(nb >= 2 && BF >= 0, DDSP_B200_E_INVALID,
               "frequency_impulse_response: need n_frequencies >= 2 (got %d)", nb);
  if (BF == 0) return 0;
  IrGeom g = make_ir_geom(nb, window_size);
  const size_t smem = sizeof(float) * ((size_t)g.S0 + (size_t)kIrFrames * nb);
  DDSP_REQUIRE(smem <= kMaxDynSmem, DDSP_B200_E_UNSUPPORTED,
               "frequency_impulse_response: n_frequencies=%d too large", nb);
  int rc = set_smem(ir_kernel, smem, "frequency_impulse_response");
  if (rc) return rc;
  const int64_t blocks = (BF + kIrFrames - 1) / kIrFrames;
  DDSP_REQUIRE(blocks < (1ll << 31), DDSP_B200_E_INVALID,
               "frequency_impulse_response: too many frames");
  ir_kernel<<<(int)blocks, kIrThreads, smem, (cudaStream_t)stream>>>(mags, ir,
                                                                     BF, g);
  DDSP_CHECK_LAUNCH("frequency_impulse_response");
  return 0;
}

int ddsp_b200_fir_time_varying(const float* audio, const float* ir, float* out,
                               int B, int N, int F, int S, int ir_batch,
                               int padding, int delay_compensation,
                               int accumulate, void* stream) {
  DDSP_REQUIRE(audio && ir && out, DDSP_B200_E_INVALID,
               "fir_time_varying: null pointer");
  DDSP_REQUIRE(B >= 0 && N >= 1 && F >= 1 && S >= 1, DDSP_B200_E_INVALID,
               "fir_time_varying: bad shape B=%d N=%d F=%d S=%d", B, N, F, S);
  // core.py:1441-1443
  DDSP_REQUIRE(ir_batch == B || ir_batch == 1, DDSP_B200_E_INVALID,
               "Batch size of audio (%d) and impulse response (%d) must be the "
               "same.", B, ir_batch);
  DDSP_REQUIRE(padding == DDSP_B200_PAD_SAME || padding == DDSP_B200_PAD_VALID,
               DDSP_B200_E_INVALID,
               "Padding must be 'valid' or 'same' (got code %d)", padding);
  // core.py:1446-1457: frame = ceil(N / F); frame(pad_end) must yield F frames
  const int frame = (N + F - 1) / F;
  const int n_audio_frames = (N + frame - 1) / frame;
  DDSP_REQUIRE(n_audio_frames == F, DDSP_B200_E_INVALID,
               "Number of Audio frames (%d) and impulse response frames (%d) do "
               "not match. For small hop size = ceil(audio_size / n_ir_frames), "
               "number of impulse response frames must be a multiple of the "
               "audio size.", n_audio_frames, F);
  if (B == 0) return 0;
  DDSP_REQUIRE(B <= 65535, DDSP_B200_E_INVALID,
               "fir_time_varying: B=%d exceeds the 65535 grid limit", B);
  // crop_and_compensate_delay (core.py:1338-1379)
  const int out_len = (padding == DDSP_B200_PAD_VALID) ? (N + S - 1) : N;
  const int start = delay_compensation < 0 ? ((S - 1) / 2 - 1)
                                           : delay_compensation;
  DDSP_REQUIRE(start >= 0, DDSP_B200_E_UNSUPPORTED,
               "fir_time_varying: impulse response of %d taps gives a negative "
               "automatic delay; pass delay_compensation >= 0", S);
  const size_t smem = sizeof(float) * ((size_t)kFirThreads + S - 1);
  DDSP_REQUIRE(smem <= kMaxDynSmem, DDSP_B200_E_UNSUPPORTED,
               "fir_time_varying: impulse response of %d taps is beyond the "
               "shared-memory FIR (long-IR convolution is not built yet)", S);
  int rc = set_smem(fir_kernel, smem, "fir_time_varying");
  if (rc) return rc;
  dim3 grid((out_len + kFirThreads - 1) / kFirThreads, B);
  fir_kernel<<<grid, kFirThreads, smem, (cudaStream_t)stream>>>(
      audio, ir, out, N, F, S, frame, ir_batch == 1 ? 0 : F * S, start, out_len,
      accumulate);
  DDSP_CHECK_LAUNCH("fir_time_varying");
  return 0;
}

int ddsp_b200_uniform_noise(float* out, int B, int N, uint64_t seed,
                            uint64_t offset, void* stream) {
  DDSP_REQUIRE(out, DDSP_B200_E_INVALID, "uniform_noise: null pointer");
  DDSP_REQUIRE(B >= 0 && N >= 0, DDSP_B200_E_INVALID, "uniform_noise: bad shape");
  if (B == 0 || N == 0) return 0;
  const int64_t n = (int64_t)B * ((N + 3) / 4);
  uniform_noise_kernel<<<grid_for(n, 256), 256, 0, (cudaStream_t)stream>>>(
      out, B, N, seed, offset);
  DDSP_CHECK_LAUNCH("uniform_noise");
  return 0;
}

size_t ddsp_b200_filtered_noise_workspace(int B, int F, int nb, int N,
                                          int window_size) {
  if (nb < 2 || B <= 0 || F <= 0 || N <= 0) return 0;
  if (noise_fused_supported(F, nb, N, window_size)) return 0;
  IrGeom g = make_ir_geom(nb, window_size);
  // generic path: IR [B,F,S] + noise [B,N]
  return sizeof(float) * ((size_t)B * F * g.S + (size_t)B * N) + 256;
}

int ddsp_b200_filtered_noise_forward(const float* mags, const float* noise,
                                     uint64_t seed, uint64_t offset,
                                     float* audio, int B, int F, int nb, int N,
                                     int window_size, int accumulate,
                                     void* workspace, size_t workspace_bytes,
                                     void* stream) {
  DDSP_REQUIRE(mags && audio, DDSP_B200_E_INVALID,
               "filtered_noise_forward: null pointer");
  DDSP_REQUIRE(B >= 0 && F >= 1 && N >= 1, DDSP_B200_E_INVALID,
               "filtered_noise_forward: bad shape B=%d F=%d N=%d", B, F, N);
  DDSP_REQUIRE(nb >= 2, DDSP_B200_E_INVALID,
               "filtered_noise_forward: need n_frequencies >= 2 (got %d)", nb);
  const int frame = (N + F - 1) / F;
  const int n_audio_frames = (N + frame - 1) / frame;
  DDSP_REQUIRE(n_audio_frames == F, DDSP_B200_E_INVALID,
               "Number of Audio frames (%d) and impulse response frames (%d) do "
               "not match. For small hop size = ceil(audio_size / n_ir_frames), "
               "number of impulse response frames must be a multiple of the "
               "audio size.", n_audio_frames, F);
  if (B == 0) return 0;
  cudaStream_t st = (cudaStream_t)stream;
  if (noise_fused_supported(F, nb, N, window_size)) {
    return launch_noise_best(mags, noise, seed, offset, audio, B, F, nb, N,
                             window_size, accumulate, st);
  }
  const size_t need = ddsp_b200_filtered_noise_workspace(B, F, nb, N, window_size);
  DDSP_REQUIRE(workspace != nullptr && workspace_bytes >= need,
               DDSP_B200_E_WORKSPACE,
               "filtered_noise_forward: workspace of %zu B needed, %zu given",
               need, workspace_bytes);
  IrGeom g = make_ir_geom(nb, window_size);
  uintptr_t base = ((uintptr_t)workspace + 255) & ~(uintptr_t)255;
  float* ir = reinterpret_cast<float*>(base);
  float* nz = ir + (size_t)B * F * g.S;
  int rc = ddsp_b200_frequency_impulse_response(mags, ir, (int64_t)B * F, nb,
                                                window_size, stream);
  if (rc) return rc;
  const float* x = noise;
  if (x == nullptr) {
    rc = ddsp_b200_uniform_noise(nz, B, N, seed, offset, stream);
    if (rc) return rc;
    x = nz;
  }
  return ddsp_b200_fir_time_varying(x, ir, audio, B, N, F, g.S, B,
                                    DDSP_B200_PAD_SAME, -1, accumulate, stream);
}

static int decoder_forward_impl(const float* amps_raw, const float* hd_raw,
                                const float* f0_hz, const float* mags_raw,
                                const float* noise, uint64_t seed, uint64_t offset,
                                float* audio, int B, int F, int K, int nb, int N,
                                float sample_rate, int amp_method,
                                int harmonic_flags, int window_size,
                                float initial_bias, void* stream, int item_base) {
  DDSP_REQUIRE(amps_raw && hd_raw && f0_hz && mags_raw && audio,
               DDSP_B200_E_INVALID, "decoder_forward: null pointer");
  DDSP_REQUIRE(B >= 0 && F >= 1 && K >= 1 && N >= 1 && nb >= 2,
               DDSP_B200_E_INVALID,
               "decoder_forward: bad shape B=%d F=%d K=%d nb=%d N=%d", B, F, K,
               nb, N);
  DDSP_REQUIRE(amp_method == DDSP_B200_AMP_WINDOW ||
                   amp_method == DDSP_B200_AMP_LINEAR,
               DDSP_B200_E_INVALID, "decoder_forward: bad amp_method %d",
               amp_method);
  DDSP_REQUIRE(harmonic_flags != 0 &&
                   (harmonic_flags & ~(DDSP_B200_CTL_SCALE | DDSP_B200_CTL_NYQUIST)) == 0,
               DDSP_B200_E_INVALID, "decoder_forward: bad harmonic_flags %d",
               harmonic_flags);
  DDSP_REQUIRE(sample_rate > 0.f, DDSP_B200_E_INVALID,
               "decoder_forward: sample_rate must be positive");
  if (B == 0) return 0;
  HarmonicParams p;
  p.f0 = f0_hz; p.amps = amps_raw; p.hd = hd_raw; p.audio = audio;
  p.B = B; p.F = F; p.K = K; p.N = N; p.hop = N / F;
  p.sample_rate = sample_rate;
  p.nyquist = sample_rate * 0.5f;
  p.inv_sr = 1.0 / (double)sample_rate;
  p.amp_method = amp_method;
  p.accumulate = 0;
  p.ctl_flags = harmonic_flags;
  p.init_phase = nullptr; p.final_phase = nullptr; p.mask_nyquist = 1;
  // The single-pass pipeline exists for the decoder regime only; everything
  // else goes through get_controls + the two *_forward calls.
  DDSP_REQUIRE(N % F == 0 && B <= 65535 && harmonic_fused_supported(p) &&
                   noise_fused_supported(F, nb, N, window_size),
               DDSP_B200_E_UNSUPPORTED,
               "decoder_forward: shape outside the fused decoder path "
               "(needs hop %% 64 == 0, n_frequencies <= %d)", kNfMaxNb);
  cudaStream_t st = (cudaStream_t)stream;
  int rc = launch_harmonic_best(p, st);
  if (rc == 1) {
    set_error("decoder_forward: harmonic tile does not fit shared memory");
    return DDSP_B200_E_UNSUPPORTED;
  }
  if (rc) return rc;
  return launch_noise_best(mags_raw, noise, seed, offset, audio, B, F, nb, N,
                           window_size, /*accumulate=*/1, st, /*raw=*/1,
                           initial_bias, item_base, /*overlap_previous=*/1);
}

int ddsp_b200_decoder_forward(const float* amps_raw, const float* hd_raw,
                              const float* f0_hz, const float* mags_raw,
                              const float* noise, uint64_t seed, uint64_t offset,
                              float* audio, int B, int F, int K, int nb, int N,
                              float sample_rate, int amp_method,
                              int harmonic_flags, int window_size,
                              float initial_bias, void* stream) {
  return decoder_forward_impl(amps_raw, hd_raw, f0_hz, mags_raw, noise, seed, offset,
                              audio, B, F, K, nb, N, sample_rate, amp_method,
                              harmonic_flags, window_size, initial_bias, stream, 0);
}

// ---- host-buffer pipeline ---------------------------------------------------
#define DDSP_CUDA_TRY(expr, what)                                         \
  do {                                                                    \
    cudaError_t e__ = (expr);                                             \
    if (e__ != cudaSuccess) {                                             \
      ::ddsp::set_error("%s: %s", what, cudaGetErrorString(e__));         \
      return DDSP_B200_E_CUDA;                                            \
    }                                                                     \
  } while (0)

int ddsp_b200_host_pipeline_create(ddsp_b200_host_pipeline** out, int max_B, int F,
                                   int K, int nb, int N, int max_chunks) {
  DDSP_REQUIRE(out != nullptr, DDSP_B200_E_INVALID, "host_pipeline_create: null out");
  *out = nullptr;
  DDSP_REQUIRE(max_B >= 1 && F >= 1 && K >= 1 && nb >= 2 && N >= 1 && max_chunks >= 1,
               DDSP_B200_E_INVALID,
               "host_pipeline_create: bad shape max_B=%d F=%d K=%d nb=%d N=%d chunks=%d",
               max_B, F, K, nb, N, max_chunks);
  HostPipeline* hp = new HostPipeline();
  auto fail = [&](const char* what, cudaError_t e) {
    set_error("host_pipeline_create: %s: %s", what, cudaGetErrorString(e));
    host_pipeline_free(hp);
    return DDSP_B200_E_CUDA;
  };
  cudaError_t e = cudaGetDevice(&hp->device);
  if (e != cudaSuccess) { hp->device = -1; return fail("cudaGetDevice", e); }
  hp->max_B = max_B; hp->F = F; hp->K = K; hp->nb = nb; hp->N = N;
  hp->max_chunks = std::min(max_chunks, max_B);
  // every sub-buffer starts on a 256-byte boundary (TMA bulk copies want 16)
  auto pad = [](size_t n) { return (n + 63) & ~(size_t)63; };
  const size_t n_amps = pad((size_t)max_B * F), n_hd = pad((size_t)max_B * F * K),
               n_mags = pad((size_t)max_B * F * nb), n_audio = pad((size_t)max_B * N);
  const size_t total = 2 * n_amps + n_hd + n_mags + n_audio;
  if ((e = cudaMalloc(&hp->d_base, total * sizeof(float))) != cudaSuccess)
    return fail("cudaMalloc(staging)", e);
  hp->d_amps = hp->d_base;
  hp->d_f0 = hp->d_amps + n_amps;
  hp->d_hd = hp->d_f0 + n_amps;
  hp->d_mags = hp->d_hd + n_hd;
  hp->d_audio = hp->d_mags + n_mags;
  if ((e = cudaStreamCreateWithFlags(&hp->s_h2d, cudaStreamNonBlocking)) != cudaSuccess)
    return fail("cudaStreamCreate", e);
  if ((e = cudaStreamCreateWithFlags(&hp->s_h2d2, cudaStreamNonBlocking)) != cudaSuccess)
    return fail("cudaStreamCreate", e);
  if ((e = cudaStreamCreateWithFlags(&hp->s_d2h, cudaStreamNonBlocking)) != cudaSuccess)
    return fail("cudaStreamCreate", e);
  if ((e = cudaEventCreateWithFlags(&hp->ev_start, cudaEventDisableTiming)) != cudaSuccess)
    return fail("cudaEventCreate", e);
  if ((e = cudaEventCreateWithFlags(&hp->ev_done, cudaEventDisableTiming)) != cudaSuccess)
    return fail("cudaEventCreate", e);
  for (int c = 0; c < hp->max_chunks; ++c) {
    cudaEvent_t a = nullptr, b = nullptr;
    if ((e = cudaEventCreateWithFlags(&a, cudaEventDisableTiming)) != cudaSuccess)
      return fail("cudaEventCreate", e);
    hp->ev_h2d.push_back(a);
    if ((e = cudaEventCreateWithFlags(&b, cudaEventDisableTiming)) != cudaSuccess)
      return fail("cudaEventCreate", e);
    hp->ev_comp.push_back(b);
    cudaEvent_t a2 = nullptr;
    if ((e = cudaEventCreateWithFlags(&a2, cudaEventDisableTiming)) != cudaSuccess)
      return fail("cudaEventCreate", e);
    hp->ev_h2d2.push_back(a2);
  }
  *out = reinterpret_cast<ddsp_b200_host_pipeline*>(hp);
  return 0;
}

int ddsp_b200_host_pipeline_destroy(ddsp_b200_host_pipeline* handle) {
  host_pipeline_free(reinterpret_cast<HostPipeline*>(handle));
  return 0;
}

int ddsp_b200_decoder_forward_host(ddsp_b200_host_pipeline* handle,
                                   const float* amps_raw, const float* hd_raw,
                                   const float* f0_hz, const float* mags_raw,
                                   uint64_t seed, uint64_t offset, float* audio,
                                   int B, int n_chunks, float sample_rate,
                                   int amp_method, int harmonic_flags,
                                   int window_size, float initial_bias,
                                   void* stream) {
  HostPipeline* hp = reinterpret_cast<HostPipeline*>(handle);
  DDSP_REQUIRE(hp != nullptr, DDSP_B200_E_INVALID, "decoder_forward_host: null handle");
  DDSP_REQUIRE(amps_raw && hd_raw && f0_hz && mags_raw && audio, DDSP_B200_E_INVALID,
               "decoder_forward_host: null pointer");
  DDSP_REQUIRE(B >= 0 && B <= hp->max_B, DDSP_B200_E_INVALID,
               "decoder_forward_host: B=%d outside [0, %d]", B, hp->max_B);
  if (B == 0) return 0;
  int dev = 0;
  DDSP_CUDA_TRY(cudaGetDevice(&dev), "decoder_forward_host: cudaGetDevice");
  DDSP_REQUIRE(dev == hp->device, DDSP_B200_E_INVALID,
               "decoder_forward_host: pipeline belongs to device %d, current is %d",
               hp->device, dev);
  n_chunks = std::max(1, std::min(std::min(std::min(n_chunks, hp->max_chunks), B), 64));
  const int F = hp->F, K = hp->K, nb = hp->nb, N = hp->N;
  cudaStream_t st = (cudaStream_t)stream;
  // Order this call after whatever the caller queued on `st`, and after the
  // previous call's last device->host copy (the staging buffers are reused).
  DDSP_CUDA_TRY(cudaEventRecord(hp->ev_start, st), "decoder_forward_host: event");
  DDSP_CUDA_TRY(cudaStreamWaitEvent(hp->s_h2d, hp->ev_start, 0), "decoder_forward_host: wait");
  DDSP_CUDA_TRY(cudaStreamWaitEvent(hp->s_h2d2, hp->ev_start, 0), "decoder_forward_host: wait");
  if (hp->used) {
    DDSP_CUDA_TRY(cudaStreamWaitEvent(hp->s_h2d, hp->ev_done, 0), "decoder_forward_host: wait");
    DDSP_CUDA_TRY(cudaStreamWaitEvent(hp->s_h2d2, hp->ev_done, 0), "decoder_forward_host: wait");
  }
  hp->used = true;
  // Two host->device streams (harmonic_distribution on one; magnitudes and the
  // small per-frame vectors on the other): a copy costs ~10 us of set-up however
  // small it is, and on one stream those set-ups do not overlap the previous
  // transfer - two streams keep the link busy while one of them sets up.  The
  // per-frame vectors go over once for the whole batch.
  DDSP_CUDA_TRY(cudaMemcpyAsync(hp->d_f0, f0_hz, sizeof(float) * (size_t)B * F,
                                cudaMemcpyHostToDevice, hp->s_h2d2), "decoder_forward_host: H2D f0");
  DDSP_CUDA_TRY(cudaMemcpyAsync(hp->d_amps, amps_raw, sizeof(float) * (size_t)B * F,
                                cudaMemcpyHostToDevice, hp->s_h2d2), "decoder_forward_host: H2D amps");
  // Chunk sizes halve: the call ends with the compute + device->host copy of the
  // LAST chunk (nothing left to overlap them with), so that one should be small,
  // while few chunks keep the per-chunk submission cost down.
  int sizes[64];
  int n_c = 0;
  for (int b0 = 0; b0 < B; ++n_c) {
    const int left = B - b0;
    sizes[n_c] = (n_c == n_chunks - 1 || n_c == 63) ? left : std::max(1, (left + 1) / 2);
    b0 += sizes[n_c];
  }
  // First queue EVERY host->device copy: the copy engines then never wait for
  // this thread to get through the launches and event calls of earlier chunks
  // (~35 us of driver time per chunk, longer than a small chunk's transfer).
  for (int c = 0, b0 = 0; c < n_c; b0 += sizes[c], ++c) {
    const int nbi = sizes[c];
    const size_t o1 = (size_t)b0 * F;
    DDSP_CUDA_TRY(cudaMemcpyAsync(hp->d_hd + o1 * K, hd_raw + o1 * K,
                                  sizeof(float) * (size_t)nbi * F * K,
                                  cudaMemcpyHostToDevice, hp->s_h2d), "decoder_forward_host: H2D hd");
    DDSP_CUDA_TRY(cudaEventRecord(hp->ev_h2d[c], hp->s_h2d), "decoder_forward_host: event");
    DDSP_CUDA_TRY(cudaMemcpyAsync(hp->d_mags + o1 * nb, mags_raw + o1 * nb,
                                  sizeof(float) * (size_t)nbi * F * nb,
                                  cudaMemcpyHostToDevice, hp->s_h2d2), "decoder_forward_host: H2D mags");
    DDSP_CUDA_TRY(cudaEventRecord(hp->ev_h2d2[c], hp->s_h2d2), "decoder_forward_host: event");
  }
  for (int c = 0, b0 = 0; c < n_c; b0 += sizes[c], ++c) {
    const int nbi = sizes[c];
    const size_t o1 = (size_t)b0 * F;
    DDSP_CUDA_TRY(cudaStreamWaitEvent(st, hp->ev_h2d[c], 0), "decoder_forward_host: wait");
    DDSP_CUDA_TRY(cudaStreamWaitEvent(st, hp->ev_h2d2[c], 0), "decoder_forward_host: wait");
    int rc = decoder_forward_impl(hp->d_amps + o1, hp->d_hd + o1 * K, hp->d_f0 + o1,
                                  hp->d_mags + o1 * nb, nullptr, seed, offset,
                                  hp->d_audio + (size_t)b0 * N, nbi, F, K, nb, N,
                                  sample_rate, amp_method, harmonic_flags, window_size,
                                  initial_bias, stream, b0);
    if (rc) return rc;
    DDSP_CUDA_TRY(cudaEventRecord(hp->ev_comp[c], st), "decoder_forward_host: event");
    DDSP_CUDA_TRY(cudaStreamWaitEvent(hp->s_d2h, hp->ev_comp[c], 0), "decoder_forward_host: wait");
    DDSP_CUDA_TRY(cudaMemcpyAsync(audio + (size_t)b0 * N, hp->d_audio + (size_t)b0 * N,
                                  sizeof(float) * (size_t)nbi * N, cudaMemcpyDeviceToHost,
                                  hp->s_d2h), "decoder_forward_host: D2H audio");
  }
  DDSP_CUDA_TRY(cudaEventRecord(hp->ev_done, hp->s_d2h), "decoder_forward_host: event");
  // The caller's stream completes when the audio is in host memory.
  DDSP_CUDA_TRY(cudaStreamWaitEvent(st, hp->ev_done, 0), "decoder_forward_host: wait");
  return 0;
}

int ddsp_b200_harmonic_backward(const float* f0_hz, const float* grad_audio,
                                float* g0, float* g1, int B, int F, int K, int N,
                                float sample_rate, int amp_method, void* stream) {
  DDSP_REQUIRE(f0_hz && grad_audio && g0 && g1, DDSP_B200_E_INVALID,
               "harmonic_backward: null pointer");
  DDSP_REQUIRE(B >= 0 && F >= 1 && K >= 1 && N >= 1 && N % F == 0,
               DDSP_B200_E_INVALID,
               "harmonic_backward: bad shape B=%d F=%d K=%d N=%d", B, F, K, N);
  DDSP_REQUIRE(amp_method == DDSP_B200_AMP_WINDOW ||
                   amp_method == DDSP_B200_AMP_LINEAR,
               DDSP_B200_E_INVALID, "harmonic_backward: bad amp_method %d",
               amp_method);
  DDSP_REQUIRE(sample_rate > 0.f, DDSP_B200_E_INVALID,
               "harmonic_backward: sample_rate must be positive");
  if (B == 0) return 0;
  HarmonicParams p;
  p.f0 = f0_hz; p.amps = nullptr; p.hd = nullptr; p.audio = nullptr;
  p.B = B; p.F = F; p.K = K; p.N = N; p.hop = N / F;
  p.sample_rate = sample_rate; p.nyquist = sample_rate * 0.5f;
  p.inv_sr = 1.0 / (double)sample_rate;
  p.amp_method = amp_method; p.accumulate = 0; p.ctl_flags = 0; p.Kp = K;
  p.init_phase = nullptr; p.final_phase = nullptr; p.mask_nyquist = 1;
  DDSP_REQUIRE(p.hop % 64 == 0 && p.hop <= 8192 && B <= 65535,
               DDSP_B200_E_UNSUPPORTED,
               "harmonic_backward: needs hop %% 64 == 0 (hop = %d)", p.hop);
  cudaStream_t st = (cudaStream_t)stream;
  static const bool use_v1 = [] {
    const char* e = getenv("DDSP_B200_HARM_BWD");
    return e != nullptr && strcmp(e, "v1") == 0;
  }();
  if (!use_v1 && harmonic_backward2_supported(p))
    return launch_harmonic_backward2(p, grad_audio, g0, g1, st);
  const size_t gbytes = sizeof(float) * (size_t)B * F * K;
  DDSP_CUDA_TRY(cudaMemsetAsync(g0, 0, gbytes, st), "harmonic_backward: memset g0");
  DDSP_CUDA_TRY(cudaMemsetAsync(g1, 0, gbytes, st), "harmonic_backward: memset g1");
  p.FT = std::max(1, std::min(F, 2048 / p.hop));
  const size_t smem = harmonic_backward_smem(p.FT, p.hop);
  dim3 grid((F + p.FT - 1) / p.FT, B);
  if (amp_method == DDSP_B200_AMP_WINDOW) {
    int rc = set_smem(harmonic_backward_kernel<true>, smem, "harmonic_backward");
    if (rc) return rc;
    harmonic_backward_kernel<true><<<grid, kHbThreads, smem, st>>>(p, grad_audio, g0, g1);
  } else {
    int rc = set_smem(harmonic_backward_kernel<false>, smem, "harmonic_backward");
    if (rc) return rc;
    harmonic_backward_kernel<false><<<grid, kHbThreads, smem, st>>>(p, grad_audio, g0, g1);
  }
  DDSP_CHECK_LAUNCH("harmonic_backward");
  return 0;
}

int ddsp_b200_harmonic_backward_f0(const float* f0_hz, const float* amps,
                                   const float* hd, const float* grad_audio,
                                   float* d_f0, int B, int F, int K, int N,
                                   float sample_rate, int amp_method,
                                   void* workspace, size_t workspace_bytes,
                                   void* stream) {
  DDSP_REQUIRE(f0_hz && amps && grad_audio && d_f0, DDSP_B200_E_INVALID,
               "harmonic_backward_f0: null pointer");
  DDSP_REQUIRE(B >= 0 && F >= 1 && K >= 1 && N >= 1 && N % F == 0, DDSP_B200_E_INVALID,
               "harmonic_backward_f0: bad shape B=%d F=%d K=%d N=%d", B, F, K, N);
  DDSP_REQUIRE(hd != nullptr || K == 1, DDSP_B200_E_INVALID,
               "harmonic_backward_f0: harmonic_distribution is NULL but K=%d", K);
  DDSP_REQUIRE(amp_method == DDSP_B200_AMP_WINDOW || amp_method == DDSP_B200_AMP_LINEAR,
               DDSP_B200_E_INVALID, "harmonic_backward_f0: bad amp_method %d", amp_method);
  DDSP_REQUIRE(sample_rate > 0.f, DDSP_B200_E_INVALID,
               "harmonic_backward_f0: sample_rate must be positive");
  if (B == 0) return 0;
  DDSP_REQUIRE(B <= 65535, DDSP_B200_E_INVALID,
               "harmonic_backward_f0: B=%d exceeds the 65535 grid limit", B);
  const size_t need = sizeof(float) * 3 * (size_t)B * F;
  DDSP_REQUIRE(workspace != nullptr && workspace_bytes >= need, DDSP_B200_E_WORKSPACE,
               "harmonic_backward_f0: workspace of %zu B needed, %zu given", need,
               workspace_bytes);
  HarmonicParams p;
  p.f0 = f0_hz; p.amps = amps; p.hd = hd; p.audio = nullptr;
  p.B = B; p.F = F; p.K = K; p.N = N; p.hop = N / F;
  p.sample_rate = sample_rate; p.nyquist = sample_rate * 0.5f;
  p.inv_sr = 1.0 / (double)sample_rate;
  p.amp_method = amp_method; p.accumulate = 0; p.ctl_flags = 0;
  p.init_phase = nullptr; p.final_phase = nullptr; p.mask_nyquist = 1;
  p.Kp = (K + 3) & ~3;
  int FT = std::max(1, std::min(F, 2048 / p.hop));
  while (FT > 1 && harmonic_df0_smem(FT, p.Kp) > kMaxDynSmem) FT = (FT + 1) / 2;
  DDSP_REQUIRE(harmonic_df0_smem(FT, p.Kp) <= kMaxDynSmem, DDSP_B200_E_UNSUPPORTED,
               "harmonic_backward_f0: K=%d needs too much shared memory", K);
  p.FT = FT;
  const size_t smem = harmonic_df0_smem(FT, p.Kp);
  cudaStream_t st = (cudaStream_t)stream;
  float* sq = reinterpret_cast<float*>(workspace);
  dim3 grid((F + FT - 1) / FT, B);
  if (amp_method == DDSP_B200_AMP_WINDOW) {
    int rc = set_smem(harmonic_df0_kernel<true>, smem, "harmonic_backward_f0");
    if (rc) return rc;
    harmonic_df0_kernel<true><<<grid, kDf0Threads, smem, st>>>(p, grad_audio, sq);
  } else {
    int rc = set_smem(harmonic_df0_kernel<false>, smem, "harmonic_backward_f0");
    if (rc) return rc;
    harmonic_df0_kernel<false><<<grid, kDf0Threads, smem, st>>>(p, grad_audio, sq);
  }
  DDSP_CHECK_LAUNCH("harmonic_backward_f0");
  harmonic_df0_finalize<<<(B + 127) / 128, 128, 0, st>>>(sq, d_f0, B, F, p.hop,
                                                       (float)p.inv_sr);
  DDSP_CHECK_LAUNCH("harmonic_backward_f0(finalize)");
  return 0;
}

int ddsp_b200_harmonic_controls_backward(const float* amps_raw, const float* hd_raw,
                                         const float* f0_hz, const float* g0,
                                         const float* g1, float* d_amps_raw,
                                         float* d_hd_raw, int B, int F, int K,
                                         float sample_rate, int flags, void* stream) {
  DDSP_REQUIRE(amps_raw && hd_raw && f0_hz && g0 && g1 && d_amps_raw && d_hd_raw,
               DDSP_B200_E_INVALID, "harmonic_controls_backward: null pointer");
  DDSP_REQUIRE(B >= 0 && F >= 1 && K >= 1, DDSP_B200_E_INVALID,
               "harmonic_controls_backward: bad shape B=%d F=%d K=%d", B, F, K);
  const int64_t rows = (int64_t)B * F;
  if (rows == 0) return 0;
  DDSP_REQUIRE(rows < (1ll << 31) / 32, DDSP_B200_E_INVALID,
               "harmonic_controls_backward: B*F too large");
  const int threads = 256;
  const int blocks = (int)((rows * 32 + threads - 1) / threads);
  harmonic_controls_backward_kernel<<<blocks, threads, 0, (cudaStream_t)stream>>>(
      amps_raw, hd_raw, f0_hz, g0, g1, d_amps_raw, d_hd_raw, (int)rows, F, K,
      sample_rate * 0.5f, flags);
  DDSP_CHECK_LAUNCH("harmonic_controls_backward");
  return 0;
}

int ddsp_b200_noise_controls_backward(const float* mags_raw, const float* d_mags,
                                      float* d_raw, int64_t n, float initial_bias,
                                      void* stream) {
  DDSP_REQUIRE(mags_raw && d_mags && d_raw, DDSP_B200_E_INVALID,
               "noise_controls_backward: null pointer");
  DDSP_REQUIRE(n >= 0, DDSP_B200_E_INVALID, "noise_controls_backward: n < 0");
  if (n == 0) return 0;
  noise_controls_backward_kernel<<<grid_for(n, 256), 256, 0, (cudaStream_t)stream>>>(
      mags_raw, d_mags, d_raw, n, initial_bias);
  DDSP_CHECK_LAUNCH("noise_controls_backward");
  return 0;
}

int ddsp_b200_filtered_noise_backward(const float* grad_audio, const float* noise,
                                      uint64_t seed, uint64_t offset, float* dmags,
                                      int B, int F, int nb, int N, int window_size,
                                      void* stream) {
  DDSP_REQUIRE(grad_audio && dmags, DDSP_B200_E_INVALID,
               "filtered_noise_backward: null pointer");
  DDSP_REQUIRE(B >= 0 && F >= 1 && N >= 1 && nb >= 2, DDSP_B200_E_INVALID,
               "filtered_noise_backward: bad shape B=%d F=%d nb=%d N=%d", B, F, nb, N);
  const int frame = (N + F - 1) / F;
  DDSP_REQUIRE((N + frame - 1) / frame == F, DDSP_B200_E_INVALID,
               "filtered_noise_backward: %d frames do not tile %d samples", F, N);
  if (B == 0) return 0;
  NoiseBwdParams p;
  p.grad = grad_audio; p.noise = noise; p.dmags = dmags;
  p.seed = seed; p.offset = offset;
  p.B = B; p.F = F; p.nb = nb; p.N = N; p.frame = frame;
  p.g = make_ir_geom(nb, window_size);
  p.S = p.g.S;
  p.start = (p.S - 1) / 2 - 1;
  DDSP_REQUIRE(p.start >= 0, DDSP_B200_E_UNSUPPORTED,
               "filtered_noise_backward: impulse response too short");
  p.ylen = frame + p.S - 1;
  p.nh = p.g.S0 / 2 + 1;
  p.xS = (((frame + 15) & ~15) + 1) | 1;
  p.gS = (((frame + 15) & ~15) + p.S + 17) | 1;
  p.hS = (p.S + p.nh) | 1;
  p.tiles_per_item = (F + 31) / 32;
  const long long n_tiles = (long long)B * p.tiles_per_item;
  DDSP_REQUIRE(n_tiles < (1ll << 31), DDSP_B200_E_INVALID,
               "filtered_noise_backward: too many tiles");
  p.n_tiles = (int)n_tiles;
  p.eo_tab = (nb == 65 && p.g.S0 == 128 && p.nh == 65) ? 1 : 0;
  const size_t smem = sizeof(float) * ((size_t)p.g.S0 + p.S + 32 * (size_t)(p.xS + p.gS + p.hS) +
                                       (p.eo_tab ? (size_t)p.nh * kEoStride : 0));
  DDSP_REQUIRE(smem <= kMaxDynSmem, DDSP_B200_E_UNSUPPORTED,
               "filtered_noise_backward: shape needs %zu B of shared memory", smem);
  int rc = set_smem(noise_backward_kernel, smem, "filtered_noise_backward");
  if (rc) return rc;
  const int per_sm = smem <= 100 * 1024 ? 2 : 1;
  const int grid = (int)std::min<long long>(n_tiles, (long long)kNumSMs * per_sm);
  noise_backward_kernel<<<grid, kNbThreads, smem, (cudaStream_t)stream>>>(p);
  DDSP_CHECK_LAUNCH("filtered_noise_backward");
  return 0;
}

size_t ddsp_b200_oscillator_bank_workspace(int B, int N, int K) {
  if (B <= 0 || N <= 0 || K <= 0) return 0;
  const size_t n_chunks = ((size_t)N + kObChunk - 1) / kObChunk;
  return sizeof(unsigned long long) * (size_t)B * n_chunks * K + 256;
}

int ddsp_b200_oscillator_bank(const float* frequency_envelopes,
                              const float* amplitude_envelopes, float* out, int B,
                              int N, int K, float sample_rate, int sum_sinusoids,
                              void* workspace, size_t workspace_bytes,
                              void* stream) {
  DDSP_REQUIRE(frequency_envelopes && amplitude_envelopes && out,
               DDSP_B200_E_INVALID, "oscillator_bank: null pointer");
  DDSP_REQUIRE(B >= 0 && N >= 1 && K >= 1, DDSP_B200_E_INVALID,
               "oscillator_bank: bad shape B=%d N=%d K=%d", B, N, K);
  DDSP_REQUIRE(sample_rate > 0.f, DDSP_B200_E_INVALID,
               "oscillator_bank: sample_rate must be positive");
  if (B == 0) return 0;
  DDSP_REQUIRE(B <= 65535, DDSP_B200_E_INVALID,
               "oscillator_bank: B=%d exceeds the 65535 grid limit", B);
  const size_t need = ddsp_b200_oscillator_bank_workspace(B, N, K);
  DDSP_REQUIRE(workspace != nullptr && workspace_bytes >= need, DDSP_B200_E_WORKSPACE,
               "oscillator_bank: workspace of %zu B needed, %zu given", need,
               workspace_bytes);
  unsigned long long* sums = reinterpret_cast<unsigned long long*>(
      ((uintptr_t)workspace + 255) & ~(uintptr_t)255);
  const int n_chunks = (N + kObChunk - 1) / kObChunk;
  const double inv_sr = 1.0 / (double)sample_rate;
  cudaStream_t st = (cudaStream_t)stream;
  dim3 grid(n_chunks, B);
  oscbank_chunk_sums<<<grid, kObThreads, 0, st>>>(frequency_envelopes, sums, N, K,
                                                 n_chunks, inv_sr);
  DDSP_CHECK_LAUNCH("oscillator_bank(chunk sums)");
  const int64_t BK = (int64_t)B * K;
  oscbank_scan_chunks<<<(int)((BK + kObThreads - 1) / kObThreads), kObThreads, 0, st>>>(
      sums, K, n_chunks, BK);
  DDSP_CHECK_LAUNCH("oscillator_bank(scan)");
  if (sum_sinusoids)
    oscbank_apply<true><<<grid, kObThreads, 0, st>>>(
        frequency_envelopes, amplitude_envelopes, sums, out, N, K, n_chunks, inv_sr,
        sample_rate * 0.5f);
  else
    oscbank_apply<false><<<grid, kObThreads, 0, st>>>(
        frequency_envelopes, amplitude_envelopes, sums, out, N, K, n_chunks, inv_sr,
        sample_rate * 0.5f);
  DDSP_CHECK_LAUNCH("oscillator_bank(apply)");
  return 0;
}

size_t ddsp_b200_fft_convolve_lti_workspace(int B, int N, int S, int ir_batch) {
  if (B <= 0 || N <= 0 || S <= 0 || (ir_batch != 1 && ir_batch != B)) return 0;
  const lc::Geom g = lc::geom(N, S);
  const size_t z = (size_t)B * g.n_in * lc::M, h = (size_t)ir_batch * g.P * lc::M,
               w = (size_t)B * g.w_len;
  return sizeof(float2) * (z + h + w) + 256;
}

int ddsp_b200_fft_convolve_lti(const float* audio, const float* impulse_response,
                               float* out, int B, int N, int S, int ir_batch,
                               int start, int out_len, int accumulate, int flags,
                               void* workspace, size_t workspace_bytes, void* stream) {
  DDSP_REQUIRE(audio && impulse_response && out, DDSP_B200_E_INVALID,
               "fft_convolve_lti: null pointer");
  DDSP_REQUIRE(B >= 0 && N >= 1 && S >= 1, DDSP_B200_E_INVALID,
               "fft_convolve_lti: bad shape B=%d N=%d S=%d", B, N, S);
  // core.py:1441-1443
  DDSP_REQUIRE(ir_batch == B || ir_batch == 1, DDSP_B200_E_INVALID,
               "Batch size of audio (%d) and impulse response (%d) must be the same.",
               B, ir_batch);
  DDSP_REQUIRE(start >= 0 && out_len >= 0 &&
                   (long long)start + out_len <= (long long)N + S - 1,
               DDSP_B200_E_INVALID,
               "fft_convolve_lti: crop [%d, %d) leaves the convolution of length %lld",
               start, start + out_len, (long long)N + S - 1);
  if (B == 0 || out_len == 0) return 0;
  DDSP_REQUIRE(B <= 65535, DDSP_B200_E_INVALID,
               "fft_convolve_lti: B=%d exceeds the 65535 grid limit", B);
  const size_t need = ddsp_b200_fft_convolve_lti_workspace(B, N, S, ir_batch);
  DDSP_REQUIRE(workspace != nullptr && workspace_bytes >= need, DDSP_B200_E_WORKSPACE,
               "fft_convolve_lti: workspace of %zu B needed, %zu given", need,
               workspace_bytes);
  const lc::Geom g = lc::geom(N, S);
  float2* Z = reinterpret_cast<float2*>(((uintptr_t)workspace + 255) & ~(uintptr_t)255);
  float2* H = Z + (size_t)B * g.n_in * lc::M;
  float2* W = H + (size_t)ir_batch * g.P * lc::M;
  cudaStream_t st = (cudaStream_t)stream;
  DDSP_REQUIRE((flags & ~3) == 0, DDSP_B200_E_INVALID,
               "fft_convolve_lti: bad flags %d", flags);
  lc::lc_fft_blocks<<<dim3(g.P, ir_batch), lc::THREADS, 0, st>>>(
      impulse_response, H, S, 0, g.P, 1, (flags & DDSP_B200_LTI_REVERSE_IR) ? 1 : 0);
  DDSP_CHECK_LAUNCH("fft_convolve_lti(ir spectra)");
  lc::lc_fft_blocks<<<dim3(g.n_in, B), lc::THREADS, 0, st>>>(
      audio, Z, N, g.n2, g.n_in, 0, (flags & DDSP_B200_LTI_REVERSE_AUDIO) ? 1 : 0);
  DDSP_CHECK_LAUNCH("fft_convolve_lti(audio spectra)");
  // w blocks the crop reads: positions [start, start + out_len) through the real
  // half and [start - n2, start + out_len - n2) through the imaginary half
  const int lo_pos = std::max(0, start - g.n2);
  const int hi_pos = std::min(g.w_len, start + out_len);      // exclusive
  const int j_first = lo_pos / lc::L;
  const int j_last = std::min(g.n_out - 1, (hi_pos - 1) / lc::L);
  const int n_blocks = j_last - j_first + 1;
  {
    int rc = set_smem(lc::lc_mac_ifft, lc::kMacSmem, "fft_convolve_lti");
    if (rc) return rc;
  }
  lc::lc_mac_ifft<<<dim3((n_blocks + lc::JT - 1) / lc::JT, B), lc::THREADS, lc::kMacSmem,
                    st>>>(
      Z, H, W, g.n_in, g.P, g.n_out, ir_batch == 1 ? 0 : g.P * lc::M, j_first, n_blocks);
  DDSP_CHECK_LAUNCH("fft_convolve_lti(multiply-accumulate + inverse)");
  const int cgrid = std::min((out_len + 255) / 256, 8 * kNumSMs);
  lc::lc_combine<<<dim3(cgrid, B), 256, 0, st>>>(W, out, g.n2, g.w_len, start, out_len,
                                               N + S - 1, accumulate, j_first * lc::L,
                                               (j_last + 1) * lc::L);
  DDSP_CHECK_LAUNCH("fft_convolve_lti(combine)");
  return 0;
}

int ddsp_b200_angular_cumsum(const float* angular_frequency, float* phase, int B,
                             int N, int C, int chunk_size, int mode,
                             void* workspace, size_t workspace_bytes, void* stream) {
  DDSP_REQUIRE(angular_frequency && phase, DDSP_B200_E_INVALID,
               "angular_cumsum: null pointer");
  DDSP_REQUIRE(B >= 0 && N >= 1 && C >= 1, DDSP_B200_E_INVALID,
               "angular_cumsum: bad shape B=%d N=%d C=%d", B, N, C);
  DDSP_REQUIRE(mode >= 0 && mode <= 2, DDSP_B200_E_INVALID,
               "angular_cumsum: bad mode %d", mode);
  DDSP_REQUIRE(mode != 2 || chunk_size >= 1, DDSP_B200_E_INVALID,
               "angular_cumsum: chunk_size must be positive");
  if (B == 0) return 0;
  cudaStream_t st = (cudaStream_t)stream;
  if (mode != 0) {
    const int64_t BC = (int64_t)B * C;
    tf_sequential_cumsum<<<(int)((BC + 127) / 128), 128, 0, st>>>(
        angular_frequency, nullptr, phase, B, N, C, mode, chunk_size, 0, 1.0f);
    DDSP_CHECK_LAUNCH("angular_cumsum(tf_sequential)");
    return 0;
  }
  DDSP_REQUIRE(B <= 65535, DDSP_B200_E_INVALID,
               "angular_cumsum: B=%d exceeds the 65535 grid limit", B);
  const size_t need = ddsp_b200_oscillator_bank_workspace(B, N, C);
  DDSP_REQUIRE(workspace != nullptr && workspace_bytes >= need, DDSP_B200_E_WORKSPACE,
               "angular_cumsum: workspace of %zu B needed, %zu given", need,
               workspace_bytes);
  unsigned long long* sums = reinterpret_cast<unsigned long long*>(
      ((uintptr_t)workspace + 255) & ~(uintptr_t)255);
  const int n_chunks = (N + kObChunk - 1) / kObChunk;
  const double inv_two_pi = 0.15915494309189535;
  dim3 grid(n_chunks, B);
  oscbank_chunk_sums<<<grid, kObThreads, 0, st>>>(angular_frequency, sums, N, C,
                                                 n_chunks, inv_two_pi);
  DDSP_CHECK_LAUNCH("angular_cumsum(chunk sums)");
  const int64_t BK = (int64_t)B * C;
  oscbank_scan_chunks<<<(int)((BK + kObThreads - 1) / kObThreads), kObThreads, 0, st>>>(
      sums, C, n_chunks, BK);
  DDSP_CHECK_LAUNCH("angular_cumsum(scan)");
  oscbank_phase_out<<<grid, kObThreads, 0, st>>>(angular_frequency, sums, phase, N, C,
                                                n_chunks, inv_two_pi);
  DDSP_CHECK_LAUNCH("angular_cumsum(apply)");
  return 0;
}

int ddsp_b200_oscillator_bank_tf_sequential(const float* frequency_envelopes,
                                            const float* amplitude_envelopes,
                                            float* out, int B, int N, int K,
                                            float sample_rate, int use_angular_cumsum,
                                            int chunk_size, void* stream) {
  DDSP_REQUIRE(frequency_envelopes && amplitude_envelopes && out, DDSP_B200_E_INVALID,
               "oscillator_bank_tf_sequential: null pointer");
  DDSP_REQUIRE(B >= 0 && N >= 1 && K >= 1 && chunk_size >= 1 && sample_rate > 0.f,
               DDSP_B200_E_INVALID, "oscillator_bank_tf_sequential: bad arguments");
  if (B == 0) return 0;
  const int64_t BK = (int64_t)B * K;
  tf_sequential_cumsum<<<(int)((BK + 127) / 128), 128, 0, (cudaStream_t)stream>>>(
      frequency_envelopes, amplitude_envelopes, out, B, N, K,
      use_angular_cumsum ? 2 : 1, chunk_size, 1, sample_rate);
  DDSP_CHECK_LAUNCH("oscillator_bank_tf_sequential");
  return 0;
}

static int sinus_tile_frames(int F, int K) {
  int FT = std::min(16, F);
  while (FT > 1 && sf_smem(FT, K).total > kMaxDynSmem) FT = (FT + 1) / 2;
  return FT;
}

size_t ddsp_b200_sinusoidal_workspace(int B, int F, int K) {
  if (B <= 0 || F <= 0 || K <= 0) return 0;
  const int FT = sinus_tile_frames(F, K);
  const size_t n_tiles = ((size_t)F + FT - 1) / FT;
  return sizeof(unsigned long long) * (size_t)B * n_tiles * K + 256;
}

int ddsp_b200_sinusoidal_forward(const float* frequencies, const float* amplitudes,
                                 float* audio, int B, int F, int K, int N,
                                 float sample_rate, int amp_method, int accumulate,
                                 void* workspace, size_t workspace_bytes,
                                 void* stream) {
  DDSP_REQUIRE(frequencies && amplitudes && audio, DDSP_B200_E_INVALID,
               "sinusoidal_forward: null pointer");
  DDSP_REQUIRE(B >= 0 && F >= 1 && K >= 1 && N >= 1, DDSP_B200_E_INVALID,
               "sinusoidal_forward: bad shape B=%d F=%d K=%d N=%d", B, F, K, N);
  DDSP_REQUIRE(amp_method == DDSP_B200_AMP_WINDOW || amp_method == DDSP_B200_AMP_LINEAR,
               DDSP_B200_E_INVALID, "sinusoidal_forward: bad amp_method %d", amp_method);
  DDSP_REQUIRE(N % F == 0, DDSP_B200_E_INVALID,
               "sinusoidal_forward: n_samples (%d) must be divisible by the number "
               "of frames (%d)", N, F);
  DDSP_REQUIRE(amp_method != DDSP_B200_AMP_WINDOW || F < N, DDSP_B200_E_INVALID,
               "sinusoidal_forward: window upsampling cannot downsample (frames %d "
               ">= timesteps %d)", F, N);
  DDSP_REQUIRE(sample_rate > 0.f, DDSP_B200_E_INVALID,
               "sinusoidal_forward: sample_rate must be positive");
  if (B == 0) return 0;
  DDSP_REQUIRE(B <= 65535, DDSP_B200_E_INVALID,
               "sinusoidal_forward: B=%d exceeds the 65535 grid limit", B);
  const int FT = sinus_tile_frames(F, K);
  const SfSmem L = sf_smem(FT, K);
  DDSP_REQUIRE(L.total <= kMaxDynSmem, DDSP_B200_E_UNSUPPORTED,
               "sinusoidal_forward: K=%d needs more shared memory than one CTA has", K);
  const size_t need = ddsp_b200_sinusoidal_workspace(B, F, K);
  DDSP_REQUIRE(workspace != nullptr && workspace_bytes >= need, DDSP_B200_E_WORKSPACE,
               "sinusoidal_forward: workspace of %zu B needed, %zu given", need,
               workspace_bytes);
  unsigned long long* sums = reinterpret_cast<unsigned long long*>(
      ((uintptr_t)workspace + 255) & ~(uintptr_t)255);
  const int n_tiles = (F + FT - 1) / FT;
  const int hop = N / F;
  const double inv_sr = 1.0 / (double)sample_rate;
  cudaStream_t st = (cudaStream_t)stream;
  dim3 grid(n_tiles, B);
  sinus_tile_sums<<<grid, kSfThreads, 0, st>>>(frequencies, sums, F, K, hop, FT, n_tiles,
                                              inv_sr);
  DDSP_CHECK_LAUNCH("sinusoidal_forward(tile sums)");
  const int64_t BK = (int64_t)B * K;
  oscbank_scan_chunks<<<(int)((BK + kObThreads - 1) / kObThreads), kObThreads, 0, st>>>(
      sums, K, n_tiles, BK);
  DDSP_CHECK_LAUNCH("sinusoidal_forward(scan)");
  if (amp_method == DDSP_B200_AMP_WINDOW) {
    int rc = set_smem(sinus_apply<true>, L.total, "sinusoidal_forward");
    if (rc) return rc;
    sinus_apply<true><<<grid, kSfThreads, L.total, st>>>(
        frequencies, amplitudes, sums, audio, F, K, N, hop, FT, n_tiles, inv_sr,
        sample_rate * 0.5f, accumulate);
  } else {
    int rc = set_smem(sinus_apply<false>, L.total, "sinusoidal_forward");
    if (rc) return rc;
    sinus_apply<false><<<grid, kSfThreads, L.total, st>>>(
        frequencies, amplitudes, sums, audio, F, K, N, hop, FT, n_tiles, inv_sr,
        sample_rate * 0.5f, accumulate);
  }
  DDSP_CHECK_LAUNCH("sinusoidal_forward(apply)");
  return 0;
}

// ---- wavetable synthesis (wavetable.cuh) -------------------------------------
static inline size_t wt_align(size_t x) { return (x + 255) & ~(size_t)255; }

// Backward warp tasks walk at most kWtSeg samples; a row is read by the samples
// of two table intervals (at most 2 ceil(N / R)).
static int wt_nseg(int R, int N) {
  const long long span = 2 * (((long long)N + R - 1) / R);
  return (int)std::max<long long>(1, (span + kWtSeg - 1) / kWtSeg);
}

// Backward CTA: nw warp tasks, nw + 1 staged rows and nw accumulator rows.
static int wt_bwd_warps(int W) {
  for (int nw = 4; nw >= 1; nw >>= 1)
    if ((size_t)(2 * nw + 1) * W * sizeof(float) <= kMaxDynSmem) return nw;
  return 0;
}

size_t ddsp_b200_wavetable_workspace(int B, int F, int R, int W, int N, int backward) {
  if (B <= 0 || F <= 0 || R <= 0 || W <= 0 || N <= 0) return 0;
  size_t n = 256 + wt_align(sizeof(WtRec) * (size_t)B * F);
  if (backward) {
    n += wt_align(sizeof(float) * (size_t)B * N);
    const int nseg = wt_nseg(R, N);
    if (nseg > 1) n += wt_align(sizeof(float) * (size_t)B * R * nseg * W);
  }
  return n;
}

static int wt_check(const char* name, int B, int F, int R, int W, int N,
                    float sample_rate) {
  DDSP_REQUIRE(B >= 0 && F >= 1 && R >= 1 && W >= 1 && N >= 1, DDSP_B200_E_INVALID,
               "%s: bad shape B=%d F=%d R=%d W=%d N=%d", name, B, F, R, W, N);
  DDSP_REQUIRE(N % F == 0, DDSP_B200_E_INVALID,
               "%s: n_samples (%d) must be divisible by the number of frames (%d)",
               name, N, F);
  DDSP_REQUIRE(sample_rate > 0.f, DDSP_B200_E_INVALID,
               "%s: sample_rate must be positive", name);
  DDSP_REQUIRE(B <= 65535, DDSP_B200_E_INVALID,
               "%s: B=%d exceeds the 65535 grid limit", name, B);
  return 0;
}

int ddsp_b200_wavetable_forward(const float* f0_hz, const float* amps,
                                const float* tables, float* audio, int B, int F, int R,
                                int W, int N, float sample_rate, int scale,
                                int accumulate, void* workspace, size_t workspace_bytes,
                                void* stream) {
  DDSP_REQUIRE(f0_hz && amps && tables && audio, DDSP_B200_E_INVALID,
               "wavetable_forward: null pointer");
  int rc = wt_check("wavetable_forward", B, F, R, W, N, sample_rate);
  if (rc) return rc;
  if (B == 0) return 0;
  const int ring = (int)std::min<size_t>(4, kMaxDynSmem / (sizeof(float) * (size_t)W));
  DDSP_REQUIRE(ring >= 2, DDSP_B200_E_UNSUPPORTED,
               "wavetable_forward: a wavetable of %d samples does not fit two rows of "
               "shared memory", W);
  const size_t need = ddsp_b200_wavetable_workspace(B, F, R, W, N, 0);
  DDSP_REQUIRE(workspace != nullptr && workspace_bytes >= need, DDSP_B200_E_WORKSPACE,
               "wavetable_forward: workspace of %zu B needed, %zu given", need,
               workspace_bytes);
  WtRec* recs = reinterpret_cast<WtRec*>(((uintptr_t)workspace + 255) & ~(uintptr_t)255);
  cudaStream_t st = (cudaStream_t)stream;
  const int hop = N / F;
  wt_phase_records<<<B, 32, 0, st>>>(f0_hz, recs, F, hop, 1.0 / (double)sample_rate);
  DDSP_CHECK_LAUNCH("wavetable_forward(phase records)");

  WtParams p;
  p.tables = tables; p.amps = amps; p.rec = recs; p.out = audio;
  p.B = B; p.F = F; p.R = R; p.W = W; p.N = N; p.hop = hop;
  p.ring = ring; p.scale = scale ? 1 : 0; p.accumulate = accumulate ? 1 : 0;
  p.inv_hop = 1.0f / (float)hop;
  p.inv_n = 1.0f / (float)N;
  // ~16 table intervals per CTA, enough CTAs to cover the chip
  const long long spi = ((long long)N + R - 1) / R;
  long long tc = std::min<long long>(8192, std::max<long long>(512, 16 * spi));
  while (tc > 512 && (long long)B * ((N + tc - 1) / tc) < 4ll * kNumSMs) tc /= 2;
  p.t_chunk = (int)tc;
  const size_t smem = 128 + sizeof(float) * (size_t)ring * W;
  dim3 grid((unsigned)((N + tc - 1) / tc), B);
  const bool tma = (W % 4 == 0) && (((uintptr_t)tables & 15) == 0);
  if (tma) {
    rc = set_smem(wt_forward<true>, smem, "wavetable_forward");
    if (rc) return rc;
    wt_forward<true><<<grid, kWtThreads, smem, st>>>(p);
  } else {
    rc = set_smem(wt_forward<false>, smem, "wavetable_forward");
    if (rc) return rc;
    wt_forward<false><<<grid, kWtThreads, smem, st>>>(p);
  }
  DDSP_CHECK_LAUNCH("wavetable_forward");
  return 0;
}

int ddsp_b200_wavetable_backward(const float* f0_hz, const float* amps,
                                 const float* tables, const float* grad_audio,
                                 float* d_amps, float* d_tables, int B, int F, int R,
                                 int W, int N, float sample_rate, int scale,
                                 void* workspace, size_t workspace_bytes, void* stream) {
  DDSP_REQUIRE(f0_hz && amps && tables && grad_audio && d_amps && d_tables,
               DDSP_B200_E_INVALID, "wavetable_backward: null pointer");
  int rc = wt_check("wavetable_backward", B, F, R, W, N, sample_rate);
  if (rc) return rc;
  if (B == 0) return 0;
  const int nw = wt_bwd_warps(W);
  DDSP_REQUIRE(nw > 0, DDSP_B200_E_UNSUPPORTED,
               "wavetable_backward: a wavetable of %d samples needs more shared memory "
               "than one CTA has", W);
  const size_t need = ddsp_b200_wavetable_workspace(B, F, R, W, N, 1);
  DDSP_REQUIRE(workspace != nullptr && workspace_bytes >= need, DDSP_B200_E_WORKSPACE,
               "wavetable_backward: workspace of %zu B needed, %zu given", need,
               workspace_bytes);
  uintptr_t base = ((uintptr_t)workspace + 255) & ~(uintptr_t)255;
  WtRec* recs = reinterpret_cast<WtRec*>(base);
  base += wt_align(sizeof(WtRec) * (size_t)B * F);
  float* gl = reinterpret_cast<float*>(base);
  base += wt_align(sizeof(float) * (size_t)B * N);
  const int nseg = wt_nseg(R, N);
  float* parts = nseg > 1 ? reinterpret_cast<float*>(base) : nullptr;
  cudaStream_t st = (cudaStream_t)stream;
  const int hop = N / F;
  wt_phase_records<<<B, 32, 0, st>>>(f0_hz, recs, F, hop, 1.0 / (double)sample_rate);
  DDSP_CHECK_LAUNCH("wavetable_backward(phase records)");

  WtBwdParams p;
  p.tables = tables; p.amps = amps; p.rec = recs; p.grad = grad_audio; p.gl = gl;
  p.d_tables = d_tables; p.parts = parts;
  p.B = B; p.F = F; p.R = R; p.W = W; p.N = N; p.hop = hop;
  p.nseg = nseg; p.nw = nw; p.scale = scale ? 1 : 0;
  p.inv_hop = 1.0f / (float)hop;
  p.inv_n = 1.0f / (float)N;
  const long long n_tasks = (long long)R * nseg;
  DDSP_REQUIRE((n_tasks + nw - 1) / nw < (1ll << 31), DDSP_B200_E_INVALID,
               "wavetable_backward: too many table rows");
  const size_t smem = sizeof(float) * (size_t)(2 * nw + 1) * W;
  rc = set_smem(wt_backward, smem, "wavetable_backward");
  if (rc) return rc;
  wt_backward<<<dim3((unsigned)((n_tasks + nw - 1) / nw), B), 32 * nw, smem, st>>>(p);
  DDSP_CHECK_LAUNCH("wavetable_backward");
  if (nseg > 1) {
    const long long n = (long long)B * R * W;
    wt_reduce_parts<<<grid_for(n, 256), 256, 0, st>>>(parts, tables, d_tables,
                                                      (long long)B * R, nseg, W,
                                                      p.scale);
    DDSP_CHECK_LAUNCH("wavetable_backward(partial rows)");
  }
  const long long warps = (long long)B * F;
  wt_amp_grad<<<(unsigned)((warps * 32 + 255) / 256), 256, 0, st>>>(
      gl, amps, d_amps, B, F, N, hop, p.inv_hop, p.scale);
  DDSP_CHECK_LAUNCH("wavetable_backward(amplitudes)");
  return 0;
}

int ddsp_b200_linear_lookup(const float* phase, const float* tables, float* out, int B,
                            int N, int W, int per_sample, void* stream) {
  DDSP_REQUIRE(phase && tables && out, DDSP_B200_E_INVALID, "linear_lookup: null pointer");
  DDSP_REQUIRE(B >= 0 && N >= 0 && W >= 1, DDSP_B200_E_INVALID,
               "linear_lookup: bad shape B=%d N=%d W=%d", B, N, W);
  const long long total = (long long)B * N;
  if (total == 0) return 0;
  wt_linear_lookup<<<grid_for(total, 256), 256, 0, (cudaStream_t)stream>>>(
      phase, tables, out, B, N, W, per_sample ? 1 : 0);
  DDSP_CHECK_LAUNCH("linear_lookup");
  return 0;
}

// ---- modulated delay (mod_delay.cuh) -----------------------------------------
static int md_tiles(int N) { return (N + kMdTile - 1) / kMdTile; }

size_t ddsp_b200_mod_delay_workspace(int B, int N, int L) {
  if (B <= 0 || N <= 0 || L <= 0) return 0;
  const size_t tiles = (size_t)md_tiles(N);
  const size_t H = (size_t)std::min(L, kMdTile);
  return 256 + wt_align(sizeof(float) * (size_t)B * tiles) + wt_align(sizeof(int) * (size_t)B) +
         sizeof(unsigned long long) * (size_t)B * tiles * H;
}

static int md_setup(const char* name, MdParams& p, const float* audio, const float* gain,
                    const float* phase, int B, int N, int L, double phase_scale,
                    double phase_offset, int scale, int add_dry) {
  DDSP_REQUIRE(audio && phase, DDSP_B200_E_INVALID, "%s: null pointer", name);
  DDSP_REQUIRE(B >= 0 && N >= 1 && L >= 1, DDSP_B200_E_INVALID,
               "%s: bad shape B=%d N=%d max_length=%d", name, B, N, L);
  DDSP_REQUIRE(B <= 65535, DDSP_B200_E_INVALID, "%s: B=%d exceeds the 65535 grid limit",
               name, B);
  DDSP_REQUIRE(N <= INT32_MAX - kMdTile, DDSP_B200_E_INVALID, "%s: N=%d too long", name, N);
  p = MdParams{};
  p.audio = audio; p.gain = gain; p.phase = phase;
  p.B = B; p.N = N; p.L = L;
  p.H = std::min(L, kMdTile);
  p.tiles = md_tiles(N);
  p.p_scale = phase_scale * (double)L;
  p.p_offset = phase_offset * (double)L;
  p.scale = scale ? 1 : 0;
  p.add_dry = add_dry ? 1 : 0;
  return 0;
}

int ddsp_b200_mod_delay_forward(const float* audio, const float* gain, const float* phase,
                                float* out, int B, int N, int L, double phase_scale,
                                double phase_offset, int scale, int add_dry,
                                void* stream) {
  MdParams p;
  int rc = md_setup("mod_delay_forward", p, audio, gain, phase, B, N, L, phase_scale,
                    phase_offset, scale, add_dry);
  if (rc) return rc;
  DDSP_REQUIRE(out, DDSP_B200_E_INVALID, "mod_delay_forward: null pointer");
  if (B == 0) return 0;
  p.out = out;
  cudaStream_t st = (cudaStream_t)stream;
  const dim3 grid((unsigned)p.tiles, (unsigned)B);
  if (L <= kMdStageMax) {
    const size_t smem = sizeof(float) * ((size_t)kMdTile + L - 1);
    rc = set_smem(md_forward<true>, smem, "mod_delay_forward");
    if (rc) return rc;
    md_forward<true><<<grid, kMdThreads, smem, st>>>(p);
  } else {
    md_forward<false><<<grid, kMdThreads, 0, st>>>(p);
  }
  DDSP_CHECK_LAUNCH("mod_delay_forward");
  return 0;
}

int ddsp_b200_mod_delay_backward(const float* audio, const float* gain, const float* phase,
                                 const float* grad_out, float* d_audio, float* d_gain,
                                 float* d_phase, int B, int N, int L, double phase_scale,
                                 double phase_offset, int scale, int add_dry,
                                 void* workspace, size_t workspace_bytes, void* stream) {
  MdParams p;
  int rc = md_setup("mod_delay_backward", p, audio, gain, phase, B, N, L, phase_scale,
                    phase_offset, scale, add_dry);
  if (rc) return rc;
  DDSP_REQUIRE(grad_out && d_audio && d_phase && (d_gain || !gain), DDSP_B200_E_INVALID,
               "mod_delay_backward: null pointer");
  if (B == 0) return 0;
  const size_t need = ddsp_b200_mod_delay_workspace(B, N, L);
  DDSP_REQUIRE(workspace != nullptr && workspace_bytes >= need, DDSP_B200_E_WORKSPACE,
               "mod_delay_backward: workspace of %zu B needed, %zu given", need,
               workspace_bytes);
  uintptr_t base = ((uintptr_t)workspace + 255) & ~(uintptr_t)255;
  p.tmax = reinterpret_cast<float*>(base);
  base += wt_align(sizeof(float) * (size_t)B * p.tiles);
  p.kexp = reinterpret_cast<int*>(base);
  base += wt_align(sizeof(int) * (size_t)B);
  p.halo = reinterpret_cast<unsigned long long*>(base);
  p.grad = grad_out; p.out = d_audio; p.d_gain = gain ? d_gain : nullptr; p.d_phase = d_phase;
  cudaStream_t st = (cudaStream_t)stream;
  const dim3 grid((unsigned)p.tiles, (unsigned)B);
  md_bwd_max<<<grid, kMdThreads, 0, st>>>(p);
  DDSP_CHECK_LAUNCH("mod_delay_backward(max)");
  size_t smem = sizeof(unsigned long long) * kMdTile;
  if (L <= kMdStageMax) {
    smem += sizeof(float) * ((size_t)kMdTile + L - 1);
    rc = set_smem(md_backward<true>, smem, "mod_delay_backward");
    if (rc) return rc;
    md_backward<true><<<grid, kMdThreads, smem, st>>>(p);
  } else {
    rc = set_smem(md_backward<false>, smem, "mod_delay_backward");
    if (rc) return rc;
    md_backward<false><<<grid, kMdThreads, smem, st>>>(p);
  }
  DDSP_CHECK_LAUNCH("mod_delay_backward");
  if (p.tiles > 1) {
    const long long n = (long long)B * (p.tiles - 1) * p.H;
    md_bwd_finish<<<grid_for(n, 256), 256, 0, st>>>(p);
    DDSP_CHECK_LAUNCH("mod_delay_backward(halo)");
  }
  return 0;
}

int ddsp_b200_sigmoid(const float* x, float* y, int64_t n, void* stream) {
  DDSP_REQUIRE(x && y, DDSP_B200_E_INVALID, "sigmoid: null pointer");
  DDSP_REQUIRE(n >= 0, DDSP_B200_E_INVALID, "sigmoid: n < 0");
  if (n == 0) return 0;
  sigmoid_kernel<<<grid_for(n, 256), 256, 0, (cudaStream_t)stream>>>(x, y, n);
  DDSP_CHECK_LAUNCH("sigmoid");
  return 0;
}

int ddsp_b200_resample(const float* in, float* out, int B, int F, int C, int N,
                       int method, int add_endpoint, void* stream) {
  DDSP_REQUIRE(in && out, DDSP_B200_E_INVALID, "resample: null pointer");
  DDSP_REQUIRE(B >= 0 && F >= 1 && C >= 1 && N >= 1, DDSP_B200_E_INVALID,
               "resample: bad shape B=%d F=%d C=%d N=%d", B, F, C, N);
  DDSP_REQUIRE(method >= 0 && method <= 3, DDSP_B200_E_INVALID,
               "resample: bad method %d", method);
  if (method == 0) {
    // upsample_with_windows (core.py:676-693)
    const int n_frames = add_endpoint ? F + 1 : F;
    const int n_intervals = n_frames - 1;
    DDSP_REQUIRE(n_frames < N, DDSP_B200_E_INVALID,
                 "Upsample with windows cannot be used for downsampling"
                 "More input frames (%d) than output timesteps (%d)", n_frames, N);
    DDSP_REQUIRE(n_intervals > 0 && N % n_intervals == 0, DDSP_B200_E_INVALID,
                 "For upsampling, the target the number of timesteps must be "
                 "divisible by the number of input frames%s. (timesteps:%d, "
                 "frames:%d, add_endpoint=%s).", add_endpoint ? "" : " - 1", N,
                 n_frames, add_endpoint ? "True" : "False");
  }
  if (B == 0) return 0;
  const int64_t total = (int64_t)B * N * C;
  resample_kernel<<<grid_for(total, 256, 16), 256, 0, (cudaStream_t)stream>>>(
      in, out, B, F, C, N, method, add_endpoint);
  DDSP_CHECK_LAUNCH("resample");
  return 0;
}

int ddsp_b200_add(const float* a, const float* b, float* out, int64_t n,
                  void* stream) {
  DDSP_REQUIRE(a && b && out, DDSP_B200_E_INVALID, "add: null pointer");
  DDSP_REQUIRE(n >= 0, DDSP_B200_E_INVALID, "add: n < 0");
  if (n == 0) return 0;
  add_kernel<<<grid_for(n, 256), 256, 0, (cudaStream_t)stream>>>(a, b, out, n);
  DDSP_CHECK_LAUNCH("add");
  return 0;
}


// ---- spectrogram-loss pieces -------------------------------------------------
int ddsp_b200_frame_window(const float* audio, const float* window, float* frames,
                           int B, int N, int n_frames, int frame_size, int frame_step,
                           void* stream) {
  DDSP_REQUIRE(audio && window && frames, DDSP_B200_E_INVALID, "frame_window: null pointer");
  DDSP_REQUIRE(B >= 0 && N >= 1 && n_frames >= 1 && frame_size >= 4 && frame_size % 4 == 0 &&
                   frame_step >= 1 && B <= 65535,
               DDSP_B200_E_INVALID, "frame_window: bad shape B=%d N=%d T=%d n=%d step=%d", B,
               N, n_frames, frame_size, frame_step);
  DDSP_REQUIRE((((uintptr_t)window | (uintptr_t)frames) & 15) == 0, DDSP_B200_E_INVALID,
               "frame_window: window / frames must be 16-byte aligned");
  if (B == 0) return 0;
  const long long quads = ((long long)n_frames * frame_size) / 4;
  dim3 grid((unsigned)((quads + 255) / 256), B);
  frame_window_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(audio, window, frames, N, n_frames,
                                                            frame_size, frame_step);
  DDSP_CHECK_LAUNCH("frame_window");
  return 0;
}

int ddsp_b200_frame_window_adjoint(const float* grad_frames, const float* window,
                                   float* grad_audio, int B, int N, int n_frames,
                                   int frame_size, int frame_step,
                                   const float* scale_device, int accumulate,
                                   void* stream) {
  DDSP_REQUIRE(grad_frames && window && grad_audio, DDSP_B200_E_INVALID,
               "frame_window_adjoint: null pointer");
  DDSP_REQUIRE(B >= 0 && N >= 1 && n_frames >= 1 && frame_size >= 1 && frame_step >= 1 &&
                   B <= 65535,
               DDSP_B200_E_INVALID, "frame_window_adjoint: bad shape");
  if (B == 0) return 0;
  dim3 grid((N + 255) / 256, B);
  frame_window_adjoint_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(
      grad_frames, window, grad_audio, N, n_frames, frame_size, frame_step,
      scale_device, accumulate);
  DDSP_CHECK_LAUNCH("frame_window_adjoint");
  return 0;
}

int ddsp_b200_spectral_l1(const float* stft_target, const float* stft_value,
                          float* grad_value, double* sums, int64_t n_bins_total,
                          float mag_weight, float logmag_weight, int n_bins,
                          int irfft_size, void* stream) {
  DDSP_REQUIRE(stft_target && stft_value && grad_value && sums, DDSP_B200_E_INVALID,
               "spectral_l1: null pointer");
  DDSP_REQUIRE(n_bins_total >= 1 && n_bins >= 1 && n_bins_total % n_bins == 0 &&
                   (irfft_size == 0 || irfft_size == -1 || irfft_size == 2 * (n_bins - 1)),
               DDSP_B200_E_INVALID, "spectral_l1: bad sizes (total %lld, bins %d, irfft %d)",
               (long long)n_bins_total, n_bins, irfft_size);
  DDSP_REQUIRE((((uintptr_t)stft_target | (uintptr_t)stft_value | (uintptr_t)grad_value) & 15) == 0,
               DDSP_B200_E_INVALID, "spectral_l1: tensors must be 16-byte aligned");
  const long long blocks = std::min<long long>((n_bins_total / 2 + 255) / 256 + 1, 8ll * kNumSMs);
  spectral_l1_kernel<<<(unsigned)blocks, 256, 0, (cudaStream_t)stream>>>(
      reinterpret_cast<const float2*>(stft_target), reinterpret_cast<const float2*>(stft_value),
      reinterpret_cast<float2*>(grad_value), sums, n_bins_total, mag_weight, logmag_weight,
      1.0f / (float)n_bins_total, 1e-5f, n_bins, irfft_size);
  DDSP_CHECK_LAUNCH("spectral_l1");
  return 0;
}

#ifdef DDSP_NR_TIMING
// measurement builds only (tools/noise_timing.py): the noise_ring phase counters of
// the last launch, [148 CTAs][32 warps][8 phases] cycles
int ddsp_b200_debug_noise_timing(unsigned* host_out) {
  cudaError_t e = cudaMemcpyFromSymbol(host_out, ddsp::nr_::g_nr_timing,
                                       sizeof(unsigned) * kNumSMs * 32 * 8);
  return e == cudaSuccess ? 0 : DDSP_B200_E_CUDA;
}
#endif

}  // extern "C"
