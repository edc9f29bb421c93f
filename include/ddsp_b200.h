/*
 * ddsp_b200.h - C ABI of libddsp_b200.so (hand-written sm_100a kernels for the
 * DDSP Harmonic + FilteredNoise decoder signal path).
 *
 * The reference (magenta/ddsp v3.7.0) has no FFI: its operator API is the Python
 * Processor / ProcessorGroup protocol (ddsp/processors.py:37-158).  Every entry
 * point below replaces one or more reference *functions*; the file:line each one
 * stands for is cited.  The Python layer in ddsp_b200/ binds these with ctypes
 * and re-creates the reference classes on top (see INTEGRATION.md).
 *
 * Conventions
 *   - All tensors are contiguous row-major float32 in DEVICE memory of the
 *     current CUDA device.  Controls are [B, F, C]; audio is [B, N].
 *   - The caller allocates every input, output and workspace.  The library never
 *     allocates, frees or retains a pointer past the call (one exception, with
 *     explicit create/destroy: ddsp_b200_host_pipeline, below).
 *   - `stream` is a cudaStream_t passed as void*.  Calls are asynchronous and
 *     re-entrant; there is no global mutable state (the last-error string is
 *     thread-local).
 *   - Return value: 0 = ok, negative = DDSP_B200_E_* below.  Shape/argument
 *     errors are detected BEFORE any launch.
 */
#ifndef DDSP_B200_H_
#define DDSP_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define DDSP_B200_VERSION 200 /* 0.2.0 */

enum {
  DDSP_B200_OK = 0,
  DDSP_B200_E_INVALID = -1,   /* bad argument / shape (maps to ValueError)    */
  DDSP_B200_E_UNSUPPORTED = -2, /* valid in the reference, not built here yet */
  DDSP_B200_E_CUDA = -3,      /* CUDA runtime error (launch failed)           */
  DDSP_B200_E_WORKSPACE = -4  /* workspace too small                          */
};

/* amp_method: how frame-rate amplitudes become audio-rate (core.py:573-714). */
enum {
  DDSP_B200_AMP_WINDOW = 0,   /* upsample_with_windows, Hann OLA (default)    */
  DDSP_B200_AMP_LINEAR = 1    /* tf v1 bilinear, add_endpoint=True            */
};

/* phase_mode of the oscillator bank.  Both accumulate *wrapped* phase exactly
 * (64-bit fixed-point turns), i.e. the intent of core.angular_cumsum
 * (core.py:799-866); they differ only in how sin(k*phi) is evaluated. */
enum {
  DDSP_B200_PHASE_RECURRENCE = 0, /* Reinsch recurrence over harmonics (fast) */
  DDSP_B200_PHASE_DIRECT = 1      /* one sin per oscillator (validation)      */
};

/* flags of ddsp_b200_harmonic_controls */
enum {
  DDSP_B200_CTL_SCALE = 1,            /* apply exp_sigmoid (scale_fn)          */
  DDSP_B200_CTL_NYQUIST = 2           /* normalize_below_nyquist=True          */
};

/* padding of ddsp_b200_fir_time_varying (core.py:1338-1379) */
enum { DDSP_B200_PAD_SAME = 0, DDSP_B200_PAD_VALID = 1 };

int ddsp_b200_version(void);
/* Thread-local description of the last non-zero return on this thread. */
const char* ddsp_b200_last_error(void);
/* Number of kernels this THREAD has launched through the library so far
 * (thread-local diagnostic counter; bench.py reports it as gpu_launches). */
uint64_t ddsp_b200_launch_count(void);

/* Harmonic.get_controls (synths.py:94-121): exp_sigmoid (core.py:386-404) on
 * amplitudes and harmonic_distribution, Nyquist mask + row normalisation
 * (core.normalize_harmonics, core.py:894-907; safe_divide core.py:207-210).
 * amps_in/out [B,F,1]; hd_in/out [B,F,K]; f0_hz [B,F,1]. In-place is allowed. */
int ddsp_b200_harmonic_controls(const float* amps_in, const float* hd_in,
                                const float* f0_hz, float* amps_out,
                                float* hd_out, int B, int F, int K,
                                float sample_rate, int flags, void* stream);

/* Harmonic.get_signal = core.harmonic_synthesis (core.py:1048-1111) with
 * harmonic_shifts=None: get_harmonic_frequencies (1028-1045), resample 'linear'
 * of f0*k (573-642), resample amp*hd by amp_method (645-714), oscillator_bank
 * (911-962) incl. audio-rate remove_above_nyquist (869-891).
 * f0_hz [B,F,1], amps [B,F,1], hd [B,F,K] or NULL (K must be 1), audio [B,N].
 * N must be a multiple of F.  accumulate!=0: audio += result (fused Add).    */
int ddsp_b200_harmonic_forward(const float* f0_hz, const float* amps,
                               const float* hd, float* audio, int B, int F,
                               int K, int N, float sample_rate, int amp_method,
                               int phase_mode, int accumulate, void* stream);

/* core.streaming_harmonic_synthesis after its normalize_harmonics call =
 * resample f0 ('linear') and amplitudes (amp_method) + harmonic_oscillator_bank
 * (core.py:1151-1163, 966-1025): phase = cumsum(omega) + initial_phase, harmonic
 * k uses k * phase, NO audio-rate Nyquist mask, and the phase after the last
 * sample is returned (wrapped cumsum in [0, 2 pi) + initial_phase, as
 * angular_cumsum gives).  hd must already be normalize_harmonics'ed
 * (ddsp_b200_harmonic_controls with DDSP_B200_CTL_NYQUIST only).
 * initial_phase [B] radians or NULL; final_phase [B] or NULL. */
int ddsp_b200_streaming_harmonic_forward(const float* f0_hz, const float* amps,
                                         const float* hd, const float* initial_phase,
                                         float* audio, float* final_phase, int B,
                                         int F, int K, int N, float sample_rate,
                                         int amp_method, void* stream);

/* FilteredNoise.get_controls (synths.py:165-179): exp_sigmoid(x + bias). */
int ddsp_b200_noise_controls(const float* mag_in, float* mag_out, int64_t n,
                             float initial_bias, int apply_scale, void* stream);

/* core.frequency_impulse_response + apply_window_to_impulse_response
 * (core.py:1534-1565, 1477-1531).  mags [BF, nb] -> ir [BF, S] with
 * S = ddsp_b200_ir_size(nb, window_size). */
int ddsp_b200_ir_size(int nb, int window_size);
int ddsp_b200_frequency_impulse_response(const float* mags, float* ir,
                                         int64_t BF, int nb, int window_size,
                                         void* stream);

/* core.fft_convolve (core.py:1382-1473) restated as the equivalent direct-form
 * time-varying FIR (get_fft_size / rfft / irfft / overlap_and_add /
 * crop_and_compensate_delay folded into index math).  audio [B,N]; ir
 * [ir_batch(1 or B), F, S]; out [B, N] ('same') or [B, N+S-1] ('valid').
 * delay_compensation < 0 -> (S-1)/2 - 1 as in the reference.
 * accumulate!=0: out += result. */
int ddsp_b200_fir_time_varying(const float* audio, const float* ir, float* out,
                               int B, int N, int F, int S, int ir_batch,
                               int padding, int delay_compensation,
                               int accumulate, void* stream);

/* Uniform noise in [-1, 1): Philox4x32-10, counter = (i/4, b, offset), key =
 * seed.  Stands in for tf.random.uniform at synths.py:192-193. out [B,N]. */
int ddsp_b200_uniform_noise(float* out, int B, int N, uint64_t seed,
                            uint64_t offset, void* stream);

/* FilteredNoise.get_signal (synths.py:181-196) = noise -> frequency_filter
 * (core.py:1628-1655), fused: IRs are built in shared memory, never in HBM.
 * mags [B,F,nb]; noise [B,N] or NULL (NULL: in-kernel Philox(seed, offset));
 * audio [B,N].  accumulate!=0: audio += result (the fused processors.Add,
 * processors.py:174-176).  workspace: ddsp_b200_filtered_noise_workspace()
 * bytes (0 for the fused path; may be NULL then). */
size_t ddsp_b200_filtered_noise_workspace(int B, int F, int nb, int N,
                                          int window_size);
int ddsp_b200_filtered_noise_forward(const float* mags, const float* noise,
                                     uint64_t seed, uint64_t offset,
                                     float* audio, int B, int F, int nb, int N,
                                     int window_size, int accumulate,
                                     void* workspace, size_t workspace_bytes,
                                     void* stream);

/* The whole `ae.gin` decoder (ae.gin:47-72) from RAW network outputs in two
 * launches: ProcessorGroup.__call__ (processors.py:121-131) for the DAG
 * Harmonic -> FilteredNoise -> Add with scale_fn = exp_sigmoid.  Both
 * get_controls (synths.py:94-121, 165-179) are applied while the frame tiles
 * are staged in shared memory (controls never reach HBM), the noise kernel adds
 * into the harmonic audio (processors.py:174-176).  harmonic_flags:
 * DDSP_B200_CTL_SCALE | DDSP_B200_CTL_NYQUIST as in harmonic_controls.
 * Returns DDSP_B200_E_UNSUPPORTED outside the decoder regime (hop % 64 == 0,
 * n_frequencies <= 80); callers then use the per-processor entry points. */
int ddsp_b200_decoder_forward(const float* amps_raw, const float* hd_raw,
                              const float* f0_hz, const float* mags_raw,
                              const float* noise, uint64_t seed, uint64_t offset,
                              float* audio, int B, int F, int K, int nb, int N,
                              float sample_rate, int amp_method,
                              int harmonic_flags, int window_size,
                              float initial_bias, void* stream);

/* The same decoder for HOST buffers - what a caller of the reference's
 * ProcessorGroup.__call__ holds when its network outputs are numpy arrays
 * (processors_test.py:35-42) and it wants numpy audio back.  The batch is cut
 * into at most n_chunks groups of items whose sizes halve (16, 8, 4, 4 of 32:
 * the tail of the call is the last chunk's compute + copy-out, so it is kept
 * small); chunk c's host->device copies, its two kernels and its device->host
 * audio copy run on three streams and overlap with the neighbouring chunks', so
 * the call costs about max(H2D, compute, D2H) instead of their sum.  Results are identical to ddsp_b200_decoder_forward on the whole
 * batch (the Philox item index of a chunk's rows is offset accordingly).
 *
 * The pipeline handle owns one device staging allocation for max_B items of
 * shape (F, K, nb, N), two copy streams and the events - the only objects this
 * library ever allocates; *_destroy releases them.  A handle belongs to the
 * device that was current at creation and serialises its own calls.
 * amps_raw/f0_hz [B,F,1], hd_raw [B,F,K], mags_raw [B,F,nb], audio [B,N]: HOST
 * pointers, pinned (cudaHostAlloc / cudaHostRegister) for the copies to be
 * asynchronous.  The call returns once everything is queued; `stream` completes
 * when the audio is in host memory. */
typedef struct ddsp_b200_host_pipeline ddsp_b200_host_pipeline;
int ddsp_b200_host_pipeline_create(ddsp_b200_host_pipeline** out, int max_B, int F,
                                   int K, int nb, int N, int max_chunks);
int ddsp_b200_host_pipeline_destroy(ddsp_b200_host_pipeline* pipeline);
int ddsp_b200_decoder_forward_host(ddsp_b200_host_pipeline* pipeline,
                                   const float* amps_raw, const float* hd_raw,
                                   const float* f0_hz, const float* mags_raw,
                                   uint64_t seed, uint64_t offset, float* audio,
                                   int B, int n_chunks, float sample_rate,
                                   int amp_method, int harmonic_flags,
                                   int window_size, float initial_bias,
                                   void* stream);

/* Backward of Harmonic.get_signal w.r.t. the frame-rate harmonic amplitudes
 * ha = amplitudes * harmonic_distribution (the transpose of core.py:1096-1111;
 * the reference gets it from TF autodiff).  grad_audio [B,N] -> g0, g1 [B,F,K]:
 *   g0[i,k] = sum_{t in frame i} grad(t) w0(r) m_k(t) sin(k phi(t)),  g1 with w1;
 *   dL/dha[i,k] = g0[i,k] + g1[i-1,k] (+ g1[F-1,k] when i == F-1).
 * The frame-rate recombination is left to the caller.  d f0 is not built. */
int ddsp_b200_harmonic_backward(const float* f0_hz, const float* grad_audio,
                                float* g0, float* g1, int B, int F, int K, int N,
                                float sample_rate, int amp_method, void* stream);

/* d f0 of core.harmonic_synthesis (what the reference gets from TF autodiff through
 * the phase cumsum, core.py:947-958; needed by models/inverse_synthesis.py:84-117).
 * f0_hz, amps [B,F,1], hd [B,F,K] are synthesizer CONTROLS; grad_audio [B,N] ->
 * d_f0 [B,F].  workspace: 12 * B * F bytes (per-frame partial sums). */
int ddsp_b200_harmonic_backward_f0(const float* f0_hz, const float* amps,
                                   const float* hd, const float* grad_audio,
                                   float* d_f0, int B, int F, int K, int N,
                                   float sample_rate, int amp_method,
                                   void* workspace, size_t workspace_bytes,
                                   void* stream);

/* Backward of Harmonic.get_controls (synths.py:94-121) fused with the frame-rate
 * recombination of ddsp_b200_harmonic_backward's g0 / g1: from the RAW network
 * outputs (amps_raw [B,F,1], hd_raw [B,F,K]) and f0_hz to d amps_raw, d hd_raw -
 * exp_sigmoid' (core.py:386-404), the Nyquist mask and the row normalisation
 * (core.py:894-907, 207-210) transposed.  flags as ddsp_b200_harmonic_controls. */
int ddsp_b200_harmonic_controls_backward(const float* amps_raw, const float* hd_raw,
                                         const float* f0_hz, const float* g0,
                                         const float* g1, float* d_amps_raw,
                                         float* d_hd_raw, int B, int F, int K,
                                         float sample_rate, int flags, void* stream);

/* Backward of FilteredNoise.get_controls (synths.py:165-179):
 * d raw = d magnitudes * exp_sigmoid'(raw + initial_bias), n elements. */
int ddsp_b200_noise_controls_backward(const float* mags_raw, const float* d_mags,
                                      float* d_raw, int64_t n, float initial_bias,
                                      void* stream);

/* Backward of FilteredNoise.get_signal w.r.t. magnitudes (controls): the
 * transpose of core.frequency_filter (core.py:1628-1655) for the same noise
 * (caller-supplied, or the Philox stream of (seed, offset)).
 * grad_audio [B,N] -> dmags [B,F,nb]. */
int ddsp_b200_filtered_noise_backward(const float* grad_audio, const float* noise,
                                      uint64_t seed, uint64_t offset, float* dmags,
                                      int B, int F, int nb, int N, int window_size,
                                      void* stream);

/* core.oscillator_bank (core.py:911-962) on audio-rate envelopes [B,N,K]:
 * Nyquist mask, exact wrapped phase accumulation (three-pass chunked scan in
 * 64-bit fixed point), amp * sin(phase), summed over k when sum_sinusoids != 0
 * (out [B,N]) or not (out [B,N,K]).  workspace: *_workspace(B,N,K) bytes. */
size_t ddsp_b200_oscillator_bank_workspace(int B, int N, int K);
int ddsp_b200_oscillator_bank(const float* frequency_envelopes,
                              const float* amplitude_envelopes, float* out, int B,
                              int N, int K, float sample_rate, int sum_sinusoids,
                              void* workspace, size_t workspace_bytes,
                              void* stream);

/* core.fft_convolve (core.py:1382-1473) with ONE impulse response per item of any
 * length (the LTI case: effects.Reverb, effects.py:103-117, 48000 taps): uniformly
 * partitioned overlap-save convolution, 1024-sample blocks, hand-written 2048-point
 * FFTs.  audio [B,N], impulse_response [ir_batch (1 or B), S] -> out [B,out_len] =
 * full convolution [start, start + out_len) (crop_and_compensate_delay,
 * core.py:1338-1379; start + out_len <= N + S - 1).  workspace:
 * ddsp_b200_fft_convolve_lti_workspace(B, N, S, ir_batch) bytes.
 * flags: DDSP_B200_LTI_REVERSE_AUDIO / _IR read that operand back to front - the
 * backward pass is the same convolution on time-reversed signals:
 *   d audio = (g * reverse(ir)) [S-1-start, +N),  d ir = (g * reverse(audio)) [N-1-start, +S). */
enum { DDSP_B200_LTI_REVERSE_AUDIO = 1, DDSP_B200_LTI_REVERSE_IR = 2 };
size_t ddsp_b200_fft_convolve_lti_workspace(int B, int N, int S, int ir_batch);
int ddsp_b200_fft_convolve_lti(const float* audio, const float* impulse_response,
                               float* out, int B, int N, int S, int ir_batch,
                               int start, int out_len, int accumulate, int flags,
                               void* workspace, size_t workspace_bytes, void* stream);

/* core.angular_cumsum (core.py:799-866) and tf.cumsum (core.py:955) on
 * [B,N,C] float32 (C = product of the trailing axes).  mode:
 *   0  exact: the wrapped running sum in 64-bit fixed point (what angular_cumsum
 *      approximates), radians in [0, 2 pi); three-pass scan, workspace =
 *      ddsp_b200_oscillator_bank_workspace(B,N,C) bytes;
 *   1  tf_sequential, tf.cumsum: float32 running sum in the reference's order;
 *   2  tf_sequential, angular_cumsum: float32, chunked by chunk_size with the
 *      reference's mod-2pi stitching (debug mode: reproduces TensorFlow's own
 *      float32 error, one thread per (b, c) - small shapes).
 * ddsp_b200_oscillator_bank_tf_sequential is core.oscillator_bank evaluated that
 * way end to end (omega = f * 2pi / sr in float32, modes 1 / 2, Nyquist mask,
 * amp * sin(phase)); out is [B,N,K], the sum over k is left to the caller. */
int ddsp_b200_angular_cumsum(const float* angular_frequency, float* phase, int B,
                             int N, int C, int chunk_size, int mode,
                             void* workspace, size_t workspace_bytes, void* stream);
int ddsp_b200_oscillator_bank_tf_sequential(const float* frequency_envelopes,
                                            const float* amplitude_envelopes,
                                            float* out, int B, int N, int K,
                                            float sample_rate, int use_angular_cumsum,
                                            int chunk_size, void* stream);

/* Frame-rate oscillator bank with per-sinusoid frequencies: the fusion of
 * resample(frequencies) + resample(amplitudes, amp_method) + oscillator_bank
 * for synths.Sinusoidal.get_signal (synths.py:305-323) and for
 * core.harmonic_synthesis with harmonic_shifts (core.py:1084-1111; the caller
 * forms f0 * k * (1 + shifts) and amp * hd at frame rate, as the reference does).
 * frequencies, amplitudes [B,F,K] -> audio [B,N] (summed over k), N % F == 0.
 * workspace: ddsp_b200_sinusoidal_workspace(B,F,K) bytes. */
size_t ddsp_b200_sinusoidal_workspace(int B, int F, int K);
int ddsp_b200_sinusoidal_forward(const float* frequencies, const float* amplitudes,
                                 float* audio, int B, int F, int K, int N,
                                 float sample_rate, int amp_method, int accumulate,
                                 void* workspace, size_t workspace_bytes,
                                 void* stream);

/* Wavetable synthesis: core.wavetable_synthesis / synths.Wavetable.get_signal
 * (core.py:1212-1282, synths.py:238-257) in one pass over the frame-rate tables.
 * f0_hz, amps [B,F] (hop N/F, N % F == 0; F == N: audio-rate controls, hop 1),
 * tables [B,R,W]: R table frames linearly interpolated in time (src = t R / N,
 * last frame held); R == 1 is a static table.  The phase is the EXCLUSIVE cumsum
 * of f0/sr mod 1 (64-bit fixed point), amps are Hann-upsampled ('window').
 * scale != 0: amps and tables are raw network outputs and exp_sigmoid
 * (Wavetable.get_controls, synths.py:212-236) is applied inside the kernel, with
 * the same device function as ddsp_b200_noise_controls.
 * workspace: ddsp_b200_wavetable_workspace(B,F,R,W,N,0) bytes (forward) or
 * (...,1) (backward).
 * backward: grad_audio [B,N] -> d_amps [B,F], d_tables [B,R,W] (w.r.t. the raw
 * inputs when scale != 0); deterministic, every element written once.  f0 gets
 * no gradient. */
size_t ddsp_b200_wavetable_workspace(int B, int F, int R, int W, int N, int backward);
int ddsp_b200_wavetable_forward(const float* f0_hz, const float* amps,
                                const float* tables, float* audio, int B, int F, int R,
                                int W, int N, float sample_rate, int scale,
                                int accumulate, void* workspace, size_t workspace_bytes,
                                void* stream);
int ddsp_b200_wavetable_backward(const float* f0_hz, const float* amps,
                                 const float* tables, const float* grad_audio,
                                 float* d_amps, float* d_tables, int B, int F, int R,
                                 int W, int N, float sample_rate, int scale,
                                 void* workspace, size_t workspace_bytes, void* stream);
/* core.linear_lookup (core.py:1168-1209): phase [B,N] (any value), tables [B,W]
 * (per_sample = 0) or [B,N,W] (per_sample = 1) -> out [B,N]. */
int ddsp_b200_linear_lookup(const float* phase, const float* tables, float* out, int B,
                            int N, int W, int per_sample, void* stream);

/* Modulated delay: core.variable_length_delay / effects.ModDelay.get_signal
 * (core.py:1285-1313, effects.py:328-393) in one pass over the audio.
 * audio, phase [B,N], gain [B,N] or NULL (gain 1), L = max_length >= 1.  Sample n
 * reads the entries e_k = audio[n-k] (0 <= k < L, zero before the start) and
 * e_L = e_0 with linear_lookup's rule at position (phase*phase_scale +
 * phase_offset)*L (double), times gain, + audio[n] when add_dry.
 * variable_length_delay is phase_scale 1, phase_offset 0, no gain, no add_dry.
 * scale != 0: gain and phase are raw network outputs and exp_sigmoid / sigmoid
 * (ModDelay.get_controls' defaults) are applied inside the kernel, with the same
 * device functions as ddsp_b200_noise_controls and ddsp_b200_sigmoid.
 * backward: grad_out [B,N] -> d_audio [B,N], d_gain [B,N] (when gain), d_phase
 * [B,N] (w.r.t. the raw inputs when scale != 0).  d_audio is summed in 64-bit
 * fixed point with integer atomics: bit-reproducible, no float atomics.
 * workspace: ddsp_b200_mod_delay_workspace(B,N,L) bytes (backward only). */
size_t ddsp_b200_mod_delay_workspace(int B, int N, int L);
int ddsp_b200_mod_delay_forward(const float* audio, const float* gain, const float* phase,
                                float* out, int B, int N, int L, double phase_scale,
                                double phase_offset, int scale, int add_dry,
                                void* stream);
int ddsp_b200_mod_delay_backward(const float* audio, const float* gain, const float* phase,
                                 const float* grad_out, float* d_audio, float* d_gain,
                                 float* d_phase, int B, int N, int L, double phase_scale,
                                 double phase_offset, int scale, int add_dry,
                                 void* workspace, size_t workspace_bytes, void* stream);
/* tf.nn.sigmoid elementwise (core.sigmoid, ModDelay's default phase_scale_fn),
 * n elements. */
int ddsp_b200_sigmoid(const float* x, float* y, int64_t n, void* stream);

/* core.resample / core.upsample_with_windows (core.py:573-714) stand-alone:
 * in [B,F,C] -> out [B,N,C].  method: 0 'window', 1 'linear', 2 'nearest',
 * 3 'cubic' (tf.compat.v1 bicubic, Keys A = -0.75).  add_endpoint as in the
 * reference.  4-D inputs [B,F,n_freq,C] are the 3-D case with n_freq*C channels
 * (the reference resizes the n_freq axis to itself, core.py:616-621). */
int ddsp_b200_resample(const float* in, float* out, int B, int F, int C, int N,
                       int method, int add_endpoint, void* stream);

/* Pieces of losses.SpectralLoss (losses.py:130-243) around cuFFT.
 * frame_window: tf.signal.stft's framing + periodic Hann window with pad_end=True
 * (spectral_ops.py:34-47): audio [B,N] -> frames [B, n_frames, frame_size],
 * frames[b,t,i] = window[i] * audio[b, t*frame_step + i] (0 past the end).
 * frame_window_adjoint: its transpose, grad_frames -> grad_audio [B,N], times the
 * optional DEVICE scalar *scale_device (NULL = 1), added to grad_audio when
 * accumulate != 0 (the FFT sizes of the multi-scale loss share one buffer).
 * spectral_l1: for complex STFTs [n_bins_total] (interleaved re/im) of target and
 * value: sums[0] += sum |mag_t - mag_v|, sums[1] += sum |safe_log mag_t -
 * safe_log mag_v| (core.py:213-216), and grad_value = d/dX_v of
 * mag_weight * mean|.| + logmag_weight * mean|.| (losses.py:102-127, 'L1').
 * n_bins = bins per frame.  irfft_size = 0: grad_value is the plain gradient;
 * irfft_size = 2 (n_bins - 1): it is pre-scaled so that irfft(grad_value,
 * irfft_size) is the gradient w.r.t. the real frames (the transpose of rfft);
 * irfft_size = -1: the same for an UNNORMALISED inverse transform (no 1/n pass).
 * sums must be zeroed by the caller. */
int ddsp_b200_frame_window(const float* audio, const float* window, float* frames,
                           int B, int N, int n_frames, int frame_size, int frame_step,
                           void* stream);
int ddsp_b200_frame_window_adjoint(const float* grad_frames, const float* window,
                                   float* grad_audio, int B, int N, int n_frames,
                                   int frame_size, int frame_step,
                                   const float* scale_device, int accumulate,
                                   void* stream);
int ddsp_b200_spectral_l1(const float* stft_target, const float* stft_value,
                          float* grad_value, double* sums, int64_t n_bins_total,
                          float mag_weight, float logmag_weight, int n_bins,
                          int irfft_size, void* stream);

/* processors.Add.get_signal (processors.py:174-176). out may alias a or b. */
int ddsp_b200_add(const float* a, const float* b, float* out, int64_t n,
                  void* stream);

#ifdef __cplusplus
}
#endif
#endif /* DDSP_B200_H_ */
