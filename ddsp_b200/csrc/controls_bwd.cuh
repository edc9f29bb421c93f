// Backward of the frame-rate controls (synths.Harmonic.get_controls,
// synths.py:94-121; synths.FilteredNoise.get_controls, synths.py:165-179) and the
// d f0 path of the harmonic synthesizer - the pieces that let the C4 training step
// (decoder forward + backward through SpectralLoss) run from RAW network outputs
// without a single frame-rate torch op.  The reference gets all of this from TF
// autodiff through core.exp_sigmoid (core.py:386-404), core.normalize_harmonics
// (core.py:894-907) and core.oscillator_bank's cumsum (core.py:947-958).
#pragma once
#include "common.cuh"
#include "harmonic.cuh"

namespace ddsp {

// exp_sigmoid(x) = 2 sigmoid(x)^ln10 + 1e-7 and its derivative
//   y' = (y - 1e-7) ln10 (1 - sigmoid(x)),  1 - sigmoid(x) = t / (1 + t), t = e^-x
// (t = inf, x << 0, is taken as the limit 1).
__device__ __forceinline__ float exp_sigmoid_grad(float x, float* y_out) {
  const float kLog2e = 1.4426950408889634f;
  const float kLn10 = 2.302585092994046f;
  const float t = ex2_approx(-x * kLog2e);
  float l;
  asm("lg2.approx.ftz.f32 %0, %1;" : "=f"(l) : "f"(1.0f + t));
  const float core = 2.0f * ex2_approx(-kLn10 * l);          // y - 1e-7
  *y_out = core + 1e-7f;
  const float one_minus_sig = (t < 1e30f) ? t * __frcp_rn(1.0f + t) : 1.0f;
  return core * kLn10 * one_minus_sig;
}

// sigmoid_f and its derivative s (1 - s), taken as t s^2 (t = e^-x) for x >= 0
// where 1 - s would cancel.
__device__ __forceinline__ float sigmoid_grad(float x, float* y_out) {
  const float t = ex2_approx(-x * 1.4426950408889634f);
  const float s = __frcp_rn(1.0f + t);
  *y_out = s;
  return x < 0.f ? s * (1.0f - s) : t * s * s;
}

// One warp per (b, i) row.
//   dha[k]   = g0[i,k] + g1[i-1,k] (i > 0) + g1[F-1,k] (i == F-1)      (backward.cuh)
//   n        = e / sum(e), e = exp_sigmoid(hd_raw) on the live prefix (f0 k < sr/2)
//   d amp    = sum_k dha[k] n[k];   d n[k] = dha[k] amp
//   d e[k]   = (d n[k] - sum_j d n[j] n[j]) / sum(e)
//   d hd_raw = d e * exp_sigmoid'(hd_raw);  d amps_raw = d amp * exp_sigmoid'(amps_raw)
// flags: DDSP_B200_CTL_SCALE (exp_sigmoid applied), DDSP_B200_CTL_NYQUIST.
__global__ void __launch_bounds__(256)
harmonic_controls_backward_kernel(const float* __restrict__ amps_raw,
                                  const float* __restrict__ hd_raw,
                                  const float* __restrict__ f0,
                                  const float* __restrict__ g0,
                                  const float* __restrict__ g1,
                                  float* __restrict__ d_amps_raw,
                                  float* __restrict__ d_hd_raw, int rows, int F, int K,
                                  float nyquist, int flags) {
  const int row = (int)(((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5);
  const int lane = threadIdx.x & 31;
  if (row >= rows) return;
  const int i = row % F;
  const bool scale = flags & DDSP_B200_CTL_SCALE;
  const float f = f0[row];
  int live = K;
  if ((flags & DDSP_B200_CTL_NYQUIST) && f > 0.f) {
    int k = (int)fminf(nyquist / f, (float)K);
    while (k < K && __fmul_rn(f, (float)(k + 1)) < nyquist) ++k;
    while (k > 0 && !(__fmul_rn(f, (float)k) < nyquist)) --k;
    live = k;
  }
  const float* hr = hd_raw + (size_t)row * K;
  const float* g0r = g0 + (size_t)row * K;
  const float* g1p = (i > 0) ? g1 + (size_t)(row - 1) * K : nullptr;
  const float* g1l = (i == F - 1) ? g1 + (size_t)row * K : nullptr;
  float* dr = d_hd_raw + (size_t)row * K;

  float amp = amps_raw[row], damp_dx = 1.0f;
  if (scale) damp_dx = exp_sigmoid_grad(amp, &amp);

  // pass 1: sum(e), sum(dha e)
  float se = 0.f, sde = 0.f;
  for (int k = lane; k < live; k += 32) {
    float e = hr[k];
    if (scale) e = exp_sigmoid_f(e);
    float d = g0r[k];
    if (g1p) d += g1p[k];
    if (g1l) d += g1l[k];
    se += e;
    sde = fmaf(d, e, sde);
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    se += __shfl_xor_sync(0xffffffffu, se, o);
    sde += __shfl_xor_sync(0xffffffffu, sde, o);
  }
  const float denom = (se == 0.0f) ? 1e-7f : se;          // safe_divide, core.py:207-210
  const float inv = 1.0f / denom;
  const float dot = sde * inv;                             // sum_k dha[k] n[k] = d amp
  // with the safe denominator a constant (se == 0) there is no coupling term
  const float couple = (se == 0.0f) ? 0.f : dot;
  // pass 2
  for (int k = lane; k < K; k += 32) {
    float out = 0.f;
    if (k < live) {
      float y = hr[k], dy = 1.0f;
      if (scale) dy = exp_sigmoid_grad(y, &y);
      float d = g0r[k];
      if (g1p) d += g1p[k];
      if (g1l) d += g1l[k];
      out = amp * (d - couple) * inv * dy;
    }
    dr[k] = out;
  }
  if (lane == 0) d_amps_raw[row] = dot * damp_dx;
}

// FilteredNoise.get_controls backward: magnitudes = exp_sigmoid(raw + bias).
__global__ void __launch_bounds__(256)
noise_controls_backward_kernel(const float* __restrict__ mags_raw,
                               const float* __restrict__ dmags, float* __restrict__ d_raw,
                               int64_t n, float bias) {
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (; i < n; i += stride) {
    float y;
    const float dy = exp_sigmoid_grad(mags_raw[i] + bias, &y);
    d_raw[i] = dmags[i] * dy;
  }
}

// ---------------------------------------------------------------------------
// d f0 of core.harmonic_synthesis.  With phi in turns,
//   d audio(t) / d phi(t) = 2 pi sum_k k a_k(t) m_k(t) cos(2 pi k phi(t)),
//   c(t) = g(t) * that;  sr * phi(t) is a linear function of the frame values f0[j]
// (the transpose of resample('linear') followed by cumsum), which for a sample at
// offset r of frame i gives weights alpha = (hop+1)/2 and beta = (hop-1)/2 for the
// completed frames and p0(r) = (r+1) - r(r+1)/(2 hop), p1(r) = r(r+1)/(2 hop) for the
// current one.  Pass 1 (this kernel) reduces per frame
//   S_i = sum_r c,  Q0_i = sum_r c p0(r),  Q1_i = sum_r c p1(r);
// pass 2 (harmonic_df0_finalize) is the frame-rate suffix sum.
// Controls here are the synthesizer controls (amplitudes, normalised
// harmonic_distribution).  One thread per sample, one sincospif per oscillator.
// ---------------------------------------------------------------------------
constexpr int kDf0Threads = 256;

template <bool WINDOW>
__global__ void __launch_bounds__(kDf0Threads)
harmonic_df0_kernel(HarmonicParams p, const float* __restrict__ grad,
                    float* __restrict__ sq /* [B, F, 3] */) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  const int FT = p.FT, Kp = p.Kp, K = p.K, F = p.F, hop = p.hop;
  unsigned long long* sP = reinterpret_cast<unsigned long long*>(smem_raw);
  unsigned long long* sA = sP + FT;
  unsigned long long* sD = sA + FT;
  unsigned long long* sRed = sD + FT;
  float* sF0 = reinterpret_cast<float*>(sRed + 8);
  float* sAmp = sF0 + (FT + 1);
  float* sAcc = sAmp + (FT + 1);                 // [FT][3]
  float* sX = sAcc + 3 * FT + ((3 * FT) & 1);
  const int b = blockIdx.y;
  const int i0 = blockIdx.x * FT;
  const int nfr = min(FT, F - i0);
  const int tid = threadIdx.x;
  const float* f0b = p.f0 + (size_t)b * F;
  const float* ampb = p.amps + (size_t)b * F;

  unsigned long long part = 0;
  for (int j = tid; j < i0; j += kDf0Threads) {
    double a0 = (double)f0b[j] * p.inv_sr;
    double a1 = (double)f0b[min(j + 1, F - 1)] * p.inv_sr;
    part += turns_to_fix64((double)hop * a0 + (a1 - a0) * (0.5 * (hop - 1)));
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) part += __shfl_xor_sync(0xffffffffu, part, o);
  if ((tid & 31) == 0) sRed[tid >> 5] = part;
  for (int j = tid; j <= nfr; j += kDf0Threads) {
    int g = min(i0 + j, F - 1);
    sF0[j] = f0b[g];
    sAmp[j] = ampb[g];
  }
  for (int j = tid; j < 3 * FT; j += kDf0Threads) sAcc[j] = 0.f;
  if (p.hd != nullptr) {
    const float* hdb = p.hd + ((size_t)b * F + i0) * K;
    const int rows_in = min(nfr + 1, F - i0);
    for (int idx = tid; idx < rows_in * K; idx += kDf0Threads) {
      int r = idx / K, c = idx - r * K;
      sX[r * Kp + c] = hdb[idx];
    }
    if (rows_in < nfr + 1) {
      for (int c = tid; c < K; c += kDf0Threads)
        sX[nfr * Kp + c] = hdb[(size_t)(nfr - 1) * K + c];
    }
  } else {
    for (int j = tid; j <= nfr; j += kDf0Threads) sX[j * Kp] = 1.0f;
  }
  __syncthreads();
  if (tid == 0) {
    unsigned long long P = 0;
    for (int w = 0; w < kDf0Threads / 32; ++w) P += sRed[w];
    for (int j = 0; j < nfr; ++j) {
      double a0 = (double)sF0[j] * p.inv_sr;
      double a1 = (double)sF0[j + 1] * p.inv_sr;
      sP[j] = P;
      sA[j] = turns_to_fix64(a0);
      sD[j] = turns_to_fix64((a1 - a0) / (double)hop);
      P += turns_to_fix64((double)hop * a0 + (a1 - a0) * (0.5 * (hop - 1)));
    }
  }
  __syncthreads();

  const int n_tile = nfr * hop;
  const float inv_hop = 1.0f / (float)hop;
  const float* gb = grad + (size_t)b * p.N + (size_t)i0 * hop;
  const int n_iter = (n_tile + kDf0Threads - 1) / kDf0Threads;
  for (int it = 0; it < n_iter; ++it) {
    const int lt = it * kDf0Threads + tid;
    const bool ok = lt < n_tile;
    const int li = ok ? lt / hop : 0;
    float c = 0.f, q0 = 0.f, q1 = 0.f;
    if (ok) {
      const int r = lt - li * hop;
      const float frac = (float)r * inv_hop;
      const float f_lo = sF0[li], f_hi = sF0[li + 1];
      unsigned long long ph = sP[li] + (unsigned long long)(r + 1) * sA[li] +
          (unsigned long long)(((long long)r * (r + 1)) >> 1) * sD[li];
      const uint32_t p32 = (uint32_t)((ph + 0x80000000ull) >> 32);
      float w1 = WINDOW ? (0.5f - 0.5f * cospif(frac)) : frac;
      const float w0 = (1.0f - w1) * sAmp[li];
      w1 *= sAmp[li + 1];
      const float* x0 = sX + li * Kp;
      const float* x1 = x0 + Kp;
      const bool monotone = (f_lo >= 1.0f) && (f_hi >= 1.0f);
      const int klive = monotone ? live_harmonics(f_lo, f_hi, frac, K, p.nyquist) : K;
      float acc = 0.f;
      uint32_t pk = 0;
      for (int k = 1; k <= klive; ++k) {
        pk += p32;
        float a = x0[k - 1] * w0 + x1[k - 1] * w1;
        if (!monotone && !(ref_harmonic_freq(f_lo, f_hi, frac, k) < p.nyquist)) a = 0.f;
        acc = fmaf(a * (float)k, cospif((float)(int)pk * 4.656612873077393e-10f), acc);
      }
      c = gb[lt] * 6.283185307179586f * acc;
      const float tri = (float)r * (float)(r + 1) * (0.5f * inv_hop);
      q1 = c * tri;
      q0 = c * ((float)(r + 1) - tri);
    }
    // per-frame reduction: a warp whose lanes all sit in one frame reduces by
    // shuffles; otherwise shared-memory atomics
    const unsigned full = 0xffffffffu;
    const int li0 = __shfl_sync(full, li, 0);
    const bool same = __all_sync(full, ok && li == li0);
    if (same) {
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) {
        c += __shfl_xor_sync(full, c, o);
        q0 += __shfl_xor_sync(full, q0, o);
        q1 += __shfl_xor_sync(full, q1, o);
      }
      if ((tid & 31) == 0) {
        atomicAdd(&sAcc[3 * li0 + 0], c);
        atomicAdd(&sAcc[3 * li0 + 1], q0);
        atomicAdd(&sAcc[3 * li0 + 2], q1);
      }
    } else if (ok) {
      atomicAdd(&sAcc[3 * li + 0], c);
      atomicAdd(&sAcc[3 * li + 1], q0);
      atomicAdd(&sAcc[3 * li + 2], q1);
    }
  }
  __syncthreads();
  for (int j = tid; j < 3 * nfr; j += kDf0Threads)
    sq[((size_t)b * F + i0) * 3 + j] = sAcc[j];
}

inline size_t harmonic_df0_smem(int FT, int Kp) {
  return sizeof(unsigned long long) * (3 * (size_t)FT + 8) +
         sizeof(float) * (2 * (size_t)(FT + 1) + 3 * (size_t)FT + 1 +
                          (size_t)(FT + 1) * Kp);
}

// pass 2: one thread per batch item walks the frames backwards.
//   d f0[j] = inv_sr [ (alpha + beta [j>=1]) Suf_j + beta [j>=1] S_j + Q0_j
//                      + Q1_{j-1} [j>=1] + Q1_{F-1} [j == F-1] ],  Suf_j = sum_{i>j} S_i
__global__ void __launch_bounds__(128)
harmonic_df0_finalize(const float* __restrict__ sq, float* __restrict__ d_f0, int B,
                      int F, int hop, float inv_sr) {
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= B) return;
  const float alpha = 0.5f * (float)(hop + 1), beta = 0.5f * (float)(hop - 1);
  const float* s = sq + (size_t)b * F * 3;
  float* out = d_f0 + (size_t)b * F;
  double suf = 0.0;
  for (int j = F - 1; j >= 0; --j) {
    const float S = s[3 * j], Q0 = s[3 * j + 1];
    double v = (double)(alpha + (j >= 1 ? beta : 0.f)) * suf + (double)Q0;
    if (j >= 1) v += (double)beta * S + (double)s[3 * (j - 1) + 2];
    if (j == F - 1) v += (double)s[3 * j + 2];
    out[j] = (float)(v * (double)inv_sr);
    suf += (double)S;
  }
}

}  // namespace ddsp
