// Modulated delay: core.variable_length_delay (core.py:1285-1313) and
// effects.ModDelay.get_signal (effects.py:328-393) without the reference's
// [B, N, L] frames and [B, N, L + 1] lookup weights.
//
// Per batch item, L = max_length, sample n:
//   e_k(n)  = x[n - k] for 0 <= k < L (x[m < 0] = 0: the reference zero-pads L - 1
//             samples in front), e_L(n) = e_0(n) = x[n] (linear_lookup wraps)
//   p(n)    = (phase(n) a + c) L, one double FMA (a = 1, c = 0 for the bare delay;
//             a = depth / (center + depth), c = center / (center + depth) for ModDelay)
//   wet(n)  = linear_lookup's two taps of e(n) at p(n) (lookup_taps, wavetable.cuh)
//   out(n)  = gain(n) wet(n) [+ x[n] with add_dry]
// With `scale`, gain and phase are raw network outputs: exp_sigmoid_f and
// sigmoid_f (common.cuh) are applied here, the functions behind core.exp_sigmoid
// and core.sigmoid.  DESIGN.md section 3.12 has the derivation and the measured
// bound.
#pragma once
#include "common.cuh"
#include "controls_bwd.cuh"
#include "wavetable.cuh"

namespace ddsp {

constexpr int kMdThreads = 256;
constexpr int kMdPer = 8;                          // samples per thread
constexpr int kMdTile = kMdThreads * kMdPer;       // samples per CTA
constexpr int kMdStageMax = 4096;                  // L up to this: history in smem

struct MdParams {
  const float* __restrict__ audio;    // [B, N]
  const float* __restrict__ gain;     // [B, N] or null (gain 1)
  const float* __restrict__ phase;    // [B, N]
  const float* __restrict__ grad;     // backward: [B, N]
  float* __restrict__ out;            // forward: [B, N]; backward: d_audio
  float* __restrict__ d_gain;         // backward, null without gain
  float* __restrict__ d_phase;        // backward
  float* __restrict__ tmax;           // backward workspace: [B, tiles] max |g gain|
  int* __restrict__ kexp;             // backward workspace: [B] fixed-point exponent
  unsigned long long* __restrict__ halo;   // backward workspace: [B, tiles, H]
  double p_scale, p_offset;           // p = phase p_scale + p_offset = (phase a + c) L
  int B, N, L, H, tiles;
  int scale, add_dry;
};

// Audio sample m of the current item: from the staged history (m >= h0) or through
// L1 / L2; zero before the start.
template <bool STAGE>
__device__ __forceinline__ float md_x(const float* __restrict__ hist,
                                      const float* __restrict__ xb, int h0, int m) {
  if (STAGE) return hist[m - h0];
  return m >= 0 ? __ldg(xb + m) : 0.f;
}

// Stage x[h0 .. n1) (zeros before 0) into shared memory.
__device__ __forceinline__ void md_stage(float* __restrict__ hist,
                                         const float* __restrict__ xb, int h0, int n1) {
  for (int i = threadIdx.x; i < n1 - h0; i += kMdThreads) {
    const int m = h0 + i;
    hist[i] = m >= 0 ? xb[m] : 0.f;
  }
}

// ---- forward ----------------------------------------------------------------------
// A CTA owns kMdTile samples of one item.  The controls of all its samples are
// loaded first (8 per thread in flight), then, with STAGE, the tile and its L - 1
// samples of history land in shared memory; otherwise the taps are read through
// L1 / L2.
template <bool STAGE>
__global__ void __launch_bounds__(kMdThreads)
md_forward(MdParams p) {
  extern __shared__ float md_hist[];
  const int b = blockIdx.y, tid = threadIdx.x;
  const int L = p.L;
  const int n0 = blockIdx.x * kMdTile;
  const int n1 = min(p.N, n0 + kMdTile);
  const size_t row = (size_t)b * p.N;
  const float* __restrict__ xb = p.audio + row;
  const int h0 = n0 - L + 1;

  float ph[kMdPer], gn[kMdPer];
#pragma unroll
  for (int u = 0; u < kMdPer; ++u) {
    const int n = n0 + u * kMdThreads + tid;
    ph[u] = n < n1 ? p.phase[row + n] : 0.f;
    gn[u] = (p.gain != nullptr && n < n1) ? p.gain[row + n] : 1.f;
  }
  if (STAGE) {
    md_stage(md_hist, xb, h0, n1);
    __syncthreads();
  }
#pragma unroll
  for (int u = 0; u < kMdPer; ++u) {
    const int n = n0 + u * kMdThreads + tid;
    if (n < n1) {
      float phase = ph[u], gain = gn[u];
      if (p.scale) {
        phase = sigmoid_f(phase);
        if (p.gain != nullptr) gain = exp_sigmoid_f(gain);
      }
      const LookupTaps t = lookup_taps(fma((double)phase, p.p_scale, p.p_offset), L);
      const float e0 = t.ok0 ? md_x<STAGE>(md_hist, xb, h0, n - t.j0) : 0.f;
      const float e1 = t.ok1 ? md_x<STAGE>(md_hist, xb, h0, n - t.j1) : 0.f;
      float y = fmaf((float)t.fr, e1, (float)(1.0 - t.fr) * e0);
      if (p.gain != nullptr) y *= gain;
      if (p.add_dry) y += md_x<STAGE>(md_hist, xb, h0, n);
      p.out[row + n] = y;
    }
  }
}

// ---- backward ---------------------------------------------------------------------
// d_audio is the transpose of the two-tap gather: sample n adds g gain (1 - fr) to
// x[n - j0] and g gain fr to x[n - j1], every target in [n - L + 1, n].  To make the
// sum independent of the order of the adds, each contribution is rounded once to a
// 64-bit fixed-point number, q = rint(c 2^s), and summed with integer atomics, which
// commute.  2^s is per item: with M = max |g gain| over the item,
// |d_audio_wet[m]| <= (L + 1) M, so s = 62 - ceil(log2((L + 1) M)) keeps every total
// below 2^62; wrap-around in partial sums cancels exactly.  The rounding error is
// at most (L + 1) 2^-s <= (L + 1)^2 M 2^-62 per target.
//
// Pass 1 (md_bwd_max): per tile, max |g gain| -> tmax; zero the tile's halo slots.
// Pass 2 (md_backward): per tile, d_gain and d_phase per sample; the d_audio
//   contributions to targets in the tile go to shared-memory u64 atomics, those to
//   earlier tiles (the halo) to global u64 atomics in `halo`.  Targets of a tile
//   that no later tile can reach (all but its last H = min(L, kMdTile) samples, and
//   all of the item's last tile) are final and written here; the others are added
//   into `halo`.
// Pass 3 (md_bwd_finish): the halo slots -> d_audio.
// Halo slot of target m in tile t < tiles - 1: [b, t, m - t kMdTile - (kMdTile - H)].

// max that keeps a NaN (fmaxf drops it), so a NaN gradient reaches md_fix_exp
__device__ __forceinline__ float md_max(float a, float b) {
  return (a != a || b != b) ? __int_as_float(0x7fc00000) : fmaxf(a, b);
}

__device__ __forceinline__ float block_max_256(float v, float* red) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = md_max(v, __shfl_xor_sync(0xffffffffu, v, o));
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = v;
  __syncthreads();
  v = red[0];
#pragma unroll
  for (int w = 1; w < kMdThreads / 32; ++w) v = md_max(v, red[w]);
  return v;
}

__global__ void __launch_bounds__(kMdThreads)
md_bwd_max(MdParams p) {
  __shared__ float red[kMdThreads / 32];
  const int b = blockIdx.y, tile = blockIdx.x, tid = threadIdx.x;
  const int n0 = tile * kMdTile;
  const int n1 = min(p.N, n0 + kMdTile);
  const size_t row = (size_t)b * p.N;
  float m = 0.f;
  for (int n = n0 + tid; n < n1; n += kMdThreads) {
    float gain = 1.f;
    if (p.gain != nullptr) {
      gain = p.gain[row + n];
      if (p.scale) gain = exp_sigmoid_f(gain);
    }
    m = md_max(m, fabsf(p.grad[row + n] * gain));
  }
  m = block_max_256(m, red);
  if (tid == 0) p.tmax[(size_t)b * p.tiles + tile] = m;
  if (tile < p.tiles - 1) {
    unsigned long long* h = p.halo + ((size_t)b * p.tiles + tile) * p.H;
    for (int i = tid; i < p.H; i += kMdThreads) h[i] = 0ull;
  }
}

// Exponent s of the fixed-point scale 2^s of item b (see above); kMdNonFinite
// when the item's g gain is not finite (its d_audio is then NaN).
constexpr int kMdNonFinite = -100000;

__device__ __forceinline__ int md_fix_exp(float M, int L) {
  if (!(M <= 3.402823466e38f)) return kMdNonFinite;
  int e;
  frexp((double)(L + 1) * (double)M, &e);    // (L + 1) M < 2^e
  return 62 - e;
}

template <bool STAGE>
__global__ void __launch_bounds__(kMdThreads)
md_backward(MdParams p) {
  extern __shared__ __align__(16) unsigned char md_smem[];
  unsigned long long* acc = reinterpret_cast<unsigned long long*>(md_smem);
  float* hist = reinterpret_cast<float*>(md_smem + sizeof(unsigned long long) * kMdTile);
  __shared__ float red[kMdThreads / 32];
  const int b = blockIdx.y, tile = blockIdx.x, tid = threadIdx.x;
  const int L = p.L;
  const int n0 = tile * kMdTile;
  const int n1 = min(p.N, n0 + kMdTile);
  const size_t row = (size_t)b * p.N;
  const float* __restrict__ xb = p.audio + row;
  const int h0 = n0 - L + 1;

  float M = 0.f;
  for (int t = tid; t < p.tiles; t += kMdThreads)
    M = md_max(M, p.tmax[(size_t)b * p.tiles + t]);
  for (int i = tid; i < kMdTile; i += kMdThreads) acc[i] = 0ull;
  if (STAGE) md_stage(hist, xb, h0, n1);
  M = block_max_256(M, red);                 // also the barrier for acc / hist
  const int s = md_fix_exp(M, L);
  const double fix = ldexp(1.0, s);
  if (tile == 0 && tid == 0) p.kexp[b] = s;
  unsigned long long* halo_b = p.halo + (size_t)b * p.tiles * p.H;
  const int recv0 = kMdTile - p.H;           // first halo-receiving offset in a tile
  const float dp_scale = (float)p.p_scale;

  auto scatter = [&](int m, double c) {
    if (m < 0) return;                       // the zero padding
    const unsigned long long q = (unsigned long long)__double2ll_rn(c * fix);
    if (m >= n0) {
      atomicAdd(acc + (m - n0), q);
    } else {
      const int t = m / kMdTile;
      atomicAdd(halo_b + (size_t)t * p.H + (m - t * kMdTile - recv0), q);
    }
  };

#pragma unroll 2
  for (int u = 0; u < kMdPer; ++u) {
    const int n = n0 + u * kMdThreads + tid;
    if (n < n1) {
      const float g = p.grad[row + n];
      float phase = p.phase[row + n], dphase = 1.f;
      if (p.scale) dphase = sigmoid_grad(phase, &phase);
      float gain = 1.f, dgain = 1.f;
      if (p.gain != nullptr) {
        gain = p.gain[row + n];
        if (p.scale) dgain = exp_sigmoid_grad(gain, &gain);
      }
      const LookupTaps t = lookup_taps(fma((double)phase, p.p_scale, p.p_offset), L);
      const float e0 = t.ok0 ? md_x<STAGE>(hist, xb, h0, n - t.j0) : 0.f;
      const float e1 = t.ok1 ? md_x<STAGE>(hist, xb, h0, n - t.j1) : 0.f;
      const float wet = fmaf((float)t.fr, e1, (float)(1.0 - t.fr) * e0);
      const float gg = g * gain;
      if (p.gain != nullptr) p.d_gain[row + n] = g * wet * dgain;
      p.d_phase[row + n] = gg * (e1 - e0) * dp_scale * dphase;
      if (t.ok0) scatter(n - t.j0, (double)gg * (1.0 - t.fr));
      if (t.ok1) scatter(n - t.j1, (double)gg * t.fr);
    }
  }
  __syncthreads();

  const bool last = tile == p.tiles - 1;
  const double inv = ldexp(1.0, -s);
  for (int i = tid; i < n1 - n0; i += kMdThreads) {
    const unsigned long long v = acc[i];
    if (!last && i >= recv0) {
      if (v) atomicAdd(halo_b + (size_t)tile * p.H + (i - recv0), v);
    } else {
      double d = s == kMdNonFinite ? nan("") : (double)(long long)v * inv;
      if (p.add_dry) d += (double)p.grad[row + n0 + i];
      p.out[row + n0 + i] = (float)d;
    }
  }
}

__global__ void __launch_bounds__(256)
md_bwd_finish(MdParams p) {
  const long long per_item = (long long)(p.tiles - 1) * p.H;
  const long long total = (long long)p.B * per_item;
  for (long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x; idx < total;
       idx += (long long)gridDim.x * blockDim.x) {
    const int b = (int)(idx / per_item);
    const long long r = idx - (long long)b * per_item;
    const int t = (int)(r / p.H), i = (int)(r - (long long)t * p.H);
    const size_t m = (size_t)b * p.N + (size_t)t * kMdTile + (kMdTile - p.H) + i;
    const unsigned long long v = p.halo[((size_t)b * p.tiles + t) * p.H + i];
    const int s = p.kexp[b];
    double d = s == kMdNonFinite ? nan("") : (double)(long long)v * ldexp(1.0, -s);
    if (p.add_dry) d += (double)p.grad[m];
    p.out[m] = (float)d;
  }
}

// ---- core.sigmoid -----------------------------------------------------------------
__global__ void __launch_bounds__(256)
sigmoid_kernel(const float* __restrict__ in, float* __restrict__ out, int64_t n) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n;
       i += (int64_t)gridDim.x * blockDim.x)
    out[i] = sigmoid_f(in[i]);
}

}  // namespace ddsp
