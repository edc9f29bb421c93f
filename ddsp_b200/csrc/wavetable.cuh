// Wavetable synthesizer: core.wavetable_synthesis / synths.Wavetable.get_signal
// (core.py:1212-1282, synths.py:238-257) and core.linear_lookup (core.py:1168-1209)
// without the reference's [B, N, W] tensors.
//
// Per batch item, hop = N / F (amplitude and f0 frames), R table frames of W
// entries (R == 1: a static table), sample t:
//   f0(t)   = v1 bilinear of the frame f0 (frame F := F-1)
//   phi(t)  = sum_{m<t} f0(m)/sr mod 1     (EXCLUSIVE cumsum, phi(0) = 0)
//           = P_i + r a_i + (a_{i+1}-a_i)/hop * r(r-1)/2,   i = t / hop, r = t % hop
//   j, fr   = floor / fraction of phi * W (64-bit fixed-point phase: j is the high
//             word of phi * W, fr its low word), jn = (j + 1) mod W
//   row     = lo = floor(t R / N), hi = min(lo + 1, R - 1), ft = (t R mod N) / N
//             (the table resample src = t R / N as an exact rational)
//   L(t)    = (1-ft) [T_lo[j] + fr (T_lo[jn] - T_lo[j])] + ft [same on T_hi]
//   amp(t)  = A_i (1 - w1) + A_{i+1} w1,   w1 = 0.5 - 0.5 cos(pi r / hop)  (Hann OLA)
//   out(t)  = L(t) amp(t)
// DESIGN.md section 3.11 has the derivation and the measured bound.
#pragma once
#include "common.cuh"
#include "controls_bwd.cuh"

namespace ddsp {

constexpr int kWtThreads = 128;      // forward CTA
constexpr int kWtSeg = 2048;         // backward: samples per warp task (at most)

struct __align__(8) WtRec {
  unsigned long long P, A, D;        // frame phase (exclusive), slope, curvature
};

struct WtParams {
  const float* __restrict__ tables;  // [B, R, W]
  const float* __restrict__ amps;    // [B, F]
  const WtRec* __restrict__ rec;     // [B, F]
  float* __restrict__ out;           // [B, N]
  int B, F, R, W, N, hop;
  int t_chunk;                       // forward: samples per CTA
  int ring;                          // forward: shared-memory row slots
  int scale;                         // amps / tables are raw: exp_sigmoid them
  int accumulate;
  float inv_hop, inv_n;
};

__device__ __forceinline__ void fence_proxy_async_smem() {
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}

__device__ __forceinline__ float wt_window_w1(int r, float inv_hop) {
  return 0.5f - 0.5f * cospif((float)r * inv_hop);
}

// Exclusive phase of sample r of the frame, 64-bit fixed-point turns.
__device__ __forceinline__ unsigned long long wt_phase(const WtRec& rc, int r) {
  return rc.P + (unsigned long long)r * rc.A +
         (unsigned long long)(((long long)r * (r - 1)) >> 1) * rc.D;
}

// Table index and interpolation fraction of phase ph for a table of W entries.
__device__ __forceinline__ void wt_index(unsigned long long ph, unsigned W, unsigned& j,
                                         unsigned& jn, float& fr) {
  j = (unsigned)__umul64hi(ph, (unsigned long long)W);
  const unsigned long long low = ph * (unsigned long long)W;
  fr = (float)(unsigned)(low >> 40) * 5.9604644775390625e-8f;     // 2^-24
  jn = (j + 1 == W) ? 0u : j + 1;
}

__device__ __forceinline__ long long ceil_div_ll(long long a, long long b) {
  return (a + b - 1) / b;
}

// ---- pass 1: per-frame phase records (one warp per item) ----------------------
__global__ void __launch_bounds__(32)
wt_phase_records(const float* __restrict__ f0, WtRec* __restrict__ rec, int F, int hop,
                 double inv_sr) {
  const int b = blockIdx.x, lane = threadIdx.x;
  const float* fb = f0 + (size_t)b * F;
  WtRec* rb = rec + (size_t)b * F;
  unsigned long long carry = 0;
  for (int base = 0; base < F; base += 32) {
    const int i = base + lane;
    unsigned long long tot = 0, A = 0, D = 0;
    if (i < F) {
      const double a0 = (double)fb[i] * inv_sr;
      const double a1 = (double)fb[min(i + 1, F - 1)] * inv_sr;
      A = turns_to_fix64(a0);
      D = turns_to_fix64((a1 - a0) / (double)hop);
      tot = turns_to_fix64((double)hop * a0 + (a1 - a0) * (0.5 * (hop - 1)));
    }
    unsigned long long incl = tot;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const unsigned long long v = __shfl_up_sync(0xffffffffu, incl, o);
      if (lane >= o) incl += v;
    }
    if (i < F) rb[i] = WtRec{carry + incl - tot, A, D};
    carry += __shfl_sync(0xffffffffu, incl, 31);
  }
}

// ---- pass 2: forward ------------------------------------------------------------
// A CTA owns samples [t0, t1) of one item and walks the table intervals k that
// cover them (samples with lo == k).  Rows r_first .. r_last stream through a ring
// of `ring` shared-memory slots: TMA bulk copies issued `ring` rows ahead (TMA),
// or plain loads when the row is needed (W % 4 != 0 or a misaligned table).  With
// `scale` every row is exp_sigmoid'ed once in shared memory after it lands.
template <bool TMA>
__global__ void __launch_bounds__(kWtThreads)
wt_forward(WtParams p) {
  extern __shared__ __align__(128) unsigned char wt_smem[];
  unsigned long long* bars = reinterpret_cast<unsigned long long*>(wt_smem);
  float* rows = reinterpret_cast<float*>(wt_smem + 128);
  const int b = blockIdx.y, tid = threadIdx.x;
  const int W = p.W, R = p.R, ring = p.ring;
  const long long N = p.N;
  const int t0 = blockIdx.x * p.t_chunk;
  const int t1 = min(p.N, t0 + p.t_chunk);
  const int r_first = (int)((long long)t0 * R / N);
  const int k_last = (int)((long long)(t1 - 1) * R / N);
  const int r_last = min(k_last + 1, R - 1);
  const float* tb = p.tables + (size_t)b * R * W;
  const uint32_t row_bytes = (uint32_t)W * 4u;

  auto slot_ptr = [&](int r) { return rows + (size_t)((r - r_first) % ring) * W; };
  auto issue = [&](int r) {
    unsigned long long* bar = bars + (r - r_first) % ring;
    mbar_expect_tx(bar, row_bytes);
    tma_bulk_g2s(slot_ptr(r), tb + (size_t)r * W, row_bytes, bar);
  };
  // make row r readable by the whole CTA (controls, exp_sigmoid'ed if raw)
  auto acquire = [&](int r) {
    float* s = slot_ptr(r);
    if (TMA) {
      mbar_wait(bars + (r - r_first) % ring, (uint32_t)(((r - r_first) / ring) & 1));
      if (p.scale)
        for (int e = tid; e < W; e += kWtThreads) s[e] = exp_sigmoid_f(s[e]);
    } else {
      const float* g = tb + (size_t)r * W;
      for (int e = tid; e < W; e += kWtThreads) {
        const float v = g[e];
        s[e] = p.scale ? exp_sigmoid_f(v) : v;
      }
    }
    __syncthreads();
  };

  if (TMA) {
    if (tid == 0) {
      for (int s = 0; s < ring; ++s) mbar_init(bars + s, 1);
    }
    __syncthreads();
    if (tid == 0) {
      for (int q = 0; q < ring && r_first + q <= r_last; ++q) issue(r_first + q);
    }
  }
  acquire(r_first);

  const float* ampb = p.amps + (size_t)b * p.F;
  const WtRec* recb = p.rec + (size_t)b * p.F;
  float* outb = p.out + (size_t)b * p.N;
  for (int k = r_first; k <= k_last; ++k) {
    const int kh = min(k + 1, R - 1);
    if (kh != k) acquire(kh);
    const float* T0 = slot_ptr(k);
    const float* T1 = slot_ptr(kh);
    const int ts = (int)max((long long)t0, ceil_div_ll((long long)k * N, R));
    const int te = (int)min((long long)t1, ceil_div_ll((long long)(k + 1) * N, R));
    for (int t = ts + tid; t < te; t += kWtThreads) {
      const int i = t / p.hop, r = t - i * p.hop;
      const WtRec rc = recb[i];
      unsigned j, jn;
      float fr;
      wt_index(wt_phase(rc, r), (unsigned)W, j, jn, fr);
      const float x0 = T0[j], x1 = T1[j];
      const float v0 = fmaf(fr, T0[jn] - x0, x0);
      const float v1 = fmaf(fr, T1[jn] - x1, x1);
      const float ft = (float)((long long)t * R - (long long)k * N) * p.inv_n;
      const float L = fmaf(ft, v1 - v0, v0);
      float a0 = ampb[i], a1 = ampb[min(i + 1, p.F - 1)];
      if (p.scale) {
        a0 = exp_sigmoid_f(a0);
        a1 = exp_sigmoid_f(a1);
      }
      const float w1 = wt_window_w1(r, p.inv_hop);
      float y = L * fmaf(a1, w1, a0 * (1.0f - w1));
      if (p.accumulate) y += outb[t];
      outb[t] = y;
    }
    __syncthreads();                     // slot of row k is free again
    if (TMA && tid == 0 && k + ring <= r_last) {
      fence_proxy_async_smem();          // generic writes (scale) before the async refill
      issue(k + ring);
    }
  }
}

// ---- backward ---------------------------------------------------------------------
// Gather form: a warp task (b, row k, segment s) walks, in sample order, the samples
// of segment s of the samples that read row k (intervals k-1 and k), recomputes
// their phases, and accumulates the row's gradient in shared memory.  Same-entry
// lanes are resolved with __match_any_sync and summed in lane order, so the result
// is bit-reproducible and every gradient element is written once (to d_tables, or
// to a partial row when a row has more than one segment: static tables, few table
// frames).  The task whose row is lo(t) also writes g(t) L(t) for the amplitude
// gradient.
struct WtBwdParams {
  const float* __restrict__ tables;  // [B, R, W] (raw when scale)
  const float* __restrict__ amps;    // [B, F] (raw when scale)
  const WtRec* __restrict__ rec;     // [B, F]
  const float* __restrict__ grad;    // [B, N]
  float* __restrict__ gl;            // [B, N] workspace: g(t) L(t)
  float* __restrict__ d_tables;      // [B, R, W]
  float* __restrict__ parts;         // [B, R, nseg, W] workspace (nseg > 1)
  int B, F, R, W, N, hop, nseg, nw, scale;
  float inv_hop, inv_n;
};

__device__ __forceinline__ void warp_scatter_add(float* acc, unsigned idx, float v,
                                                 bool valid, int lane) {
  const unsigned key = valid ? idx : 0xffffffffu;
  const unsigned peers = __match_any_sync(0xffffffffu, key);
  const unsigned maxn = __reduce_max_sync(0xffffffffu, (unsigned)__popc(peers));
  float sum = v;
  if (maxn > 1) {
    sum = 0.f;
    unsigned m = peers;
    for (unsigned it = 0; it < maxn; ++it) {
      const int src = m ? __ffs(m) - 1 : lane;
      const float x = __shfl_sync(0xffffffffu, v, src);
      if (m) {
        sum += x;
        m &= m - 1;
      }
    }
  }
  if (valid && lane == __ffs(peers) - 1) acc[idx] += sum;
  __syncwarp();
}

__device__ __forceinline__ long long wt_row_start(int k, int R, long long N) {
  return ceil_div_ll((long long)k * N, R);   // first sample with lo >= k
}

// Stage n controls (exp_sigmoid'ed when raw) into shared memory: 16-byte loads,
// several in flight per thread, where the rows allow.
__device__ __forceinline__ void wt_stage_rows(float* __restrict__ stage,
                                           const float* __restrict__ src, int n,
                                           int scale) {
  if ((n & 3) == 0 && (((uintptr_t)src) & 15) == 0) {
    for (int e = threadIdx.x; e < n / 4; e += blockDim.x) {
      float4 v = reinterpret_cast<const float4*>(src)[e];
      if (scale) {
        v.x = exp_sigmoid_f(v.x); v.y = exp_sigmoid_f(v.y);
        v.z = exp_sigmoid_f(v.z); v.w = exp_sigmoid_f(v.w);
      }
      reinterpret_cast<float4*>(stage)[e] = v;
    }
  } else {
    for (int e = threadIdx.x; e < n; e += blockDim.x) {
      const float v = src[e];
      stage[e] = scale ? exp_sigmoid_f(v) : v;
    }
  }
}

__global__ void __launch_bounds__(128, 1)
wt_backward(WtBwdParams p) {
  extern __shared__ __align__(16) float smem_f[];
  const int b = blockIdx.y, warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int W = p.W, R = p.R, nseg = p.nseg;
  const long long N = p.N;
  const int n_tasks = R * nseg;
  const int task0 = blockIdx.x * p.nw;
  const int k_first = task0 / nseg;
  const int k_end = min(R - 1, (min(task0 + p.nw, n_tasks) - 1) / nseg + 1);   // inclusive
  const int n_stage = k_end - k_first + 1;
  float* stage = smem_f;                                 // n_stage rows (controls)
  float* acc = smem_f + (size_t)(p.nw + 1) * W + (size_t)warp * W;
  const float* tb = p.tables + (size_t)b * R * W;

  wt_stage_rows(stage, tb + (size_t)k_first * W, n_stage * W, p.scale);
  for (int e = lane; e < W; e += 32) acc[e] = 0.f;
  __syncthreads();

  const int task = task0 + warp;
  if (task >= n_tasks) return;
  const int k = task / nseg, s = task - k * nseg;
  const long long u0 = wt_row_start(max(k - 1, 0), R, N);
  const long long u1 = wt_row_start(k + 1, R, N) < N ? wt_row_start(k + 1, R, N) : N;
  const long long ts_k = wt_row_start(k, R, N);
  const long long seg0 = u0 + (long long)s * kWtSeg;
  const long long seg1 = min(u1, seg0 + kWtSeg);
  const int kh = min(k + 1, R - 1);
  const float* T0 = stage + (size_t)(k - k_first) * W;
  const float* T1 = stage + (size_t)(kh - k_first) * W;
  const float* ampb = p.amps + (size_t)b * p.F;
  const WtRec* recb = p.rec + (size_t)b * p.F;
  const float* gb = p.grad + (size_t)b * N;
  float* glb = p.gl + (size_t)b * N;

  for (long long tb0 = seg0; tb0 < seg1; tb0 += 32) {
    const long long tl = tb0 + lane;
    const bool valid = tl < seg1;
    const int t = valid ? (int)tl : (int)seg0;
    const bool is_lo = t >= ts_k;                 // lo(t) == k, else lo(t) == k - 1
    const int lo = is_lo ? k : k - 1;
    const int hi = min(lo + 1, R - 1);
    const float ft = (float)((long long)t * R - (long long)lo * N) * p.inv_n;
    const float wk = (is_lo ? 1.0f - ft : 0.f) + (hi == k ? ft : 0.f);
    const int i = t / p.hop, r = t - i * p.hop;
    unsigned j, jn;
    float fr;
    wt_index(wt_phase(recb[i], r), (unsigned)W, j, jn, fr);
    float a0 = ampb[i], a1 = ampb[min(i + 1, p.F - 1)];
    if (p.scale) {
      a0 = exp_sigmoid_f(a0);
      a1 = exp_sigmoid_f(a1);
    }
    const float w1 = wt_window_w1(r, p.inv_hop);
    const float g = valid ? gb[t] : 0.f;
    const float c = g * fmaf(a1, w1, a0 * (1.0f - w1)) * wk;
    if (valid && is_lo) {
      const float x0 = T0[j], x1 = T1[j];
      const float v0 = fmaf(fr, T0[jn] - x0, x0);
      const float v1 = fmaf(fr, T1[jn] - x1, x1);
      glb[t] = g * fmaf(ft, v1 - v0, v0);
    }
    warp_scatter_add(acc, j, c * (1.0f - fr), valid, lane);
    warp_scatter_add(acc, jn, c * fr, valid, lane);
  }

  if (nseg == 1) {
    float* dst = p.d_tables + ((size_t)b * R + k) * W;
    const float* raw = tb + (size_t)k * W;
    for (int e = lane; e < W; e += 32) {
      float d = acc[e];
      if (p.scale) {
        float y;
        d *= exp_sigmoid_grad(raw[e], &y);
      }
      dst[e] = d;
    }
  } else {
    float* dst = p.parts + (((size_t)b * R + k) * nseg + s) * W;
    for (int e = lane; e < W; e += 32) dst[e] = acc[e];
  }
}

// Sum of the partial rows in segment order (+ the exp_sigmoid derivative).
__global__ void __launch_bounds__(256)
wt_reduce_parts(const float* __restrict__ parts, const float* __restrict__ tables,
                float* __restrict__ d_tables, long long n_rows, int nseg, int W,
                int scale) {
  const long long total = n_rows * W;
  for (long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x; idx < total;
       idx += (long long)gridDim.x * blockDim.x) {
    const long long row = idx / W;
    const int e = (int)(idx - row * W);
    const float* pr = parts + (size_t)row * nseg * W + e;
    float d = 0.f;
    for (int s = 0; s < nseg; ++s) d += pr[(size_t)s * W];
    if (scale) {
      float y;
      d *= exp_sigmoid_grad(tables[idx], &y);
    }
    d_tables[idx] = d;
  }
}

// d amplitudes: the transpose of the Hann overlap-add, one warp per (b, frame),
// a fixed-order tree over the lanes.
__global__ void __launch_bounds__(256)
wt_amp_grad(const float* __restrict__ gl, const float* __restrict__ amps,
            float* __restrict__ d_amps, int B, int F, int N, int hop, float inv_hop,
            int scale) {
  const long long wid = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (wid >= (long long)B * F) return;
  const int b = (int)(wid / F), i = (int)(wid - (long long)b * F);
  const float* g = gl + (size_t)b * N;
  float acc = 0.f;
  for (int r = lane; r < hop; r += 32) {
    const float w1 = wt_window_w1(r, inv_hop);
    acc += g[(size_t)i * hop + r] * (1.0f - w1);
    if (i > 0) acc += g[(size_t)(i - 1) * hop + r] * w1;
    if (i == F - 1) acc += g[(size_t)i * hop + r] * w1;
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
  if (lane == 0) {
    if (scale) {
      float y;
      acc *= exp_sigmoid_grad(amps[wid], &y);
    }
    d_amps[wid] = acc;
  }
}

// ---- core.linear_lookup's interpolation rule ---------------------------------------
// A table of W + 1 entries whose entry W is entry 0, read at position x = phase W
// (in double): entries floor(x) and floor(x) + 1 weigh 1 - frac and frac, and an
// entry outside [0, W] weighs zero - the reference's relu(1 - |phase - j/W| W).
// The indices come back in [0, W) (entry W as 0, an entry outside the table as 0
// with ok = false), so both are always readable.  wt_linear_lookup and the
// variable-length delay (mod_delay.cuh) both read their tables through this.
struct LookupTaps {
  int j0, j1;          // entry indices in [0, W)
  bool ok0, ok1;       // inside [0, W]: weights 1 - fr and fr, else zero
  double fr;
};

__device__ __forceinline__ LookupTaps lookup_taps(double x, int W) {
  LookupTaps t;
  const double fl = floor(x);
  t.fr = x - fl;
  t.ok0 = fl >= 0.0 && fl <= (double)W;
  t.ok1 = fl + 1.0 >= 0.0 && fl + 1.0 <= (double)W;
  const int j0 = t.ok0 ? (int)fl : 0;
  const int j1 = t.ok1 ? (int)(fl + 1.0) : 0;
  t.j0 = j0 == W ? 0 : j0;
  t.j1 = j1 == W ? 0 : j1;
  return t;
}

// ---- stand-alone core.linear_lookup ----------------------------------------------
// phase [B, N] (any real value), tables [B, W] (static) or [B, N, W].
__global__ void __launch_bounds__(256)
wt_linear_lookup(const float* __restrict__ phase, const float* __restrict__ tables,
                 float* __restrict__ out, int B, int N, int W, int per_sample) {
  const long long total = (long long)B * N;
  for (long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x; idx < total;
       idx += (long long)gridDim.x * blockDim.x) {
    const long long b = idx / N;
    const float* T = tables + (per_sample ? (size_t)idx * W : (size_t)b * W);
    const LookupTaps t = lookup_taps((double)phase[idx] * (double)W, W);
    double acc = 0.0;
    if (t.ok0) acc += (1.0 - t.fr) * (double)T[t.j0];
    if (t.ok1) acc += t.fr * (double)T[t.j1];
    out[idx] = (float)acc;
  }
}

}  // namespace ddsp
