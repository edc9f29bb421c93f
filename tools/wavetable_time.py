"""Times the wavetable synthesizer on the GPU and writes profiles/wavetable_timing.txt.

  python tools/wavetable_time.py [--out PATH] [--iters 10]

Event-timed forward (raw path: exp_sigmoid in the kernel; controls path) and
backward (raw) at B = 32 and 256, F = F_wt = 1000, W = 2048, N = 64000, with the
achieved fraction of the HBM peak bench.py uses (MEASURED_PEAKS.json hbm_gbs, else
its 6650 GB/s fallback), and the reference-shaped decomposition (tables resampled to
[B, N, W], then linear_lookup) at a batch where that fits.  Every input set is larger
than the 126 MB L2, so each timed pass streams its tables from HBM.
"""
import argparse
import json
import os
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from ddsp_b200 import autograd, core  # noqa: E402

F, W, N = 1000, 2048, 64000


def peak_gbs():
  path = os.path.join(ROOT, 'MEASURED_PEAKS.json')
  if os.path.exists(path):
    with open(path) as f:
      return float(json.load(f)['hbm_gbs']), 'measured (MEASURED_PEAKS.json)'
  return 6650.0, 'bench.py fallback'


def gpu_info():
  name = torch.cuda.get_device_name(0)
  try:
    q = subprocess.run(['nvidia-smi', '--query-gpu=power.limit,clocks.max.sm',
                        '--format=csv,noheader', '-i', '0'], capture_output=True,
                       text=True, timeout=30).stdout.strip()
  except (OSError, subprocess.SubprocessError) as e:
    q = 'nvidia-smi unavailable (%s)' % e
  return name, q


def time_ms(fn, iters):
  for _ in range(2):
    fn()
  torch.cuda.synchronize()
  e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
  e0.record()
  for _ in range(iters):
    fn()
  e1.record()
  torch.cuda.synchronize()
  return e0.elapsed_time(e1) / iters


def inputs(b, seed=0):
  g = torch.Generator(device='cuda').manual_seed(seed)
  amps = torch.randn((b, F, 1), device='cuda', generator=g)
  tables = torch.randn((b, F, W), device='cuda', generator=g)
  f0 = (80.0 + 720.0 * torch.rand((b, 1, 1), device='cuda', generator=g)).expand(
      b, F, 1).contiguous()
  return amps, tables, f0


def main():
  ap = argparse.ArgumentParser()
  ap.add_argument('--out', default=os.path.join(ROOT, 'profiles', 'wavetable_timing.txt'))
  ap.add_argument('--iters', type=int, default=10)
  args = ap.parse_args()
  assert torch.cuda.is_available(), 'wavetable_time.py needs a CUDA device'
  peak, peak_src = peak_gbs()
  name, power = gpu_info()
  fwd_bytes = 4 * (F * W + 2 * F + N)            # per item
  bwd_bytes = 4 * (2 * F * W + N + 3 * F)        # per item
  lines = ['GPU: %s; power.limit, clocks.max.sm: %s' % (name, power),
           'HBM peak used for the fraction: %.0f GB/s (%s)' % (peak, peak_src),
           'shape per item: F = F_wt = %d, W = %d, N = %d' % (F, W, N),
           'algorithmic bytes per item: forward 4 (F_wt W + 2 F + N) = %d; '
           'backward 4 (2 F_wt W + N + 3 F) = %d (tables read, d tables written, '
           'grad read, f0 / amps read, d amps written)' % (fwd_bytes, bwd_bytes), '']
  for b in (32, 256):
    amps, tables, f0 = inputs(b)
    ctl_a, ctl_t = core.exp_sigmoid(amps), core.exp_sigmoid(tables)
    grad = torch.randn((b, N), device='cuda')
    a_req = amps.clone().requires_grad_()
    t_req = tables.clone().requires_grad_()
    y = autograd.wavetable_train(a_req, t_req, f0, n_samples=N)

    def bwd():
      torch.autograd.backward(y, grad, retain_graph=True)
      a_req.grad = None
      t_req.grad = None

    runs = [('forward, raw outputs (exp_sigmoid fused)',
             lambda: core.wavetable_raw(amps, tables, f0, n_samples=N), fwd_bytes),
            ('forward, controls',
             lambda: core.wavetable_synthesis(f0, ctl_a, ctl_t, n_samples=N), fwd_bytes),
            ('backward, raw outputs', bwd, bwd_bytes)]
    for label, fn, nbytes in runs:
      ms = time_ms(fn, args.iters)
      gbs = b * nbytes / (ms * 1e-3) / 1e9
      lines.append('B=%-3d %-44s %8.3f ms  %7.0f GB/s  %.3f of peak' % (
          b, label, ms, gbs, gbs / peak))
    del y, a_req, t_req, grad, ctl_a, ctl_t, amps, tables, f0
    torch.cuda.empty_cache()
  b = 32
  amps, tables, f0 = inputs(b)
  ctl_a, ctl_t = core.exp_sigmoid(amps), core.exp_sigmoid(tables)

  def reference_shaped():
    tab_n = core.resample(ctl_t, N)                                   # [B, N, W]
    amp_env = core.resample(ctl_a, N, method='window')[:, :, 0]
    phase = torch.cumsum(core.resample(f0, N)[:, :, 0] / 16000.0, dim=1)
    phase = torch.remainder(phase - phase[:, :1], 1.0)
    return core.linear_lookup(phase, tab_n) * amp_env

  ms_ref = time_ms(reference_shaped, 3)
  ms_fused = time_ms(lambda: core.wavetable_synthesis(f0, ctl_a, ctl_t, n_samples=N),
                     args.iters)
  lines += ['', 'reference-shaped decomposition at B=%d (resample tables to [B, N, W] = '
            '%.1f GB, window-resample amps, cumsum phase, linear_lookup): %.3f ms; '
            'fused controls path %.3f ms (%.1fx)' % (
                b, b * N * W * 4 / 1e9, ms_ref, ms_fused, ms_ref / ms_fused)]
  text = '\n'.join(lines) + '\n'
  print(text, end='')
  os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
  with open(args.out, 'w') as f:
    f.write(text)


if __name__ == '__main__':
  main()
