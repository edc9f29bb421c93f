"""Times the modulated delay on the GPU and writes profiles/mod_delay_timing.txt.

  python tools/mod_delay_time.py [--out PATH] [--iters 20]

Event-timed forward (raw path: exp_sigmoid / sigmoid in the kernel; controls
path) and backward (raw) at B = 32 and 256, N = 64000, L = 400 (ModDelay()'s
default) and L = 16000 (1 s at 16 kHz), with the achieved fraction of the HBM peak
bench.py uses (MEASURED_PEAKS.json hbm_gbs, else its 6650 GB/s fallback), and the
reference-shaped decomposition (audio unfolded to [B, N, L], then
core.linear_lookup) at a small batch.  Every timed pass cycles through enough
input sets to exceed the 126 MB L2, so each pass streams from HBM.
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

N = 64000
L2_BYTES = 126 << 20
FWD_B = 16    # per sample: audio, gain, phase read, out written
BWD_B = 28    # per sample: audio, gain, phase, grad read, d audio / gain / phase written


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


def time_ms(fns, iters):
  """Mean time of one call, cycling through the callables (one per input set)."""
  for fn in fns:
    fn()
  torch.cuda.synchronize()
  e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
  e0.record()
  for i in range(iters):
    fns[i % len(fns)]()
  e1.record()
  torch.cuda.synchronize()
  return e0.elapsed_time(e1) / iters


def input_sets(b, seed=0):
  n_sets = max(1, -(-2 * L2_BYTES // (12 * b * N)))
  g = torch.Generator(device='cuda').manual_seed(seed)
  return [(torch.randn((b, N), device='cuda', generator=g),
           torch.randn((b, N, 1), device='cuda', generator=g),
           2.0 * torch.randn((b, N, 1), device='cuda', generator=g))
          for _ in range(n_sets)]


def main():
  ap = argparse.ArgumentParser()
  ap.add_argument('--out', default=os.path.join(ROOT, 'profiles', 'mod_delay_timing.txt'))
  ap.add_argument('--iters', type=int, default=20)
  args = ap.parse_args()
  assert torch.cuda.is_available(), 'mod_delay_time.py needs a CUDA device'
  peak, peak_src = peak_gbs()
  name, power = gpu_info()
  lines = ['GPU: %s; power.limit, clocks.max.sm: %s' % (name, power),
           'HBM peak used for the fraction: %.0f GB/s (%s)' % (peak, peak_src),
           'shape: N = %d; L = max_length (ModDelay(): 400)' % N,
           'algorithmic bytes per sample: forward %d (audio, gain, phase read, out '
           'written); backward %d (audio, gain, phase, grad read, d audio, d gain, '
           'd phase written; workspace traffic not counted)' % (FWD_B, BWD_B),
           'inputs cycled over sets totalling more than 2 x 126 MB (L2)', '']
  for L, center, depth in ((400, 15.0, 10.0), (16000, 600.0, 400.0)):
    max_length, a, c = int(16000 / 1000.0 * (center + depth)), depth / (center + depth), \
        center / (center + depth)
    assert max_length == L
    for b in (32, 256):
      sets = input_sets(b)
      ctl = [(x, core.exp_sigmoid(gn), core.sigmoid(ph)) for x, gn, ph in sets]
      grad = torch.randn((b, N), device='cuda')
      graphs = []
      for x, gn, ph in sets:
        xr, gr, pr = (t.clone().requires_grad_() for t in (x, gn, ph))
        graphs.append((autograd.mod_delay_train(xr, gr, pr, center, depth), xr, gr, pr))

      def bwd_fn(item):
        y, xr, gr, pr = item

        def run():
          torch.autograd.backward(y, grad, retain_graph=True)
          xr.grad = gr.grad = pr.grad = None
        return run

      runs = [
          ('forward, raw outputs (sigmoids fused)',
           [lambda s=s: core.mod_delay(s[0], s[1], s[2], L, a, c, True, True)
            for s in sets], FWD_B),
          ('forward, controls',
           [lambda s=s: core.mod_delay(s[0], s[1], s[2], L, a, c, True, False)
            for s in ctl], FWD_B),
          ('backward, raw outputs', [bwd_fn(item) for item in graphs], BWD_B)]
      for label, fns, nbytes in runs:
        ms = time_ms(fns, args.iters)
        gbs = b * N * nbytes / (ms * 1e-3) / 1e9
        lines.append('L=%-5d B=%-3d %-40s %8.3f ms  %7.0f GB/s  %.3f of peak' % (
            L, b, label, ms, gbs, gbs / peak))
      del sets, ctl, graphs, grad
      torch.cuda.empty_cache()
  # the reference's shape: frames [B, N, L] of the zero-padded audio, reversed, then
  # linear_lookup (which appends entry 0) - on this library's kernels
  b, L = 4, 400
  x, gn, ph = input_sets(b)[0]
  gain, phase = core.exp_sigmoid(gn)[:, :, 0], core.sigmoid(ph)[:, :, 0]

  def reference_shaped():
    padded = torch.nn.functional.pad(x, (L - 1, 0))
    frames = padded.unfold(1, L, 1).flip(-1).contiguous()       # [B, N, L]
    wet = core.linear_lookup(phase * 0.4 + 0.6, frames)
    return wet * gain + x

  ms_ref = time_ms([reference_shaped], 3)
  ms_fused = time_ms([lambda: core.mod_delay(x, gain, phase, L, 0.4, 0.6)], args.iters)
  lines += ['', 'reference-shaped decomposition at B=%d, L=%d (frames [B, N, L] = %.2f GB, '
            'linear_lookup, gain, dry): %.3f ms; fused controls path %.3f ms (%.1fx; '
            'the fused input set fits L2 here)' % (
                b, L, b * N * L * 4 / 1e9, ms_ref, ms_fused, ms_ref / ms_fused)]
  text = '\n'.join(lines) + '\n'
  print(text, end='')
  os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
  with open(args.out, 'w') as f:
    f.write(text)


if __name__ == '__main__':
  main()
