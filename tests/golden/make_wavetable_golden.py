"""Writes tests/golden/wavetable.npz: outputs of the UNMODIFIED reference's
wavetable synthesizer (ddsp/core.py:1167-1282, ddsp/synths.py:199-257) on the
NumPy TensorFlow shim, narrow (float32) and wide (float64), on the seeded cases of
`cases()` (the tests regenerate the inputs from there).

Needs the reference sources, like make_golden.py:

  python tests/golden/make_wavetable_golden.py          # rewrite the fixture
  python tests/golden/make_wavetable_golden.py --check  # regenerate and compare
"""
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))
from oracle import ref_on_shim                                       # noqa: E402
from tests.golden.make_golden import _both, compare, pack_outputs   # noqa: E402

PATH = os.path.join(HERE, 'wavetable.npz')
FULL = dict(B=1, F=1000, W=2048, N=64000)


def _f0(rng, b, f, n, sample_rate=16000):
  t = np.arange(f) * (n / f) / sample_rate
  base = rng.uniform(80.0, 800.0, (b, 1))
  ph = rng.uniform(0, 2 * np.pi, (b, 1))
  return (base * (1.0 + 0.03 * np.sin(2 * np.pi * 5.0 * t[None, :] + ph)))[..., None] \
      .astype(np.float32)


def cases():
  """name -> (kind, arrays, kwargs).  kind: 'synth' = Wavetable(**kwargs) on raw
  outputs (amps, tables, f0); 'synthesis' = core.wavetable_synthesis(f0, amps,
  tables, **kwargs) on controls; 'lookup' = core.linear_lookup(phase, tables);
  'hd' = core.harmonic_distribution_to_wavetable(hd, **kwargs)."""
  rng = np.random.default_rng(2024)
  out = {}

  def raw(b, f, fw, w, n):
    return (rng.standard_normal((b, f, 1)).astype(np.float32),
            rng.standard_normal((b, fw, w)).astype(np.float32), _f0(rng, b, f, n))

  # the processor from raw network outputs (get_controls + get_signal)
  out['synth'] = ('synth', raw(2, 50, 50, 256, 3200), dict(n_samples=3200))
  # one table frame: a static table after the reference's resample
  out['synth_one_table'] = ('synth', raw(2, 40, 1, 128, 3200), dict(n_samples=3200))
  # non-power-of-two hop (75) and a table length that is not a multiple of 4
  out['synth_hop75'] = ('synth', raw(2, 40, 40, 130, 3000), dict(n_samples=3000))

  def ctl(b, f, fw, w, n):
    a, t, f0 = raw(b, f, fw, w, n)
    return (f0, np.abs(a) + 0.1, np.tanh(t))

  # 200 table frames over 100 control frames (core_test.py:630-634)
  out['synthesis_fwt200'] = ('synthesis', ctl(2, 100, 200, 256, 1600),
                             dict(n_samples=1600, sample_rate=16000))
  f0, a, t = ctl(2, 50, 1, 96, 1600)
  out['synthesis_2d'] = ('synthesis', (f0, a, t[:, 0, :]),
                         dict(n_samples=1600, sample_rate=16000))
  out['synthesis_fwt7'] = ('synthesis', ctl(1, 32, 7, 64, 2048),
                           dict(n_samples=2048, sample_rate=16000))

  W = 64
  ends = np.array([0.0, 1.0, 1.0 - 1e-7, -0.3 / W, 1.0 + 0.3 / W, -0.5, 1.5,
                   -1.0 / W, 1.0 + 1.0 / W, 0.5 / W], np.float32)
  ph = np.concatenate([ends, rng.uniform(-0.2, 1.2, 54).astype(np.float32)])
  ph = np.stack([ph, ph[::-1]])[:, :, None]
  out['lookup_2d'] = ('lookup', (ph, rng.standard_normal((2, W)).astype(np.float32)), {})
  out['lookup_3d'] = ('lookup', (ph[:, :, 0], rng.standard_normal(
      (2, ph.shape[1], W)).astype(np.float32)), {})

  out['hd_10_of_64'] = ('hd', (rng.uniform(0, 1, (2, 3, 10)).astype(np.float32),),
                        dict(n_wavetable=64))
  out['hd_32_of_64'] = ('hd', (rng.uniform(0, 1, (1, 2, 32)).astype(np.float32),),
                        dict(n_wavetable=64))
  return out


def full_inputs():
  """The full-length item: Wavetable() on raw outputs, F = F_wt = 1000,
  W = 2048, N = 64000."""
  rng = np.random.default_rng(77)
  b, f, w, n = FULL['B'], FULL['F'], FULL['W'], FULL['N']
  return (rng.standard_normal((b, f, 1)).astype(np.float32),
          rng.standard_normal((b, f, w)).astype(np.float32), _f0(rng, b, f, n))


def run_case(ddsp, kind, arrays, kw):
  if kind == 'synth':
    return ddsp.synths.Wavetable(**kw)(*arrays)
  if kind == 'synthesis':
    return ddsp.core.wavetable_synthesis(*arrays, **kw)
  if kind == 'lookup':
    return ddsp.core.linear_lookup(*arrays)
  return ddsp.core.harmonic_distribution_to_wavetable(*arrays, **kw)


def wavetable():
  ddsp = ref_on_shim.load()
  out = {}
  for name, (kind, arrays, kw) in cases().items():
    n, w = _both(lambda: run_case(ddsp, kind, arrays, kw))  # pylint: disable=cell-var-from-loop
    out[name + '_f32'] = np.asarray(n, np.float32)
    out[name + '_wide'] = np.asarray(w, np.float64)
  n, w = _both(lambda: ddsp.synths.Wavetable(n_samples=FULL['N'])(*full_inputs()))
  n, w = np.asarray(n, np.float64), np.asarray(w, np.float64)
  peak = np.abs(w).max()
  out['full_narrow_wide_maxrel'] = np.float64(np.abs(n - w).max() / peak)
  out['full_narrow_wide_l2rel'] = np.float64(np.sqrt(((n - w)**2).sum() / (w * w).sum()))
  packed = pack_outputs({'full_wide': w, 'full_f32': n})
  out.update({'full_' + k: v for k, v in packed.items()})
  return out


if __name__ == '__main__':
  got = wavetable()
  if '--check' in sys.argv:
    compare('wavetable', got, np.load(PATH))
    print('ok    wavetable')
  else:
    np.savez_compressed(PATH, **got)
    print('wrote wavetable %.0f kB' % (os.path.getsize(PATH) / 1e3))
