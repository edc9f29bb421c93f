"""Writes tests/golden/mod_delay.npz: outputs of the UNMODIFIED reference's
modulated delay (ddsp/core.py:1285-1313 variable_length_delay, ddsp/effects.py:
328-393 ModDelay) on the NumPy TensorFlow shim, narrow (float32) and wide
(float64), on the seeded cases of `cases()` (the tests regenerate the inputs
from there).

Needs the reference sources, like make_golden.py:

  python tests/golden/make_mod_delay_golden.py          # rewrite the fixture
  python tests/golden/make_mod_delay_golden.py --check  # regenerate and compare
"""
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))
from oracle import ref_on_shim                                       # noqa: E402
from tests.golden.make_golden import _both, compare, pack_outputs   # noqa: E402

PATH = os.path.join(HERE, 'mod_delay.npz')
FULL = dict(B=1, N=64000)

# effects.ModDelay constructor arguments of the 1_synths_and_effects tutorial
TUTORIAL = {'flanger': dict(center_ms=0.75, depth_ms=0.75, mod_rate=0.25),
            'chorus': dict(center_ms=25.0, depth_ms=1.0, mod_rate=2.0),
            'vibrato': dict(center_ms=25.0, depth_ms=12.5, mod_rate=5.0)}


def audio_like(rng, b, n, sample_rate=16000):
  """A few partials plus noise: a signal whose history matters at every lag."""
  t = np.arange(n) / sample_rate
  f = rng.uniform(80.0, 900.0, (b, 3, 1))
  ph = rng.uniform(0.0, 2 * np.pi, (b, 3, 1))
  x = np.sin(2 * np.pi * f * t[None, None, :] + ph).sum(axis=1) / 3.0
  return (x + 0.1 * rng.standard_normal((b, n))).astype(np.float32)


def special_phases(L):
  """Phases at the edges of linear_lookup's rule for a delay of L samples."""
  return np.array([0.0, 1.0, 1.0 - 1e-7, 0.3 / L, -0.3 / L, 1.0 + 0.3 / L,
                   1.0 - 0.3 / L, -1.0 / L, 1.0 + 1.0 / L, -1.5 / L, 1.0 + 1.5 / L,
                   1.0 / L, (L // 2) / L, (L - 1) / L, -0.5, 1.5], np.float32)


def delay_phases(rng, b, n, L):
  ph = rng.uniform(-0.2, 1.2, (b, n)).astype(np.float32)
  sp = special_phases(L)
  idx = np.arange(0, n, 5)
  ph[:, idx] = np.resize(sp, idx.size)[None, :]
  return ph[:, :, None]


def tutorial_phase(mod_rate, n, sample_rate=16000):
  """The tutorial's sin_phase: sin(linspace(0, mod_rate n / sr 2 pi, n))."""
  ph = np.sin(np.linspace(0.0, mod_rate * (n / sample_rate) * 2.0 * np.pi, n))
  return ph.astype(np.float32)[None, :, None]


def cases():
  """name -> (kind, arrays, kwargs).  kind: 'mod_delay' = ModDelay(**kwargs)
  (audio, gain, phase); 'delay' = core.variable_length_delay(phase, audio,
  **kwargs)."""
  rng = np.random.default_rng(2025)
  out = {}

  def raw(b, n, two_d=False):
    a = audio_like(rng, b, n)
    g = rng.standard_normal((b, n, 1)).astype(np.float32)
    p = (2.0 * rng.standard_normal((b, n, 1))).astype(np.float32)
    if two_d:
      g, p = g[:, :, 0], p[:, :, 0]
    return a, g, p

  # ModDelay() on raw network outputs (get_controls + get_signal)
  out['moddelay_default'] = ('mod_delay', raw(2, 8000), {})
  out['moddelay_no_dry'] = ('mod_delay', raw(2, 3000), dict(add_dry=False))
  out['moddelay_2d_controls'] = ('mod_delay', raw(2, 3000, two_d=True), {})
  # 15 ms at 44.1 kHz: max_length = int(661.5) = 661
  out['moddelay_44k1'] = ('mod_delay', raw(2, 3000),
                          dict(center_ms=10.0, depth_ms=5.0, sample_rate=44100))
  out['moddelay_center_lt_depth'] = ('mod_delay', raw(2, 3000),
                                     dict(center_ms=2.0, depth_ms=8.0))
  # the tutorial's flanger / chorus / vibrato: controls given, no scaling
  for name, t in TUTORIAL.items():
    n = 4000
    a = audio_like(rng, 1, n)
    out['tutorial_' + name] = ('mod_delay', (a, np.ones((1, n, 1), np.float32),
                                             tutorial_phase(t['mod_rate'], n)),
                               dict(center_ms=t['center_ms'], depth_ms=t['depth_ms'],
                                    gain_scale_fn=None, phase_scale_fn=None))
  # variable_length_delay across max_length, including max_length > n_samples
  for L, n in ((1, 600), (2, 600), (7, 600), (400, 1600), (500, 300)):
    out['delay_L%d' % L] = ('delay', (delay_phases(rng, 2, n, L), audio_like(rng, 2, n)),
                            dict(max_length=L))
  # 2-D phase
  ph = delay_phases(rng, 2, 800, 24)[:, :, 0]
  out['delay_2d_phase'] = ('delay', (ph, audio_like(rng, 2, 800)), dict(max_length=24))
  return out


def full_inputs():
  """The full-length item: ModDelay() on raw outputs, N = 64000."""
  rng = np.random.default_rng(78)
  b, n = FULL['B'], FULL['N']
  return (audio_like(rng, b, n), rng.standard_normal((b, n, 1)).astype(np.float32),
          (2.0 * rng.standard_normal((b, n, 1))).astype(np.float32))


def run_case(ddsp, kind, arrays, kw):
  if kind == 'mod_delay':
    kw = dict(kw)
    for key in ('gain_scale_fn', 'phase_scale_fn'):
      if key in kw and kw[key] is not None:
        raise ValueError('only None stands in for a scale function here')
    return ddsp.effects.ModDelay(**kw)(*arrays)
  return ddsp.core.variable_length_delay(*arrays, **kw)


def mod_delay():
  ddsp = ref_on_shim.load()
  out = {}
  for name, (kind, arrays, kw) in cases().items():
    n, w = _both(lambda: run_case(ddsp, kind, arrays, kw))  # pylint: disable=cell-var-from-loop
    out[name + '_f32'] = np.asarray(n, np.float32)
    out[name + '_wide'] = np.asarray(w, np.float64)
  n, w = _both(lambda: ddsp.effects.ModDelay()(*full_inputs()))
  n, w = np.asarray(n, np.float64), np.asarray(w, np.float64)
  peak = np.abs(w).max()
  out['full_narrow_wide_maxrel'] = np.float64(np.abs(n - w).max() / peak)
  out['full_narrow_wide_l2rel'] = np.float64(np.sqrt(((n - w)**2).sum() / (w * w).sum()))
  packed = pack_outputs({'full_wide': w, 'full_f32': n})
  out.update({'full_' + k: v for k, v in packed.items()})
  return out


if __name__ == '__main__':
  got = mod_delay()
  if '--check' in sys.argv:
    compare('mod_delay', got, np.load(PATH))
    print('ok    mod_delay')
  else:
    np.savez_compressed(PATH, **got)
    print('wrote mod_delay %.0f kB' % (os.path.getsize(PATH) / 1e3))
