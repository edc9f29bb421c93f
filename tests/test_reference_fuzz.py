"""Randomised cross-check of the oracle against the UNMODIFIED reference (CPU).

The golden fixtures pin the oracle on the path's configurations; this sweeps the
argument space around them - shapes, paddings, delays, odd / even / degenerate filter
windows, every amplitude resampling method, both phase accumulators, sample rates,
optional arguments - in the reference's "wide" mode (its own code evaluated in float64)
against the oracle's float64 mode.  It is how the odd-window Hann discrepancy was found.

The arguments are drawn from fixed seeds by the fuzz_*_cases generators of
tests/golden/make_golden.py; the reference's results on them are in
tests/golden/reference_fuzz.npz (each output's shape, peak and L2 norm, and up to
make_golden.SAMPLE of its elements), and test_reference_pin.py checks that file
against a fresh reference run wherever the reference sources are present.
"""
import os

import numpy as np
import pytest

from oracle import ddsp_oracle as o
from tests.golden import make_golden as mg

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), 'golden')


@pytest.fixture(scope='module')
def ref():
  return mg.unpack_outputs(np.load(os.path.join(GOLD, 'reference_fuzz.npz')))


def _close(got, want, tol, what):
  """The whole of `got` against a stored reference output: same shape, the stored
  elements within tol * max(1, peak), and peak and L2 norm within what that
  elementwise bound allows."""
  shape, values, peak, l2 = want
  got = np.asarray(got, np.float64)
  assert got.shape == shape, (what, got.shape, shape)
  if got.size:
    bound = tol * max(1.0, peak)
    assert np.abs(got.ravel()[mg.sample_index(got.size)] - values).max() <= bound, what
    assert abs(np.abs(got).max() - peak) <= bound, what
    assert abs(np.sqrt((got * got).sum()) - l2) <= bound * np.sqrt(got.size), what


def _w(x):
  return None if x is None else x.astype(np.float64)


def test_fft_convolve_shapes_paddings_delays(ref):
  checked = 0
  for i, c in enumerate(mg.fuzz_fft_convolve_cases()):
    want = ref['fft_convolve_%d' % i]
    kw = dict(padding=c['padding'], delay_compensation=c['delay_compensation'])
    if want is None:            # the reference raises on these arguments
      with pytest.raises(Exception):
        o.fft_convolve(_w(c['a']), _w(c['ir']), **kw)
      continue
    got = o.fft_convolve(_w(c['a']), _w(c['ir']), **kw)
    _close(got, want, 1e-9, ('fft_convolve', c['a'].shape, c['ir'].shape, kw))
    checked += 1
  assert checked >= 12


def test_frequency_filter_windows(ref):
  for i, c in enumerate(mg.fuzz_frequency_filter_cases()):
    got = o.frequency_filter(_w(c['audio']), _w(c['magnitudes']),
                             window_size=c['window_size'])
    _close(got, ref['frequency_filter_%d' % i], 1e-9,
           ('frequency_filter', c['audio'].shape, c['magnitudes'].shape, c['window_size']))


def test_harmonic_synthesis_argument_space(ref):
  for i, c in enumerate(mg.fuzz_harmonic_synthesis_cases()):
    got = o.harmonic_synthesis(_w(c['f0']), _w(c['amp']), harmonic_shifts=_w(c['shifts']),
                               harmonic_distribution=_w(c['hd']), n_samples=c['n_samples'],
                               sample_rate=c['sample_rate'], amp_resample_method=c['method'],
                               use_angular_cumsum=c['use_angular_cumsum'], dtype=np.float64)
    _close(got, ref['harmonic_synthesis_%d' % i], 2e-7,
           ('harmonic_synthesis', i, c['f0'].shape, c['n_samples'], c['method'],
            c['use_angular_cumsum'], c['sample_rate']))


def test_controls_oscillators_streaming_and_scalers(ref):
  for i, (kind, c) in enumerate(mg.fuzz_misc_cases()):
    key = '%s_%d' % (kind, i)
    if kind == 'get_controls':
      got = o.harmonic_get_controls(_w(c['a']), _w(c['h']), _w(c['f0']),
                                    sample_rate=c['sample_rate'], scale=c['scale'],
                                    normalize_below_nyquist=c['nyquist'], dtype=np.float64)
      for name in ('amplitudes', 'harmonic_distribution', 'f0_hz'):
        _close(got[name], ref['%s_%s' % (key, name)], 1e-12, (key, name))
    elif kind == 'oscillator_bank':
      got = o.oscillator_bank(_w(c['fe']), _w(c['ae']), sample_rate=c['sample_rate'],
                              sum_sinusoids=c['sum_sinusoids'],
                              use_angular_cumsum=c['use_angular_cumsum'], dtype=np.float64)
      _close(got, ref[key], 1e-8, key)
    elif kind == 'streaming':           # carried phase
      got = o.streaming_harmonic_synthesis(_w(c['f0']), _w(c['amp']), _w(c['hd']),
                                           _w(c['phase']), n_samples=c['n_samples'],
                                           sample_rate=16000, amp_resample_method=c['method'],
                                           dtype=np.float64)
      _close(got[0], ref[key + '_audio'], 1e-8, key)
      shape, values, _, _ = ref[key + '_phase']
      phase = np.asarray(got[1], np.float64)
      assert phase.shape == shape and values.size == phase.size, key
      d = np.angle(np.exp(1j * (phase.ravel() - values)))    # on the circle
      assert np.abs(d).max() <= 1e-8, key
    elif kind == 'scalers':
      _close(o.exp_sigmoid(_w(c['x']), c['exponent'], c['max_value'], c['threshold'],
                           dtype=np.float64), ref[key + '_exp_sigmoid'], 1e-12, key)
      _close(o.frequencies_sigmoid(_w(c['fr']), depth=c['depth'], dtype=np.float64),
             ref[key + '_sigmoid'], 1e-9, key)
      _close(o.frequencies_softmax(_w(c['fr']), depth=c['depth'], dtype=np.float64),
             ref[key + '_softmax'], 1e-9, key)
    else:                               # Sinusoidal
      ctl = o.sinusoidal_get_controls(_w(c['a']), _w(c['fr']), dtype=np.float64)
      got = o.sinusoidal_get_signal(ctl['amplitudes'], ctl['frequencies'], c['n_samples'],
                                    amp_resample_method=c['method'], dtype=np.float64)
      _close(got, ref[key], 1e-8, key)
