"""NumPy restatement of the reference's wavetable synthesizer (ddsp/core.py:1167-1282,
ddsp/synths.py:199-257): the arbiter of the wavetable tests.

float64 mode is the gather form: phase -> two table entries -> linear weights, and
two table rows -> linear time weights.  No [batch, n_samples, n_wavetable] array is
built, so a full-length item stays cheap.  float32 mode follows TensorFlow's order
(float32 index math of the v1 bilinear resize, sequential float32 exclusive cumsum,
the literal distance-weight form of linear_lookup); it materialises the audio-rate
tables and is meant for the short cases.
"""
import numpy as np

from oracle import ddsp_oracle as o


def _lookup_gather(phase, tab, rows=None):
  """linear_lookup rule in float64.  phase [B, N]; tab [B, R, W]; sample t reads
  row rows[t] (default: row t when R == N, row 0 when R == 1).  Entry W is entry
  0; entries outside [0, W] weigh zero."""
  W = tab.shape[-1]
  ext = np.concatenate([tab, tab[..., :1]], axis=-1)
  x = phase * W
  j0 = np.floor(x)
  fr = x - j0
  j0 = j0.astype(np.int64)
  if rows is None:
    rows = np.arange(phase.shape[1]) if tab.shape[1] > 1 else np.zeros(phase.shape[1], np.int64)
  rows = np.broadcast_to(np.asarray(rows)[None, :], phase.shape)
  bidx = np.arange(phase.shape[0])[:, None]
  out = np.zeros(phase.shape, np.float64)
  for j, w in ((j0, 1.0 - fr), (j0 + 1, fr)):
    ok = (j >= 0) & (j <= W)
    v = ext[bidx, rows, np.clip(j, 0, W)]
    out += np.where(ok, w * v, 0.0)
  return out


def _lookup_tf(phase, tab, dtype):
  """linear_lookup as written (core.py:1168-1209), in `dtype`."""
  ext = np.concatenate([tab, tab[..., :1]], axis=-1).astype(dtype)
  n = ext.shape[-1]
  grid = np.linspace(0.0, 1.0, n).astype(dtype)
  dist = np.abs(phase[..., None].astype(dtype) - grid[None, None, :]).astype(dtype)
  dist = (dist * dtype(n - 1)).astype(dtype)
  weights = np.maximum(dtype(1.0) - dist, dtype(0.0)).astype(dtype)
  return (weights * ext).astype(dtype).sum(-1, dtype=dtype)


def linear_lookup(phase, wavetables, dtype=np.float64):
  """core.linear_lookup: phase [B, N] or [B, N, 1]; wavetables [B, W] or
  [B, N, W] -> [B, N]."""
  phase = np.asarray(phase, dtype)
  tab = np.asarray(wavetables, dtype)
  if tab.ndim == 2:
    tab = tab[:, None, :]
  if phase.ndim == 3:
    phase = phase[:, :, 0]
  if dtype == np.float32:
    return _lookup_tf(phase, tab, np.float32)
  return _lookup_gather(phase, tab)


def harmonic_distribution_to_wavetable(harmonic_distribution, n_wavetable=2048,
                                       dtype=np.float64):
  """core.harmonic_distribution_to_wavetable: (W/2) irfft([0, hd, 0...])."""
  hd = np.asarray(harmonic_distribution, np.float64)
  n_harmonics = hd.shape[-1]
  n_pad = int(n_wavetable / 2 - n_harmonics)
  if n_pad < 0:
    raise ValueError(f'harmonic_distribution_to_wavetable: {n_harmonics} harmonics do '
                     f'not fit a wavetable of {n_wavetable} samples (at most '
                     f'{n_wavetable // 2}).')
  fft_in = np.pad(hd, [(0, 0), (0, 0), (1, n_pad)])
  return (np.fft.irfft(fft_in, axis=-1) * (n_wavetable / 2)).astype(dtype)


def _check_window(n_frames, n_samples):
  # upsample_with_windows (core.py:676-693), add_endpoint=True
  if n_frames + 1 >= n_samples:
    raise ValueError('Upsample with windows cannot be used for downsampling'
                     'More input frames ({}) than output timesteps ({})'.format(
                         n_frames + 1, n_samples))
  if n_samples % n_frames != 0:
    raise ValueError(
        'For upsampling, the target the number of timesteps must be divisible '
        'by the number of input frames. (timesteps:{}, frames:{}, '
        'add_endpoint=True).'.format(n_samples, n_frames + 1))


def wavetable_synthesis(frequencies, amplitudes, wavetables, n_samples=64000,
                        sample_rate=16000, dtype=np.float64):
  """core.wavetable_synthesis (core.py:1229-1282)."""
  f = np.asarray(frequencies, dtype)
  a = np.asarray(amplitudes, dtype)
  tab = np.asarray(wavetables, dtype)
  _check_window(a.shape[1], n_samples)
  amp_env = o.upsample_with_windows(a, n_samples, dtype=dtype)[:, :, 0]
  f_env = o.resample(f, n_samples, dtype=dtype,
                     tf_index_math=dtype == np.float32)[:, :, 0]
  vel = (f_env / dtype(sample_rate)).astype(dtype)
  if dtype == np.float32:
    phase = np.cumsum(vel, axis=1, dtype=np.float32)
    phase = np.concatenate([np.zeros_like(phase[:, :1]), phase[:, :-1]], axis=1)
    phase = np.mod(phase, np.float32(1.0)).astype(np.float32)
    if tab.ndim == 3 and tab.shape[1] > 1:
      tab = o.resample(tab, n_samples, dtype=np.float32, tf_index_math=True)
    elif tab.ndim == 2:
      tab = tab[:, None, :]
    return (_lookup_tf(phase, tab, np.float32) * amp_env).astype(np.float32)
  phase = np.cumsum(vel, axis=1)
  phase = np.concatenate([np.zeros_like(phase[:, :1]), phase[:, :-1]], axis=1) % 1.0
  if tab.ndim == 2:
    tab = tab[:, None, :]
  if tab.shape[1] == 1:
    return _lookup_gather(phase, tab) * amp_env
  lo, hi, frac = o._bilinear_indices(tab.shape[1], n_samples, False, False)  # pylint: disable=protected-access
  v_lo = _lookup_gather(phase, tab, lo)
  v_hi = _lookup_gather(phase, tab, hi)
  return (v_lo + (v_hi - v_lo) * frac[None, :]) * amp_env


def wavetable_get_controls(amplitudes, wavetables, f0_hz, scale=True,
                           dtype=np.float64):
  """synths.Wavetable.get_controls (synths.py:212-236): exp_sigmoid on the
  amplitudes and the wavetables, f0 unchanged."""
  a = np.asarray(amplitudes, dtype)
  w = np.asarray(wavetables, dtype)
  if scale:
    a = o.exp_sigmoid(a, dtype=dtype)
    w = o.exp_sigmoid(w, dtype=dtype)
  return {'amplitudes': a, 'wavetables': w, 'f0_hz': np.asarray(f0_hz, dtype)}


def wavetable_get_signal(amplitudes, wavetables, f0_hz, n_samples=64000,
                         sample_rate=16000, dtype=np.float64):
  """synths.Wavetable.get_signal (synths.py:238-257).  The reference first
  resamples the tables to n_samples; wavetable_synthesis then resamples n_samples
  to n_samples, the identity.  A 2-D table [B, W] is resampled along its only
  axis into a static table of n_samples entries, as the reference does."""
  w = np.asarray(wavetables, dtype)
  if w.ndim == 2:
    w = o.resample(w, n_samples, dtype=dtype, tf_index_math=dtype == np.float32)
  elif dtype == np.float32 and w.shape[1] > 1:
    pass                                   # resampled inside wavetable_synthesis
  return wavetable_synthesis(f0_hz, amplitudes, w, n_samples, sample_rate, dtype)


def wavetable(amplitudes, wavetables, f0_hz, n_samples=64000, sample_rate=16000,
              scale=True, dtype=np.float64):
  """Wavetable(...)(amplitudes, wavetables, f0_hz): get_controls then get_signal."""
  c = wavetable_get_controls(amplitudes, wavetables, f0_hz, scale, dtype)
  return wavetable_get_signal(c['amplitudes'], c['wavetables'], c['f0_hz'],
                              n_samples, sample_rate, dtype)
