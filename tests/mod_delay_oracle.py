"""NumPy restatement of the reference's modulated delay (ddsp/core.py:1285-1313
variable_length_delay, ddsp/effects.py:328-393 ModDelay): the arbiter of the
mod-delay tests.

float64 mode is the gather form: the position p = phase' L in double, then
linear_lookup's two taps of the time-reversed history (entry k of sample n is
x[n - k], zero before the start; entry L is entry 0).  No [batch, n_samples,
max_length] array is built, so a full-length item stays cheap.  float32 mode
follows TensorFlow's order (zero pad, frames, reversal, linspace distances,
relu weights, reduce_sum), materialises the frames and is meant for the short
cases.
"""
import numpy as np

from oracle import ddsp_oracle as o


def sigmoid(x, dtype=np.float64):
  """tf.nn.sigmoid: 1 / (1 + exp(-x))."""
  x = np.asarray(x, dtype)
  one = np.asarray(1, dtype)
  return (one / (one + np.exp(-x))).astype(dtype)


def _delay_gather(phase, audio, L):
  """float64 gather form; phase [B, N] (already mapped), audio [B, N]."""
  b, n = audio.shape
  x = phase * float(L)
  fl = np.floor(x)
  fr = x - fl
  idx = np.arange(n)[None, :]
  bi = np.arange(b)[:, None]
  out = np.zeros((b, n), np.float64)
  for j, w in ((fl, 1.0 - fr), (fl + 1.0, fr)):
    ok = (j >= 0) & (j <= L)
    k = np.where(ok, j, 0).astype(np.int64)
    k = np.where(k == L, 0, k)                  # entry L is entry 0
    m = idx - k
    v = np.where(m >= 0, audio[bi, np.clip(m, 0, n - 1)], 0.0)
    out += np.where(ok, w * v, 0.0)
  return out


def _delay_tf(phase, audio, L):
  """variable_length_delay as written, in float32: pad L - 1 zeros in front,
  frames of L with step 1, reversed, then linear_lookup (core.py:1168-1209)."""
  f32 = np.float32
  b, n = audio.shape
  padded = np.concatenate([np.zeros((b, L - 1), f32), audio.astype(f32)], axis=1)
  frames = padded[:, np.arange(n)[:, None] + np.arange(L)[None, :]][..., ::-1]
  tab = np.concatenate([frames, frames[..., :1]], axis=-1)
  nw = L + 1
  delta = f32(1.0) / f32(nw - 1)
  grid = np.concatenate([f32(0.0) + delta * np.arange(nw - 1, dtype=f32),
                         np.ones(1, f32)]).astype(f32)
  dist = np.abs(phase.astype(f32)[..., None] - grid[None, None, :]).astype(f32)
  dist = (dist * f32(nw - 1)).astype(f32)
  weights = np.maximum(f32(1.0) - dist, f32(0.0)).astype(f32)
  return (weights * tab).astype(f32).sum(-1, dtype=f32)


def variable_length_delay(phase, audio, max_length=512, dtype=np.float64):
  """core.variable_length_delay: phase [B, N] or [B, N, 1], audio [B, N]."""
  phase = np.asarray(phase, dtype)
  audio = np.asarray(audio, dtype)
  if phase.ndim == 3:
    phase = phase[:, :, 0]
  if dtype == np.float32:
    return _delay_tf(phase, audio, int(max_length))
  return _delay_gather(phase, audio, int(max_length))


def delay_map(center_ms=15.0, depth_ms=10.0, sample_rate=16000):
  """effects.py:381-386: (max_length, depth_phase, center_phase)."""
  max_delay_ms = center_ms + depth_ms
  return (int(sample_rate / 1000.0 * max_delay_ms), depth_ms / max_delay_ms,
          center_ms / max_delay_ms)


def mod_delay(audio, gain, phase, center_ms=15.0, depth_ms=10.0, sample_rate=16000,
              scale=True, add_dry=True, dtype=np.float64, map_dtype=None):
  """ModDelay(...)(audio, gain, phase): get_controls (exp_sigmoid / sigmoid when
  scale, else none) then get_signal.

  map_dtype: the precision of phase * depth_phase + center_phase (effects.py:386).
  The reference evaluates it in the type of the phase it holds: a tensor from
  get_controls (dtype), or, with phase_scale_fn=None, the caller's float32 NumPy
  array, which stays float32 (the tutorial's route; pass np.float32)."""
  audio = np.asarray(audio, dtype)
  gain = np.asarray(gain, dtype)
  phase = np.asarray(phase, dtype)
  if scale:
    gain = o.exp_sigmoid(gain, dtype=dtype)
    phase = sigmoid(phase, dtype)
  max_length, depth_phase, center_phase = delay_map(center_ms, depth_ms, sample_rate)
  md = map_dtype or dtype
  phase = (phase.astype(md) * md(depth_phase) + md(center_phase)).astype(dtype)
  wet = variable_length_delay(phase, audio, max_length, dtype)
  if gain.ndim == 3:
    gain = gain[..., 0]
  wet = (wet * gain).astype(dtype)
  return (wet + audio).astype(dtype) if add_dry else wet
