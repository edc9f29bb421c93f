"""Host-side mirror of the hot-path functions of `ddsp/core.py`.

Same names, argument meaning and error behaviour as the reference (file:line
cited per function); the arithmetic happens in libddsp_b200.so (hand-written
sm_100a kernels) through the ctypes C ABI in `_lib.py`.  torch is plumbing:
device memory and streams.  There is no CPU fallback.
"""
from collections import abc
from typing import Any, Dict, Optional, Sequence, Text

import numpy as np
import torch

from ddsp_b200 import _lib

AMP_METHODS = {'window': _lib.AMP_WINDOW, 'linear': _lib.AMP_LINEAR}


# ----------------------------------------------------------------------------
# Utility functions (core.py:30-129)
# ----------------------------------------------------------------------------
def _device():
  if not torch.cuda.is_available():
    raise RuntimeError(
        'ddsp_b200 needs a CUDA device (B200, sm_100a); there is no CPU '
        'fallback.')
  return torch.device('cuda', torch.cuda.current_device())


def torch_float32(x, device=None):
  """`tf_float32` (core.py:31-36): a contiguous float32 CUDA tensor."""
  if isinstance(x, torch.Tensor):
    if x.is_cuda and device is None:
      return x.to(torch.float32).contiguous()
    return x.to(device=device or _device(), dtype=torch.float32).contiguous()
  return torch.as_tensor(np.asarray(x, dtype=np.float32),
                         device=device or _device()).contiguous()


tf_float32 = torch_float32  # the reference's name for the same coercion


def make_iterable(x):
  """core.py:39-47."""
  if x is None:
    return []
  elif isinstance(x, (np.ndarray, torch.Tensor)):
    return [x]
  else:
    return x if isinstance(x, abc.Iterable) else [x]


def to_dict(x, keys):
  """core.py:50-61."""
  if isinstance(x, dict):
    return x
  else:
    x = make_iterable(x)
    if len(keys) != len(x):
      raise ValueError(f'Keys: {keys} must be the same length as {x}')
    return dict(zip(keys, x))


def nested_keys(nested_dict: Dict[Text, Any], delimiter: Text = '/',
                prefix: Text = '') -> Sequence[Text]:
  """core.py:78-102."""
  keys = []
  for k, v in nested_dict.items():
    key = k if not prefix else f'{prefix}{delimiter}{k}'
    if not isinstance(v, dict):
      keys.append(key)
    else:
      keys += nested_keys(v, prefix=key)
  return keys


def nested_lookup(nested_key: Text, nested_dict: Dict[Text, Any],
                  delimiter: Text = '/'):
  """core.py:105-129."""
  keys = nested_key.split(delimiter)
  value = nested_dict
  for key in keys:
    try:
      value = value[key]
    except KeyError:
      raise KeyError(f'Key \'{key}\' as a part of nested key \'{nested_key}\' '
                     'not found during nested dictionary lookup, out of '
                     f'available keys: {nested_keys(nested_dict)}')
  return value


def _shape(x):
  """Static shape of a tensor / array / nested list, without touching a GPU."""
  return tuple(x.shape) if hasattr(x, 'shape') else tuple(np.shape(x))


def _stream():
  return torch.cuda.current_stream().cuda_stream


class _on_device_of:
  """Context: make the device of the operands current (so the launch goes to
  THAT device's current stream), after checking they all live on one device."""

  def __init__(self, *tensors):
    devs = {t.device for t in tensors if isinstance(t, torch.Tensor)}
    if len(devs) > 1:
      raise ValueError('ddsp_b200: operands live on different devices: %s'
                       % sorted(str(d) for d in devs))
    dev = devs.pop() if devs else _device()
    if dev.type != 'cuda':
      raise ValueError('ddsp_b200: operands must be CUDA tensors, got %s' % dev)
    self._ctx = torch.cuda.device(dev)

  def __enter__(self):
    return self._ctx.__enter__()

  def __exit__(self, *exc):
    return self._ctx.__exit__(*exc)


def _check_out(out, shape, like, name='out'):
  """`out=` of the synthesizers is written by a kernel: B*N floats at data_ptr."""
  if (not isinstance(out, torch.Tensor) or not out.is_cuda or
      out.dtype != torch.float32 or not out.is_contiguous() or
      tuple(out.shape) != tuple(shape) or out.device != like.device):
    raise ValueError(
        f'{name} must be a contiguous float32 CUDA tensor of shape {tuple(shape)} '
        f'on {like.device}; got {type(out).__name__}'
        + (f' {tuple(out.shape)} {out.dtype} {out.device}' if isinstance(out, torch.Tensor) else ''))


def _no_grad_path(name, *tensors):
  """The kernels behind `core.*` / Processor / ProcessorGroup do not record an
  autograd graph.  A training loop that relies on gradients must go through
  ddsp_b200.autograd (decoder_train / HarmonicSynthesisFn / FilteredNoiseFn);
  silently returning detached audio would train nothing."""
  if torch.is_grad_enabled() and any(
      isinstance(t, torch.Tensor) and t.requires_grad for t in tensors):
    raise RuntimeError(
        f'ddsp_b200.core.{name}: an input requires grad, but this call is the '
        'inference path and returns detached audio.  Use ddsp_b200.autograd.'
        'decoder_train / HarmonicSynthesisFn / FilteredNoiseFn (CUDA backward '
        'kernels), or wrap the call in torch.no_grad().')


def _ptr(t):
  return 0 if t is None else t.data_ptr()


# ----------------------------------------------------------------------------
# Scaling (core.py:386-404) - used by callers that want the bare function; the
# processors call the fused controls kernels instead.
# ----------------------------------------------------------------------------
def exp_sigmoid(x, exponent=10.0, max_value=2.0, threshold=1e-7):
  """core.py:386-404.  Default arguments run the CUDA controls kernel."""
  x = torch_float32(x)
  if (exponent, max_value, threshold) == (10.0, 2.0, 1e-7) and not (
      torch.is_grad_enabled() and x.requires_grad):
    out = torch.empty_like(x)
    with _on_device_of(x):
      _lib.check(_lib.load().ddsp_b200_noise_controls(
          _ptr(x), _ptr(out), x.numel(), 0.0, 1, _stream()))
    return out
  return max_value * torch.sigmoid(x)**float(np.log(exponent)) + threshold


def sigmoid(x):
  """tf.nn.sigmoid, the default phase_scale_fn of effects.ModDelay
  (effects.py:331-344): 1 / (1 + e^-x) in the CUDA kernel `ddsp_b200_sigmoid`.
  Its device function is the one ModDelay's one-launch path applies to raw
  outputs, so both routes give the same bits.  An input that requires grad goes
  through torch.sigmoid."""
  x = torch_float32(x)
  if torch.is_grad_enabled() and x.requires_grad:
    return torch.sigmoid(x)
  out = torch.empty_like(x)
  with _on_device_of(x):
    _lib.check(_lib.load().ddsp_b200_sigmoid(_ptr(x), _ptr(out), x.numel(), _stream()))
  return out


# ----------------------------------------------------------------------------
# Frequency scaling of network outputs (core.py:207-348, 414-508) - frame-rate
# torch ops (a few thousand elements per item), device-agnostic.
# ----------------------------------------------------------------------------
def _as_f32(x):
  if torch.is_tensor(x):
    return x.to(torch.float32)
  return torch.as_tensor(np.asarray(x, dtype=np.float32))


def safe_log(x, eps=1e-5):
  """core.safe_log (core.py:213-216)."""
  x = _as_f32(x)
  return torch.log(torch.where(x <= 0.0, torch.full_like(x, eps), x))


def logb(x, base=2.0, eps=1e-5):
  """core.logb (core.py:219-221): safe_divide(safe_log(x), safe_log(base))."""
  den = safe_log(base, eps)
  den = torch.where(den == 0.0, torch.full_like(den, eps), den)
  return safe_log(x, eps) / den


def midi_to_hz(notes, midi_zero_silence: bool = False):
  """core.midi_to_hz (core.py:280-297)."""
  notes = _as_f32(notes)
  hz = 440.0 * (2.0 ** ((notes - 69.0) / 12.0))
  if midi_zero_silence:
    hz = torch.where(notes == 0.0, torch.zeros_like(hz), hz)
  return hz


def hz_to_midi(frequencies):
  """core.hz_to_midi (core.py:300-306): 0 Hz maps to MIDI 0."""
  frequencies = _as_f32(frequencies)
  notes = 12.0 * (logb(frequencies, 2.0) - logb(440.0, 2.0)) + 69.0
  return torch.where(frequencies <= 0.0, torch.zeros_like(notes), notes)


def unit_to_midi(unit, midi_min=20.0, midi_max=90.0, clip: bool = False):
  """core.unit_to_midi (core.py:309-315)."""
  unit = _as_f32(unit)
  unit = torch.clamp(unit, 0.0, 1.0) if clip else unit
  return midi_min + (midi_max - midi_min) * unit


def midi_to_unit(midi, midi_min=20.0, midi_max=90.0, clip: bool = False):
  """core.midi_to_unit (core.py:318-324)."""
  unit = (_as_f32(midi) - midi_min) / (midi_max - midi_min)
  return torch.clamp(unit, 0.0, 1.0) if clip else unit


def unit_to_hz(unit, hz_min, hz_max, clip: bool = False):
  """core.unit_to_hz (core.py:327-336): logarithmic map of [0, 1]."""
  midi = unit_to_midi(unit, midi_min=hz_to_midi(hz_min), midi_max=hz_to_midi(hz_max),
                      clip=clip)
  return midi_to_hz(midi)


def hz_to_unit(hz, hz_min, hz_max, clip: bool = False):
  """core.hz_to_unit (core.py:339-348)."""
  return midi_to_unit(hz_to_midi(hz), midi_min=hz_to_midi(hz_min),
                      midi_max=hz_to_midi(hz_max), clip=clip)


def _add_depth_axis(freqs, depth: int = 1):
  """core._add_depth_axis (core.py:414-420): [B, T, N*D] -> [B, T, N, D]."""
  b, t, combined = freqs.shape
  return freqs.reshape(b, t, int(combined) // depth, depth)


def frequencies_softmax(freqs, depth: int = 1, hz_min: float = 20.0,
                        hz_max: float = 8000.0):
  """core.frequencies_softmax (core.py:424-457)."""
  freqs = torch_float32(freqs, device=freqs.device if torch.is_tensor(freqs) else 'cpu')
  if freqs.dim() == 3:
    freqs = _add_depth_axis(freqs, depth)
  else:
    depth = int(freqs.shape[-1])
  f_probs = torch.softmax(freqs, dim=-1)
  unit_bins = torch.linspace(0.0, 1.0, depth, device=freqs.device)
  unit_bins = unit_bins[None, None, None, :]
  f_unit = torch.sum(unit_bins * f_probs, dim=-1)
  return unit_to_hz(f_unit, hz_min=hz_min, hz_max=hz_max)


def frequencies_sigmoid(freqs, depth: int = 1, hz_min: float = 0.0,
                        hz_max: float = 8000.0):
  """core.frequencies_sigmoid (core.py:460-507): a sum of `depth` sigmoids, each
  mapped logarithmically onto a slice of [hz_min, hz_max]."""
  freqs = torch_float32(freqs, device=freqs.device if torch.is_tensor(freqs) else 'cpu')
  if freqs.dim() == 3:
    freqs = _add_depth_axis(freqs, depth)
  else:
    depth = int(freqs.shape[-1])
  f_probs = torch.sigmoid(freqs)
  hz_scales = []
  hz_min_copy = hz_min
  remainder = hz_max - hz_min
  scale_factor = remainder**(1.0 / depth)
  for i in range(depth):
    if i == (depth - 1):
      hz_max = remainder
      hz_min = hz_min_copy
    else:
      hz_max = remainder * (1.0 - 1.0 / scale_factor)
      hz_min = 0
      remainder -= hz_max
    hz_scales.append(unit_to_hz(f_probs[..., i], hz_min=hz_min, hz_max=hz_max))
  return torch.sum(torch.stack(hz_scales, dim=-1), dim=-1)


# ----------------------------------------------------------------------------
# Resampling (core.py:573-714) - stand-alone ops (the synthesizers fuse them)
# ----------------------------------------------------------------------------
_RESAMPLE_METHODS = {'window': 0, 'linear': 1, 'nearest': 2, 'cubic': 3}


def _resample_3d(inputs, n_timesteps, method, add_endpoint):
  inputs = torch_float32(inputs)
  b, f, c = inputs.shape
  out = torch.empty((b, int(n_timesteps), c), dtype=torch.float32,
                    device=inputs.device)
  with _on_device_of(inputs):
    _lib.check(_lib.load().ddsp_b200_resample(
        _ptr(inputs), _ptr(out), b, f, c, int(n_timesteps),
        _RESAMPLE_METHODS[method], int(bool(add_endpoint)), _stream()))
  return out


def upsample_with_windows(inputs, n_timesteps: int, add_endpoint: bool = True):
  """core.upsample_with_windows (core.py:645-714)."""
  shape = _shape(inputs)
  if len(shape) != 3:
    raise ValueError('Upsample_with_windows() only supports 3 dimensions, '
                     'not {}.'.format(list(shape)))
  n_frames = shape[1] + (1 if add_endpoint else 0)
  n_intervals = n_frames - 1
  if n_frames >= n_timesteps:
    raise ValueError('Upsample with windows cannot be used for downsampling'
                     'More input frames ({}) than output timesteps ({})'.format(
                         n_frames, n_timesteps))
  if n_intervals <= 0 or n_timesteps % n_intervals != 0.0:
    minus_one = '' if add_endpoint else ' - 1'
    raise ValueError(
        'For upsampling, the target the number of timesteps must be divisible '
        'by the number of input frames{}. (timesteps:{}, frames:{}, '
        'add_endpoint={}).'.format(minus_one, n_timesteps, n_frames, add_endpoint))
  return _resample_3d(inputs, n_timesteps, 'window', add_endpoint)


def resample(inputs, n_timesteps: int, method: Text = 'linear',
             add_endpoint: bool = True):
  """core.resample (core.py:573-642) for 1-D / 2-D / 3-D / 4-D inputs, methods
  'nearest', 'linear', 'cubic' (tf.compat.v1 image kernels) and 'window'."""
  shape = _shape(inputs)
  if method not in ('nearest', 'linear', 'cubic', 'window'):
    raise ValueError('Method ({}) is invalid. Must be one of {}.'.format(
        method, "['nearest', 'linear', 'cubic', 'window']"))
  if len(shape) not in (1, 2, 3, 4):
    raise ValueError(f'resample takes 1-D to 4-D inputs, got shape {list(shape)}.')
  x = torch_float32(inputs)
  if len(shape) == 1:
    x = x[None, :, None]
  elif len(shape) == 2:
    x = x[:, :, None]
  elif len(shape) == 4:
    if method == 'window':
      # upsample_with_windows only takes 3-D (core.py:670-672)
      raise ValueError('Upsample_with_windows() only supports 3 dimensions, '
                       'not {}.'.format(list(shape)))
    # core.py:616-621 resizes [n_frames, n_freq] to [n_timesteps, n_freq]: the
    # n_freq axis maps onto itself, so this is the 3-D case over n_freq*channels.
    x = x.reshape(shape[0], shape[1], shape[2] * shape[3])
  if method == 'window':
    out = upsample_with_windows(x, n_timesteps, add_endpoint)
  else:
    out = _resample_3d(x, n_timesteps, method, add_endpoint)
  if len(shape) == 1:
    out = out[0, :, 0]
  elif len(shape) == 2:
    out = out[:, :, 0]
  elif len(shape) == 4:
    out = out.reshape(shape[0], int(n_timesteps), shape[2], shape[3])
  return out


# ----------------------------------------------------------------------------
# Harmonic synthesis (core.py:1048-1111)
# ----------------------------------------------------------------------------
def harmonic_controls(amplitudes, harmonic_distribution, f0_hz, sample_rate,
                      scale=True, normalize_below_nyquist=True):
  """synths.Harmonic.get_controls arithmetic (synths.py:94-121): exp_sigmoid,
  core.normalize_harmonics (core.py:894-907)."""
  sa, sh, sf = _shape(amplitudes), _shape(harmonic_distribution), _shape(f0_hz)
  if len(sh) != 3 or len(sa) != 3 or len(sf) != 3:
    raise ValueError('Harmonic controls must be 3-D [batch, frames, channels]; '
                     f'got {sa}, {sh}, {sf}.')
  b, f, k = sh
  if sa != (b, f, 1) or sf != (b, f, 1):
    raise ValueError(
        f'amplitudes {sa} and f0_hz {sf} must be [{b}, {f}, 1] to match '
        f'harmonic_distribution {sh}.')
  amplitudes = torch_float32(amplitudes)
  hd = torch_float32(harmonic_distribution)
  f0_hz = torch_float32(f0_hz)
  amps_out = torch.empty_like(amplitudes)
  hd_out = torch.empty_like(hd)
  flags = ((_lib.CTL_SCALE if scale else 0) |
           (_lib.CTL_NYQUIST if normalize_below_nyquist else 0))
  _no_grad_path('harmonic_controls', amplitudes, hd, f0_hz)
  with _on_device_of(amplitudes, hd, f0_hz):
    _lib.check(_lib.load().ddsp_b200_harmonic_controls(
        _ptr(amplitudes), _ptr(hd), _ptr(f0_hz), _ptr(amps_out), _ptr(hd_out),
        b, f, k, float(sample_rate), flags, _stream()))
  return amps_out, hd_out


def safe_divide(numerator, denominator, eps=1e-7):
  """core.safe_divide (core.py:207-210)."""
  safe = torch.where(denominator == 0.0, torch.full_like(denominator, eps),
                     denominator)
  return numerator / safe


def get_harmonic_frequencies(frequencies, n_harmonics: int):
  """core.get_harmonic_frequencies (core.py:1028-1045): f0 * [1..K]."""
  frequencies = torch_float32(frequencies)
  ratios = torch.linspace(1.0, float(n_harmonics), int(n_harmonics),
                          device=frequencies.device)
  return frequencies * ratios[None, None, :]


def remove_above_nyquist(frequency_envelopes, amplitude_envelopes,
                         sample_rate: int = 16000):
  """core.remove_above_nyquist (core.py:869-891)."""
  frequency_envelopes = torch_float32(frequency_envelopes)
  amplitude_envelopes = torch_float32(amplitude_envelopes)
  return torch.where(frequency_envelopes >= sample_rate / 2.0,
                     torch.zeros_like(amplitude_envelopes), amplitude_envelopes)


def normalize_harmonics(harmonic_distribution, f0_hz=None, sample_rate=None):
  """core.normalize_harmonics (core.py:894-907) on the controls kernel."""
  sh = _shape(harmonic_distribution)
  if len(sh) != 3:
    raise ValueError(f'harmonic_distribution must be 3-D, got {sh}.')
  b, f, _ = sh
  mask = sample_rate is not None and f0_hz is not None
  if f0_hz is None:
    f0_hz = torch.zeros((b, f, 1), dtype=torch.float32, device=_device())
  amps = torch.zeros((b, f, 1), dtype=torch.float32, device=_device())
  _, hd = harmonic_controls(amps, harmonic_distribution, f0_hz,
                            sample_rate if mask else 2.0, scale=False,
                            normalize_below_nyquist=mask)
  return hd


def angular_cumsum(angular_frequency, chunk_size: int = 1000,
                   tf_sequential: bool = False):
  """core.angular_cumsum (core.py:799-866): accumulated phase in [0, 2 pi) of an
  angular frequency [batch, time, ...] in radians per sample.

  Default: the wrapped running sum computed EXACTLY (64-bit fixed-point turns,
  three-pass scan) - the quantity the reference's chunked float32 cumsum
  approximates; `chunk_size` does not matter then.  tf_sequential=True reproduces
  the reference's own float32 arithmetic in its own order (chunks of
  `chunk_size`, mod-2pi stitching) - a debug mode for comparing against
  TensorFlow, one thread per (batch, channel)."""
  x = torch_float32(angular_frequency)
  shape = tuple(x.shape)
  if len(shape) < 2:
    raise ValueError(f'angular_frequency must be [batch, time, ...], got {list(shape)}.')
  b, n = shape[0], shape[1]
  c = 1
  for d in shape[2:]:
    c *= int(d)
  x3 = x.reshape(b, n, max(c, 1))
  out = torch.empty_like(x3)
  lib = _lib.load()
  with _on_device_of(x3):
    if tf_sequential:
      _lib.check(lib.ddsp_b200_angular_cumsum(
          _ptr(x3), _ptr(out), b, n, max(c, 1), int(chunk_size), 2, None, 0,
          _stream()))
    else:
      nbytes = lib.ddsp_b200_oscillator_bank_workspace(b, n, max(c, 1))
      ws = torch.empty((max(nbytes, 1),), dtype=torch.uint8, device=x3.device)
      _lib.check(lib.ddsp_b200_angular_cumsum(
          _ptr(x3), _ptr(out), b, n, max(c, 1), int(chunk_size), 0, _ptr(ws),
          nbytes, _stream()))
  return out.reshape(shape)


def oscillator_bank(frequency_envelopes, amplitude_envelopes,
                    sample_rate: int = 16000, sum_sinusoids: bool = True,
                    use_angular_cumsum: bool = False,
                    phase_mode: Text = 'exact'):
  """core.oscillator_bank (core.py:911-962) on audio-rate envelopes
  [batch, n_samples, n_sinusoids].

  phase_mode='exact' (default): phase is accumulated wrapped and exactly (64-bit
  fixed point) whatever `use_angular_cumsum` says - both reference modes
  approximate this.  phase_mode='tf_sequential': the reference's own float32
  arithmetic in its own order - tf.cumsum, or angular_cumsum (chunks of 1000)
  when use_angular_cumsum - reproducing TensorFlow's phase error (debug)."""
  if phase_mode not in ('exact', 'tf_sequential'):
    raise ValueError(f"phase_mode must be 'exact' or 'tf_sequential', got {phase_mode!r}.")
  sf, sa = _shape(frequency_envelopes), _shape(amplitude_envelopes)
  if len(sf) != 3 or sf != sa:
    raise ValueError(f'frequency_envelopes {sf} and amplitude_envelopes {sa} must '
                     'both be [batch, n_samples, n_sinusoids].')
  b, n, k = sf
  f = torch_float32(frequency_envelopes)
  a = torch_float32(amplitude_envelopes)
  _no_grad_path('oscillator_bank', f, a)
  lib = _lib.load()
  with _on_device_of(f, a):
    if phase_mode == 'tf_sequential':
      wavs = torch.empty((b, n, k), dtype=torch.float32, device=f.device)
      _lib.check(lib.ddsp_b200_oscillator_bank_tf_sequential(
          _ptr(f), _ptr(a), _ptr(wavs), b, n, k, float(sample_rate),
          int(bool(use_angular_cumsum)), 1000, _stream()))
      return wavs.sum(-1) if sum_sinusoids else wavs
    out = torch.empty((b, n) if sum_sinusoids else (b, n, k), dtype=torch.float32,
                      device=f.device)
    nbytes = lib.ddsp_b200_oscillator_bank_workspace(b, n, k)
    ws = torch.empty((max(nbytes, 1),), dtype=torch.uint8, device=f.device)
    _lib.check(lib.ddsp_b200_oscillator_bank(
        _ptr(f), _ptr(a), _ptr(out), b, n, k, float(sample_rate),
        int(bool(sum_sinusoids)), _ptr(ws), nbytes, _stream()))
  return out


def sinusoidal_synthesis(frequencies, amplitudes, n_samples: int = 64000,
                         sample_rate: int = 16000,
                         amp_resample_method: Text = 'window', out=None,
                         accumulate: bool = False):
  """Frame-rate bank of sinusoids with per-sinusoid frequencies
  [batch, n_frames, n_sinusoids] -> audio [batch, n_samples]: the fused form of
  resample + resample + core.oscillator_bank (synths.py:305-323) - the
  [batch, n_samples, n_sinusoids] envelopes are never materialised."""
  sf, sa = _shape(frequencies), _shape(amplitudes)
  if len(sf) != 3 or sf != sa:
    raise ValueError(f'frequencies {sf} and amplitudes {sa} must both be '
                     '[batch, n_frames, n_sinusoids].')
  b, f, k = sf
  n_samples = int(n_samples)
  freqs = torch_float32(frequencies)
  amps = torch_float32(amplitudes)
  _no_grad_path('sinusoidal_synthesis', freqs, amps)
  if out is None:
    out = torch.empty((b, n_samples), dtype=torch.float32, device=freqs.device)
    accumulate = False
  else:
    _check_out(out, (b, n_samples), freqs)
  lib = _lib.load()
  with _on_device_of(freqs, amps, out):
    nbytes = lib.ddsp_b200_sinusoidal_workspace(b, f, k)
    ws = torch.empty((max(nbytes, 1),), dtype=torch.uint8, device=freqs.device)
    _lib.check(lib.ddsp_b200_sinusoidal_forward(
        _ptr(freqs), _ptr(amps), _ptr(out), b, f, k, n_samples, float(sample_rate),
        AMP_METHODS[amp_resample_method], int(bool(accumulate)), _ptr(ws), nbytes,
        _stream()))
  return out


# ----------------------------------------------------------------------------
# Wavetable synthesis (core.py:1167-1282)
# ----------------------------------------------------------------------------
def linear_lookup(phase, wavetables):
  """core.linear_lookup (core.py:1168-1209): phase [batch, n_samples] or
  [batch, n_samples, 1]; wavetables [batch, n_wavetable] or
  [batch, n_samples, n_wavetable] -> [batch, n_samples].

  Entry n_wavetable is entry 0 and the weight on entry j is
  relu(1 - |phase - j / n_wavetable| * n_wavetable): linear interpolation at
  phase * n_wavetable, with entries outside [0, n_wavetable] weighing zero - so
  a phase below 0 or above 1 fades to silence within one entry, as in the
  reference.  One gather kernel (`ddsp_b200_linear_lookup`); inference only."""
  sp, sw = _shape(phase), _shape(wavetables)
  if len(sp) == 3 and sp[2] == 1:
    sp = sp[:2]
  if len(sp) != 2 or len(sw) not in (2, 3) or sw[0] != sp[0] or (
      len(sw) == 3 and sw[1] not in (1, sp[1])):
    raise ValueError(f'phase {_shape(phase)} must be [batch, n_samples(, 1)] and '
                     f'wavetables {sw} [batch, n_wavetable] or [batch, n_samples, '
                     'n_wavetable].')
  b, n = sp
  w = int(sw[-1])
  ph = torch_float32(phase).reshape(b, n)
  tab = torch_float32(wavetables)
  if len(sw) == 3 and sw[1] == 1 and n != 1:
    sw = sw[:1] + sw[2:]              # one table frame broadcasts over time
    tab = tab.reshape(b, w)
  _no_grad_path('linear_lookup', ph, tab)
  out = torch.empty((b, n), dtype=torch.float32, device=ph.device)
  with _on_device_of(ph, tab):
    _lib.check(_lib.load().ddsp_b200_linear_lookup(
        _ptr(ph), _ptr(tab), _ptr(out), b, n, w, int(len(sw) == 3), _stream()))
  return out


def harmonic_distribution_to_wavetable(harmonic_distribution, n_wavetable=2048):
  """core.harmonic_distribution_to_wavetable (core.py:1212-1226):
  (n_wavetable / 2) * irfft([0, hd, 0, ...]) on torch.fft (a frame-rate helper, off
  the synthesis path).  The reference pads with n_wavetable / 2 - n_harmonics
  zeros, which fails for more harmonics than that; this raises a ValueError."""
  sh = _shape(harmonic_distribution)
  if len(sh) != 3:
    raise ValueError(f'harmonic_distribution must be [batch, time, n_harmonics], '
                     f'got {sh}.')
  n_pad = int(n_wavetable / 2 - sh[-1])
  if n_pad < 0:
    raise ValueError(f'harmonic_distribution_to_wavetable: {sh[-1]} harmonics do not '
                     f'fit a wavetable of {n_wavetable} samples (at most '
                     f'{int(n_wavetable) // 2}).')
  hd = torch_float32(harmonic_distribution)
  fft_in = torch.nn.functional.pad(hd, (1, n_pad))
  return torch.fft.irfft(fft_in.to(torch.complex64), dim=-1) * (n_wavetable / 2)


def _wavetable_shapes(frequencies, amplitudes, wavetables, n_samples):
  """Shape checks and the reference's ValueErrors of wavetable_synthesis, before
  any device work.  Returns (b, f0 frames, amp frames, table frames, W)."""
  sf, sa, sw = _shape(frequencies), _shape(amplitudes), _shape(wavetables)
  if len(sf) != 3 or len(sa) != 3 or sf[2] != 1 or sa[2] != 1 or sf[0] != sa[0]:
    raise ValueError(f'frequencies {sf} and amplitudes {sa} must be '
                     '[batch, n_frames, 1].')
  if len(sw) not in (2, 3) or sw[0] != sf[0]:
    raise ValueError(f'wavetables {sw} must be [batch, n_wavetable] or '
                     '[batch, n_frames, n_wavetable].')
  fa = sa[1]
  if fa + 1 >= n_samples:
    # core.py:682-685 (the amplitudes are resampled with 'window')
    raise ValueError('Upsample with windows cannot be used for downsampling'
                     'More input frames ({}) than output timesteps ({})'.format(
                         fa + 1, n_samples))
  if n_samples % fa != 0:
    # core.py:687-693
    raise ValueError(
        'For upsampling, the target the number of timesteps must be divisible '
        'by the number of input frames. (timesteps:{}, frames:{}, '
        'add_endpoint=True).'.format(n_samples, fa + 1))
  r = 1 if len(sw) == 2 else sw[1]
  return sf[0], sf[1], fa, r, sw[-1]


def _wavetable_launch(f0, amps, tables, n_samples, sample_rate, scale, out, accumulate):
  """ddsp_b200_wavetable_forward on [B,F,1] controls (equal frame counts, F | N)
  and [B,R,W] tables."""
  b, f = f0.shape[0], f0.shape[1]
  r, w = tables.shape[1], tables.shape[2]
  lib = _lib.load()
  with _on_device_of(f0, amps, tables, out):
    nbytes = lib.ddsp_b200_wavetable_workspace(b, f, r, w, n_samples, 0)
    ws = torch.empty((max(nbytes, 1),), dtype=torch.uint8, device=f0.device)
    _lib.check(lib.ddsp_b200_wavetable_forward(
        _ptr(f0), _ptr(amps), _ptr(tables), _ptr(out), b, f, r, w, n_samples,
        float(sample_rate), int(bool(scale)), int(bool(accumulate)), _ptr(ws), nbytes,
        _stream()))
  return out


def wavetable_synthesis(frequencies, amplitudes, wavetables, n_samples: int = 64000,
                        sample_rate: int = 16000, out=None, accumulate: bool = False):
  """core.wavetable_synthesis (core.py:1229-1282): frame-rate f0 [batch, frames, 1]
  and amplitudes [batch, frames, 1], wavetables [batch, n_wavetable] (static) or
  [batch, table_frames, n_wavetable] -> audio [batch, n_samples].

  One kernel (`ddsp_b200_wavetable_forward`) reads the frame-rate tables: the
  reference's audio-rate tables and its [batch, n_samples, n_wavetable + 1] lookup
  weights are never formed.  The phase is the exclusive cumsum of f0 / sr mod 1,
  accumulated exactly (64-bit fixed point).  When f0 and the amplitudes have
  different frame counts, or n_samples is not a multiple of f0's, both are first
  brought to audio rate with the resample kernel."""
  n_samples = int(n_samples)
  b, ff, fa, _, _ = _wavetable_shapes(frequencies, amplitudes, wavetables, n_samples)
  f0 = torch_float32(frequencies)
  amps = torch_float32(amplitudes)
  tables = torch_float32(wavetables)
  _no_grad_path('wavetable_synthesis', f0, amps, tables)
  if tables.dim() == 2:
    tables = tables[:, None, :]
  if out is None:
    out = torch.empty((b, n_samples), dtype=torch.float32, device=f0.device)
    accumulate = False
  else:
    _check_out(out, (b, n_samples), f0)
  if ff != fa or n_samples % ff != 0:
    with _on_device_of(f0, amps):
      f0 = resample(f0, n_samples)
      amps = resample(amps, n_samples, method='window')
  return _wavetable_launch(f0, amps, tables, n_samples, sample_rate, False, out,
                           accumulate)


def wavetable_raw(amplitudes, wavetables, f0_hz, n_samples: int = 64000,
                  sample_rate: int = 16000, out=None, accumulate: bool = False):
  """synths.Wavetable()(...) with the default exp_sigmoid scaling from RAW network
  outputs in one launch: exp_sigmoid is applied to the amplitudes and to each
  table row as it lands in shared memory (bit-identical to get_signal of
  get_controls).  Needs f0 and amplitudes on the same frames, a multiple of which
  n_samples is, and 3-D tables."""
  n_samples = int(n_samples)
  b, ff, fa, _, _ = _wavetable_shapes(f0_hz, amplitudes, wavetables, n_samples)
  if ff != fa or len(_shape(wavetables)) != 3:
    raise ValueError('wavetable_raw needs f0 and amplitudes on the same frames and '
                     '[batch, frames, n_wavetable] tables.')
  f0 = torch_float32(f0_hz)
  amps = torch_float32(amplitudes)
  tables = torch_float32(wavetables)
  _no_grad_path('wavetable_raw', f0, amps, tables)
  if out is None:
    out = torch.empty((b, n_samples), dtype=torch.float32, device=f0.device)
    accumulate = False
  else:
    _check_out(out, (b, n_samples), f0)
  return _wavetable_launch(f0, amps, tables, n_samples, sample_rate, True, out,
                           accumulate)


# ----------------------------------------------------------------------------
# Variable-length delay (core.py:1285-1313) and ModDelay's signal
# ----------------------------------------------------------------------------
def _delay_controls(name, audio, controls):
  """Shape checks of the delay before any device work: audio [batch, n_samples],
  each control [batch, n_samples] or [batch, n_samples, 1].  Returns (b, n)."""
  sa = _shape(audio)
  if len(sa) != 2:
    raise ValueError(f'{name}: audio must be [batch, n_samples], got {sa}.')
  for key, x in controls.items():
    sx = _shape(x)
    if len(sx) == 3 and sx[2] == 1:
      sx = sx[:2]
    if sx != sa:
      raise ValueError(f'{name}: {key} {_shape(x)} must be [batch, n_samples] or '
                       f'[batch, n_samples, 1] with audio {sa}.')
  return sa


def _check_max_length(name, max_length):
  if int(max_length) != max_length or int(max_length) < 1:
    raise ValueError(f'{name}: max_length must be an integer >= 1, got {max_length}.')
  return int(max_length)


def _mod_delay_launch(audio, gain, phase, max_length, phase_scale, phase_offset,
                      scale, add_dry):
  """ddsp_b200_mod_delay_forward on checked inputs; gain may be None."""
  b, n = audio.shape
  out = torch.empty((b, n), dtype=torch.float32, device=audio.device)
  with _on_device_of(audio, gain, phase):
    _lib.check(_lib.load().ddsp_b200_mod_delay_forward(
        _ptr(audio), _ptr(gain), _ptr(phase), _ptr(out), b, n, int(max_length),
        float(phase_scale), float(phase_offset), int(bool(scale)), int(bool(add_dry)),
        _stream()))
  return out


def variable_length_delay(phase, audio, max_length: int = 512):
  """core.variable_length_delay (core.py:1285-1313): phase [batch, n_samples(, 1)],
  audio [batch, n_samples] -> [batch, n_samples].

  Sample n reads its own history e_k = audio[n - k] (0 <= k < max_length, zero
  before the start) with linear_lookup's rule at phase * max_length; entry
  max_length is entry 0, so phase 1 gives the undelayed sample and a phase further
  outside [0, 1] is silent, as in the reference.  One kernel
  (`ddsp_b200_mod_delay_forward`); the reference's [batch, n_samples, max_length]
  frames are never formed.  Inference only (see autograd.variable_length_delay)."""
  max_length = _check_max_length('variable_length_delay', max_length)
  b, n = _delay_controls('variable_length_delay', audio, {'phase': phase})
  ph = torch_float32(phase).reshape(b, n)
  x = torch_float32(audio)
  _no_grad_path('variable_length_delay', ph, x)
  return _mod_delay_launch(x, None, ph, max_length, 1.0, 0.0, False, False)


def mod_delay(audio, gain, phase, max_length, phase_scale, phase_offset,
              add_dry=True, scale=False):
  """effects.ModDelay.get_signal (effects.py:369-393) in one launch:
  variable_length_delay(phase * phase_scale + phase_offset, audio, max_length)
  * gain (+ audio with add_dry).  scale=True: gain and phase are raw network
  outputs, and exp_sigmoid / sigmoid (ModDelay.get_controls' defaults) run inside
  the kernel, bit-identical to applying core.exp_sigmoid / core.sigmoid first."""
  max_length = _check_max_length('ModDelay', max_length)
  b, n = _delay_controls('ModDelay', audio, {'gain': gain, 'phase': phase})
  x = torch_float32(audio)
  g = torch_float32(gain).reshape(b, n)
  ph = torch_float32(phase).reshape(b, n)
  _no_grad_path('mod_delay', x, g, ph)
  return _mod_delay_launch(x, g, ph, max_length, phase_scale, phase_offset, scale,
                           add_dry)


def harmonic_synthesis(frequencies,
                       amplitudes,
                       harmonic_shifts=None,
                       harmonic_distribution=None,
                       n_samples: int = 64000,
                       sample_rate: int = 16000,
                       amp_resample_method: Text = 'window',
                       use_angular_cumsum: bool = False,
                       out: Optional[torch.Tensor] = None,
                       accumulate: bool = False,
                       phase_mode: Text = 'recurrence'):
  """core.harmonic_synthesis (core.py:1048-1111).

  The common case (no harmonic_shifts, 'window' / 'linear' amplitudes, n_samples
  a multiple of the frame count) is ONE fused kernel.  With `harmonic_shifts`
  (core.py:1084-1093) the harmonics are no longer integer multiples of one
  phase: f0 * k * (1 + shift) and amp * hd are formed at frame rate, as the
  reference does, and the frame-rate oscillator bank with per-sinusoid phases
  (`sinusoidal_synthesis`) takes over.  'nearest' / 'cubic' amplitudes and
  non-integer hops take the reference's own decomposition on our kernels:
  `resample` + `resample` + `oscillator_bank` (audio-rate envelopes exist then).

  Phase is accumulated wrapped and exactly (64-bit fixed point) whatever
  `use_angular_cumsum` says - that is what angular_cumsum approximates
  (core.py:803-817; DESIGN.md "phase").  phase_mode: 'recurrence' (default) /
  'direct' choose how sin(k phi) is evaluated in the fused kernel;
  'tf_sequential' reproduces TensorFlow's float32 phase arithmetic in its own
  order (tf.cumsum, or angular_cumsum if use_angular_cumsum) - a debug mode for
  small shapes that materialises the envelopes.
  """
  if amp_resample_method not in ('nearest', 'linear', 'cubic', 'window'):
    # core.py:632-634
    raise ValueError('Method ({}) is invalid. Must be one of {}.'.format(
        amp_resample_method, "['nearest', 'linear', 'cubic', 'window']"))
  if phase_mode not in ('recurrence', 'direct', 'tf_sequential'):
    raise ValueError("phase_mode must be 'recurrence', 'direct' or "
                     f"'tf_sequential', got {phase_mode!r}.")
  sf, sa = _shape(frequencies), _shape(amplitudes)
  if len(sf) != 3 or len(sa) != 3:
    # core.py:670-672 (the window upsampler only takes 3-D inputs)
    raise ValueError('Upsample_with_windows() only supports 3 dimensions, '
                     'not {}.'.format(list(sa)))
  b, f, _ = sf
  if sa != (b, f, 1) or sf != (b, f, 1):
    raise ValueError(f'frequencies {sf} and amplitudes {sa} must both be '
                     f'[batch, n_frames, 1].')
  k = 1
  if harmonic_distribution is not None:
    sh = _shape(harmonic_distribution)
    if len(sh) != 3 or sh[:2] != (b, f):
      raise ValueError(f'harmonic_distribution {sh} must be [{b}, {f}, '
                       'n_harmonics].')
    k = int(sh[-1])
  if harmonic_shifts is not None:
    ss = _shape(harmonic_shifts)
    if len(ss) != 3 or ss[:2] != (b, f) or (harmonic_distribution is not None
                                             and ss[-1] != k):
      raise ValueError(f'harmonic_shifts {ss} must be [{b}, {f}, n_harmonics'
                       f'{"=" + str(k) if harmonic_distribution is not None else ""}].')
    k = int(ss[-1])
  n_samples = int(n_samples)
  if amp_resample_method == 'window':
    if f >= n_samples:
      # core.py:682-685
      raise ValueError('Upsample with windows cannot be used for downsampling'
                       'More input frames ({}) than output timesteps ({})'.format(
                           f + 1, n_samples))
    if n_samples % f != 0:
      # core.py:687-693
      raise ValueError(
          'For upsampling, the target the number of timesteps must be divisible '
          'by the number of input frames{}. (timesteps:{}, frames:{}, '
          'add_endpoint={}).'.format('', n_samples, f + 1, True))
  frequencies = torch_float32(frequencies)
  amplitudes = torch_float32(amplitudes)
  if harmonic_distribution is not None:
    harmonic_distribution = torch_float32(harmonic_distribution)
  if harmonic_shifts is not None:
    harmonic_shifts = torch_float32(harmonic_shifts)
  _no_grad_path('harmonic_synthesis', frequencies, amplitudes, harmonic_distribution,
                harmonic_shifts)
  if out is not None:
    _check_out(out, (b, n_samples), frequencies)
  else:
    accumulate = False

  fused_ok = (amp_resample_method in AMP_METHODS and n_samples % f == 0 and
              phase_mode != 'tf_sequential')
  if harmonic_shifts is None and fused_ok:
    mode = {'recurrence': _lib.PHASE_RECURRENCE, 'direct': _lib.PHASE_DIRECT}[
        phase_mode]
    if out is None:
      out = torch.empty((b, n_samples), dtype=torch.float32,
                        device=frequencies.device)
    with _on_device_of(frequencies, amplitudes, harmonic_distribution, out):
      _lib.check(_lib.load().ddsp_b200_harmonic_forward(
          _ptr(frequencies), _ptr(amplitudes), _ptr(harmonic_distribution),
          _ptr(out), b, f, k, n_samples, float(sample_rate),
          AMP_METHODS[amp_resample_method], mode, int(bool(accumulate)), _stream()))
    return out

  # frame-rate harmonic frequencies / amplitudes, float32 op for op as the
  # reference (core.py:1091-1099): (f0 * k) * (1 + shifts), amplitudes * hd
  with _on_device_of(frequencies, amplitudes, harmonic_distribution, harmonic_shifts):
    harmonic_frequencies = get_harmonic_frequencies(frequencies, k)
    if harmonic_shifts is not None:
      harmonic_frequencies = harmonic_frequencies * (1.0 + harmonic_shifts)
    harmonic_amplitudes = (amplitudes * harmonic_distribution
                           if harmonic_distribution is not None
                           else amplitudes.expand(b, f, k).contiguous())
    if fused_ok:
      return sinusoidal_synthesis(harmonic_frequencies, harmonic_amplitudes,
                                  n_samples=n_samples, sample_rate=sample_rate,
                                  amp_resample_method=amp_resample_method, out=out,
                                  accumulate=accumulate)
    # core.py:1101-1110 on the stand-alone kernels (audio-rate envelopes exist)
    frequency_envelopes = resample(harmonic_frequencies, n_samples)
    amplitude_envelopes = resample(harmonic_amplitudes, n_samples,
                                   method=amp_resample_method)
    audio = oscillator_bank(
        frequency_envelopes, amplitude_envelopes, sample_rate=sample_rate,
        use_angular_cumsum=use_angular_cumsum,
        phase_mode='tf_sequential' if phase_mode == 'tf_sequential' else 'exact')
  if out is None:
    return audio
  if accumulate:
    out += audio
  else:
    out.copy_(audio)
  return out


def streaming_harmonic_synthesis(frequencies,
                                 amplitudes,
                                 harmonic_distribution=None,
                                 initial_phase=None,
                                 n_samples: int = 64000,
                                 sample_rate: int = 16000,
                                 amp_resample_method: Text = 'linear'):
  """core.streaming_harmonic_synthesis (core.py:1114-1164): single-f0 harmonic
  bank with a carried phase.  Returns (audio [B, n_samples], final_phase
  [B, 1, 1]) - feed final_phase back as initial_phase for the next hop
  (training/inference.py:463-478)."""
  sf, sa = _shape(frequencies), _shape(amplitudes)
  if len(sf) != 3 or len(sa) != 3 or sa != sf or sf[2] != 1:
    raise ValueError(f'frequencies {sf} and amplitudes {sa} must both be '
                     '[batch, n_frames, 1].')
  if amp_resample_method not in ('nearest', 'linear', 'cubic', 'window'):
    raise ValueError('Method ({}) is invalid. Must be one of {}.'.format(
        amp_resample_method, "['nearest', 'linear', 'cubic', 'window']"))
  if amp_resample_method not in AMP_METHODS:
    raise NotImplementedError(amp_resample_method)
  b, f, _ = sf
  n_samples = int(n_samples)
  if n_samples % f != 0:
    raise NotImplementedError(
        f'n_samples ({n_samples}) must be a multiple of the number of frames ({f}).')
  frequencies = torch_float32(frequencies)
  amplitudes = torch_float32(amplitudes)
  k = 1
  hd = None
  lib = _lib.load()
  if harmonic_distribution is not None:
    hd = torch_float32(harmonic_distribution)
    k = int(hd.shape[-1])
    # normalize_harmonics (core.py:1143-1146): Nyquist mask + row normalisation
    hd_n = torch.empty_like(hd)
    amp_copy = torch.empty_like(amplitudes)
    _lib.check(lib.ddsp_b200_harmonic_controls(
        _ptr(amplitudes), _ptr(hd), _ptr(frequencies), _ptr(amp_copy), _ptr(hd_n),
        b, f, k, float(sample_rate), _lib.CTL_NYQUIST, _stream()))
    hd = hd_n
  init = None
  if initial_phase is not None:
    init = torch_float32(initial_phase).reshape(b).contiguous()
  audio = torch.empty((b, n_samples), dtype=torch.float32, device=frequencies.device)
  final_phase = torch.empty((b,), dtype=torch.float32, device=frequencies.device)
  _lib.check(lib.ddsp_b200_streaming_harmonic_forward(
      _ptr(frequencies), _ptr(amplitudes), _ptr(hd), _ptr(init), _ptr(audio),
      _ptr(final_phase), b, f, k, n_samples, float(sample_rate),
      AMP_METHODS[amp_resample_method], _stream()))
  return audio, final_phase.reshape(b, 1, 1)


# ----------------------------------------------------------------------------
# Time-varying FIR / filtered noise (core.py:1316-1655)
# ----------------------------------------------------------------------------
def get_fft_size(frame_size: int, ir_size: int, power_of_2: bool = True) -> int:
  """core.py:1317-1335 (kept for API parity; the CUDA path is time-domain)."""
  convolved_frame_size = ir_size + frame_size - 1
  if power_of_2:
    return int(2**np.ceil(np.log2(convolved_frame_size)))
  raise NotImplementedError('power_of_2=False needs scipy.fftpack.')


def frequency_impulse_response(magnitudes, window_size: int = 0):
  """core.frequency_impulse_response (core.py:1534-1565)."""
  nb = int(_shape(magnitudes)[-1])
  lib = _lib.load()
  s = lib.ddsp_b200_ir_size(nb, int(window_size))
  if s < 0:
    raise ValueError(f'frequency_impulse_response needs >= 2 frequencies, got {nb}.')
  magnitudes = torch_float32(magnitudes)
  ir = torch.empty(tuple(magnitudes.shape[:-1]) + (s,), dtype=torch.float32,
                   device=magnitudes.device)
  bf = magnitudes.numel() // nb
  _lib.check(lib.ddsp_b200_frequency_impulse_response(
      _ptr(magnitudes), _ptr(ir), bf, nb, int(window_size), _stream()))
  return ir


def apply_window_to_impulse_response(impulse_response, window_size: int = 0,
                                     causal: bool = False):
  """core.apply_window_to_impulse_response (core.py:1477-1531) for callers of the
  reference function: zero-phase (or `causal`) impulse responses [..., ir_size] ->
  Hann-windowed, causal form, cropped to `window_size` (made odd) when that is
  shorter.  Frame-rate torch ops on whatever device the input lives on; the
  synthesis path never calls it - `frequency_impulse_response` and the fused noise
  kernels build the windowed taps straight from the magnitudes."""
  ir = _as_f32(impulse_response)
  if causal:
    ir = torch.fft.fftshift(ir, dim=-1)
  ir_size = int(ir.shape[-1])
  if window_size <= 0 or window_size > ir_size:
    window_size = ir_size
  # tf.signal.hann_window: periodic for even lengths, symmetric for odd ones
  window = torch.hann_window(window_size, periodic=(window_size % 2 == 0),
                             dtype=torch.float32, device=ir.device)
  padding = ir_size - window_size
  if padding > 0:
    half_idx = (window_size + 1) // 2
    window = torch.cat([window[half_idx:],
                        torch.zeros(padding, dtype=torch.float32, device=ir.device),
                        window[:half_idx]], dim=0)
  else:
    window = torch.fft.fftshift(window, dim=-1)
  ir = window * ir
  if padding > 0:
    first_half_start = (ir_size - (half_idx - 1)) + 1
    second_half_end = half_idx + 1
    ir = torch.cat([ir[..., first_half_start:], ir[..., :second_half_end]], dim=-1)
  else:
    ir = torch.fft.fftshift(ir, dim=-1)
  return ir


def crop_and_compensate_delay(audio, audio_size: int, ir_size: int, padding: Text,
                              delay_compensation: int):
  """core.crop_and_compensate_delay (core.py:1338-1379): the slice
  `audio[:, start:-end]` of a convolution output, with the reference's ValueError and
  its Python slice semantics (an `end` of 0 gives an empty result).  A view - no
  kernel; `fft_convolve` applies the same index arithmetic (`_crop_range`) inside its
  kernels instead of materialising the uncropped signal."""
  if not isinstance(audio, torch.Tensor):
    audio = torch.as_tensor(np.asarray(audio, dtype=np.float32))
  start, _, _ = _crop_range(int(audio.shape[-1]), audio_size, ir_size, padding,
                            delay_compensation)
  crop_size = ir_size + audio_size - 1 if padding == 'valid' else audio_size
  end = (int(audio.shape[-1]) - crop_size) - start
  return audio[:, start:-end]


def _crop_range(total_size, audio_size, ir_size, padding, delay_compensation):
  """Index arithmetic of crop_and_compensate_delay (core.py:1338-1379),
  including Python's slice semantics of `audio[:, start:-end]`."""
  if padding == 'valid':
    crop_size = ir_size + audio_size - 1
  elif padding == 'same':
    crop_size = audio_size
  else:
    raise ValueError('Padding must be \'valid\' or \'same\', instead '
                     'of {}.'.format(padding))
  crop = total_size - crop_size
  start = ((ir_size - 1) // 2 - 1 if delay_compensation < 0
           else delay_compensation)
  end = crop - start
  rng = range(total_size)[start:-end]
  return start, len(rng), crop_size


# Impulse responses longer than this take a frequency-domain formulation instead of
# the direct-form FIR kernel: the direct form costs audio_size * ir_size MACs per
# item - the cross-over is a few thousand taps.  One long IR per item (the Reverb
# case: 48000 taps, effects.py:28-117; SURVEY 8f-3) runs the hand-written
# partitioned overlap-save convolution `ddsp_b200_fft_convolve_lti`.
FFT_CONVOLVE_MIN_IR = 2048


def _fft_convolve_cufft(audio, impulse_response, n_ir_frames, frame_size, fft_size,
                        start, crop_size):
  """The reference's own algorithm (core.py:1445-1473) on torch.fft: frame (hop =
  frame_size, zero padded), rfft both, multiply, irfft, overlap-add, crop."""
  b, n = audio.shape
  pad = n_ir_frames * frame_size - n
  frames = torch.nn.functional.pad(audio, (0, pad)).reshape(b, n_ir_frames, frame_size)
  audio_fft = torch.fft.rfft(frames, n=fft_size, dim=-1)
  ir_fft = torch.fft.rfft(impulse_response, n=fft_size, dim=-1)   # broadcasts batch 1
  frames_out = torch.fft.irfft(audio_fft * ir_fft, n=fft_size, dim=-1)
  if n_ir_frames == 1:
    total = frames_out[:, 0, :]
  else:
    total_size = (n_ir_frames - 1) * frame_size + fft_size
    total = torch.nn.functional.fold(
        frames_out.transpose(1, 2), output_size=(total_size, 1),
        kernel_size=(fft_size, 1), stride=(frame_size, 1))[:, 0, :, 0]
  return total[:, start:start + crop_size].contiguous()


def fft_convolve_lti(audio, impulse_response, start, out_len, out=None,
                     accumulate=False, reverse_audio=False, reverse_ir=False):
  """Full linear convolution of audio [B, N] with ONE impulse response per item
  [1 or B, S], cropped to [start, start + out_len): `ddsp_b200_fft_convolve_lti`
  (partitioned overlap-save, hand-written FFTs).  reverse_*: read that operand back
  to front (what the backward pass needs)."""
  b, n = audio.shape
  ir_batch, s_len = impulse_response.shape
  if out is None:
    out = torch.empty((b, out_len), dtype=torch.float32, device=audio.device)
    accumulate = False
  lib = _lib.load()
  flags = ((_lib.LTI_REVERSE_AUDIO if reverse_audio else 0) |
           (_lib.LTI_REVERSE_IR if reverse_ir else 0))
  with _on_device_of(audio, impulse_response, out):
    nbytes = lib.ddsp_b200_fft_convolve_lti_workspace(b, n, s_len, ir_batch)
    ws = torch.empty((max(nbytes, 1),), dtype=torch.uint8, device=audio.device)
    _lib.check(lib.ddsp_b200_fft_convolve_lti(
        _ptr(audio), _ptr(impulse_response), _ptr(out), b, n, s_len, ir_batch,
        int(start), int(out_len), int(bool(accumulate)), flags, _ptr(ws), nbytes,
        _stream()))
  return out


def fft_convolve(audio, impulse_response, padding: Text = 'same',
                 delay_compensation: int = -1, out=None, accumulate=False):
  """core.fft_convolve (core.py:1382-1473).

  Computed as the mathematically identical direct-form time-varying FIR
  (frame / rfft / multiply / irfft / overlap_and_add / crop folded into index
  math; SURVEY.md A.6) - the name is kept for drop-in compatibility.
  """
  sa, si = _shape(audio), _shape(impulse_response)
  if len(sa) != 2 or len(si) not in (2, 3):
    raise ValueError(f'audio must be [batch, time] and impulse_response 2-D or '
                     f'3-D; got {sa} and {si}.')
  batch_size, audio_size = sa
  if len(si) == 2:
    si = (si[0], 1, si[1])
  ir_batch, n_ir_frames, ir_size = si
  if not (ir_batch == 1 and batch_size > 1) and batch_size != ir_batch:
    # core.py:1441-1443
    raise ValueError('Batch size of audio ({}) and impulse response ({}) must '
                     'be the same.'.format(batch_size, ir_batch))
  frame_size = int(np.ceil(audio_size / n_ir_frames))
  n_audio_frames = -(-audio_size // frame_size)
  if n_audio_frames != n_ir_frames:
    # core.py:1452-1457
    raise ValueError(
        'Number of Audio frames ({}) and impulse response frames ({}) do not '
        'match. For small hop size = ceil(audio_size / n_ir_frames), '
        'number of impulse response frames must be a multiple of the audio '
        'size.'.format(n_audio_frames, n_ir_frames))
  fft_size = get_fft_size(frame_size, ir_size, power_of_2=True)
  total_size = (n_ir_frames - 1) * frame_size + fft_size
  start, out_len, crop_size = _crop_range(total_size, audio_size, ir_size,
                                          padding, delay_compensation)
  if out_len != crop_size:
    # The reference's `audio[:, start:-end]` degenerates when end <= 0 (e.g.
    # end == 0 yields an empty tensor).  Reproduce the empty case; refuse the
    # rest rather than guess.
    if out_len == 0:
      return torch.empty((batch_size, 0), dtype=torch.float32, device=_device())
    raise NotImplementedError(
        'crop_and_compensate_delay slice is degenerate for this shape '
        f'(start={start}, total={total_size}, crop={crop_size}).')
  audio = torch_float32(audio)
  impulse_response = torch_float32(impulse_response).reshape(si)
  if ir_size >= FFT_CONVOLVE_MIN_IR and n_ir_frames == 1:
    # one long impulse response per item (effects.Reverb): hand-written
    # partitioned overlap-save convolution (csrc/longconv.cuh)
    ir2 = impulse_response.reshape(ir_batch, ir_size).contiguous()
    if torch.is_grad_enabled() and (audio.requires_grad or ir2.requires_grad):
      # trainable reverb (effects.py:70-79): forward and backward are the same
      # kernels (the backward on time-reversed operands)
      from ddsp_b200 import autograd as _ag
      wet = _ag.FftConvolveLtiFn.apply(audio, ir2, int(start), int(crop_size))
      if out is None:
        return wet
      _check_out(out, (batch_size, crop_size), audio)
      if accumulate:
        out += wet
      else:
        out.copy_(wet)
      return out
    if out is not None:
      _check_out(out, (batch_size, crop_size), audio)
    return fft_convolve_lti(audio, ir2, int(start), int(crop_size), out=out,
                            accumulate=accumulate)
  if ir_size >= FFT_CONVOLVE_MIN_IR:
    # time-varying filter with long impulse responses (several IR frames of >= 2048
    # taps): no reference configuration does this; the reference's own framed
    # algorithm on cuFFT
    wet = _fft_convolve_cufft(audio, impulse_response, n_ir_frames, frame_size,
                              fft_size, int(start), int(crop_size))
    if out is None:
      return wet
    _check_out(out, tuple(wet.shape), audio)
    if accumulate:
      out += wet
    else:
      out.copy_(wet)
    return out
  if out is None:
    out = torch.empty((batch_size, crop_size), dtype=torch.float32,
                      device=audio.device)
    accumulate = False
  else:
    _check_out(out, (batch_size, crop_size), audio)
  impulse_response = impulse_response.contiguous()
  _no_grad_path('fft_convolve', audio, impulse_response)
  with _on_device_of(audio, impulse_response, out):
    _lib.check(_lib.load().ddsp_b200_fir_time_varying(
        _ptr(audio), _ptr(impulse_response), _ptr(out), batch_size,
        audio_size, n_ir_frames, ir_size, ir_batch,
        _lib.PAD_SAME if padding == 'same' else _lib.PAD_VALID,
        int(start), int(bool(accumulate)), _stream()))
  return out


def frequency_filter(audio, magnitudes, window_size: int = 0,
                     padding: Text = 'same'):
  """core.frequency_filter (core.py:1628-1655)."""
  impulse_response = frequency_impulse_response(magnitudes,
                                                window_size=window_size)
  return fft_convolve(audio, impulse_response, padding=padding)


def uniform_noise(batch_size, n_samples, seed=0, offset=0, device=None):
  """Stand-in for tf.random.uniform([B, N], -1, 1) (synths.py:192-193):
  Philox4x32-10 keyed by `seed`, counter (sample/4, batch, offset)."""
  out = torch.empty((batch_size, n_samples), dtype=torch.float32,
                    device=device or _device())
  _lib.check(_lib.load().ddsp_b200_uniform_noise(
      _ptr(out), batch_size, n_samples, int(seed) & (2**64 - 1),
      int(offset) & (2**64 - 1), _stream()))
  return out


def filtered_noise(magnitudes, n_samples, window_size=257, noise=None, seed=0,
                   offset=0, out=None, accumulate=False):
  """FilteredNoise.get_signal arithmetic (synths.py:181-196): uniform noise ->
  core.frequency_filter (core.py:1628-1655), fused where the shape allows."""
  sm = _shape(magnitudes)
  if len(sm) != 3:
    raise ValueError('magnitudes must be [batch, n_frames, n_filter_banks], got '
                     f'{sm}.')
  b, f, nb = sm
  n_samples = int(n_samples)
  if noise is not None and _shape(noise) != (b, n_samples):
    raise ValueError(f'noise must be [{b}, {n_samples}], got {_shape(noise)}.')
  frame_size = int(np.ceil(n_samples / f))
  n_audio_frames = -(-n_samples // frame_size)
  if n_audio_frames != f:
    # core.py:1452-1457
    raise ValueError(
        'Number of Audio frames ({}) and impulse response frames ({}) do not '
        'match. For small hop size = ceil(audio_size / n_ir_frames), '
        'number of impulse response frames must be a multiple of the audio '
        'size.'.format(n_audio_frames, f))
  lib = _lib.load()
  magnitudes = torch_float32(magnitudes)
  if noise is not None:
    noise = torch_float32(noise)
  if out is None:
    out = torch.empty((b, n_samples), dtype=torch.float32,
                      device=magnitudes.device)
    accumulate = False
  else:
    _check_out(out, (b, n_samples), magnitudes)
  _no_grad_path('filtered_noise', magnitudes)
  with _on_device_of(magnitudes, noise, out):
    ws_bytes = lib.ddsp_b200_filtered_noise_workspace(b, f, nb, n_samples,
                                                      int(window_size))
    workspace = (torch.empty((ws_bytes,), dtype=torch.uint8,
                             device=magnitudes.device) if ws_bytes else None)
    _lib.check(lib.ddsp_b200_filtered_noise_forward(
        _ptr(magnitudes), _ptr(noise), int(seed) & (2**64 - 1),
        int(offset) & (2**64 - 1), _ptr(out), b, f, nb, n_samples,
        int(window_size), int(bool(accumulate)), _ptr(workspace), ws_bytes,
        _stream()))
  return out


def decoder_forward(amps, harmonic_distribution, f0_hz, noise_magnitudes,
                    n_samples, sample_rate=16000, amp_resample_method='window',
                    normalize_below_nyquist=True, window_size=0,
                    initial_bias=-5.0, noise=None, seed=0, offset=0):
  """The `ae.gin` DAG (ae.gin:47-72) from RAW network outputs, two launches:
  Harmonic (exp_sigmoid scaling + Nyquist normalisation fused into the tile
  staging) then FilteredNoise (exp_sigmoid fused likewise) accumulating into the
  same audio buffer (= processors.Add).  Raises NotImplementedError outside the
  fused regime; ProcessorGroup then runs the per-processor path."""
  sh = _shape(harmonic_distribution)
  sm = _shape(noise_magnitudes)
  if len(sh) != 3 or len(sm) != 3:
    raise ValueError(f'decoder inputs must be 3-D, got {sh} and {sm}.')
  b, f, k = sh
  if _shape(amps) != (b, f, 1) or _shape(f0_hz) != (b, f, 1) or sm[:2] != (b, f):
    raise ValueError(
        f'decoder inputs disagree: amps {_shape(amps)}, f0_hz {_shape(f0_hz)}, '
        f'harmonic_distribution {sh}, noise_magnitudes {sm}.')
  if amp_resample_method not in AMP_METHODS:
    raise NotImplementedError(amp_resample_method)
  n_samples = int(n_samples)
  if noise is not None and _shape(noise) != (b, n_samples):
    raise ValueError(f'noise must be [{b}, {n_samples}], got {_shape(noise)}.')
  amps = torch_float32(amps)
  hd = torch_float32(harmonic_distribution)
  f0_hz = torch_float32(f0_hz)
  mags = torch_float32(noise_magnitudes)
  if noise is not None:
    noise = torch_float32(noise)
  _no_grad_path('decoder_forward', amps, hd, f0_hz, mags)
  out = torch.empty((b, n_samples), dtype=torch.float32, device=hd.device)
  flags = _lib.CTL_SCALE | (_lib.CTL_NYQUIST if normalize_below_nyquist else 0)
  with _on_device_of(amps, hd, f0_hz, mags, noise):
    _lib.check(_lib.load().ddsp_b200_decoder_forward(
        _ptr(amps), _ptr(hd), _ptr(f0_hz), _ptr(mags), _ptr(noise),
        int(seed) & (2**64 - 1), int(offset) & (2**64 - 1), _ptr(out), b, f, k,
        sm[2], n_samples, float(sample_rate), AMP_METHODS[amp_resample_method],
        flags, int(window_size), float(initial_bias), _stream()))
  return out


def noise_controls(magnitudes, initial_bias=-5.0, scale=True):
  """FilteredNoise.get_controls arithmetic (synths.py:165-179)."""
  magnitudes = torch_float32(magnitudes)
  _no_grad_path('noise_controls', magnitudes)
  out = torch.empty_like(magnitudes)
  with _on_device_of(magnitudes):
    _lib.check(_lib.load().ddsp_b200_noise_controls(
        _ptr(magnitudes), _ptr(out), magnitudes.numel(), float(initial_bias),
        int(bool(scale)), _stream()))
  return out


def add(signal_one, signal_two, out=None):
  """processors.Add.get_signal (processors.py:174-176)."""
  a = torch_float32(signal_one)
  b = torch_float32(signal_two)
  if a.shape != b.shape:
    a, b = torch.broadcast_tensors(a, b)
    a, b = a.contiguous(), b.contiguous()
  if out is None:
    out = torch.empty_like(a)
  _lib.check(_lib.load().ddsp_b200_add(_ptr(a), _ptr(b), _ptr(out), a.numel(),
                                       _stream()))
  return out
