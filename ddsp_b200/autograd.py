"""Differentiable wrappers of the synthesis kernels (C4: decoder forward +
backward through SpectralLoss).

The reference differentiates through every TF op of `core.harmonic_synthesis` /
`core.frequency_filter`; here forward and backward are the hand-written CUDA
kernels, exposed as `torch.autograd.Function`s:

  * `HarmonicSynthesisFn`  - d amplitudes, d harmonic_distribution, d f0 (the
    phase path, `models/inverse_synthesis.py:84-117`; computed only when f0
    requires grad);
  * `FilteredNoiseFn`      - d magnitudes (the filter is linear in them);
  * `DecoderFn` / `decoder_train` - the whole `ae.gin` decoder from RAW network
    outputs: forward is the fused two-kernel pipeline (`get_controls` in shared
    memory), backward is the two synthesizer backward kernels plus the
    `get_controls` backward kernels - no frame-rate torch op on either pass.

`harmonic_controls` / `exp_sigmoid` below are the same `get_controls` arithmetic as
differentiable torch ops, kept for callers that compose their own graphs.
"""
import math

import torch

from ddsp_b200 import _lib
from ddsp_b200 import core


def _stream():
  return torch.cuda.current_stream().cuda_stream


class HarmonicSynthesisFn(torch.autograd.Function):
  """core.harmonic_synthesis (core.py:1048-1111), differentiable in
  amplitudes and harmonic_distribution."""

  @staticmethod
  def forward(ctx, f0_hz, amplitudes, harmonic_distribution, n_samples,
              sample_rate, amp_resample_method):
    f0_hz = core.torch_float32(f0_hz)
    amplitudes = core.torch_float32(amplitudes)
    harmonic_distribution = core.torch_float32(harmonic_distribution)
    ctx.save_for_backward(f0_hz, amplitudes, harmonic_distribution)
    ctx.cfg = (int(n_samples), float(sample_rate), amp_resample_method)
    return core.harmonic_synthesis(
        f0_hz, amplitudes, harmonic_distribution=harmonic_distribution,
        n_samples=n_samples, sample_rate=sample_rate,
        amp_resample_method=amp_resample_method)

  @staticmethod
  def backward(ctx, grad_audio):
    f0_hz, amplitudes, hd = ctx.saved_tensors
    n_samples, sample_rate, method = ctx.cfg
    b, f, k = hd.shape
    grad_audio = grad_audio.contiguous().to(torch.float32)
    g0 = torch.empty_like(hd)
    g1 = torch.empty_like(hd)
    _lib.check(_lib.load().ddsp_b200_harmonic_backward(
        f0_hz.data_ptr(), grad_audio.data_ptr(), g0.data_ptr(), g1.data_ptr(),
        b, f, k, n_samples, sample_rate, core.AMP_METHODS[method], _stream()))
    # dL/d(amp * hd)[i] = g0[i] + g1[i-1], frame F being a copy of frame F-1
    dha = g0
    dha[:, 1:] += g1[:, :-1]
    dha[:, -1] += g1[:, -1]
    d_hd = dha * amplitudes
    d_amp = (dha * hd).sum(-1, keepdim=True)
    d_f0 = None
    if ctx.needs_input_grad[0]:
      d_f0 = _harmonic_d_f0(f0_hz, amplitudes, hd, grad_audio, n_samples, sample_rate,
                            method)
    return d_f0, d_amp, d_hd, None, None, None


def _harmonic_d_f0(f0_hz, amplitudes, hd, grad_audio, n_samples, sample_rate, method):
  """dL/d f0_hz [B, F, 1] through the phase (`ddsp_b200_harmonic_backward_f0`)."""
  b, f, k = hd.shape
  d_f0 = torch.empty((b, f, 1), dtype=torch.float32, device=hd.device)
  nbytes = 12 * b * f
  ws = torch.empty((max(nbytes, 1),), dtype=torch.uint8, device=hd.device)
  _lib.check(_lib.load().ddsp_b200_harmonic_backward_f0(
      f0_hz.data_ptr(), amplitudes.data_ptr(), hd.data_ptr(), grad_audio.data_ptr(),
      d_f0.data_ptr(), b, f, k, n_samples, sample_rate, core.AMP_METHODS[method],
      ws.data_ptr(), nbytes, _stream()))
  return d_f0


class DecoderFn(torch.autograd.Function):
  """The `ae.gin` decoder (ae.gin:47-72) from raw network outputs, forward and
  backward entirely in the CUDA library.  Gradients: amps, harmonic_distribution,
  noise_magnitudes always; f0_hz when it requires grad."""

  @staticmethod
  def forward(ctx, amps, harmonic_distribution, f0_hz, noise_magnitudes, n_samples,
              sample_rate, amp_resample_method, normalize_below_nyquist, window_size,
              initial_bias, noise, seed, offset):
    amps = core.torch_float32(amps)
    hd = core.torch_float32(harmonic_distribution)
    f0_hz = core.torch_float32(f0_hz)
    mags = core.torch_float32(noise_magnitudes)
    noise = None if noise is None else core.torch_float32(noise)
    ctx.save_for_backward(amps, hd, f0_hz, mags)
    ctx.noise = noise
    ctx.cfg = (int(n_samples), float(sample_rate), amp_resample_method,
               bool(normalize_below_nyquist), int(window_size), float(initial_bias),
               int(seed), int(offset))
    return core.decoder_forward(
        amps, hd, f0_hz, mags, n_samples, sample_rate=sample_rate,
        amp_resample_method=amp_resample_method,
        normalize_below_nyquist=normalize_below_nyquist, window_size=window_size,
        initial_bias=initial_bias, noise=noise, seed=seed, offset=offset)

  @staticmethod
  def backward(ctx, grad_audio):
    amps, hd, f0_hz, mags = ctx.saved_tensors
    n_samples, sample_rate, method, nyq, window_size, bias, seed, offset = ctx.cfg
    b, f, k = hd.shape
    nb = mags.shape[-1]
    lib = _lib.load()
    st = _stream()
    g = grad_audio.contiguous().to(torch.float32)
    flags = _lib.CTL_SCALE | (_lib.CTL_NYQUIST if nyq else 0)
    # harmonic: sample-rate reductions, then get_controls transposed at frame rate
    g0 = torch.empty_like(hd)
    g1 = torch.empty_like(hd)
    _lib.check(lib.ddsp_b200_harmonic_backward(
        f0_hz.data_ptr(), g.data_ptr(), g0.data_ptr(), g1.data_ptr(), b, f, k,
        n_samples, sample_rate, core.AMP_METHODS[method], st))
    d_amps = torch.empty_like(amps)
    d_hd = torch.empty_like(hd)
    _lib.check(lib.ddsp_b200_harmonic_controls_backward(
        amps.data_ptr(), hd.data_ptr(), f0_hz.data_ptr(), g0.data_ptr(), g1.data_ptr(),
        d_amps.data_ptr(), d_hd.data_ptr(), b, f, k, sample_rate, flags, st))
    # noise: the filter is linear in the magnitudes
    dmags = torch.empty_like(mags)
    _lib.check(lib.ddsp_b200_filtered_noise_backward(
        g.data_ptr(), 0 if ctx.noise is None else ctx.noise.data_ptr(),
        seed & (2**64 - 1), offset & (2**64 - 1), dmags.data_ptr(), b, f, nb,
        n_samples, window_size, st))
    d_mags = torch.empty_like(mags)
    _lib.check(lib.ddsp_b200_noise_controls_backward(
        mags.data_ptr(), dmags.data_ptr(), d_mags.data_ptr(), mags.numel(), bias, st))
    d_f0 = None
    if ctx.needs_input_grad[2]:
      # the phase path needs the synthesizer controls: one controls launch
      a_ctl, h_ctl = core.harmonic_controls(amps, hd, f0_hz, sample_rate, scale=True,
                                            normalize_below_nyquist=nyq)
      d_f0 = _harmonic_d_f0(f0_hz, a_ctl, h_ctl, g, n_samples, sample_rate, method)
    return (d_amps, d_hd, d_f0, d_mags) + (None,) * 9


class FftConvolveLtiFn(torch.autograd.Function):
  """core.fft_convolve with one long impulse response per item (effects.Reverb,
  effects.py:103-117), differentiable in both operands:
    y[n]      = sum_s h[s] x[n + start - s]
    dL/dx[m]  = (g * reverse(h)) [m + S - 1 - start]
    dL/dh[s]  = (g * reverse(x)) [s + N - 1 - start]     (summed over the batch when
                                                          the IR is shared)
  - three calls of the same partitioned overlap-save kernels."""

  @staticmethod
  def forward(ctx, audio, ir, start, out_len):
    audio = core.torch_float32(audio)
    ir = core.torch_float32(ir)
    ctx.save_for_backward(audio, ir)
    ctx.cfg = (int(start), int(out_len))
    return core.fft_convolve_lti(audio, ir, start, out_len)

  @staticmethod
  def backward(ctx, g):
    audio, ir = ctx.saved_tensors
    start, out_len = ctx.cfg
    b, n = audio.shape
    ir_batch, s = ir.shape
    g = g.contiguous().to(torch.float32)
    d_audio = d_ir = None
    if ctx.needs_input_grad[0]:
      off = s - 1 - start
      if off >= 0:
        d_audio = core.fft_convolve_lti(g, ir, off, n, reverse_ir=True)
      else:      # crop starts beyond the IR length: shift through a padded gradient
        gp = torch.nn.functional.pad(g, (-off, 0))
        d_audio = core.fft_convolve_lti(gp, ir, 0, n, reverse_ir=True)
    if ctx.needs_input_grad[1]:
      off = n - 1 - start
      if off >= 0:
        d_ir = core.fft_convolve_lti(g, audio, off, s, reverse_ir=True)
      else:
        gp = torch.nn.functional.pad(g, (-off, 0))
        d_ir = core.fft_convolve_lti(gp, audio, 0, s, reverse_ir=True)
      if ir_batch == 1 and b > 1:
        d_ir = d_ir.sum(0, keepdim=True)
    return d_audio, d_ir, None, None


class FilteredNoiseFn(torch.autograd.Function):
  """FilteredNoise.get_signal (synths.py:181-196), differentiable in magnitudes."""

  @staticmethod
  def forward(ctx, magnitudes, n_samples, window_size, noise, seed, offset):
    magnitudes = core.torch_float32(magnitudes)
    ctx.cfg = (int(n_samples), int(window_size), int(seed), int(offset),
               tuple(magnitudes.shape))
    ctx.noise = None if noise is None else core.torch_float32(noise)
    return core.filtered_noise(magnitudes, n_samples, window_size=window_size,
                               noise=ctx.noise, seed=seed, offset=offset)

  @staticmethod
  def backward(ctx, grad_audio):
    n_samples, window_size, seed, offset, (b, f, nb) = ctx.cfg
    grad_audio = grad_audio.contiguous().to(torch.float32)
    dmags = torch.empty((b, f, nb), dtype=torch.float32, device=grad_audio.device)
    _lib.check(_lib.load().ddsp_b200_filtered_noise_backward(
        grad_audio.data_ptr(), 0 if ctx.noise is None else ctx.noise.data_ptr(),
        seed & (2**64 - 1), offset & (2**64 - 1), dmags.data_ptr(), b, f, nb,
        n_samples, window_size, _stream()))
    return dmags, None, None, None, None, None


def exp_sigmoid(x, exponent=10.0, max_value=2.0, threshold=1e-7):
  """core.exp_sigmoid (core.py:386-404) as differentiable torch ops."""
  return max_value * torch.sigmoid(x)**math.log(exponent) + threshold


def harmonic_controls(amps, harmonic_distribution, f0_hz, sample_rate=16000,
                      normalize_below_nyquist=True):
  """Harmonic.get_controls (synths.py:94-121) as differentiable torch ops."""
  amps = exp_sigmoid(amps)
  hd = exp_sigmoid(harmonic_distribution)
  if normalize_below_nyquist:
    k = hd.shape[-1]
    ratios = torch.linspace(1.0, float(k), k, device=hd.device, dtype=hd.dtype)
    hd = torch.where(f0_hz * ratios >= sample_rate / 2.0, torch.zeros_like(hd), hd)
  denom = hd.sum(-1, keepdim=True)
  denom = torch.where(denom == 0.0, torch.full_like(denom, 1e-7), denom)
  return amps, hd / denom


def decoder_train(amps, harmonic_distribution, f0_hz, noise_magnitudes,
                  n_samples=64000, sample_rate=16000, window_size=0,
                  initial_bias=-5.0, noise=None, seed=0, offset=0,
                  amp_resample_method='window', normalize_below_nyquist=True):
  """The `ae.gin` decoder (ae.gin:47-72) with gradients to amps,
  harmonic_distribution, noise_magnitudes (and f0_hz if it requires grad) - one
  autograd node: fused forward pipeline, CUDA backward kernels for the two
  synthesizers and both `get_controls`."""
  return DecoderFn.apply(amps, harmonic_distribution, f0_hz, noise_magnitudes,
                         n_samples, sample_rate, amp_resample_method,
                         normalize_below_nyquist, window_size, initial_bias, noise,
                         seed, offset)


def decoder_train_unfused(amps, harmonic_distribution, f0_hz, noise_magnitudes,
                          n_samples=64000, sample_rate=16000, window_size=0,
                          initial_bias=-5.0, noise=None, seed=0, offset=0):
  """The same decoder with `get_controls` as differentiable torch ops around the two
  synthesizer Functions (the round-1 route; kept as a cross-check of DecoderFn)."""
  dev = core._device()
  amps = core.torch_float32(amps, dev) if not isinstance(amps, torch.Tensor) else amps
  a, h = harmonic_controls(amps, harmonic_distribution, f0_hz, sample_rate)
  harm = HarmonicSynthesisFn.apply(f0_hz, a, h, n_samples, sample_rate, 'window')
  mags = exp_sigmoid(noise_magnitudes + initial_bias)
  nz = FilteredNoiseFn.apply(mags, n_samples, window_size, noise, seed, offset)
  return harm + nz


class WavetableSynthesisFn(torch.autograd.Function):
  """core.wavetable_synthesis (core.py:1229-1282), differentiable in the
  amplitudes and the wavetables.  scale=True: amplitudes and wavetables are RAW
  network outputs and Wavetable.get_controls' exp_sigmoid (synths.py:212-236) is
  part of the node, forward and backward.  Backward is
  `ddsp_b200_wavetable_backward` (gather form, bit-reproducible).  f0 gets no
  gradient: an f0 that requires grad is refused."""

  @staticmethod
  def forward(ctx, f0_hz, amplitudes, wavetables, n_samples, sample_rate, scale):
    n_samples = int(n_samples)
    b, ff, fa, _, _ = core._wavetable_shapes(f0_hz, amplitudes, wavetables, n_samples)  # pylint: disable=protected-access
    if ff != fa:
      raise NotImplementedError(
          f'WavetableSynthesisFn needs f0 and amplitudes on the same frames '
          f'(got {ff} and {fa}).')
    f0 = core.torch_float32(f0_hz)
    amps = core.torch_float32(amplitudes)
    tables = core.torch_float32(wavetables)
    tables3 = tables if tables.dim() == 3 else tables[:, None, :]
    ctx.save_for_backward(f0, amps, tables3)
    ctx.cfg = (n_samples, float(sample_rate), bool(scale), tuple(tables.shape))
    out = torch.empty((b, n_samples), dtype=torch.float32, device=f0.device)
    return core._wavetable_launch(f0, amps, tables3, n_samples, sample_rate,  # pylint: disable=protected-access
                                  scale, out, False)

  @staticmethod
  def backward(ctx, grad_audio):
    f0, amps, tables = ctx.saved_tensors
    n_samples, sample_rate, scale, tshape = ctx.cfg
    b, f = f0.shape[0], f0.shape[1]
    r, w = tables.shape[1], tables.shape[2]
    grad_audio = grad_audio.contiguous().to(torch.float32)
    d_amps = torch.empty_like(amps)
    d_tables = torch.empty_like(tables)
    lib = _lib.load()
    with core._on_device_of(f0, amps, tables, grad_audio):  # pylint: disable=protected-access
      nbytes = lib.ddsp_b200_wavetable_workspace(b, f, r, w, n_samples, 1)
      ws = torch.empty((max(nbytes, 1),), dtype=torch.uint8, device=f0.device)
      _lib.check(lib.ddsp_b200_wavetable_backward(
          f0.data_ptr(), amps.data_ptr(), tables.data_ptr(), grad_audio.data_ptr(),
          d_amps.data_ptr(), d_tables.data_ptr(), b, f, r, w, n_samples, sample_rate,
          int(scale), ws.data_ptr(), nbytes, _stream()))
    return None, d_amps, d_tables.reshape(tshape), None, None, None


def _refuse_f0_grad(f0_hz):
  if isinstance(f0_hz, torch.Tensor) and f0_hz.requires_grad and torch.is_grad_enabled():
    raise NotImplementedError(
        'ddsp_b200 wavetable synthesis has no gradient with respect to f0_hz (the '
        'reference models do not learn f0 through a wavetable); pass '
        'f0_hz.detach().')


def wavetable_synthesis(frequencies, amplitudes, wavetables, n_samples=64000,
                        sample_rate=16000):
  """core.wavetable_synthesis on CONTROLS with gradients to amplitudes and
  wavetables."""
  _refuse_f0_grad(frequencies)
  return WavetableSynthesisFn.apply(frequencies, amplitudes, wavetables, n_samples,
                                    sample_rate, False)


def wavetable_train(amps_raw, wavetables_raw, f0_hz, n_samples=64000,
                    sample_rate=16000):
  """synths.Wavetable() (exp_sigmoid scaling) from RAW network outputs with
  gradients to both: one forward launch, one backward pass."""
  _refuse_f0_grad(f0_hz)
  return WavetableSynthesisFn.apply(f0_hz, amps_raw, wavetables_raw, n_samples,
                                    sample_rate, True)


class ModDelayFn(torch.autograd.Function):
  """core.variable_length_delay (core.py:1285-1313) and effects.ModDelay's
  signal (effects.py:367-393), differentiable in the audio, the gain and the
  phase.  gain may be None (the bare delay).  scale=True: gain and phase are RAW
  network outputs and ModDelay.get_controls' exp_sigmoid / sigmoid are part of
  the node, forward and backward.  Backward is `ddsp_b200_mod_delay_backward`:
  d audio is the transpose of the two-tap gather, summed in 64-bit fixed point
  (bit-reproducible); d phase is g gain L (e_{j+1} - e_j) times the phase map's
  slope, and it jumps where the position crosses an integer."""

  @staticmethod
  def forward(ctx, audio, gain, phase, max_length, phase_scale, phase_offset, scale,
              add_dry):
    name = 'ModDelay' if gain is not None else 'variable_length_delay'
    max_length = core._check_max_length(name, max_length)  # pylint: disable=protected-access
    controls = {'phase': phase} if gain is None else {'gain': gain, 'phase': phase}
    b, n = core._delay_controls(name, audio, controls)  # pylint: disable=protected-access
    x = core.torch_float32(audio)
    g = None if gain is None else core.torch_float32(gain).reshape(b, n)
    ph = core.torch_float32(phase).reshape(b, n)
    ctx.save_for_backward(x, g, ph)
    ctx.cfg = (max_length, float(phase_scale), float(phase_offset), bool(scale),
               bool(add_dry), None if gain is None else tuple(gain.shape),
               tuple(phase.shape))
    return core._mod_delay_launch(x, g, ph, max_length, phase_scale, phase_offset,  # pylint: disable=protected-access
                                  scale, add_dry)

  @staticmethod
  def backward(ctx, grad_out):
    x, g, ph = ctx.saved_tensors
    max_length, phase_scale, phase_offset, scale, add_dry, gshape, pshape = ctx.cfg
    b, n = x.shape
    grad_out = grad_out.contiguous().to(torch.float32)
    d_audio = torch.empty_like(x)
    d_gain = None if g is None else torch.empty_like(g)
    d_phase = torch.empty_like(ph)
    lib = _lib.load()
    with core._on_device_of(x, g, ph, grad_out):  # pylint: disable=protected-access
      nbytes = lib.ddsp_b200_mod_delay_workspace(b, n, max_length)
      ws = torch.empty((max(nbytes, 1),), dtype=torch.uint8, device=x.device)
      _lib.check(lib.ddsp_b200_mod_delay_backward(
          x.data_ptr(), 0 if g is None else g.data_ptr(), ph.data_ptr(),
          grad_out.data_ptr(), d_audio.data_ptr(),
          0 if d_gain is None else d_gain.data_ptr(), d_phase.data_ptr(), b, n,
          max_length, phase_scale, phase_offset, int(scale), int(add_dry),
          ws.data_ptr(), nbytes, _stream()))
    if d_gain is not None:
      d_gain = d_gain.reshape(gshape)
    return (d_audio, d_gain, d_phase.reshape(pshape), None, None, None, None, None)


def variable_length_delay(phase, audio, max_length=512):
  """core.variable_length_delay on controls with gradients to the phase and the
  audio."""
  return ModDelayFn.apply(audio, None, phase, max_length, 1.0, 0.0, False, False)


def mod_delay_train(audio, gain_raw, phase_raw, center_ms=15.0, depth_ms=10.0,
                    sample_rate=16000, add_dry=True):
  """effects.ModDelay() (exp_sigmoid gain, sigmoid phase) from RAW network outputs
  with gradients to the audio and both controls: one forward launch, one backward
  pass.  The audio's gradient reaches the synthesizer upstream."""
  from ddsp_b200 import effects  # local import: effects imports core only
  md = effects.ModDelay(center_ms=center_ms, depth_ms=depth_ms, sample_rate=sample_rate,
                        add_dry=add_dry)
  max_length, depth_phase, center_phase = md.delay_map()
  return ModDelayFn.apply(audio, gain_raw, phase_raw, max_length, depth_phase,
                          center_phase, True, add_dry)
