"""Harmonic and FilteredNoise synthesizers with the reference's constructor
arguments, method names and dict keys (`ddsp/synths.py:55-196`)."""
import itertools

from ddsp_b200 import core
from ddsp_b200 import processors


class Harmonic(processors.Processor):
  """Synthesize audio with a bank of harmonic sinusoidal oscillators
  (synths.py:55-146)."""

  def __init__(self,
               n_samples=64000,
               sample_rate=16000,
               scale_fn=core.exp_sigmoid,
               normalize_below_nyquist=True,
               amp_resample_method='window',
               use_angular_cumsum=False,
               name='harmonic'):
    super().__init__(name=name)
    self.n_samples = n_samples
    self.sample_rate = sample_rate
    self.scale_fn = scale_fn
    self.normalize_below_nyquist = normalize_below_nyquist
    self.amp_resample_method = amp_resample_method
    self.use_angular_cumsum = use_angular_cumsum

  def get_controls(self, amplitudes, harmonic_distribution, f0_hz):
    """synths.py:94-121.  exp_sigmoid scaling, Nyquist masking and row
    normalisation run as one kernel; any other scale_fn is applied by calling
    it (as the reference does) before the mask/normalise kernel."""
    f0_hz = core.torch_float32(f0_hz)
    fused_scale = self.scale_fn is core.exp_sigmoid
    if self.scale_fn is not None and not fused_scale:
      amplitudes = self.scale_fn(core.torch_float32(amplitudes))
      harmonic_distribution = self.scale_fn(
          core.torch_float32(harmonic_distribution))
    amplitudes, harmonic_distribution = core.harmonic_controls(
        amplitudes, harmonic_distribution, f0_hz, self.sample_rate,
        scale=fused_scale, normalize_below_nyquist=self.normalize_below_nyquist)
    return {'amplitudes': amplitudes,
            'harmonic_distribution': harmonic_distribution,
            'f0_hz': f0_hz}

  def get_signal(self, amplitudes, harmonic_distribution, f0_hz, out=None,
                 accumulate=False):
    """synths.py:123-146."""
    return core.harmonic_synthesis(
        frequencies=f0_hz,
        amplitudes=amplitudes,
        harmonic_distribution=harmonic_distribution,
        n_samples=self.n_samples,
        sample_rate=self.sample_rate,
        amp_resample_method=self.amp_resample_method,
        use_angular_cumsum=self.use_angular_cumsum,
        out=out, accumulate=accumulate)


class FilteredNoise(processors.Processor):
  """Synthesize audio by filtering white noise (synths.py:149-196).

  The reference draws fresh `tf.random.uniform` noise per call
  (synths.py:192-193).  Here the noise is Philox4x32-10 generated inside the
  filter kernel, keyed by `seed` with a per-call counter so successive calls
  differ; pass `noise=` to get_signal to inject a specific noise tensor
  (parity tests do).
  """

  def __init__(self,
               n_samples=64000,
               window_size=257,
               scale_fn=core.exp_sigmoid,
               initial_bias=-5.0,
               name='filtered_noise',
               seed=0):
    super().__init__(name=name)
    self.n_samples = n_samples
    self.window_size = window_size
    self.scale_fn = scale_fn
    self.initial_bias = initial_bias
    self.seed = seed
    self._calls = itertools.count()
    # Test hook: a [B, n_samples] tensor used instead of the Philox stream.
    self.injected_noise = None

  def next_offset(self):
    """Per-call Philox counter offset, so successive calls draw fresh noise."""
    return next(self._calls)

  def get_controls(self, magnitudes):
    """synths.py:165-179."""
    if self.scale_fn is core.exp_sigmoid:
      magnitudes = core.noise_controls(magnitudes, self.initial_bias, scale=True)
    elif self.scale_fn is not None:
      magnitudes = self.scale_fn(
          core.torch_float32(magnitudes) + self.initial_bias)
    else:
      magnitudes = core.torch_float32(magnitudes)
    return {'magnitudes': magnitudes}

  def get_signal(self, magnitudes, noise=None, out=None, accumulate=False,
                 offset=None):
    """synths.py:181-196."""
    if noise is None:
      noise = self.injected_noise
    return core.filtered_noise(
        magnitudes, self.n_samples, window_size=self.window_size, noise=noise,
        seed=self.seed, offset=self.next_offset() if offset is None else offset,
        out=out, accumulate=accumulate)


class Wavetable(processors.Processor):
  """Synthesize audio from a series of wavetables (synths.py:199-257).

  get_signal passes the frame-rate tables straight to one fused kernel
  (`ddsp_b200_wavetable_forward`); the reference's audio-rate tables
  [batch, n_samples, n_wavetable] never exist.  Called for the signal only with
  the default exp_sigmoid scaling, the processor runs get_controls inside that
  kernel (one launch from raw network outputs)."""

  def __init__(self,
               n_samples=64000,
               sample_rate=16000,
               scale_fn=core.exp_sigmoid,
               name='wavetable'):
    super().__init__(name=name)
    self.n_samples = n_samples
    self.sample_rate = sample_rate
    self.scale_fn = scale_fn

  def call(self, amplitudes, wavetables, f0_hz, return_outputs_dict=False, **kwargs):
    for k in ['training', 'mask']:
      kwargs.pop(k, None)
    sa, sw, sf = core._shape(amplitudes), core._shape(wavetables), core._shape(f0_hz)  # pylint: disable=protected-access
    if (not return_outputs_dict and not kwargs and self.scale_fn is core.exp_sigmoid
        and len(sw) == 3 and len(sa) == 3 and len(sf) == 3 and sa[:2] == sf[:2]):
      return core.wavetable_raw(amplitudes, wavetables, f0_hz,
                                n_samples=self.n_samples, sample_rate=self.sample_rate)
    return super().call(amplitudes, wavetables, f0_hz,
                        return_outputs_dict=return_outputs_dict, **kwargs)

  def get_controls(self, amplitudes, wavetables, f0_hz):
    """synths.py:212-236: scale_fn on the amplitudes and the wavetables."""
    if self.scale_fn is not None:
      amplitudes = self.scale_fn(core.torch_float32(amplitudes))
      wavetables = self.scale_fn(core.torch_float32(wavetables))
    return {'amplitudes': amplitudes,
            'wavetables': wavetables,
            'f0_hz': f0_hz}

  def get_signal(self, amplitudes, wavetables, f0_hz, out=None, accumulate=False):
    """synths.py:238-257.  The reference resamples 3-D tables to n_samples before
    wavetable_synthesis (which then resamples n_samples to n_samples, the
    identity): the kernel interpolates the frame-rate tables itself.  A 2-D table
    [batch, n_wavetable] is resampled along its only axis into a static table of
    n_samples entries, as in the reference."""
    if len(core._shape(wavetables)) == 2:  # pylint: disable=protected-access
      wavetables = core.resample(wavetables, self.n_samples)
    return core.wavetable_synthesis(f0_hz, amplitudes, wavetables,
                                    n_samples=self.n_samples,
                                    sample_rate=self.sample_rate, out=out,
                                    accumulate=accumulate)


class Sinusoidal(processors.Processor):
  """Bank of arbitrary sinusoidal oscillators (synths.py:260-323).

  get_controls is frame-rate torch arithmetic; get_signal is one fused frame-rate
  oscillator bank with per-sinusoid exact phases
  (`ddsp_b200_sinusoidal_forward`) - the [batch, n_samples, n_sinusoids]
  envelopes of the reference are never materialised."""

  def __init__(self,
               n_samples=64000,
               sample_rate=16000,
               amp_scale_fn=core.exp_sigmoid,
               amp_resample_method='window',
               freq_scale_fn=core.frequencies_sigmoid,
               name='sinusoidal'):
    super().__init__(name=name)
    self.n_samples = n_samples
    self.sample_rate = sample_rate
    self.amp_scale_fn = amp_scale_fn
    self.amp_resample_method = amp_resample_method
    self.freq_scale_fn = freq_scale_fn

  def get_controls(self, amplitudes, frequencies):
    """synths.py:277-303."""
    amplitudes = core.torch_float32(amplitudes)
    frequencies = core.torch_float32(frequencies)
    if self.amp_scale_fn is not None:
      amplitudes = self.amp_scale_fn(amplitudes)
    if self.freq_scale_fn is not None:
      frequencies = self.freq_scale_fn(frequencies)
      amplitudes = core.remove_above_nyquist(frequencies, amplitudes,
                                             self.sample_rate)
    return {'amplitudes': amplitudes, 'frequencies': frequencies}

  def get_signal(self, amplitudes, frequencies):
    """synths.py:305-323.  One fused frame-rate kernel when the hop is an integer
    and the amplitudes are resampled by 'window' / 'linear'; otherwise the
    reference's own decomposition on the stand-alone kernels."""
    sa = core._shape(amplitudes)  # pylint: disable=protected-access
    if (self.amp_resample_method in core.AMP_METHODS and len(sa) == 3 and
        sa[1] > 0 and self.n_samples % sa[1] == 0 and
        (self.amp_resample_method != 'window' or sa[1] < self.n_samples)):
      return core.sinusoidal_synthesis(
          frequencies, amplitudes, n_samples=self.n_samples,
          sample_rate=self.sample_rate,
          amp_resample_method=self.amp_resample_method)
    amplitude_envelopes = core.resample(amplitudes, self.n_samples,
                                        method=self.amp_resample_method)
    frequency_envelopes = core.resample(frequencies, self.n_samples)
    return core.oscillator_bank(frequency_envelopes=frequency_envelopes,
                                amplitude_envelopes=amplitude_envelopes,
                                sample_rate=self.sample_rate)
