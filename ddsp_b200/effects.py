"""Effects processors that consume the decoder's audio: `Reverb`,
`FilteredNoiseReverb`, `FIRFilter` and `ModDelay` with the reference's
constructors and semantics (`ddsp/effects.py:28-117, 202-278, 283-393`; SURVEY
8f-3; the next node after `Add` in `solo_instrument.gin:26-40`).

`Reverb` is a long linear time-invariant convolution (48000-tap impulse
response): `core.fft_convolve` routes one impulse response of 2048 taps and more
per item to the hand-written partitioned overlap-save convolution
(csrc/longconv.cuh); `FilteredNoiseReverb` draws that impulse response from a
`FilteredNoise` synthesizer; `FIRFilter` is the time-varying filter of
`FilteredNoise` applied to given audio and runs on the IR + FIR kernels.
`ModDelay` (chorus, flanger, vibrato) reads two taps of the audio's own history
per sample in one kernel (csrc/mod_delay.cuh)."""
import torch

from ddsp_b200 import core
from ddsp_b200 import processors
from ddsp_b200 import synths


class Reverb(processors.Processor):
  """Convolutional (FIR) reverb (effects.py:28-117)."""

  def __init__(self, trainable=False, reverb_length=48000, add_dry=True,
               name='reverb'):
    super().__init__(name=name, trainable=trainable)
    self._reverb_length = reverb_length
    self._add_dry = add_dry
    self._ir = None

  def _mask_dry_ir(self, ir):
    """effects.py:50-59: zero the first tap (the dry path)."""
    if ir.dim() == 1:
      ir = ir[None, :]
    if ir.dim() == 3:
      ir = ir[:, :, 0]
    dry_mask = torch.zeros((ir.shape[0], 1), dtype=torch.float32, device=ir.device)
    return torch.cat([dry_mask, ir[:, 1:]], dim=1)

  def _match_dimensions(self, audio, ir):
    """effects.py:61-68."""
    if ir.dim() == 1:
      ir = ir[None, :]
    return ir.repeat(int(audio.shape[0]), 1)

  def build(self, device=None):
    """effects.py:70-79: the single learned impulse response, N(0, 1e-6)."""
    if self.trainable and self._ir is None:
      self._ir = (1e-6 * torch.randn(self._reverb_length, dtype=torch.float32,
                                     device=device)).requires_grad_(True)

  def get_controls(self, audio, ir=None):
    """effects.py:81-101."""
    if not self.trainable and ir is None:          # before any device work
      raise ValueError('Must provide "ir" tensor if Reverb trainable=False.')
    audio = core.torch_float32(audio)
    if self.trainable:
      self.build(audio.device)
      ir = self._match_dimensions(audio, self._ir)
    return {'audio': audio, 'ir': ir}

  def get_signal(self, audio, ir):
    """effects.py:103-117."""
    audio, ir = core.torch_float32(audio), core.torch_float32(ir)
    ir = self._mask_dry_ir(ir)
    wet = core.fft_convolve(audio, ir, padding='same', delay_compensation=0)
    return (wet + audio) if self._add_dry else wet


class FilteredNoiseReverb(Reverb):
  """Impulse response = the output of a filtered-noise synthesizer
  (effects.py:202-278): `get_controls` runs `FilteredNoise(n_samples =
  reverb_length)` on the magnitudes (given per item, or ONE learned
  [n_frames, n_filter_banks] set tiled over the batch when trainable), `get_signal`
  is `Reverb`'s."""

  def __init__(self, trainable=False, reverb_length=48000, window_size=257,
               n_frames=1000, n_filter_banks=16, scale_fn=core.exp_sigmoid,
               initial_bias=-3.0, add_dry=True, name='filtered_noise_reverb'):
    super().__init__(name=name, add_dry=add_dry, trainable=trainable)
    self._n_frames = n_frames
    self._n_filter_banks = n_filter_banks
    self._synth = synths.FilteredNoise(n_samples=reverb_length,
                                       window_size=window_size,
                                       scale_fn=scale_fn,
                                       initial_bias=initial_bias)
    self._magnitudes = None

  def build(self, device=None):
    """effects.py:240-249: the learned magnitudes, N(0, 1e-2)."""
    if self.trainable and self._magnitudes is None:
      self._magnitudes = (1e-2 * torch.randn(
          self._n_frames, self._n_filter_banks, dtype=torch.float32,
          device=device)).requires_grad_(True)

  def _synth_ir(self, magnitudes):
    """`self._synth(magnitudes)` (effects.py:272); with gradients to the magnitudes
    when they ask for them (the synthesizer's autograd node, exp_sigmoid as
    differentiable torch ops on the [n_frames, n_filter_banks] controls)."""
    if (isinstance(magnitudes, torch.Tensor) and magnitudes.requires_grad and
        torch.is_grad_enabled()):
      from ddsp_b200 import autograd as _ag
      syn = self._synth
      if syn.scale_fn is core.exp_sigmoid:
        mags = _ag.exp_sigmoid(magnitudes + syn.initial_bias)
      elif syn.scale_fn is not None:
        mags = syn.scale_fn(magnitudes + syn.initial_bias)
      else:
        mags = magnitudes
      return _ag.FilteredNoiseFn.apply(mags, syn.n_samples, syn.window_size,
                                       syn.injected_noise, syn.seed,
                                       syn.next_offset())
    return self._synth(magnitudes)

  def get_controls(self, audio, magnitudes=None):
    """effects.py:251-277."""
    if not self.trainable and magnitudes is None:  # before any device work
      raise ValueError('Must provide "magnitudes" tensor if '
                       'FilteredNoiseReverb trainable=False.')
    audio = core.torch_float32(audio)
    if self.trainable:
      self.build(audio.device)
      magnitudes = self._magnitudes[None, :]
    ir = self._synth_ir(magnitudes)
    if self.trainable:
      ir = self._match_dimensions(audio, ir)
    return {'audio': audio, 'ir': ir}


class FIRFilter(processors.Processor):
  """Linear time-varying FIR filter (effects.py:283-325)."""

  def __init__(self, window_size=257, scale_fn=core.exp_sigmoid, name='fir_filter'):
    super().__init__(name=name)
    self.window_size = window_size
    self.scale_fn = scale_fn

  def get_controls(self, audio, magnitudes):
    if self.scale_fn is not None:
      magnitudes = self.scale_fn(core.torch_float32(magnitudes))
    return {'audio': audio, 'magnitudes': magnitudes}

  def get_signal(self, audio, magnitudes):
    return core.frequency_filter(audio, magnitudes, window_size=self.window_size)


class ModDelay(processors.Processor):
  """Modulated delay times used in chorus, flanger, and vibrato effects
  (effects.py:328-393).

  gain and phase are audio-rate controls, [batch, n_samples, 1] or
  [batch, n_samples].  get_signal is one kernel (`ddsp_b200_mod_delay_forward`):
  the reference's [batch, n_samples, max_length] frames never exist.  Called for
  the signal only with the default scale functions (core.exp_sigmoid for the gain,
  core.sigmoid for the phase), the processor runs get_controls inside that kernel
  (one launch from raw network outputs, bit-identical to the two steps).  Training
  goes through autograd.mod_delay_train."""

  def __init__(self,
               center_ms=15.0,
               depth_ms=10.0,
               sample_rate=16000,
               gain_scale_fn=core.exp_sigmoid,
               phase_scale_fn=core.sigmoid,
               add_dry=True,
               name='mod_delay'):
    super().__init__(name=name)
    self.center_ms = center_ms
    self.depth_ms = depth_ms
    self.sample_rate = sample_rate
    self.gain_scale_fn = gain_scale_fn
    self.phase_scale_fn = phase_scale_fn
    self.add_dry = add_dry

  def delay_map(self):
    """effects.py:381-386 in Python floats: (max_length, depth_phase,
    center_phase); max_length truncates, as the reference's int() does."""
    max_delay_ms = self.center_ms + self.depth_ms
    max_length_samples = int(self.sample_rate / 1000.0 * max_delay_ms)
    depth_phase = self.depth_ms / max_delay_ms
    center_phase = self.center_ms / max_delay_ms
    return max_length_samples, depth_phase, center_phase

  def call(self, audio, gain, phase, return_outputs_dict=False, **kwargs):
    for k in ['training', 'mask']:
      kwargs.pop(k, None)
    if (not return_outputs_dict and not kwargs and
        self.gain_scale_fn is core.exp_sigmoid and self.phase_scale_fn is core.sigmoid):
      max_length, depth_phase, center_phase = self.delay_map()
      return core.mod_delay(audio, gain, phase, max_length, depth_phase, center_phase,
                            add_dry=self.add_dry, scale=True)
    return super().call(audio, gain, phase, return_outputs_dict=return_outputs_dict,
                        **kwargs)

  def get_controls(self, audio, gain, phase):
    """effects.py:346-365."""
    if self.gain_scale_fn is not None:
      gain = self.gain_scale_fn(core.torch_float32(gain))
    if self.phase_scale_fn is not None:
      phase = self.phase_scale_fn(core.torch_float32(phase))
    return {'audio': audio, 'gain': gain, 'phase': phase}

  def get_signal(self, audio, gain, phase):
    """effects.py:367-393."""
    max_length, depth_phase, center_phase = self.delay_map()
    return core.mod_delay(audio, gain, phase, max_length, depth_phase, center_phase,
                          add_dry=self.add_dry, scale=False)
