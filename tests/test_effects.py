"""Reverb / FIRFilter (SURVEY 8f-3) and the long-impulse-response path of
core.fft_convolve (framed FFT convolution on torch.fft / cuFFT).

CPU: the FFT formulation against the oracle's literal restatement of
core.py:1382-1473, for single-frame (reverb) and multi-frame IRs.  GPU: the
processors against the float64 oracle through both routes of fft_convolve."""
import os

import numpy as np
import pytest
import torch

from oracle import ddsp_oracle as o
from ddsp_b200 import core


def _fft_path(audio, ir, padding, delay):
  b, n = audio.shape
  ir3 = ir if ir.ndim == 3 else ir[:, None, :]
  f, s = ir3.shape[1], ir3.shape[2]
  frame = int(np.ceil(n / f))
  fft_size = core.get_fft_size(frame, s, power_of_2=True)
  total = (f - 1) * frame + fft_size
  start, out_len, crop = core._crop_range(total, n, s, padding, delay)
  assert out_len == crop
  return core._fft_convolve_cufft(torch.from_numpy(audio), torch.from_numpy(ir3), f,
                                  frame, fft_size, int(start), int(crop)).numpy()


@pytest.mark.parametrize('n,frames,taps,padding,delay', [
    (4000, 1, 3000, 'same', 0), (4000, 1, 3000, 'same', -1), (1000, 1, 100, 'valid', -1),
    (1280, 20, 129, 'same', -1), (1280, 5, 300, 'valid', -1), (999, 1, 4096, 'same', 0)])
def test_fft_formulation_matches_oracle(n, frames, taps, padding, delay):
  rng = np.random.default_rng(n + taps)
  audio = rng.standard_normal((2, n)).astype(np.float32)
  ir = (rng.standard_normal((2, frames, taps)) / np.sqrt(taps)).astype(np.float32)
  want = o.fft_convolve(audio, ir, padding=padding, delay_compensation=delay)
  got = _fft_path(audio, ir, padding, delay)
  assert got.shape == want.shape
  assert np.abs(got - want).max() < 1e-4 * max(1.0, np.abs(want).max())


def test_reverb_value_errors_and_masking():
  """effects.py:81-101 (ValueError without an IR) and 50-59 (dry tap masked)."""
  from ddsp_b200 import effects
  rev = effects.Reverb(trainable=False)
  ir = torch.arange(1.0, 6.0)[None, :].repeat(2, 1)
  masked = rev._mask_dry_ir(ir)
  assert masked.tolist() == [[0.0, 2.0, 3.0, 4.0, 5.0]] * 2
  assert rev._mask_dry_ir(ir[..., None]).shape == (2, 5)
  assert rev._match_dimensions(torch.zeros(3, 10), torch.ones(4)).shape == (3, 4)


def test_filtered_noise_reverb_constructor_and_errors():
  """effects.py:205-238, 266-270."""
  from ddsp_b200 import effects
  rev = effects.FilteredNoiseReverb()
  assert (rev.name, rev.trainable, rev._add_dry, rev._n_frames, rev._n_filter_banks) == (
      'filtered_noise_reverb', False, True, 1000, 16)
  syn = rev._synth
  assert (syn.n_samples, syn.window_size, syn.initial_bias) == (48000, 257, -3.0)
  assert syn.scale_fn is core.exp_sigmoid
  with pytest.raises(ValueError, match='Must provide "magnitudes" tensor'):
    rev.get_controls(np.zeros((2, 100), np.float32))
  with pytest.raises(ValueError, match='Must provide "ir" tensor'):
    effects.Reverb().get_controls(np.zeros((2, 100), np.float32))


@pytest.mark.parametrize('trainable', [False, True])
def test_filtered_noise_reverb_composition_matches_reference(monkeypatch, trainable):
  """The host logic of FilteredNoiseReverb (effects.py:202-278 on top of Reverb's
  28-117) against the UNMODIFIED reference class, with the same noise and, when
  trainable, the same learned magnitudes (tests/golden/filtered_noise_reverb.npz,
  made by make_golden.py on the NumPy shim).  The CUDA kernels are replaced by the
  oracle here (they have their own parity tests): what is under test is the
  composition - scale + bias, synthesis of the impulse response, tiling of the
  single learned response, dry-tap masking, 'same' convolution with zero delay
  compensation, dry mix."""
  from ddsp_b200 import effects
  from tests.golden import make_golden as mg
  audio, mags, noise, reverb_kw = mg.filtered_noise_reverb_case(trainable)
  B, N = audio.shape
  want = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), 'golden',
                              'filtered_noise_reverb.npz'))['audio_trainable_%d' % trainable]

  # ---- ours, kernels swapped for the oracle ----
  def t32(x, device=None):
    return torch.as_tensor(np.asarray(x.detach() if isinstance(x, torch.Tensor) else x,
                                      dtype=np.float32))
  monkeypatch.setattr(core, 'torch_float32', t32)
  monkeypatch.setattr(core, 'noise_controls', lambda m, bias, scale=True: torch.from_numpy(
      o.noise_get_controls(t32(m).numpy(), initial_bias=bias, scale=scale,
                           dtype=np.float32)['magnitudes']))
  monkeypatch.setattr(core, 'filtered_noise', lambda m, n, window_size=257, noise=None, **kw:
                      torch.from_numpy(o.noise_get_signal(t32(m).numpy(), t32(noise).numpy(),
                                                          window_size=window_size,
                                                          dtype=np.float32)))
  monkeypatch.setattr(core, 'fft_convolve', lambda a, ir, padding='same',
                      delay_compensation=-1, **kw: torch.from_numpy(
                          o.fft_convolve(t32(a).numpy(), t32(ir).numpy(), padding=padding,
                                         delay_compensation=delay_compensation,
                                         dtype=np.float32)))
  rev = effects.FilteredNoiseReverb(**reverb_kw)
  rev._synth.injected_noise = torch.from_numpy(noise)
  with torch.no_grad():
    if trainable:
      rev._magnitudes = torch.from_numpy(mags[0]).requires_grad_(True)
      got = rev(audio).numpy()
    else:
      got = rev(audio, mags).numpy()
  assert got.shape == want.shape == (B, N)
  assert np.abs(got - want).max() < 2e-5 * max(1.0, np.abs(want).max())


@pytest.mark.gpu
@pytest.mark.parametrize('taps,add_dry', [(3000, True), (48000, False), (200, True)])
def test_reverb_matches_oracle(taps, add_dry):
  import ddsp_b200
  from tests.util import rel_err
  rng = np.random.default_rng(taps)
  B, N = 2, 16000
  audio = rng.standard_normal((B, N)).astype(np.float32)
  ir = (rng.standard_normal((B, taps)) * np.exp(-np.arange(taps) / (taps / 6.0)) /
        np.sqrt(taps)).astype(np.float32)
  rev = ddsp_b200.Reverb(add_dry=add_dry)
  with pytest.raises(ValueError):
    rev.get_controls(audio)
  got = rev(audio, ir).cpu().numpy()
  masked = ir.copy()
  masked[:, 0] = 0.0
  want = o.fft_convolve(audio, masked, padding='same', delay_compensation=0)
  if add_dry:
    want = want + audio
  assert got.shape == (B, N)
  emax, el2 = rel_err(got, want)
  assert emax < 1e-4 and el2 < 1e-4, (emax, el2)


@pytest.mark.gpu
def test_trainable_reverb_and_fir_filter():
  import ddsp_b200
  from tests.util import rel_err
  rng = np.random.default_rng(3)
  B, N, F, nb = 2, 6400, 100, 65
  audio = rng.standard_normal((B, N)).astype(np.float32)
  rev = ddsp_b200.Reverb(trainable=True, reverb_length=4000)
  out = rev(audio)
  assert tuple(out.shape) == (B, N) and rev._ir.requires_grad
  out.square().mean().backward()
  assert rev._ir.grad is not None and float(rev._ir.grad.abs().sum()) > 0
  mags = rng.standard_normal((B, F, nb)).astype(np.float32)
  filt = ddsp_b200.FIRFilter(window_size=257)
  got = filt(audio, mags).cpu().numpy()
  scaled = o.exp_sigmoid(mags.astype(np.float64))
  want = o.frequency_filter(audio, scaled, window_size=257)
  emax, el2 = rel_err(got, want)
  assert emax < 1e-4 and el2 < 1e-4, (emax, el2)


@pytest.mark.gpu
@pytest.mark.parametrize('B,n,taps,ir_batch,padding,delay', [
    (2, 64000, 48000, 2, 'same', 0),        # effects.Reverb at the ae.gin length
    (3, 64000, 48000, 1, 'same', 0),        # one trainable IR shared by the batch
    (2, 16000, 2048, 2, 'same', -1),        # smallest IR on this route, auto delay
    (2, 5000, 9000, 2, 'valid', 0),         # IR longer than the audio, full tail
    (1, 1023, 2049, 1, 'same', 0),          # ragged against the 1024-sample blocks
    (2, 4097, 4096, 2, 'same', 5)])
def test_long_impulse_response_convolution_kernel(B, n, taps, ir_batch, padding, delay):
  """`ddsp_b200_fft_convolve_lti` (partitioned overlap-save, hand-written FFTs)
  behind core.fft_convolve for 2-D / single-frame impulse responses >= 2048 taps,
  against the oracle's restatement of core.py:1382-1473."""
  from tests.util import rel_err
  rng = np.random.default_rng(n + taps)
  audio = rng.standard_normal((B, n)).astype(np.float32)
  ir = (rng.standard_normal((ir_batch, taps)) * np.exp(-np.arange(taps) / (taps / 5.0))
        ).astype(np.float32)
  want = o.fft_convolve(audio, np.broadcast_to(ir, (B, taps)) if ir_batch == 1 else ir,
                        padding=padding, delay_compensation=delay)
  got = core.fft_convolve(audio, ir, padding=padding, delay_compensation=delay)
  assert tuple(got.shape) == want.shape
  emax, el2 = rel_err(got.cpu().numpy(), want)
  assert emax < 1e-4 and el2 < 1e-4, (emax, el2)
  # accumulate into an existing buffer (the wet + dry sum of Reverb)
  base = torch.full(tuple(got.shape), 0.25, device='cuda')
  acc = core.fft_convolve(audio, ir, padding=padding, delay_compensation=delay,
                          out=base.clone(), accumulate=True)
  assert float((acc - (got + 0.25)).abs().max()) < 1e-5


@pytest.mark.gpu
@pytest.mark.parametrize('shared', [True, False])
def test_long_convolution_backward_matches_autograd(shared):
  """FftConvolveLtiFn (the trainable Reverb): d audio and d impulse response from
  the same kernels on reversed operands, against float64 autograd of torch.fft."""
  from ddsp_b200 import autograd as ag
  torch.manual_seed(3)
  B, n, taps, start = 3, 6000, 5000, 0
  audio = torch.randn(B, n, device='cuda')
  ir = torch.randn(1 if shared else B, taps, device='cuda') * 0.02
  g = torch.randn(B, n, device='cuda')
  a1, h1 = audio.clone().requires_grad_(True), ir.clone().requires_grad_(True)
  y = core.fft_convolve(a1, h1, padding='same', delay_compensation=start)
  (y * g).sum().backward()
  a2, h2 = audio.double().requires_grad_(True), ir.double().requires_grad_(True)
  m = n + taps - 1
  yr = torch.fft.irfft(torch.fft.rfft(a2, m) * torch.fft.rfft(h2.expand(B, taps), m), m)
  yr = yr[:, start:start + n]
  (yr * g.double()).sum().backward()
  assert float((y.double() - yr).abs().max() / yr.abs().max()) < 1e-4
  for got, want in ((a1.grad, a2.grad), (h1.grad, h2.grad)):
    err = float((got.double() - want).abs().max() / want.abs().max())
    assert err < 2e-4, err
