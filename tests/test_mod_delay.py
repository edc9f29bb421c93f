"""Modulated delay (effects.ModDelay, core.variable_length_delay).

CPU: the NumPy oracle (tests/mod_delay_oracle.py) against the reference's own
outputs in tests/golden/mod_delay.npz (narrow = float32, wide = float64), the
stated narrow-wide distance, and the ValueErrors.
GPU: the kernels against the wide outputs, the ports of the reference's own
tests (core_test.py:681-716, effects_test.py:107-117), the one-launch raw path,
determinism, the backward against float64 torch autograd, ProcessorGroup, CUDA
graph capture and the full-size memory bound."""
import os

import numpy as np
import pytest
import torch

from oracle import ref_on_shim
from tests import mod_delay_oracle as mo
from tests.golden import make_mod_delay_golden as mg
from tests.util import rel_err

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), 'golden', 'mod_delay.npz')
CASES = mg.cases()


def gold():
  return np.load(GOLD)


def oracle_case(kind, arrays, kw, dtype):
  if kind == 'delay':
    return mo.variable_length_delay(*arrays, dtype=dtype, **kw)
  kw = dict(kw)
  scale = 'gain_scale_fn' not in kw
  kw.pop('gain_scale_fn', None)
  kw.pop('phase_scale_fn', None)
  # without scale functions the reference maps the caller's float32 phase in float32
  return mo.mod_delay(*arrays, scale=scale, dtype=dtype,
                      map_dtype=None if scale else np.float32, **kw)


def unpack_full():
  from tests.golden.make_golden import unpack_outputs
  g = gold()
  return unpack_outputs({k[len('full_'):]: g[k] for k in g.files
                         if k.startswith('full_') and k[len('full_'):] in (
                             'names', 'ndim', 'dims', 'start', 'values', 'absmax', 'l2')})


# ---------------------------------------------------------------------------
# CPU
# ---------------------------------------------------------------------------
@pytest.mark.parametrize('name', sorted(CASES))
def test_oracle_float64_matches_reference_wide(name):
  kind, arrays, kw = CASES[name]
  got = oracle_case(kind, arrays, kw, np.float64)
  want = gold()[name + '_wide']
  assert got.shape == want.shape
  assert np.abs(got - want).max() <= 1e-9 * max(1.0, np.abs(want).max())


@pytest.mark.parametrize('name', sorted(CASES))
def test_oracle_float32_matches_reference_narrow(name):
  kind, arrays, kw = CASES[name]
  got = oracle_case(kind, arrays, kw, np.float32).astype(np.float64)
  want = gold()[name + '_f32'].astype(np.float64)
  ulp = np.spacing(np.float32(np.abs(want).max()))
  assert np.abs(got - want).max() <= 4 * ulp


def test_full_item_oracle_matches_reference_wide_summary():
  from tests.golden.make_golden import sample_index
  shape, values, peak, l2 = unpack_full()['full_wide']
  got = mo.mod_delay(*mg.full_inputs())
  assert got.shape == shape
  idx = sample_index(got.size)
  assert np.abs(got.ravel()[idx] - values).max() <= 1e-9 * peak
  assert abs(np.abs(got).max() - peak) <= 1e-9 * peak
  assert abs(np.sqrt((got**2).sum()) - l2) <= 1e-9 * l2


def test_reference_narrow_wide_distance_is_what_we_state():
  """DESIGN.md section 3.12: on a full default ModDelay() item the reference's own
  float32 output is 2.0e-5 max/peak and 6.0e-6 relative L2 away from its float64
  value (its float32 |phase - k/L| L), so the gate is against wide."""
  g = gold()
  assert abs(float(g['full_narrow_wide_maxrel']) - 2.0e-5) < 0.1e-5
  assert abs(float(g['full_narrow_wide_l2rel']) - 6.0e-6) < 0.1e-6


@pytest.mark.skipif(not ref_on_shim.available(),
                    reason='reference sources are only in the authoring container')
def test_fixture_is_output_of_the_unmodified_reference():
  from tests.golden.make_golden import compare
  compare('mod_delay', mg.mod_delay(), gold(), atol=0.0)


def test_value_errors_before_any_device_work():
  import ddsp_b200
  from ddsp_b200 import autograd, core
  a = np.zeros((2, 50), np.float32)
  c = np.zeros((2, 50, 1), np.float32)
  for bad in (0, -3, 2.5):
    with pytest.raises(ValueError, match='max_length'):
      core.variable_length_delay(c, a, max_length=bad)
  with pytest.raises(ValueError, match='phase'):
    core.variable_length_delay(np.zeros((2, 49, 1), np.float32), a, 8)
  with pytest.raises(ValueError, match='phase'):
    core.variable_length_delay(np.zeros((2, 50, 2), np.float32), a, 8)
  with pytest.raises(ValueError, match='audio'):
    core.variable_length_delay(c, c, 8)
  with pytest.raises(ValueError, match='gain'):
    ddsp_b200.ModDelay()(a, np.zeros((1, 50, 1), np.float32), c)
  with pytest.raises(ValueError, match='phase'):
    ddsp_b200.ModDelay(gain_scale_fn=None, phase_scale_fn=None)(a, c, c[:, :10])
  with pytest.raises(ValueError, match='max_length'):
    ddsp_b200.ModDelay(center_ms=0.01, depth_ms=0.01)(a, c, c)
  with pytest.raises(ValueError, match='max_length'):
    autograd.variable_length_delay(c, a, max_length=0)


def test_constructor_matches_reference_defaults():
  import ddsp_b200
  from ddsp_b200 import core
  md = ddsp_b200.ModDelay()
  assert (md.center_ms, md.depth_ms, md.sample_rate, md.add_dry, md.name) == (
      15.0, 10.0, 16000, True, 'mod_delay')
  assert md.gain_scale_fn is core.exp_sigmoid and md.phase_scale_fn is core.sigmoid
  assert md.delay_map() == (400, 0.4, 0.6)
  assert ddsp_b200.ModDelay(center_ms=10.0, depth_ms=5.0,
                            sample_rate=44100).delay_map()[0] == 661


# ---------------------------------------------------------------------------
# GPU
# ---------------------------------------------------------------------------
def cuda(x):
  return torch.as_tensor(np.asarray(x, np.float32)).cuda()


def run_kernel_case(kind, arrays, kw):
  import ddsp_b200
  from ddsp_b200 import core
  if kind == 'delay':
    return core.variable_length_delay(*[cuda(x) for x in arrays], **kw)
  return ddsp_b200.ModDelay(**kw)(*[cuda(x) for x in arrays])


@pytest.mark.gpu
@pytest.mark.parametrize('name', sorted(CASES))
def test_kernel_matches_reference_wide(name):
  kind, arrays, kw = CASES[name]
  got = run_kernel_case(kind, arrays, kw)
  want = gold()[name + '_wide']
  assert tuple(got.shape) == want.shape
  emax, el2 = rel_err(got.cpu().numpy(), want)
  assert emax <= 1e-4 and el2 <= 1e-4, (emax, el2)


@pytest.mark.gpu
def test_full_item_matches_reference_wide():
  import ddsp_b200
  from tests.golden.make_golden import sample_index
  shape, values, peak, l2 = unpack_full()['full_wide']
  got = ddsp_b200.ModDelay()(*[cuda(x) for x in mg.full_inputs()]).cpu().numpy()
  assert got.shape == shape
  got = got.astype(np.float64)
  assert np.abs(got.ravel()[sample_index(got.size)] - values).max() <= 1e-4 * peak
  assert abs(np.sqrt((got**2).sum()) - l2) <= 1e-4 * l2


@pytest.mark.gpu
@pytest.mark.parametrize('batch_size,n_samples,max_length', [(1, 16000, 10),
                                                              (2, 4000, 1000)])
def test_variable_length_delay_is_accurate(batch_size, n_samples, max_length):
  """core_test.py:681-716: a sine of period max_length; half delay negates, full
  delay (phase 1, entry max_length = entry 0) is the identity."""
  from ddsp_b200 import core
  n_cycles = float(n_samples) / max_length
  wav_np = np.sin(np.linspace(0, 2.0 * np.pi * n_cycles, n_samples))
  wav_np = np.tile(wav_np[np.newaxis, :], [batch_size, 1]).astype(np.float32)
  ones = np.ones_like(wav_np)[..., np.newaxis]
  for value, target in ((0.0, wav_np), (0.5, -wav_np), (1.0, wav_np)):
    got = core.variable_length_delay(cuda(value * ones), cuda(wav_np),
                                     max_length).cpu().numpy()
    difference = np.abs(target[:, max_length:] - got[:, max_length:]).mean()
    assert difference <= 1e-2, (value, difference)


@pytest.mark.gpu
def test_output_shape_is_correct():
  """effects_test.py:107-117."""
  import ddsp_b200
  processor = ddsp_b200.ModDelay()
  audio = torch.zeros((3, 16000), device='cuda')
  gain = torch.zeros((3, 16000, 1), device='cuda')
  phase = torch.zeros((3, 16000, 1), device='cuda')
  assert tuple(processor(audio, gain, phase).shape) == (3, 16000)


@pytest.mark.gpu
def test_tutorial_call_runs():
  """1_synths_and_effects: ModDelay(center, depth, None, None) on [1, N] audio."""
  import ddsp_b200
  n = 16000
  audio = mg.audio_like(np.random.default_rng(0), 1, n)
  for t in mg.TUTORIAL.values():
    md = ddsp_b200.ModDelay(center_ms=t['center_ms'], depth_ms=t['depth_ms'],
                            gain_scale_fn=None, phase_scale_fn=None)
    phase = mg.tutorial_phase(t['mod_rate'], n)
    gain = 1.0 * np.ones_like(audio)[..., np.newaxis]
    out = 0.5 * md(audio, gain, phase)
    want = 0.5 * mo.mod_delay(audio, gain, phase, t['center_ms'], t['depth_ms'],
                              scale=False)
    emax, _ = rel_err(out.cpu().numpy(), want)
    assert emax <= 1e-4


@pytest.mark.gpu
@pytest.mark.parametrize('name', ['moddelay_default', 'moddelay_2d_controls',
                                  'moddelay_no_dry', 'moddelay_44k1'])
def test_raw_call_is_bit_identical_to_get_signal_of_get_controls(name):
  import ddsp_b200
  _, arrays, kw = CASES[name]
  md = ddsp_b200.ModDelay(**kw)
  args = [cuda(x) for x in arrays]
  fused = md(*args)
  two_step = md.get_signal(**md.get_controls(*args))
  assert torch.equal(fused, two_step)
  assert torch.equal(fused, md(*args, return_outputs_dict=True)['signal'])


@pytest.mark.gpu
def test_user_scale_function_takes_the_generic_route():
  import ddsp_b200
  _, arrays, _ = CASES['moddelay_default']
  args = [cuda(x) for x in arrays]
  got = ddsp_b200.ModDelay(phase_scale_fn=torch.sigmoid)(*args)
  want = mo.mod_delay(*arrays)
  emax, el2 = rel_err(got.cpu().numpy(), want)
  assert emax <= 1e-4 and el2 <= 1e-4


@pytest.mark.gpu
def test_refuses_inputs_that_require_grad():
  import ddsp_b200
  from ddsp_b200 import core
  _, (a, g, p), _ = CASES['moddelay_no_dry']
  with pytest.raises(RuntimeError, match='autograd'):
    ddsp_b200.ModDelay()(cuda(a).requires_grad_(), cuda(g), cuda(p))
  with pytest.raises(RuntimeError, match='autograd'):
    core.variable_length_delay(cuda(p).requires_grad_(), cuda(a), 16)


# ---- backward ----------------------------------------------------------------
def exp_sigmoid64(x):
  return 2.0 * torch.sigmoid(x)**float(np.log(10.0)) + 1e-7


def torch_delay64(audio, gain, phase, L, a, c, add_dry):
  """float64 torch restatement on controls, differentiable in all three: the
  backward's arbiter.  gain may be None."""
  b, n = audio.shape
  p = (phase * a + c) * L
  fl = torch.floor(p).detach()
  fr = p - fl
  idx = torch.arange(n)[None, :]
  out = torch.zeros((b, n), dtype=torch.float64)
  for j, w in ((fl, 1.0 - fr), (fl + 1.0, fr)):
    ok = (j >= 0) & (j <= L)
    k = torch.where(ok, j, torch.zeros_like(j)).long()
    k = torch.where(k == L, torch.zeros_like(k), k)
    m = idx - k
    v = torch.gather(audio, 1, m.clamp(min=0))
    v = torch.where(m >= 0, v, torch.zeros_like(v))
    out = out + torch.where(ok, w * v, torch.zeros_like(v))
  if gain is not None:
    out = out * gain
  return out + audio if add_dry else out


def away_from_integers(phase, a, c, L, scale):
  """Nudge phases whose delay position lies within 1e-3 samples of an integer
  (d phase jumps there).  With scale, the position is that of the kernel's own
  sigmoid (core.sigmoid)."""
  from ddsp_b200 import core
  phase = phase.copy()
  for _ in range(20):
    ctl = core.sigmoid(cuda(phase)).cpu().numpy() if scale else phase
    p = (ctl.astype(np.float64) * a + c) * L
    bad = np.abs(p - np.round(p)) < 1e-3
    if not bad.any():
      return phase
    phase[bad] += np.float32(0.01 if scale else 3e-3 / (a * L))
  raise AssertionError('could not move the positions off the integers')


BWD_CASES = {
    # name: (B, N, L, with_gain, add_dry, center_ms, depth_ms)
    'delay_L400': (2, 6000, 400, False, False, 0.0, 1.0),
    'moddelay_L400': (2, 6000, 400, True, True, 15.0, 10.0),
    'moddelay_L400_wet': (2, 5000, 400, True, False, 15.0, 10.0),
    'delay_L16000': (2, 40000, 16000, False, False, 0.0, 1.0),
    'moddelay_L16000': (2, 40000, 16000, True, True, 600.0, 400.0),
    'delay_L7': (2, 3000, 7, False, True, 0.0, 1.0),
}


@pytest.mark.gpu
@pytest.mark.parametrize('scale', [True, False])
@pytest.mark.parametrize('case', sorted(BWD_CASES))
def test_backward_matches_float64_autograd_and_is_deterministic(case, scale):
  from ddsp_b200 import autograd, core
  b, n, L, with_gain, add_dry, center, depth = BWD_CASES[case]
  if scale and not with_gain:
    pytest.skip('the bare delay takes controls')
  rng = np.random.default_rng(sorted(BWD_CASES).index(case))
  audio = mg.audio_like(rng, b, n)
  if with_gain:
    L_, a, c = mo.delay_map(center, depth)
    assert L_ == L
  else:
    a, c = 1.0, 0.0
  if scale:
    gain = rng.standard_normal((b, n, 1)).astype(np.float32)
    phase = (2.0 * rng.standard_normal((b, n, 1))).astype(np.float32)
  else:
    gain = rng.uniform(0.2, 1.5, (b, n, 1)).astype(np.float32)
    phase = rng.uniform(-0.1, 1.1, (b, n, 1)).astype(np.float32)
  phase = away_from_integers(phase, a, c, L, scale)
  g = rng.standard_normal((b, n)).astype(np.float32)

  def run():
    x = cuda(audio).requires_grad_()
    ph = cuda(phase).requires_grad_()
    gn = cuda(gain).requires_grad_() if with_gain else None
    if not with_gain and not add_dry:
      y = autograd.variable_length_delay(ph, x, max_length=L)
    elif scale:
      y = autograd.mod_delay_train(x, gn, ph, center_ms=center, depth_ms=depth,
                                   add_dry=add_dry)
    else:
      y = autograd.ModDelayFn.apply(x, gn, ph, L, a, c, False, add_dry)
    y.backward(cuda(g))
    return y.detach(), x.grad, ph.grad, None if gn is None else gn.grad

  y1, dx1, dp1, dg1 = run()
  y2, dx2, dp2, dg2 = run()
  assert torch.equal(y1, y2) and torch.equal(dx1, dx2) and torch.equal(dp1, dp2)
  if with_gain:
    assert torch.equal(dg1, dg2)

  x64 = torch.from_numpy(audio).double().requires_grad_()
  p64 = torch.from_numpy(phase[:, :, 0]).double().requires_grad_()
  g64 = torch.from_numpy(gain[:, :, 0]).double().requires_grad_() if with_gain else None
  ph_ctl, gn_ctl = p64, g64
  if scale:
    # the kernel's own control values, with float64 derivatives of the scalings
    s_f = core.sigmoid(cuda(phase[:, :, 0])).cpu().double()
    e_f = core.exp_sigmoid(cuda(gain[:, :, 0])).cpu().double()
    ph_ctl = s_f + (torch.sigmoid(p64) - torch.sigmoid(p64).detach())
    gn_ctl = e_f + (exp_sigmoid64(g64) - exp_sigmoid64(g64).detach())
  y64 = torch_delay64(x64, gn_ctl, ph_ctl, L, a, c, add_dry)
  y64.backward(torch.from_numpy(g).double())
  assert rel_err(y1.cpu().numpy(), y64.detach().numpy())[0] <= 1e-5
  pairs = [('audio', dx1, x64.grad), ('phase', dp1[:, :, 0], p64.grad)]
  if with_gain:
    pairs.append(('gain', dg1[:, :, 0], g64.grad))
  for label, got, want in pairs:
    emax, el2 = rel_err(got.cpu().numpy(), want.numpy())
    assert emax <= 1e-4 and el2 <= 1e-4, (case, scale, label, emax, el2)


@pytest.mark.gpu
def test_nan_gradient_reaches_d_audio():
  from ddsp_b200 import autograd
  x = torch.randn((1, 5000), device='cuda', requires_grad=True)
  ph = torch.rand((1, 5000), device='cuda', requires_grad=True)
  y = autograd.variable_length_delay(ph, x, max_length=100)
  g = torch.zeros_like(y)
  g[0, 4000] = float('nan')
  y.backward(g)
  assert torch.isnan(x.grad).all()


# ---- composition, capture, full size -------------------------------------------
@pytest.mark.gpu
def test_processor_group_with_mod_delay_after_add():
  import ddsp_b200
  from tests.util import synth_inputs
  b, f, k, nb, n = 2, 125, 60, 65, 8000
  inp = synth_inputs(b, f, k, nb, n, seed=5)
  rng = np.random.default_rng(9)
  noise = ddsp_b200.FilteredNoise(n_samples=n, window_size=0)
  noise.injected_noise = cuda(inp['noise'])
  group = ddsp_b200.ProcessorGroup(dag=[
      (ddsp_b200.Harmonic(n_samples=n), ['amps', 'harmonic_distribution', 'f0_hz']),
      (noise, ['noise_magnitudes']),
      (ddsp_b200.Add(), ['filtered_noise/signal', 'harmonic/signal']),
      (ddsp_b200.ModDelay(), ['add/signal', 'gain', 'phase'])])
  feats = {key: cuda(inp[key]) for key in ['amps', 'harmonic_distribution', 'f0_hz',
                                           'noise_magnitudes']}
  feats['gain'] = cuda(rng.standard_normal((b, n, 1)))
  feats['phase'] = cuda(rng.standard_normal((b, n, 1)))
  audio = group(feats)
  outs = group(feats, return_outputs_dict=True)['controls']
  want = ddsp_b200.ModDelay()(outs['add']['signal'], feats['gain'], feats['phase'])
  assert torch.equal(audio, want)
  assert torch.equal(outs['mod_delay']['signal'], want)


@pytest.mark.gpu
def test_cuda_graph_replay_equals_eager():
  import ddsp_b200
  from ddsp_b200 import autograd
  _, arrays, _ = CASES['moddelay_default']
  audio, gain, phase = [cuda(x) for x in arrays]
  md = ddsp_b200.ModDelay()
  eager = md(audio, gain, phase)
  g = torch.randn_like(eager)

  def bwd():
    return autograd.ModDelayFn.backward(_Ctx(audio, gain, phase), g)

  eager_bwd = bwd()
  s = torch.cuda.Stream()
  s.wait_stream(torch.cuda.current_stream())
  with torch.cuda.stream(s):
    md(audio, gain, phase)                      # warm-up outside the capture
    bwd()
  torch.cuda.current_stream().wait_stream(s)
  graph = torch.cuda.CUDAGraph()
  with torch.cuda.graph(graph):
    static_out = md(audio, gain, phase)
    static_bwd = bwd()
  audio.mul_(0.5)
  graph.replay()
  torch.cuda.synchronize()
  assert torch.equal(static_out, md(audio, gain, phase))
  audio.mul_(2.0)
  graph.replay()
  torch.cuda.synchronize()
  assert torch.equal(static_out, eager)
  for got, want in zip(static_bwd[:3], eager_bwd[:3]):
    assert torch.equal(got, want)


class _Ctx:
  """The saved state ModDelayFn.backward reads, for ModDelay() on raw outputs."""

  def __init__(self, audio, gain, phase):
    b, n = audio.shape
    self.saved_tensors = (audio, gain.reshape(b, n), phase.reshape(b, n))
    self.cfg = (400, 0.4, 0.6, True, True, tuple(gain.shape), tuple(phase.shape))


@pytest.mark.gpu
def test_full_size_b256_memory_matches_oracle_and_is_deterministic():
  import ddsp_b200
  from ddsp_b200 import _lib, autograd
  b, n = 256, 64000
  gen = torch.Generator(device='cuda').manual_seed(0)
  audio = torch.randn((b, n), device='cuda', generator=gen)
  gain = torch.randn((b, n, 1), device='cuda', generator=gen)
  phase = 2.0 * torch.randn((b, n, 1), device='cuda', generator=gen)
  md = ddsp_b200.ModDelay()
  torch.cuda.synchronize()
  base = torch.cuda.memory_allocated()
  torch.cuda.reset_peak_memory_stats()
  y1 = md(audio, gain, phase)
  torch.cuda.synchronize()
  rise = torch.cuda.max_memory_allocated() - base
  assert rise <= 4 * b * n + (1 << 20), rise
  assert torch.equal(y1, md(audio, gain, phase))
  for item in (0, 131, 255):
    want = mo.mod_delay(audio[item:item + 1].cpu().numpy(),
                        gain[item:item + 1].cpu().numpy(),
                        phase[item:item + 1].cpu().numpy())
    emax, el2 = rel_err(y1[item:item + 1].cpu().numpy(), want)
    assert emax <= 1e-4 and el2 <= 1e-4, (item, emax, el2)
  del y1
  x = audio.requires_grad_()
  gn = gain.requires_grad_()
  ph = phase.requires_grad_()
  y = autograd.mod_delay_train(x, gn, ph)
  gout = torch.randn((b, n), device='cuda', generator=gen)
  torch.cuda.synchronize()
  base = torch.cuda.memory_allocated()
  torch.cuda.reset_peak_memory_stats()
  y.backward(gout)
  torch.cuda.synchronize()
  rise = torch.cuda.max_memory_allocated() - base
  ws = _lib.load().ddsp_b200_mod_delay_workspace(b, n, 400)
  assert rise <= 3 * 4 * b * n + ws + (1 << 20), (rise, ws)
