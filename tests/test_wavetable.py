"""Wavetable synthesizer (synths.Wavetable, core.wavetable_synthesis,
core.linear_lookup, core.harmonic_distribution_to_wavetable).

CPU: the NumPy oracle (tests/wavetable_oracle.py) against the reference's own
outputs in tests/golden/wavetable.npz (narrow = float32, wide = float64), the
float64 torch restatement the backward is checked against, and the ValueErrors.
GPU: the kernels against the wide outputs and the oracle, the ports of the
reference's own tests (core_test.py:592-675, synths_test.py:53-70), the full-size
memory bound, determinism, and the backward."""
import os

import numpy as np
import pytest
import torch

from oracle import ddsp_oracle as o
from oracle import ref_on_shim
from tests import wavetable_oracle as wo
from tests.golden import make_wavetable_golden as mwg
from tests.util import rel_err

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), 'golden', 'wavetable.npz')
CASES = mwg.cases()


def gold():
  return np.load(GOLD)


def oracle_case(kind, arrays, kw, dtype):
  if kind == 'synth':
    return wo.wavetable(*arrays, n_samples=kw['n_samples'], dtype=dtype)
  if kind == 'synthesis':
    return wo.wavetable_synthesis(*arrays, dtype=dtype, **kw)
  if kind == 'lookup':
    return wo.linear_lookup(*arrays, dtype=dtype)
  return wo.harmonic_distribution_to_wavetable(*arrays, dtype=dtype, **kw)


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


# The reference's float32 table resample and its float32 cumsum are reproduced op
# for op; two cases keep a few ulp of difference at the output peak (the 2-D table
# is resampled along its n_wavetable axis in float32, hop 75 is not a power of two).
F32_TOL = {'synth_hop75': 2e-5, 'synthesis_2d': 2e-5}


@pytest.mark.parametrize('name', sorted(CASES))
def test_oracle_float32_matches_reference_narrow(name):
  kind, arrays, kw = CASES[name]
  got = oracle_case(kind, arrays, kw, np.float32)
  want = gold()[name + '_f32']
  assert np.abs(got.astype(np.float64) - want).max() <= F32_TOL.get(name, 1e-6)


def test_full_item_oracle_matches_reference_wide_summary():
  from tests.golden.make_golden import unpack_outputs
  g = gold()
  packed = unpack_outputs({k[len('full_'):]: g[k] for k in g.files
                           if k.startswith('full_') and k[len('full_'):] in (
                               'names', 'ndim', 'dims', 'start', 'values', 'absmax',
                               'l2')})
  shape, values, peak, l2 = packed['full_wide']
  got = wo.wavetable(*mwg.full_inputs(), n_samples=mwg.FULL['N'])
  assert got.shape == shape
  from tests.golden.make_golden import sample_index
  idx = sample_index(got.size)
  assert np.abs(got.ravel()[idx] - values).max() <= 1e-9 * peak
  assert abs(np.abs(got).max() - peak) <= 1e-9 * peak
  assert abs(np.sqrt((got**2).sum()) - l2) <= 1e-9 * l2


def test_reference_narrow_wide_distance_is_what_we_state():
  """DESIGN.md section 3.11: at 64000 samples the reference's own float32 output
  is 0.83 max/peak and 0.63 relative L2 away from its float64 value (a random
  table is very sensitive to the phase), so the gate is against wide."""
  g = gold()
  assert abs(float(g['full_narrow_wide_maxrel']) - 0.83) < 0.01
  assert abs(float(g['full_narrow_wide_l2rel']) - 0.63) < 0.01


@pytest.mark.skipif(not ref_on_shim.available(),
                    reason='reference sources are only in the authoring container')
def test_fixture_is_output_of_the_unmodified_reference():
  from tests.golden.make_golden import compare
  compare('wavetable', mwg.wavetable(), gold(), atol=0.0)


def torch_wavetable64(f0, amps, tables, n_samples, sample_rate=16000, scale=False):
  """float64 torch restatement of the same rules in gather form, differentiable in
  amps and tables (the backward's arbiter)."""
  f0 = np.asarray(f0, np.float64)
  if scale:
    amps = 2.0 * torch.sigmoid(amps)**float(np.log(10.0)) + 1e-7
    tables = 2.0 * torch.sigmoid(tables)**float(np.log(10.0)) + 1e-7
  if tables.dim() == 2:
    tables = tables[:, None, :]
  b, f, _ = amps.shape
  r_tab, w = tables.shape[1], tables.shape[2]
  hop = n_samples // f
  t = np.arange(n_samples)
  i, rr = t // hop, t % hop
  w1 = torch.from_numpy(0.5 - 0.5 * np.cos(np.pi * rr / hop))
  a_ext = torch.cat([amps[:, :, 0], amps[:, -1:, 0]], dim=1)
  amp_env = a_ext[:, i] * (1 - w1) + a_ext[:, i + 1] * w1
  f_env = o.resample(f0, n_samples)[:, :, 0]
  ph = np.cumsum(f_env / sample_rate, axis=1)
  ph = np.concatenate([np.zeros((b, 1)), ph[:, :-1]], axis=1) % 1.0
  x = ph * w
  j0 = np.floor(x).astype(np.int64)
  fr = torch.from_numpy(x - j0)
  j1 = j0 + 1
  if r_tab == 1:
    lo = hi = np.zeros(n_samples, np.int64)
    ft = np.zeros(n_samples)
  else:
    lo, hi, ft = o._bilinear_indices(r_tab, n_samples, False, False)  # pylint: disable=protected-access
  ft = torch.from_numpy(np.asarray(ft, np.float64))
  ext = torch.cat([tables, tables[..., :1]], dim=-1)
  bi = torch.arange(b)[:, None]

  def v(rows):
    rows = torch.from_numpy(np.broadcast_to(rows[None, :], (b, n_samples)).copy())
    return ((1 - fr) * ext[bi, rows, torch.from_numpy(j0)] +
            fr * ext[bi, rows, torch.from_numpy(j1)])

  return (v(lo) * (1 - ft) + v(hi) * ft) * amp_env


@pytest.mark.parametrize('name', ['synth', 'synth_one_table', 'synth_hop75'])
def test_torch_restatement_matches_reference_wide(name):
  _, (a, tab, f0), kw = CASES[name]
  got = torch_wavetable64(f0, torch.from_numpy(a).double(), torch.from_numpy(tab).double(),
                          kw['n_samples'], scale=True).numpy()
  want = gold()[name + '_wide']
  assert np.abs(got - want).max() <= 1e-9 * np.abs(want).max()


def test_value_errors_before_any_device_work():
  from ddsp_b200 import core
  f0 = np.full((1, 10, 1), 100.0, np.float32)
  a = np.ones((1, 10, 1), np.float32)
  t = np.zeros((1, 10, 16), np.float32)
  with pytest.raises(ValueError, match='divisible'):
    core.wavetable_synthesis(f0, a, t, n_samples=105)
  with pytest.raises(ValueError, match='downsampling'):
    core.wavetable_synthesis(f0, a, t, n_samples=11)
  with pytest.raises(ValueError):
    core.wavetable_synthesis(f0[:, :, 0], a, t, n_samples=100)
  with pytest.raises(ValueError):
    core.wavetable_synthesis(f0, a, np.zeros((2, 16), np.float32), n_samples=100)
  with pytest.raises(ValueError, match='harmonics'):
    core.harmonic_distribution_to_wavetable(np.zeros((1, 2, 9), np.float32), 16)
  with pytest.raises(ValueError):
    core.linear_lookup(np.zeros((1, 5), np.float32), np.zeros((1, 4, 8), np.float32))
  with pytest.raises(ValueError, match='harmonics'):
    wo.harmonic_distribution_to_wavetable(np.zeros((1, 2, 9)), 16)


# ---------------------------------------------------------------------------
# GPU
# ---------------------------------------------------------------------------
def cuda(x):
  return torch.as_tensor(np.asarray(x, np.float32)).cuda()


@pytest.mark.gpu
@pytest.mark.parametrize('name', sorted(CASES))
def test_kernel_matches_reference_wide(name):
  import ddsp_b200
  from ddsp_b200 import core
  kind, arrays, kw = CASES[name]
  if kind == 'synth':
    got = ddsp_b200.Wavetable(**kw)(*[cuda(x) for x in arrays])
  elif kind == 'synthesis':
    got = core.wavetable_synthesis(*[cuda(x) for x in arrays], **kw)
  elif kind == 'lookup':
    got = core.linear_lookup(*[cuda(x) for x in arrays])
  else:
    got = core.harmonic_distribution_to_wavetable(cuda(arrays[0]), **kw)
  want = gold()[name + '_wide']
  emax, el2 = rel_err(got.cpu().numpy(), want)
  assert emax <= 1e-4 and el2 <= 1e-4, (emax, el2)


@pytest.mark.gpu
@pytest.mark.parametrize('batch_size,n_wavetable,n_frames,n_samples,n_cycles', [
    (1, 2048, 0, 10000, 1000), (2, 1024, 0, 20000, 10), (1, 2048, 1, 10000, 1000),
    (1, 2048, 10000, 10000, 1000)])
def test_linear_lookup_is_accurate(batch_size, n_wavetable, n_frames, n_samples,
                                   n_cycles):
  """core_test.py:594-627."""
  from ddsp_b200 import core
  two_pi = 2.0 * np.pi
  wavetable = np.sin(np.linspace(0, two_pi, n_wavetable).astype(np.float32))
  wavetable = np.tile(wavetable[np.newaxis, :], [batch_size, 1])
  if n_frames > 0:
    wavetable = np.tile(wavetable[:, np.newaxis, :], [1, n_frames, 1])
  phase = np.linspace(0, n_cycles, n_samples).astype(np.float32) % 1.0
  phase = np.tile(phase[np.newaxis, :, np.newaxis], [batch_size, 1, 1])
  wav_np = np.sin(two_pi * phase)[:, :, 0]
  wav = core.linear_lookup(cuda(phase), cuda(wavetable)).cpu().numpy()
  assert np.abs(wav_np - wav).mean() <= 2e-3


@pytest.mark.gpu
@pytest.mark.parametrize('batch_size,frequency,amplitude,n_wavetable,wavetable_frames', [
    (1, 440.0, 0.5, 2048, 0), (2, 1000.0, 0.1, 1024, 1), (2, 1000.0, 0.1, 1024, 200)])
def test_wavetable_synth_is_accurate(batch_size, frequency, amplitude, n_wavetable,
                                     wavetable_frames):
  """core_test.py:629-675."""
  from ddsp_b200 import core
  sample_rate, seconds, n_frames = 16000, 0.1, 100
  n_samples = int(sample_rate * seconds)
  n_cycles = seconds * frequency
  two_pi = 2.0 * np.pi
  wavetable = np.sin(np.linspace(0, two_pi, n_wavetable).astype(np.float32))
  wavetable = np.tile(wavetable[np.newaxis, :], [batch_size, 1])
  if wavetable_frames > 0:
    wavetable = np.tile(wavetable[:, np.newaxis, :], [1, wavetable_frames, 1])
  wav_np = amplitude * np.sin(two_pi * np.linspace(0, n_cycles, n_samples))
  wav_np = np.tile(wav_np[np.newaxis, :], [batch_size, 1]).astype(np.float32)
  amplitudes = np.ones([batch_size, n_frames, 1]) * amplitude
  frequencies = np.ones([batch_size, n_frames, 1]) * frequency
  wav = core.wavetable_synthesis(cuda(frequencies), cuda(amplitudes), cuda(wavetable),
                                 n_samples, sample_rate).cpu().numpy()
  pad = n_samples // n_frames
  assert np.abs(wav_np[:, pad:-pad] - wav[:, pad:-pad]).mean() <= 3e-2


@pytest.mark.gpu
def test_wavetable_output_shape_is_correct():
  """synths_test.py:55-70."""
  import ddsp_b200
  synthesizer = ddsp_b200.Wavetable(n_samples=64000, sample_rate=16000, scale_fn=None)
  amp = torch.zeros((3, 1000, 1), device='cuda') + 1.0
  wavetables = torch.zeros((3, 1000, 1024), device='cuda')
  f0_hz = torch.zeros((3, 1000, 1), device='cuda') + 440
  assert tuple(synthesizer(amp, wavetables, f0_hz).shape) == (3, 64000)


@pytest.mark.gpu
@pytest.mark.parametrize('per_sample', [False, True])
def test_linear_lookup_matches_oracle_outside_the_ends(per_sample):
  from ddsp_b200 import core
  rng = np.random.default_rng(3)
  b, n, w = 3, 777, 37
  phase = rng.uniform(-0.3, 1.3, (b, n)).astype(np.float32)
  phase[:, :6] = [0.0, 1.0, -0.5 / w, 1.0 + 0.5 / w, -2.0, 3.0]
  tab = rng.standard_normal((b, n, w) if per_sample else (b, w)).astype(np.float32)
  got = core.linear_lookup(cuda(phase), cuda(tab)).cpu().numpy()
  want = wo.linear_lookup(phase, tab)
  assert np.abs(got - want).max() <= 1e-5 * np.abs(want).max()


def _full_inputs(b, seed=0):
  g = torch.Generator(device='cuda').manual_seed(seed)
  amps = torch.randn((b, 1000, 1), device='cuda', generator=g)
  tables = torch.randn((b, 1000, 2048), device='cuda', generator=g)
  f0 = 80.0 + 720.0 * torch.rand((b, 1, 1), device='cuda', generator=g)
  vib = 1.0 + 0.03 * torch.sin(torch.arange(1000, device='cuda') * 0.02)[None, :, None]
  return amps, tables, (f0 * vib).contiguous()


@pytest.mark.gpu
def test_full_size_b256_matches_oracle_deterministic_and_never_holds_bnw():
  import ddsp_b200
  from ddsp_b200 import _lib
  b, n = 256, 64000
  amps, tables, f0 = _full_inputs(b)
  synth = ddsp_b200.Wavetable(n_samples=n)
  torch.cuda.synchronize()
  base = torch.cuda.memory_allocated()
  torch.cuda.reset_peak_memory_stats()
  y1 = synth(amps, tables, f0)
  torch.cuda.synchronize()
  rise = torch.cuda.max_memory_allocated() - base
  ws = _lib.load().ddsp_b200_wavetable_workspace(b, 1000, 1000, 2048, n, 0)
  assert rise <= 4 * b * n + ws + (1 << 20), (rise, ws)
  y2 = synth(amps, tables, f0)
  assert torch.equal(y1, y2)
  for item in (0, 137, 255):
    want = wo.wavetable(amps[item:item + 1].cpu().numpy(),
                        tables[item:item + 1].cpu().numpy(),
                        f0[item:item + 1].cpu().numpy(), n_samples=n)
    emax, el2 = rel_err(y1[item:item + 1].cpu().numpy(), want)
    assert emax <= 1e-4 and el2 <= 1e-4, (item, emax, el2)


@pytest.mark.gpu
@pytest.mark.parametrize('name', ['synth', 'synth_hop75'])
def test_raw_call_is_bit_identical_to_get_signal_of_get_controls(name):
  import ddsp_b200
  _, arrays, kw = CASES[name]
  synth = ddsp_b200.Wavetable(**kw)
  args = [cuda(x) for x in arrays]
  fused = synth(*args)
  two_step = synth.get_signal(**synth.get_controls(*args))
  assert torch.equal(fused, two_step)
  assert torch.equal(fused, synth(*args, return_outputs_dict=True)['signal'])


@pytest.mark.gpu
def test_accumulate_adds_into_out():
  from ddsp_b200 import core
  _, (f0, a, t), kw = CASES['synthesis_fwt200']
  base = torch.randn((2, 1600), device='cuda')
  out = base.clone()
  core.wavetable_synthesis(cuda(f0), cuda(a), cuda(t), out=out, accumulate=True, **kw)
  want = base + core.wavetable_synthesis(cuda(f0), cuda(a), cuda(t), **kw)
  torch.testing.assert_close(out, want, rtol=0, atol=1e-6)


BWD_CASES = {
    'same_frames': (2, 50, 50, 256, 3200),
    'fwt_ne_f': (2, 40, 130, 64, 3200),
    'static_3d': (2, 40, 1, 128, 6400),
    'hop75_w130': (2, 40, 40, 130, 3000),
    'few_table_frames': (1, 16, 2, 64, 8192),
}


@pytest.mark.gpu
@pytest.mark.parametrize('scale', [True, False])
@pytest.mark.parametrize('case', sorted(BWD_CASES))
def test_backward_matches_float64_autograd_and_is_deterministic(case, scale):
  from ddsp_b200 import autograd
  b, f, r, w, n = BWD_CASES[case]
  rng = np.random.default_rng(sorted(BWD_CASES).index(case))
  a = rng.standard_normal((b, f, 1)).astype(np.float32)
  tab = rng.standard_normal((b, r, w)).astype(np.float32)
  if not scale:
    a, tab = np.abs(a) + 0.1, np.tanh(tab)
  f0 = mwg._f0(rng, b, f, n)  # pylint: disable=protected-access
  g = rng.standard_normal((b, n)).astype(np.float32)
  fn = autograd.wavetable_train if scale else (
      lambda a_, t_, f_, **kw: autograd.wavetable_synthesis(f_, a_, t_, **kw))

  def run():
    a_t = cuda(a).requires_grad_()
    t_t = cuda(tab).requires_grad_()
    y = fn(a_t, t_t, cuda(f0), n_samples=n)
    y.backward(cuda(g))
    return y.detach(), a_t.grad, t_t.grad

  y1, da1, dt1 = run()
  _, da2, dt2 = run()
  assert torch.equal(da1, da2) and torch.equal(dt1, dt2)
  a64 = torch.from_numpy(a).double().requires_grad_()
  t64 = torch.from_numpy(tab).double().requires_grad_()
  y64 = torch_wavetable64(f0, a64, t64, n, scale=scale)
  y64.backward(torch.from_numpy(g).double())
  assert rel_err(y1.cpu().numpy(), y64.detach().numpy())[0] <= 1e-4
  for got, want in ((da1, a64.grad), (dt1, t64.grad)):
    emax, _ = rel_err(got.cpu().numpy(), want.numpy())
    assert emax <= 2e-4, (case, scale, emax)


@pytest.mark.gpu
def test_f0_requiring_grad_is_refused():
  from ddsp_b200 import autograd
  _, (a, tab, f0), kw = CASES['synth']
  f0_t = cuda(f0).requires_grad_()
  with pytest.raises(NotImplementedError, match='f0'):
    autograd.wavetable_train(cuda(a).requires_grad_(), cuda(tab), f0_t, **kw)
