"""Host-side contract tests that need no GPU: the C ABI surface, argument
validation (which happens before any launch), and the Processor /
ProcessorGroup / DAG semantics of the reference (processors_test.py, dags.py).
"""
import ctypes
import os
import re

import numpy as np
import pytest

import ddsp_b200
from ddsp_b200 import _lib, core, dags, processors, synths

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


# ---- C ABI ------------------------------------------------------------------
def _header_symbols():
  text = open(os.path.join(ROOT, 'include', 'ddsp_b200.h')).read()
  return sorted(set(re.findall(r'\b(ddsp_b200_[a-z0-9_]+)\s*\(', text)))


def test_library_exports_every_declared_symbol():
  lib = ctypes.CDLL(_lib.LIB_PATH)
  names = _header_symbols()
  assert len(names) >= 13
  for name in names:
    assert hasattr(lib, name), name
    assert name in _lib.SIGNATURES, f'{name} is not bound in _lib.SIGNATURES'
  assert set(_lib.SIGNATURES) == set(names)
  assert _lib.load().ddsp_b200_version() == 200


def test_abi_validates_before_launching():
  """Shape errors come back as E_INVALID with a message - no CUDA call made."""
  lib = _lib.load()
  fake = ctypes.c_void_p(0x1000)   # never dereferenced on the host
  # N not divisible by F
  rc = lib.ddsp_b200_harmonic_forward(fake, fake, fake, fake, 1, 7, 4, 100,
                                      16000.0, 0, 0, 0, None)
  assert rc == _lib.E_INVALID
  assert b'divisible' in lib.ddsp_b200_last_error()
  with pytest.raises(ValueError):
    _lib.check(rc)
  # NULL harmonic_distribution with K > 1
  rc = lib.ddsp_b200_harmonic_forward(fake, fake, None, fake, 1, 10, 4, 100,
                                      16000.0, 0, 0, 0, None)
  assert rc == _lib.E_INVALID
  # bad enum values
  assert lib.ddsp_b200_harmonic_forward(fake, fake, fake, fake, 1, 10, 4, 100,
                                        16000.0, 7, 0, 0, None) == _lib.E_INVALID
  assert lib.ddsp_b200_harmonic_forward(fake, fake, fake, fake, 1, 10, 4, 100,
                                        16000.0, 0, 9, 0, None) == _lib.E_INVALID
  # fir: batch mismatch / frame mismatch / bad padding (core.py:1441-1457,1367)
  assert lib.ddsp_b200_fir_time_varying(fake, fake, fake, 2, 1000, 10, 16, 3, 0,
                                        -1, 0, None) == _lib.E_INVALID
  assert b'Batch size' in lib.ddsp_b200_last_error()
  assert lib.ddsp_b200_fir_time_varying(fake, fake, fake, 1, 1000, 999, 16, 1, 0,
                                        -1, 0, None) == _lib.E_INVALID
  assert b'Number of Audio frames' in lib.ddsp_b200_last_error()
  assert lib.ddsp_b200_fir_time_varying(fake, fake, fake, 1, 1000, 10, 16, 1, 5,
                                        -1, 0, None) == _lib.E_INVALID
  # null pointers
  assert lib.ddsp_b200_add(None, fake, fake, 4, None) == _lib.E_INVALID
  assert lib.ddsp_b200_harmonic_controls(fake, fake, fake, fake, None, 1, 1, 1,
                                         16000.0, 3, None) == _lib.E_INVALID
  # too few frequencies for an irfft
  assert lib.ddsp_b200_ir_size(1, 0) == _lib.E_INVALID
  # empty batches are no-ops, not errors
  assert lib.ddsp_b200_harmonic_forward(fake, fake, fake, fake, 0, 10, 4, 640,
                                        16000.0, 0, 0, 0, None) == 0


@pytest.mark.parametrize('nb,ws,want', [(1025, 0, 2048), (1025, 257, 257),
                                        (513, 22, 21), (513, 2048, 1024),
                                        (65, 0, 128), (65, 257, 128), (100, 50, 49)])
def test_ir_size_table(nb, ws, want):
  """core_test.py:825-855: window_size if odd, -1 if even, fft size if none."""
  assert _lib.load().ddsp_b200_ir_size(nb, ws) == want


def test_missing_library_is_loud(monkeypatch):
  monkeypatch.setattr(_lib, '_lib', None)
  monkeypatch.setattr(_lib, 'LIB_PATH', '/nonexistent/libddsp_b200.so')
  with pytest.raises(RuntimeError, match='no CPU fallback'):
    _lib.load()


# ---- Python error conventions (raised before any device work) ----------------
def test_harmonic_synthesis_value_errors():
  f0 = np.zeros((1, 10, 1), np.float32)
  amp = np.zeros((1, 10, 1), np.float32)
  with pytest.raises(ValueError, match='is invalid'):        # core.py:632-634
    core.harmonic_synthesis(f0, amp, n_samples=640, amp_resample_method='bogus')
  with pytest.raises(ValueError, match='only supports 3 dimensions'):
    core.harmonic_synthesis(f0[0], amp[0], n_samples=640)    # core.py:670-672
  with pytest.raises(ValueError, match='downsampling'):      # core.py:682-685
    core.harmonic_synthesis(f0, amp, n_samples=5)
  with pytest.raises(ValueError, match='divisible'):         # core.py:687-693
    core.harmonic_synthesis(f0, amp, n_samples=645)
  with pytest.raises(ValueError, match='harmonic_shifts'):
    core.harmonic_synthesis(f0, amp, harmonic_shifts=np.zeros((1, 9, 4), np.float32),
                            n_samples=640)


def test_fft_convolve_value_errors():
  """core_test.py:787-823."""
  audio = np.zeros((1, 1000), np.float32)
  with pytest.raises(ValueError, match='Batch size'):
    core.fft_convolve(audio, np.zeros((2, 1000), np.float32))
  for padding in ('', 'saaammmeee'):
    with pytest.raises(ValueError, match='Padding'):
      core.fft_convolve(audio, audio, padding=padding)
  for n_frames in (1010, 999):
    with pytest.raises(ValueError, match='Number of Audio frames'):
      core.fft_convolve(audio, np.zeros((1, n_frames, 1000), np.float32))


def test_filtered_noise_value_errors():
  with pytest.raises(ValueError, match='Number of Audio frames'):
    core.filtered_noise(np.zeros((1, 999, 65), np.float32), 1000)
  with pytest.raises(ValueError, match='noise must be'):
    core.filtered_noise(np.zeros((1, 10, 65), np.float32), 640,
                        noise=np.zeros((1, 64), np.float32))


def test_get_fft_size():
  """core.py:1317-1335."""
  assert core.get_fft_size(64, 128) == 256
  assert core.get_fft_size(64, 257) == 512
  assert core.get_fft_size(1000, 10) == 1024


# ---- dict helpers (core.py:39-129) --------------------------------------------
def test_nested_lookup_and_to_dict():
  d = {'a': {'b': {'c': 3}}, 'x': 1}
  assert core.nested_lookup('a/b/c', d) == 3
  assert core.nested_keys(d) == ['a/b/c', 'x']
  with pytest.raises(KeyError, match='available keys'):
    core.nested_lookup('a/z', d)
  assert core.to_dict([1, 2], ['p', 'q']) == {'p': 1, 'q': 2}
  assert core.to_dict({'k': 1}, ['ignored']) == {'k': 1}
  with pytest.raises(ValueError):
    core.to_dict([1, 2, 3], ['p', 'q'])
  assert core.make_iterable(None) == []
  arr = np.zeros(3)
  assert core.make_iterable(arr)[0] is arr


# ---- Processor / ProcessorGroup / DAG (processors.py:37-176, dags.py:57-195) --
class _Scale(processors.Processor):
  """A host-only processor: lets the DAG logic run without a GPU."""

  def __init__(self, gain, name):
    super().__init__(name=name)
    self.gain = gain

  def get_controls(self, x):
    return {'x': np.asarray(x) * 1.0}

  def get_signal(self, x):
    return x * self.gain


class _HostAdd(processors.Processor):

  def __init__(self, name='add'):
    super().__init__(name=name)

  def get_controls(self, signal_one, signal_two):
    return {'signal_one': signal_one, 'signal_two': signal_two}

  def get_signal(self, signal_one, signal_two):
    return signal_one + signal_two


def test_processor_call_protocol():
  """processors.py:53-68: drops training/mask, optional outputs dict."""
  p = _Scale(3.0, 'scale')
  x = np.ones((2, 4))
  assert np.all(p(x) == 3.0)
  out = p(x, return_outputs_dict=True, training=True, mask=None)
  assert set(out) == {'signal', 'controls'} and set(out['controls']) == {'x'}
  with pytest.raises(NotImplementedError):
    processors.Processor('base').get_controls()


def test_processor_group_dag_semantics():
  """processors_test.py:57-87 key set; dags.py:149-193 outputs / 'out' alias."""
  a, b, add = _Scale(2.0, 'a'), _Scale(5.0, 'b'), _HostAdd('add')
  dag = [(a, ['inputs/u']), (b, ['v']), (add, ['a/signal', 'b/signal'])]
  group = processors.ProcessorGroup(dag=dag, name='processor_group')
  assert group.dag == [['a', ['inputs/u']], ['b', ['v']],
                       ['add', ['a/signal', 'b/signal']]]
  assert group.processors == [a, b, add] and group.a is a
  feats = {'u': np.ones((1, 3)), 'v': np.ones((1, 3))}
  outs = group.get_controls(feats)
  for key in ['u', 'v', 'inputs/u', 'a/signal', 'a/controls/x', 'b/signal',
              'b/controls/x', 'add/signal', 'add/controls/signal_one',
              'add/controls/signal_two', 'out/signal']:
    assert isinstance(core.nested_lookup(key, outs), np.ndarray), key
  assert np.all(outs['out']['signal'] == 7.0)
  assert np.all(group.get_signal(outs) == 7.0)
  assert np.all(group(feats) == 7.0)
  full = group(feats, return_outputs_dict=True)
  assert set(full) == {'signal', 'controls'}
  # string nodes resolve through kwarg processors (dags.py:104-106)
  g2 = processors.ProcessorGroup(dag=[('a', ['u']), ('add', ['a/signal', 'u'])],
                                 a=a, add=add)
  assert np.all(g2({'u': np.ones((1, 3))}) == 3.0)
  with pytest.raises(KeyError):
    group.get_controls({'u': np.ones((1, 3))})          # 'v' missing


def test_dag_layer_non_processor_modules_and_output_keys():
  """dags.py:171-186: plain modules are called, tuples zipped with output keys."""

  class Split:
    name = 'split'

    def __call__(self, x):
      return x + 1, x - 1

  layer = dags.DAGLayer([(Split(), ['x'], ['hi', 'lo'])])
  out = layer({'x': np.zeros(2)})
  assert np.all(out['split']['hi'] == 1) and np.all(out['out']['lo'] == -1)
  bad = dags.DAGLayer([(Split(), ['x'], ['only_one'])])
  with pytest.raises(ValueError):
    bad({'x': np.zeros(2)})


def test_synth_constructors_match_reference_defaults():
  """synths.py:59-66, 153-158; processors.py:166."""
  h = synths.Harmonic()
  assert (h.n_samples, h.sample_rate, h.normalize_below_nyquist,
          h.amp_resample_method, h.use_angular_cumsum, h.name) == (
              64000, 16000, True, 'window', False, 'harmonic')
  assert h.scale_fn is core.exp_sigmoid
  n = synths.FilteredNoise()
  assert (n.n_samples, n.window_size, n.initial_bias, n.name) == (
      64000, 257, -5.0, 'filtered_noise')
  assert processors.Add().name == 'add'
  assert dags.is_processor(h) and dags.is_processor(n)


def test_decoder_pattern_detection():
  h, n, add = synths.Harmonic(), synths.FilteredNoise(), processors.Add()
  g = processors.ProcessorGroup(dag=[
      (h, ['amps', 'hd', 'f0_hz']), (n, ['mags']),
      (add, ['filtered_noise/signal', 'harmonic/signal'])])
  assert g._decoder_pattern() is not None
  g2 = processors.ProcessorGroup(dag=[(h, ['amps', 'hd', 'f0_hz'])])
  assert g2._decoder_pattern() is None
  g3 = processors.ProcessorGroup(dag=[
      (h, ['amps', 'hd', 'f0_hz']), (n, ['mags']),
      (add, ['harmonic/signal', 'harmonic/signal'])])
  assert g3._decoder_pattern() is None


def test_resample_value_errors():
  """core_test.py:178-198, 295-381 - raised before any device work."""
  for dims in (1, 2, 4):
    with pytest.raises(ValueError, match='only supports 3 dimensions'):
      core.upsample_with_windows(np.ones([5] * dims, np.float32), 16000)
  for add_endpoint in (True, False):
    with pytest.raises(ValueError, match='downsampling'):
      core.upsample_with_windows(np.ones([1, 16000, 1], np.float32), 5, add_endpoint)
  with pytest.raises(ValueError, match='divisible'):
    core.upsample_with_windows(np.ones([1, 5, 1], np.float32), 16)
  with pytest.raises(ValueError, match='divisible'):
    core.upsample_with_windows(np.ones([1, 5, 1], np.float32), 15, add_endpoint=False)
  with pytest.raises(ValueError, match='is invalid'):
    core.resample(np.ones([1, 5, 1], np.float32), 10, method='bogus')


def test_host_pipeline_validates_without_a_gpu():
  """ddsp_b200_host_pipeline_*: argument errors come back as status codes before
  any CUDA call; a null handle is rejected by the forward entry point."""
  import ctypes
  lib = _lib.load()
  h = ctypes.c_void_p()
  assert lib.ddsp_b200_host_pipeline_create(ctypes.byref(h), 0, 10, 4, 5, 640, 2) == _lib.E_INVALID
  assert not h.value
  assert lib.ddsp_b200_decoder_forward_host(None, 1, 1, 1, 1, 0, 0, 1, 1, 1, 16000.0,
                                            0, 3, 0, -5.0, None) == _lib.E_INVALID
  assert b'null handle' in lib.ddsp_b200_last_error()
  assert lib.ddsp_b200_host_pipeline_destroy(None) == 0


def test_host_decoder_rejects_non_decoder_dags():
  import ddsp_b200
  harm = ddsp_b200.Harmonic(n_samples=640)
  group = ddsp_b200.ProcessorGroup(dag=[(harm, ['a', 'h', 'f'])])
  with pytest.raises(ValueError):
    ddsp_b200.HostDecoder(group, 2, 10, 4, 5)


def test_window_and_crop_helpers_match_oracle_and_reference():
  """core.apply_window_to_impulse_response (core.py:1477-1531) and
  core.crop_and_compensate_delay (1338-1379): host-side torch ops, so they run on
  the CPU - against the oracle and the unmodified reference's results
  (tests/golden/host_helpers.npz: shape, peak and L2 norm of each output and up to
  make_golden.SAMPLE of its elements)."""
  import torch
  from oracle import ddsp_oracle as o
  from tests.golden import make_golden as mg
  ref = mg.unpack_outputs(np.load(os.path.join(ROOT, 'tests', 'golden', 'host_helpers.npz')))
  for i, (kind, args) in enumerate(mg.host_helper_cases()):
    shape, values, peak, l2 = ref['%s_%d' % (kind, i)]
    if kind == 'window':
      ir, ws, causal = args
      got = core.apply_window_to_impulse_response(ir, ws, causal)
      assert isinstance(got, torch.Tensor) and not got.is_cuda
      want = o.apply_window_to_impulse_response(ir, ws, causal, dtype=np.float32)
      assert tuple(got.shape) == want.shape
      assert np.abs(got.numpy() - want).max() < 1e-6
      got = got.numpy().astype(np.float64)
      assert got.shape == shape, (args[1:], got.shape, shape)
      assert np.abs(got.ravel()[mg.sample_index(got.size)] - values).max() < 1e-6
      assert abs(np.abs(got).max() - peak) < 1e-6
      assert abs(np.sqrt((got * got).sum()) - l2) < 1e-6 * np.sqrt(got.size)
    else:
      got = core.crop_and_compensate_delay(*args).numpy()
      assert np.array_equal(got, o.crop_and_compensate_delay(*args))
      got = got.astype(np.float64)
      assert got.shape == shape, (args[1:], got.shape, shape)
      assert np.array_equal(got.ravel()[mg.sample_index(got.size)], values)
      assert (np.abs(got).max() if got.size else 0.0) == peak
      assert abs(np.sqrt((got * got).sum()) - l2) <= 1e-12 * l2   # summation order only
  with pytest.raises(ValueError, match="Padding must be 'valid' or 'same'"):
    core.crop_and_compensate_delay(np.zeros((1, 10), np.float32), 5, 3, 'full', 0)

