"""Writes tests/golden/*.npz: outputs of the UNMODIFIED REFERENCE (magenta/ddsp,
/root/reference/ddsp) on seeded inputs, for the decoder path.

How: the reference package is imported as it lies and run on the NumPy stand-in
for its TensorFlow primitives (oracle/tf_shim via oracle/ref_on_shim.py) - twice:
"narrow" (float32, the reference's own arithmetic incl. its sequential float32
phase cumsum) and "wide" (the same reference code with every float32 widened to
float64: the exact value of the reference's formulae, which is what the 1e-4
parity gate is measured against; BASELINE.md section 5 gives the distance between
the two - the reference's own phase-accumulation error).

Needs /root/reference, so it runs in the authoring container only:

  python tests/golden/make_golden.py          # rewrite every fixture
  python tests/golden/make_golden.py --check  # regenerate in memory and compare

The tests read the fixtures, so they need no reference: tests/test_reference_pin.py
(CPU: oracle vs fixtures, and fixtures vs a fresh reference run when the reference
is present), tests/test_gpu_golden.py (CUDA path vs fixtures), and
tests/test_reference_fuzz.py, test_effects.py and test_host_api.py (oracle and host
logic vs the reference on the argument sets drawn by the *_cases generators below).
Inputs are regenerated from their seeds by tests/util.synth_inputs; an input
checksum in every fixture guards against generator drift.
"""
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))
from oracle import ref_on_shim               # noqa: E402
from tests.util import synth_inputs          # noqa: E402


def checksum(inp):
  return np.float64(sum(float(np.asarray(v, np.float64).sum()) * (i + 1)
                        for i, v in enumerate(inp[k] for k in sorted(inp))))


def _both(fn):
  """fn() under the narrow and the wide shim -> (narrow, wide) numpy results."""
  tf = ref_on_shim.tf()
  out = []
  for wide in (False, True):
    tf.set_wide(wide)
    try:
      out.append(ref_on_shim.to_numpy(fn()))
    finally:
      tf.set_wide(False)
  return out


def _nyquist_margin(ddsp, inp, n_samples, k, sample_rate=16000):
  """Smallest |f_k(t) - sr/2| of the float32 frequency envelopes: the fixture is
  only meaningful if no oscillator sits within an ulp of the Nyquist decision
  (then narrow and wide would disagree by a whole oscillator at that sample)."""
  hf = ddsp.core.get_harmonic_frequencies(inp['f0_hz'], k)
  fe = ddsp.core.resample(hf, n_samples).numpy().astype(np.float64)
  return float(np.abs(fe - sample_rate / 2.0).min())


def c1_harmonic():
  """BASELINE.json configs[0]: Harmonic only, B=1, 16000 samples, 64 harmonics,
  250 frames (synths.Harmonic defaults: window resampling, Nyquist normalise)."""
  ddsp = ref_on_shim.load()
  seed = 101
  inp = synth_inputs(1, 250, 64, 65, 16000, seed=seed)
  args = (inp['amps'], inp['harmonic_distribution'], inp['f0_hz'])
  assert _nyquist_margin(ddsp, inp, 16000, 64) > 1e-2

  def run(angular):
    h = ddsp.synths.Harmonic(n_samples=16000, use_angular_cumsum=angular)
    return h(*args, return_outputs_dict=True)

  n0, w0 = _both(lambda: run(False))
  n1, _ = _both(lambda: run(True))
  return dict(
      seed=seed, input_checksum=checksum(inp),
      amplitudes=n0['controls']['amplitudes'],
      harmonic_distribution=n0['controls']['harmonic_distribution'],
      audio_ref_f32_cumsum=n0['signal'], audio_ref_f32_angular=n1['signal'],
      audio_ref_wide=w0['signal'].astype(np.float64))


def decoder_small():
  """The ae.gin DAG (ae.gin:47-72) through the reference's ProcessorGroup from raw
  network outputs, B=2, F=25, N=1600, K=100, 65 bands, injected noise."""
  ddsp = ref_on_shim.load()
  tf = ref_on_shim.tf()
  seed = 202
  B, F, K, nb, N = 2, 25, 100, 65, 1600
  inp = synth_inputs(B, F, K, nb, N, seed=seed)
  assert _nyquist_margin(ddsp, inp, N, K) > 1e-2

  def run():
    harm = ddsp.synths.Harmonic(n_samples=N, sample_rate=16000)
    noise = ddsp.synths.FilteredNoise(n_samples=N, window_size=0)
    group = ddsp.processors.ProcessorGroup(dag=[
        (harm, ['amps', 'harmonic_distribution', 'f0_hz']),
        (noise, ['noise_magnitudes']),
        (ddsp.processors.Add(), ['filtered_noise/signal', 'harmonic/signal'])])
    tf.random.inject_uniform(inp['noise'])
    feats = {k: inp[k] for k in ('amps', 'harmonic_distribution', 'f0_hz',
                                 'noise_magnitudes')}
    return group.get_controls(feats)

  n, w = _both(run)
  out = dict(seed=seed, input_checksum=checksum(inp))
  for tag, o in (('f32', n), ('wide', w)):
    out['harmonic_' + tag] = o['harmonic']['signal']
    out['filtered_noise_' + tag] = o['filtered_noise']['signal']
    out['audio_' + tag] = o['out']['signal']
  out['magnitudes'] = n['filtered_noise']['controls']['magnitudes']
  out['harmonic_distribution'] = n['harmonic']['controls']['harmonic_distribution']
  out['amplitudes'] = n['harmonic']['controls']['amplitudes']
  return out


def c2_item():
  """One batch item at the configs[1..4] shapes (F=1000, K=100, 65 bands, 64000
  samples): the reference's harmonic and filtered-noise signals, wide; stored as
  float32 (rounding 6e-8, far inside the 1e-4 gate) to keep the file small."""
  ddsp = ref_on_shim.load()
  tf = ref_on_shim.tf()
  seed = 303
  inp = synth_inputs(1, 1000, 100, 65, 64000, seed=seed)
  assert _nyquist_margin(ddsp, inp, 64000, 100) > 1e-2

  def run():
    harm = ddsp.synths.Harmonic(n_samples=64000, sample_rate=16000)
    noise = ddsp.synths.FilteredNoise(n_samples=64000, window_size=0)
    tf.random.inject_uniform(inp['noise'])
    return {'h': harm(inp['amps'], inp['harmonic_distribution'], inp['f0_hz']),
            'n': noise(inp['noise_magnitudes'])}

  n, w = _both(run)
  return dict(seed=seed, input_checksum=checksum(inp),
              harmonic_wide=w['h'].astype(np.float32),
              filtered_noise_wide=w['n'].astype(np.float32),
              # the reference's own float32 result, decimated: documents its
              # phase-accumulation error at 64000 samples
              harmonic_f32_every16=n['h'][:, ::16].astype(np.float32))


def harmonic_shifts():
  """core.harmonic_synthesis with harmonic_shifts (core.py:1084-1093), 'linear'
  and 'window' amplitudes, B=2, F=50, K=20, N=3200."""
  ddsp = ref_on_shim.load()
  seed = 404
  B, F, K, N = 2, 50, 20, 3200
  inp = synth_inputs(B, F, K, 65, N, seed=seed, f0_lo=100.0, f0_hi=500.0)
  rng = np.random.default_rng(seed)
  shifts = (0.02 * rng.standard_normal((B, F, K))).astype(np.float32)
  amps = np.abs(inp['amps']) * 0.5
  hd = np.abs(inp['harmonic_distribution'])
  hd = (hd / hd.sum(-1, keepdims=True)).astype(np.float32)
  out = dict(seed=seed, shifts=shifts, amplitudes=amps.astype(np.float32),
             harmonic_distribution=hd, f0_hz=inp['f0_hz'])
  for method in ('window', 'linear'):
    n, w = _both(lambda: ddsp.core.harmonic_synthesis(
        inp['f0_hz'], amps, harmonic_shifts=shifts, harmonic_distribution=hd,
        n_samples=N, sample_rate=16000, amp_resample_method=method))
    out['audio_f32_' + method] = n
    out['audio_wide_' + method] = w.astype(np.float64)
  return out


def resample_methods():
  """core.resample (core.py:573-642) for every method, both add_endpoint values,
  3-D and 4-D inputs, up- and down-sampling."""
  ddsp = ref_on_shim.load()
  rng = np.random.default_rng(505)
  x3 = rng.standard_normal((2, 10, 3)).astype(np.float32)
  x4 = rng.standard_normal((2, 10, 4, 3)).astype(np.float32)
  out = dict(x3=x3, x4=x4)
  for method in ('nearest', 'linear', 'cubic', 'window'):
    for ep in (True, False):
      n_up = 90 if not ep else 80      # divisible by 9 intervals / 10 frames
      n, w = _both(lambda: ddsp.core.resample(x3, n_up, method=method, add_endpoint=ep))
      out['up3_%s_%d' % (method, ep)] = n
      out['up3w_%s_%d' % (method, ep)] = w
      if method != 'window':
        out['down3_%s_%d' % (method, ep)] = _both(
            lambda: ddsp.core.resample(x3, 4, method=method, add_endpoint=ep))[0]
        out['up4_%s_%d' % (method, ep)] = _both(
            lambda: ddsp.core.resample(x4, 37, method=method, add_endpoint=ep))[0]
  return out


def angular_cumsum():
  """core.angular_cumsum (core.py:799-866) and tf.cumsum on the same angular
  frequencies, float32: [2, 2500, 3] (so the 1000-sample chunking pads)."""
  ddsp = ref_on_shim.load()
  tf = ref_on_shim.tf()
  rng = np.random.default_rng(606)
  omega = (2 * np.pi * rng.uniform(50.0, 4000.0, (2, 1, 3)) / 16000.0 *
           (1 + 0.01 * rng.standard_normal((2, 2500, 3)))).astype(np.float32)
  n, w = _both(lambda: ddsp.core.angular_cumsum(tf.convert_to_tensor(omega)))
  return dict(omega=omega, phase_f32=n, phase_wide=w.astype(np.float64))


def spectral_loss():
  """losses.SpectralLoss (losses.py:130-243) with the ae.gin weights (L1 on
  magnitudes and log magnitudes, ae.gin:39-41), B=2, N=8000."""
  ddsp = ref_on_shim.load()
  rng = np.random.default_rng(707)
  target = (0.1 * rng.standard_normal((2, 8000))).astype(np.float32)
  t = np.arange(8000) / 16000.0
  audio = (0.3 * np.sin(2 * np.pi * 220.0 * t)[None, :] * np.array([[1.0], [0.5]])
           + 0.05 * rng.standard_normal((2, 8000))).astype(np.float32)
  out = dict(target=target, audio=audio)
  for tag, kw in (('mag', dict(mag_weight=1.0, logmag_weight=0.0)),
                  ('maglog', dict(mag_weight=1.0, logmag_weight=1.0))):
    n, w = _both(lambda: ddsp.losses.SpectralLoss(**kw)(target, audio))
    out['loss_f32_' + tag] = np.float32(n)
    out['loss_wide_' + tag] = np.float64(w)
  return out


IR_CASES = [(65, 0), (65, 257), (65, 63), (65, 64), (100, 51), (100, 50), (513, 257),
            (513, 22), (1025, 257), (16, 257), (65, 3)]


def impulse_responses():
  """core.frequency_impulse_response (core.py:1534-1565) and frequency_filter
  (1628-1655) for even AND odd window sizes: tf.signal.hann_window is periodic
  for even lengths and symmetric for odd ones (window_ops._raised_cosine_window),
  which a restatement gets wrong unless it is checked on an odd window shorter than
  the impulse response (window_size=257 with more than 129 bins, e.g.)."""
  ddsp = ref_on_shim.load()
  rng = np.random.default_rng(808)
  out = {}
  for nb, ws in IR_CASES:
    m = rng.uniform(0.0, 1.0, (2, 3, nb)).astype(np.float32)
    n, w = _both(lambda: ddsp.core.frequency_impulse_response(m, ws))
    out['mags_%d_%d' % (nb, ws)] = m
    out['ir_f32_%d_%d' % (nb, ws)] = n
    out['ir_wide_%d_%d' % (nb, ws)] = w.astype(np.float64)
  noise = rng.uniform(-1.0, 1.0, (2, 960)).astype(np.float32)
  mags = rng.uniform(0.0, 1.0, (2, 20, 513)).astype(np.float32)
  n, w = _both(lambda: ddsp.core.frequency_filter(noise, mags, window_size=257))
  out.update(filter_noise=noise, filter_mags=mags, filter_f32=n,
             filter_wide=w.astype(np.float64))
  return out


SAMPLE = 512


def sample_index(size):
  """Flat indices of the stored part of an output of `size` elements: all of them
  up to SAMPLE, else a fixed seeded choice of SAMPLE."""
  if size <= SAMPLE:
    return np.arange(size)
  return np.sort(np.random.default_rng(size).choice(size, SAMPLE, replace=False))


def pack_outputs(outputs):
  """{name: array, or None where the reference raised} -> fixture entries: for
  each output its shape, its sample_index values, and its peak and L2 norm over
  every element, in a few flat arrays (one small array per output would make the
  file mostly zip headers)."""
  names, ndim, dims, start, values, absmax, l2 = [], [], [], [0], [], [], []
  for name, x in outputs.items():
    names.append(name)
    x = None if x is None else np.asarray(x, np.float64)
    ndim.append(-1 if x is None else x.ndim)
    dims.append(([] if x is None else list(x.shape)) + [0] * (4 - (0 if x is None else x.ndim)))
    v = np.zeros(0) if x is None else x.ravel()[sample_index(x.size)]
    values.append(v)
    start.append(start[-1] + v.size)
    absmax.append(np.abs(x).max() if x is not None and x.size else 0.0)
    l2.append(0.0 if x is None else np.sqrt((x * x).sum()))
  return dict(names=np.array(names), ndim=np.array(ndim, np.int64),
              dims=np.array(dims, np.int64), start=np.array(start, np.int64),
              values=np.concatenate(values), absmax=np.array(absmax),
              l2=np.array(l2))


def unpack_outputs(g):
  """pack_outputs entries -> {name: None where the reference raised, else
  (shape, sampled values, peak, L2 norm)}."""
  out = {}
  for i, name in enumerate(g['names']):
    n = int(g['ndim'][i])
    out[str(name)] = None if n < 0 else (
        tuple(int(d) for d in g['dims'][i][:n]),
        g['values'][g['start'][i]:g['start'][i + 1]], float(g['absmax'][i]),
        float(g['l2'][i]))
  return out


def fuzz_fft_convolve_cases():
  """Arguments of core.fft_convolve: shapes, both paddings, delay compensations."""
  rng = np.random.default_rng(123)
  for _ in range(24):
    b, f = int(rng.integers(1, 3)), int(rng.choice([1, 2, 5, 10, 25]))
    frame, s = int(rng.choice([1, 3, 16, 48, 64])), int(rng.choice([1, 2, 3, 10, 31, 64, 65, 128, 200]))
    pad, dc = str(rng.choice(['same', 'valid'])), int(rng.choice([-1, 0, 1, 5]))
    a = rng.standard_normal((b, f * frame)).astype(np.float32)
    ir = rng.standard_normal((b, f, s)).astype(np.float32)
    yield dict(a=a, ir=ir, padding=pad, delay_compensation=dc)


def fuzz_frequency_filter_cases():
  """core.frequency_filter with odd / even / degenerate windows."""
  rng = np.random.default_rng(124)
  for _ in range(20):
    f, frame = int(rng.choice([1, 4, 10])), int(rng.choice([8, 32, 64]))
    nb = int(rng.choice([2, 3, 9, 16, 33, 65, 100, 129, 130, 257]))
    ws = int(rng.choice([0, 1, 2, 3, 7, 8, 50, 51, 64, 65, 257]))
    a = rng.uniform(-1, 1, (1, f * frame)).astype(np.float32)
    m = rng.uniform(0, 1, (1, f, nb)).astype(np.float32)
    yield dict(audio=a, magnitudes=m, window_size=ws)


def fuzz_harmonic_synthesis_cases():
  """core.harmonic_synthesis over every amplitude resampling method, both phase
  accumulators, sample rates and the optional arguments."""
  rng = np.random.default_rng(321)
  for _ in range(14):
    b, f = int(rng.integers(1, 3)), int(rng.choice([2, 5, 10, 25]))
    hop, k = int(rng.choice([4, 16, 64, 100])), int(rng.choice([1, 3, 20, 60]))
    method = str(rng.choice(['window', 'linear', 'nearest', 'cubic']))
    uac, sr = bool(rng.integers(0, 2)), int(rng.choice([16000, 8000, 44100]))
    f0 = rng.uniform(20, sr * 0.45, (b, f, 1)).astype(np.float32)
    amp = rng.uniform(0, 1, (b, f, 1)).astype(np.float32)
    hd = rng.uniform(0, 1, (b, f, k)).astype(np.float32) if rng.integers(0, 4) else None
    shifts = (rng.uniform(-0.05, 0.05, (b, f, k)).astype(np.float32)
              if hd is not None and rng.integers(0, 2) else None)
    yield dict(f0=f0, amp=amp, hd=hd, shifts=shifts, n_samples=f * hop, sample_rate=sr,
               method=method, use_angular_cumsum=uac)


def fuzz_misc_cases():
  """(kind, arguments) for Harmonic.get_controls, oscillator_bank, streaming
  synthesis, the scaling functions and Sinusoidal, drawn from one generator."""
  rng = np.random.default_rng(999)
  for _ in range(8):                                   # Harmonic.get_controls variants
    f, k = int(rng.choice([3, 10])), int(rng.choice([1, 7, 40]))
    scale, nyq, sr = bool(rng.integers(0, 2)), bool(rng.integers(0, 2)), int(rng.choice([16000, 4000]))
    a = rng.standard_normal((1, f, 1)).astype(np.float32)
    h = rng.standard_normal((1, f, k)).astype(np.float32)
    f0 = rng.uniform(0, sr / 2, (1, f, 1)).astype(np.float32)
    if not scale:
      a, h = np.abs(a), np.abs(h)
    yield 'get_controls', dict(a=a, h=h, f0=f0, f=f, scale=scale, nyquist=nyq, sample_rate=sr)
  for _ in range(8):                                   # oscillator_bank
    b, n, k = int(rng.integers(1, 3)), int(rng.choice([50, 1000, 2500])), int(rng.choice([1, 4, 17]))
    sr, ss, uac = int(rng.choice([16000, 8000])), bool(rng.integers(0, 2)), bool(rng.integers(0, 2))
    fe = rng.uniform(0, sr * 0.6, (b, n, k)).astype(np.float32)
    ae = rng.uniform(0, 1, (b, n, k)).astype(np.float32)
    yield 'oscillator_bank', dict(fe=fe, ae=ae, sample_rate=sr, sum_sinusoids=ss,
                                  use_angular_cumsum=uac)
  for _ in range(8):                                   # streaming synthesis, carried phase
    b, f, hop = int(rng.integers(1, 3)), int(rng.choice([1, 4, 10])), int(rng.choice([16, 64]))
    k = int(rng.choice([1, 5, 30]))
    f0 = rng.uniform(50, 2000, (b, f, 1)).astype(np.float32)
    amp = rng.uniform(0, 1, (b, f, 1)).astype(np.float32)
    hd = rng.uniform(0, 1, (b, f, k)).astype(np.float32) if rng.integers(0, 3) else None
    ph = rng.uniform(0, 6.28, (b, 1, 1)).astype(np.float32) if rng.integers(0, 2) else None
    method = str(rng.choice(['linear', 'window']))
    yield 'streaming', dict(f0=f0, amp=amp, hd=hd, phase=ph, n_samples=f * hop,
                            method=method)
  for _ in range(5):                                   # scaling functions
    x = (4 * rng.standard_normal((2, 5, 7))).astype(np.float32)
    ex, mv, th = float(rng.choice([10.0, 2.0, 5.0])), float(rng.choice([2.0, 1.0])), float(rng.choice([1e-7, 1e-3]))
    depth = int(rng.choice([1, 8, 64]))
    fr = rng.standard_normal((2, 5, 3 * depth)).astype(np.float32)
    yield 'scalers', dict(x=x, exponent=ex, max_value=mv, threshold=th, fr=fr, depth=depth)
  for _ in range(4):                                   # Sinusoidal
    f, k, hop = int(rng.choice([5, 10])), int(rng.choice([1, 4, 9])), int(rng.choice([16, 64]))
    a = rng.standard_normal((1, f, k)).astype(np.float32)
    fr = rng.standard_normal((1, f, k)).astype(np.float32)
    method = str(rng.choice(['window', 'linear']))
    yield 'sinusoidal', dict(a=a, fr=fr, n_samples=f * hop, method=method)


def reference_fuzz():
  """The reference in its wide mode (its own code evaluated in float64) on the
  fuzz_*_cases arguments: what tests/test_reference_fuzz.py holds the oracle's
  float64 mode to, packed by pack_outputs under the names
  <function>_<case>[_<output>]."""
  ddsp = ref_on_shim.load()
  tf = ref_on_shim.tf()
  t = tf.convert_to_tensor
  tt = lambda x: None if x is None else t(x)  # noqa: E731

  def wide(fn):
    tf.set_wide(True)
    try:
      return ref_on_shim.to_numpy(fn())
    finally:
      tf.set_wide(False)

  out = {}
  for i, c in enumerate(fuzz_fft_convolve_cases()):
    try:
      want = wide(lambda: ddsp.core.fft_convolve(c['a'], c['ir'], padding=c['padding'],
                                                 delay_compensation=c['delay_compensation']))
    except Exception:  # pylint: disable=broad-except
      want = None
    out['fft_convolve_%d' % i] = want
  for i, c in enumerate(fuzz_frequency_filter_cases()):
    out['frequency_filter_%d' % i] = wide(lambda: ddsp.core.frequency_filter(
        c['audio'], c['magnitudes'], window_size=c['window_size']))
  for i, c in enumerate(fuzz_harmonic_synthesis_cases()):
    # tensors, so that the wide mode widens every operand (a raw float32 array in
    # `1.0 + harmonic_shifts` would be rounded by NumPy before the shim sees it)
    out['harmonic_synthesis_%d' % i] = wide(lambda: ddsp.core.harmonic_synthesis(
        t(c['f0']), t(c['amp']), harmonic_shifts=tt(c['shifts']),
        harmonic_distribution=tt(c['hd']), n_samples=c['n_samples'],
        sample_rate=c['sample_rate'], amp_resample_method=c['method'],
        use_angular_cumsum=c['use_angular_cumsum']))
  for i, (kind, c) in enumerate(fuzz_misc_cases()):
    key = '%s_%d' % (kind, i)
    if kind == 'get_controls':
      syn = ddsp.synths.Harmonic(n_samples=c['f'] * 8, sample_rate=c['sample_rate'],
                                 scale_fn=ddsp.core.exp_sigmoid if c['scale'] else None,
                                 normalize_below_nyquist=c['nyquist'])
      want = wide(lambda: syn.get_controls(c['a'], c['h'], c['f0']))
      for name in ('amplitudes', 'harmonic_distribution', 'f0_hz'):
        out['%s_%s' % (key, name)] = want[name]
    elif kind == 'oscillator_bank':
      out[key] = wide(lambda: ddsp.core.oscillator_bank(
          t(c['fe']), t(c['ae']), sample_rate=c['sample_rate'],
          sum_sinusoids=c['sum_sinusoids'], use_angular_cumsum=c['use_angular_cumsum']))
    elif kind == 'streaming':
      audio, phase = wide(lambda: list(ddsp.core.streaming_harmonic_synthesis(
          t(c['f0']), t(c['amp']), tt(c['hd']), tt(c['phase']), n_samples=c['n_samples'],
          sample_rate=16000, amp_resample_method=c['method'])))
      out[key + '_audio'], out[key + '_phase'] = audio, phase
    elif kind == 'scalers':
      out[key + '_exp_sigmoid'] = wide(lambda: ddsp.core.exp_sigmoid(
          t(c['x']), c['exponent'], c['max_value'], c['threshold']))
      out[key + '_sigmoid'] = wide(lambda: ddsp.core.frequencies_sigmoid(
          t(c['fr']), depth=c['depth']))
      out[key + '_softmax'] = wide(lambda: ddsp.core.frequencies_softmax(
          t(c['fr']), depth=c['depth']))
    else:
      syn = ddsp.synths.Sinusoidal(n_samples=c['n_samples'], sample_rate=16000,
                                   amp_resample_method=c['method'])
      out[key] = wide(lambda: syn(t(c['a']), t(c['fr'])))
  return pack_outputs(out)


WINDOW_CASES = [(128, 0, False), (128, 257, False), (128, 64, False), (128, 63, False),
                (30, 257, False), (2048, 257, True), (100, 51, True), (100, 50, False),
                (4, 0, False)]
CROP_CASES = [(64192, 64000, 128, 'same', -1), (64192, 64000, 128, 'valid', -1),
              (1009, 1000, 10, 'same', 0), (109, 10, 100, 'same', -1),
              (4095, 1000, 3000, 'same', 0), (3999, 1000, 3000, 'valid', -1)]


def host_helper_cases():
  """(kind, arguments) for core.apply_window_to_impulse_response and
  core.crop_and_compensate_delay."""
  rng = np.random.default_rng(0)
  for ir_size, ws, causal in WINDOW_CASES:
    ir = rng.standard_normal((2, 3, ir_size)).astype(np.float32)
    yield 'window', (ir, ws, causal)
  for total, n, s, pad, dc in CROP_CASES:
    a = rng.standard_normal((2, total)).astype(np.float32)
    yield 'crop', (a, n, s, pad, dc)


def host_helpers():
  """The reference's float32 results on host_helper_cases, for
  tests/test_host_api.py."""
  ddsp = ref_on_shim.load()
  out = {}
  for i, (kind, args) in enumerate(host_helper_cases()):
    fn = (ddsp.core.apply_window_to_impulse_response if kind == 'window' else
          ddsp.core.crop_and_compensate_delay)
    out['%s_%d' % (kind, i)] = ref_on_shim.to_numpy(fn(*args))
  return pack_outputs(out)


def filtered_noise_reverb_case(trainable):
  """Shapes and draws of the FilteredNoiseReverb composition check: audio, the
  magnitudes (one learned set when trainable) and the noise the synthesizer uses."""
  rng = np.random.default_rng(5)
  B, N, L, F, NB, WS = 2, 3000, 1920, 40, 16, 257
  audio = rng.standard_normal((B, N)).astype(np.float32)
  mags = rng.standard_normal((1 if trainable else B, F, NB)).astype(np.float32)
  noise = rng.uniform(-1, 1, (mags.shape[0], L)).astype(np.float32)
  kw = dict(trainable=trainable, reverb_length=L, window_size=WS, n_frames=F,
            n_filter_banks=NB)
  return audio, mags, noise, kw


def filtered_noise_reverb():
  """effects.FilteredNoiseReverb (the reference's class, float32) on
  filtered_noise_reverb_case, with its tf.random.uniform draw pinned to the case's
  noise, fixed and trainable: for tests/test_effects.py."""
  ddsp = ref_on_shim.load()
  tf = ref_on_shim.tf()
  out = {}
  for trainable in (False, True):
    audio, mags, noise, kw = filtered_noise_reverb_case(trainable)
    uniform = tf.random.uniform
    tf.random.uniform = lambda shape, minval=0, maxval=1, **_: tf.constant(noise)
    try:
      r = ddsp.effects.FilteredNoiseReverb(**kw)
      if trainable:
        r.build(None)
        r._magnitudes = tf.constant(mags[0])
        want = ref_on_shim.to_numpy(r(audio))
      else:
        want = ref_on_shim.to_numpy(r(audio, mags))
    finally:
      tf.random.uniform = uniform
    out['audio_trainable_%d' % trainable] = want
  return out


FIXTURES = dict(c1_harmonic=c1_harmonic, decoder_small=decoder_small, c2_item=c2_item,
                harmonic_shifts=harmonic_shifts, resample_methods=resample_methods,
                angular_cumsum=angular_cumsum, spectral_loss=spectral_loss,
                impulse_responses=impulse_responses, reference_fuzz=reference_fuzz,
                host_helpers=host_helpers, filtered_noise_reverb=filtered_noise_reverb)


def compare(name, got, want, atol=0.0):
  assert set(want.files) == set(got), (name, sorted(set(want.files) ^ set(got)))
  for k in want.files:
    if want[k].dtype.kind == 'U':
      np.testing.assert_array_equal(got[k], want[k], err_msg='%s/%s' % (name, k))
      continue
    np.testing.assert_allclose(np.asarray(got[k], np.float64),
                               np.asarray(want[k], np.float64), rtol=0, atol=atol,
                               err_msg='%s/%s' % (name, k))


if __name__ == '__main__':
  check = '--check' in sys.argv
  for name, fn in FIXTURES.items():
    path = os.path.join(HERE, name + '.npz')
    got = fn()
    if check:
      compare(name, got, np.load(path))
      print('ok   ', name)
    else:
      np.savez_compressed(path, **got)
      print('wrote', name, '%.0f kB' % (os.path.getsize(path) / 1e3))
