#!/usr/bin/env python
"""bench.py - audio samples/sec of the Harmonic(100)+FilteredNoise(65) decoder.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference]
                  [--dump-outputs DIR]
  python -m torch.distributed.run --nnodes=1 --nproc-per-node N \
      --master-addr 127.0.0.1 --master-port P bench.py --gpus N ...

Workload per GPU: batch 256 x 64000 samples @16 kHz, F=1000 frames, K=100
harmonics, 65 noise bands - BASELINE.json configs[2] at N=1 and configs[4]
(2048 = 256/GPU) at N=8 - the `ae.gin` DAG Harmonic -> FilteredNoise -> Add, from
raw network outputs (get_controls included), through ddsp_b200.ProcessorGroup.
One "step" = one decoder forward over one batch, replayed from a CUDA graph
captured around the public ProcessorGroup call (no Python between the kernels of
the timed region).  Weak scaling: every GPU runs the same per-GPU batch on its
own shard, no data-path collective (SURVEY.md 8e); the optional NCCL all-gather
of the audio is timed separately and reported as `all_gather`.  configs[1]
(B=32), configs[0] (Harmonic only, B=1) and configs[3] (forward + backward
through SpectralLoss, B=128) ride along as extra keys timed on rank 0.

One JSON line on stdout (rank 0).  See the task contract for the keys.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

N_SAMPLES = 64000
N_FRAMES = 1000
N_HARM = 100
N_BANDS = 65
SAMPLE_RATE = 16000
BATCH_PER_GPU = 256
L2_BYTES = 126 * 1024 * 1024

# Algorithmic bytes per batch item (BASELINE.md section 3 / SURVEY.md 8d), fp32.
BYTES_HARMONIC = 4 * (2 * N_FRAMES + N_FRAMES * N_HARM) + 4 * N_SAMPLES  # 664000
BYTES_NOISE = 4 * N_FRAMES * N_BANDS + 4 * N_SAMPLES                     # 516000
BYTES_DECODER_FUSED = (4 * (2 * N_FRAMES + N_FRAMES * N_HARM + N_FRAMES * N_BANDS)
                       + 4 * N_SAMPLES)                                  # 924000


def _measured_peaks():
  path = os.path.join(ROOT, 'MEASURED_PEAKS.json')
  if os.path.exists(path):
    with open(path) as f:
      return float(json.load(f)['hbm_gbs']), 'measured'
  return 6650.0, 'fallback'


class ClockSampler:
  """Samples SM clocks / throttle reasons through NVML while the GPU is under
  load.  The timed region of this workload is ~16 ms, so a polling
  `nvidia-smi -lms` process rarely lands a sample inside it; an in-process NVML
  thread polls every ~2 ms instead.  Samples are stamped so
  the timed window can be separated from the rest of the load window."""
  REASONS = {
      'hw_slowdown': 0x8, 'hw_thermal_slowdown': 0x40,
      'sw_thermal_slowdown': 0x20, 'sw_power_cap': 0x4,
  }

  def __init__(self, index):
    self.index = index
    self.samples = []            # (t, sm_mhz, reasons bitmask)
    self.smax = None
    self.stop_flag = False
    self.thread = None
    self.err = None
    self.t_timed = [None, None]

  def start(self):
    try:
      import pynvml
      import torch
      pynvml.nvmlInit()
      try:
        uuid = 'GPU-' + str(torch.cuda.get_device_properties(self.index).uuid)
        h = pynvml.nvmlDeviceGetHandleByUUID(uuid)
      except Exception:  # pylint: disable=broad-except
        h = pynvml.nvmlDeviceGetHandleByIndex(self.index)
      self.smax = float(pynvml.nvmlDeviceGetMaxClockInfo(h, pynvml.NVML_CLOCK_SM))
      get_reasons = getattr(pynvml, 'nvmlDeviceGetCurrentClocksEventReasons',
                            None) or pynvml.nvmlDeviceGetCurrentClocksThrottleReasons

      def loop():
        while not self.stop_flag:
          try:
            mhz = float(pynvml.nvmlDeviceGetClockInfo(h, pynvml.NVML_CLOCK_SM))
            rs = int(get_reasons(h))
            self.samples.append((time.perf_counter(), mhz, rs))
          except Exception as e:  # pylint: disable=broad-except
            self.err = repr(e)
            return
          time.sleep(0.002)     # ~8 samples in a 16 ms timed region, no GIL pressure

      self.thread = threading.Thread(target=loop, daemon=True)
      self.thread.start()
    except Exception as e:  # pylint: disable=broad-except
      self.err = repr(e)

  def mark_timed(self, which):
    self.t_timed[which] = time.perf_counter()

  def stop(self):
    self.stop_flag = True
    if self.thread is not None:
      self.thread.join(timeout=2)
    if not self.samples:
      return {'sm_mhz': None, 'sm_max_mhz': self.smax, 'samples': 0,
              'reasons': ['nvml unavailable: %s' % self.err]}
    t0, t1 = self.t_timed
    window = 'timed region'
    rows = [r for r in self.samples if t0 is not None and t1 is not None and
            t0 <= r[0] <= t1]
    if len(rows) < 3:
      # a short timed region (K steps of ~70 us): use every sample taken while
      # this process kept the GPU busy (warm-up, timed, e2e and per-kernel loops)
      rows = self.samples
      window = 'load window (warm-up + timed + e2e + per-kernel loops)'
    mask = 0
    for r in rows:
      mask |= r[2]
    reasons = sorted(k for k, bit in self.REASONS.items() if mask & bit)
    return {'sm_mhz': statistics.median(r[1] for r in rows),
            'sm_max_mhz': self.smax, 'samples': len(rows), 'window': window,
            'reasons': reasons}


DUMP_ITEMS = 64   # batch items --dump-outputs keeps (64 x 64000 float32 audio = 16 MB)


def dump_outputs(path, arrays):
  """Writes `arrays` (name -> tensor, batch first) as path/<name>.npy in float32.
  Outputs with more than DUMP_ITEMS batch items keep a fixed, seeded choice of
  DUMP_ITEMS of them, the same items in every run, so that two builds can be
  compared output for output."""
  import torch
  os.makedirs(path, exist_ok=True)
  for name, t in arrays.items():
    x = t.detach()
    if x.dim() and x.shape[0] > DUMP_ITEMS:
      idx = np.sort(np.random.default_rng(0).choice(x.shape[0], DUMP_ITEMS, replace=False))
      x = x[torch.from_numpy(idx).to(x.device)]
    np.save(os.path.join(path, name + '.npy'), x.float().cpu().numpy())


def make_host_inputs(batch, seed):
  from tests.util import synth_inputs
  inp = synth_inputs(batch, N_FRAMES, N_HARM, N_BANDS, N_SAMPLES, seed=seed)
  return {k: inp[k] for k in ['amps', 'harmonic_distribution', 'f0_hz',
                              'noise_magnitudes']}


# ----------------------------------------------------------------------------
# reference arm: the CPU port of the reference decoder, host cores only
# ----------------------------------------------------------------------------
_BEST_THREADS = []


def _pick_cpu_threads(items=8):
  """The port is memory-bound torch-CPU code: on a 128-thread host it runs several
  times SLOWER with every thread than with a fraction of them.  Use the thread
  count at which it is fastest (the sample itself, four candidates, once per process)."""
  if _BEST_THREADS:
    return _BEST_THREADS[0]
  import torch
  from oracle import ref_port_torch as rp
  n = os.cpu_count() or 1
  cands = sorted({c for c in (n, n // 2, n // 4, n // 8) if 1 <= c <= n}, reverse=True)
  inp = make_host_inputs(items, seed=98)
  t = {k: torch.from_numpy(v) for k, v in inp.items()}
  best = (None, n)
  for c in cands:
    torch.set_num_threads(c)
    t0 = time.perf_counter()
    rp.decoder(t['amps'], t['harmonic_distribution'], t['f0_hz'],
               t['noise_magnitudes'], n_samples=N_SAMPLES,
               sample_rate=SAMPLE_RATE, window_size=0)
    dt = time.perf_counter() - t0
    if best[0] is None or dt < best[0]:
      best = (dt, c)
  _BEST_THREADS.append(best[1])
  return best[1]


def cpu_reference_throughput(items, repeats=1, threads=None):
  """samples/s of oracle/ref_port_torch.decoder on `items` batch items, on the
  host thread count that serves it best (torchrun exports OMP_NUM_THREADS=1; undo
  that)."""
  import torch
  from oracle import ref_port_torch as rp
  torch.set_num_threads(threads or _pick_cpu_threads(items))
  inp = make_host_inputs(items, seed=99)
  t = {k: torch.from_numpy(v) for k, v in inp.items()}
  best = None
  for _ in range(repeats):
    t0 = time.perf_counter()
    rp.decoder(t['amps'], t['harmonic_distribution'], t['f0_hz'],
               t['noise_magnitudes'], n_samples=N_SAMPLES,
               sample_rate=SAMPLE_RATE, window_size=0)
    dt = time.perf_counter() - t0
    best = dt if best is None else min(best, dt)
  return items * N_SAMPLES / best, best, torch.get_num_threads()


def cpu_c1_throughput(c1):
  """configs[0] (Harmonic only, B=1, 16000 samples, 64 harmonics) on the CPU port."""
  import torch
  from oracle import ref_port_torch as rp
  torch.set_num_threads(max(1, min(8, os.cpu_count() or 1)))
  t = {k: torch.from_numpy(c1[k]) for k in ('amps', 'harmonic_distribution', 'f0_hz')}
  best = None
  for _ in range(5):
    t0 = time.perf_counter()
    a, h = rp.harmonic_controls(t['amps'], t['harmonic_distribution'], t['f0_hz'])
    rp.harmonic_signal(a, h, t['f0_hz'], 16000)
    dt = time.perf_counter() - t0
    best = dt if best is None else min(best, dt)
  return 16000 / best


def run_reference(args):
  rank = int(os.environ.get('RANK', '0'))
  if rank != 0:
    return None  # other ranks exit 0 without work
  import torch
  # bounded sample of the B=256 workload: up to 8 items per step, fewer when the
  # caller asks for many steps, so that warm-up + timed steps stay near 2.5 min
  # (one item costs up to ~0.65 s on this class of host)
  n_calls = args.warmup + args.steps
  items = max(1, min(8, int(150.0 / (0.65 * n_calls))))
  cores = _pick_cpu_threads(items)
  rates, times = [], []
  for i in range(args.warmup + args.steps):
    rate, dt, cores = cpu_reference_throughput(items)
    if i >= args.warmup:
      rates.append(rate)
      times.append(dt)
  value = items * N_SAMPLES * len(times) / sum(times)
  line = {
      'impl': 'reference', 'metric': 'audio samples/sec (Harmonic+FilteredNoise decoder)',
      'value': value, 'unit': 'samples/s', 'n_gpus': args.gpus,
      'steps': args.steps, 'warmup': args.warmup,
      'ms_per_step': 1e3 * sum(times) / len(times), 'higher_is_better': True,
      'scaling': 'weak', 'vs_baseline': None, 'dtype': 'f32', 'data': 'synthetic',
      'config': {'workload': 'ae.gin decoder Harmonic(100)+FilteredNoise(65)+Add, '
                             'N=64000 @16kHz, F=1000 (configs[2] shapes); each step is '
                             'a bounded sample of %d of the 256 batch items - '
                             'throughput is per sample, so it compares directly' % items,
                 'batch_per_step': items, 'batch_per_gpu': BATCH_PER_GPU},
      'cpu_baseline': {'value': value, 'unit': 'samples/s', 'cores': cores,
                       'kind': 'port',
                       'sample': '%d of the 256 batch items per step (torch-CPU '
                                 'op-by-op float32 port of ddsp core/synths, '
                                 'validated against the unmodified reference run '
                                 'on oracle/tf_shim; TensorFlow is not installable '
                                 'here)' % items},
      'e2e': {'value': value, 'unit': 'samples/s', 'h2d_bytes_per_step': 0,
              'd2h_bytes_per_step': 0},
      'gpu_launches': 0,
  }
  return line


# ----------------------------------------------------------------------------
# our arm
# ----------------------------------------------------------------------------
def run_ours(args):
  import torch
  import torch.distributed as dist
  import ddsp_b200
  from ddsp_b200 import _lib, core, host as host_mod, sharding

  world = int(os.environ.get('WORLD_SIZE', '1'))
  rank = int(os.environ.get('RANK', '0'))
  local_rank = int(os.environ.get('LOCAL_RANK', '0'))
  if not torch.cuda.is_available():
    raise SystemExit('bench.py (ours) needs a CUDA device; there is no CPU path.')
  torch.cuda.set_device(local_rank)
  dev = torch.device('cuda', local_rank)
  # Pin this process to the CPUs of the GPU's NUMA node BEFORE any page-locked
  # buffer exists: pinned pages are placed where the allocating thread runs, and on
  # a two-socket 8-GPU host a far-socket buffer halves the host<->device rate.
  numa_node = host_mod.bind_to_device_numa_node(dev)
  if world > 1:
    os.environ.setdefault('MASTER_ADDR', '127.0.0.1')
    import datetime
    dist.init_process_group('nccl', device_id=dev,
                            timeout=datetime.timedelta(seconds=300))
  lib = _lib.load()
  B = args.batch

  def make_group(seed):
    harm = ddsp_b200.Harmonic(n_samples=N_SAMPLES, sample_rate=SAMPLE_RATE)
    noise = ddsp_b200.FilteredNoise(n_samples=N_SAMPLES, window_size=0, seed=seed)
    add = ddsp_b200.Add()
    return harm, noise, ddsp_b200.ProcessorGroup(dag=[
        (harm, ['amps', 'harmonic_distribution', 'f0_hz']),
        (noise, ['noise_magnitudes']),
        (add, ['filtered_noise/signal', 'harmonic/signal'])])

  harm, noise, group = make_group(rank)

  # A ring of distinct input sets larger than 2x L2 so every step reads HBM.
  host = make_host_inputs(B, seed=1234 + rank)
  set_bytes = sum(v.nbytes for v in host.values()) + 4 * B * N_SAMPLES
  n_sets = max(2, -(-2 * L2_BYTES // set_bytes))
  dev_sets = []
  for s in range(n_sets):
    d = {k: torch.from_numpy(v).to(dev) for k, v in host.items()}
    if s:
      d['amps'] = d['amps'] + 0.01 * s   # distinct contents, same statistics
    dev_sets.append(d)
  pinned = {k: torch.from_numpy(v).pin_memory() for k, v in host.items()}
  h2d_bytes = sum(v.numel() * 4 for v in pinned.values())
  out_host = torch.empty((B, N_SAMPLES), dtype=torch.float32).pin_memory()
  d2h_bytes = out_host.numel() * 4

  def barrier(collective=True):
    torch.cuda.synchronize()
    if world > 1 and collective:
      dist.barrier()
      torch.cuda.synchronize()

  def timed(fn, steps, warmup, collective=True, mark=None):
    """CUDA-event time of `steps` calls; `collective=False` for rank-local
    measurements (no barrier / all-reduce: the other ranks are not here)."""
    for i in range(warmup):
      fn(i)
    barrier(collective)
    e0 = torch.cuda.Event(enable_timing=True)
    e1 = torch.cuda.Event(enable_timing=True)
    if mark is not None:
      mark.mark_timed(0)
    e0.record()
    for i in range(steps):
      fn(warmup + i)
    e1.record()
    barrier(collective)
    if mark is not None:
      mark.mark_timed(1)
    ms = e0.elapsed_time(e1)
    if world > 1 and collective:
      tms = torch.tensor([ms], device=dev)
      dist.all_reduce(tms, op=dist.ReduceOp.MAX)
      ms = float(tms.item())
    return ms

  # -- value: whole decoder step, inputs resident in HBM ----------------------
  # The step is the public call `group(inputs)` (ProcessorGroup.__call__ over raw
  # network outputs).  It is captured once per input set in a CUDA graph
  # (torch.cuda.graph around that same call, the route a serving loop would take)
  # so that the timed region replays kernels back to back with no Python, ctypes
  # or allocator work between them; --graph 0 times the eager call instead.
  graph_note = 'eager ProcessorGroup.__call__'
  launches_per_step = None
  graphs, graph_out = [], []
  if args.graph:
    try:
      side = torch.cuda.Stream()
      side.wait_stream(torch.cuda.current_stream())
      with torch.cuda.stream(side):
        for d in dev_sets:
          group(d)
      torch.cuda.current_stream().wait_stream(side)
      torch.cuda.synchronize()
      for d in dev_sets:
        g = torch.cuda.CUDAGraph()
        c0 = lib.ddsp_b200_launch_count()
        with torch.cuda.graph(g, stream=side):
          o = group(d)
        launches_per_step = int(lib.ddsp_b200_launch_count() - c0)
        graphs.append(g)
        graph_out.append(o)
      torch.cuda.synchronize()
      graph_note = ('CUDA graph replay of ProcessorGroup.__call__ (one graph per '
                    'input set, %d kernel nodes each)' % launches_per_step)
    except Exception as e:  # pylint: disable=broad-except
      graphs, graph_out = [], []
      graph_note = 'eager ProcessorGroup.__call__ (graph capture failed: %r)' % (e,)
      torch.cuda.synchronize()

  eager_out = {}
  if graphs:
    def step_resident(i):
      graphs[i % n_sets].replay()
  else:
    def step_resident(i):
      eager_out['audio'] = group(dev_sets[i % n_sets])

  sampler = ClockSampler(local_rank)
  if rank == 0:
    sampler.start()
  c0 = lib.ddsp_b200_launch_count()
  ms_total = timed(step_resident, args.steps, args.warmup,
                   mark=sampler if rank == 0 else None)
  if graphs:
    launches_timed = launches_per_step * args.steps
  else:
    launches = lib.ddsp_b200_launch_count() - c0
    launches_timed = launches * args.steps // (args.steps + args.warmup)
  ms_per_step = ms_total / args.steps
  value = world * B * N_SAMPLES / (ms_per_step * 1e-3)
  if args.dump_outputs and rank == 0:
    # the audio of the last timed step (rank 0's shard when sharded)
    dump_outputs(args.dump_outputs, {'audio': graph_out[
        (args.warmup + args.steps - 1) % n_sets] if graphs else eager_out['audio']})

  # -- e2e: host buffers in, host audio out, copies inside the timed region ---
  # The public host-buffer call: HostDecoder = ProcessorGroup over pinned host
  # arrays through ddsp_b200_decoder_forward_host (chunked copy / compute / copy
  # pipeline on three streams).  Every step copies all inputs H2D and the whole
  # audio D2H and waits for it.
  def step_e2e_with(dec):
    return lambda i: dec(pinned, out=out_host, sync=True)   # the caller reads it

  # The PCIe link and copy engines need ~50 ms of traffic to reach full speed
  # after idling (first copies of a run move at about half rate): warm them up,
  # then pick the chunk count on this box (rank-local, short) before timing.
  cand = [args.chunks] if args.chunks > 0 else ([2, 3, 4] if B <= 64 else [4, 6, 8])
  decs = {c: ddsp_b200.HostDecoder(group, max_batch=B, n_frames=N_FRAMES,
                                   n_harmonics=N_HARM, n_bands=N_BANDS, n_chunks=c)
          for c in cand}
  t_end = time.perf_counter() + 0.15
  while time.perf_counter() < t_end:
    decs[cand[0]](pinned, out=out_host, sync=True)
  best_c, best_ms = cand[0], None
  for c in cand:
    ms = timed(step_e2e_with(decs[c]), 8, 2, collective=False) / 8
    if best_ms is None or ms < best_ms:
      best_c, best_ms = c, ms
  host_dec = decs[best_c]
  e2e_steps = max(min(args.steps, 30), 10)
  ms_e2e = timed(step_e2e_with(host_dec), e2e_steps, 3) / e2e_steps
  e2e_value = world * B * N_SAMPLES / (ms_e2e * 1e-3)

  # link floor of the same round trip: the H2D bytes alone, pinned -> device,
  # one copy per tensor (nothing else on the link), to say how far e2e is from it
  def step_h2d_only(i):
    for k, v in pinned.items():
      dev_sets[0][k].copy_(v, non_blocking=True)
  ms_h2d_floor = timed(step_h2d_only, 10, 3, collective=False) / 10

  # the same round trip without the pipeline (4 copies, one call, one copy)
  def step_e2e_serial(i):
    feats = {k: v.to(dev, non_blocking=True) for k, v in pinned.items()}
    audio = group(feats)
    out_host.copy_(audio, non_blocking=True)
    torch.cuda.current_stream().synchronize()

  ms_e2e_serial = timed(step_e2e_serial, 5, 2, collective=False) / 5
  for d in decs.values():
    d.close()

  # -- optional reassembly: NCCL all-gather of the [B, N] audio shards ---------
  all_gather = None
  if world > 1:
    shard = graph_out[0] if graph_out else group(dev_sets[0])
    def step_gather(i):
      sharding.all_gather_audio(shard, B * world)
    ms_ag = timed(step_gather, 10, 3) / 10
    all_gather = {'ms': ms_ag, 'bytes_out_per_rank': 4 * B * world * N_SAMPLES,
                  'algbw_GBps': 4 * B * world * N_SAMPLES / (ms_ag * 1e-3) / 1e9,
                  'backend': 'nccl all_gather_into_tensor over NVLink, off the '
                             'synthesis path (not in ms_per_step)'}

  # -- per-kernel durations for the roofline (rank 0 reports) -----------------
  ctl = []
  for d in dev_sets:
    hc = harm.get_controls(d['amps'], d['harmonic_distribution'], d['f0_hz'])
    nc = noise.get_controls(d['noise_magnitudes'])
    ctl.append((hc, nc))
  audio_bufs = [torch.empty((B, N_SAMPLES), dtype=torch.float32, device=dev)
                for _ in range(n_sets)]

  # single kernels through the C ABI directly (ctypes, pointers resolved once):
  # the launches are then cheaper than the kernels, so a group of them runs back
  # to back on the GPU and the event pair around the group carries no idle time
  st_ptr = torch.cuda.current_stream().cuda_stream
  hargs = [(c[0]['f0_hz'].data_ptr(), c[0]['amplitudes'].data_ptr(),
            c[0]['harmonic_distribution'].data_ptr()) for c in ctl]
  nargs = [c[1]['magnitudes'].data_ptr() for c in ctl]
  optr = [a.data_ptr() for a in audio_bufs]
  amp_method = core.AMP_METHODS[harm.amp_resample_method]

  def harm_only(i):
    j = i % n_sets
    _lib.check(lib.ddsp_b200_harmonic_forward(
        hargs[j][0], hargs[j][1], hargs[j][2], optr[j], B, N_FRAMES, N_HARM,
        N_SAMPLES, float(SAMPLE_RATE), amp_method, _lib.PHASE_RECURRENCE, 0, st_ptr))

  def noise_only(i):
    j = i % n_sets
    _lib.check(lib.ddsp_b200_filtered_noise_forward(
        nargs[j], None, 7, i, optr[j], B, N_FRAMES, N_BANDS, N_SAMPLES, 0, 1, None, 0,
        st_ptr))

  def controls_only(i):
    d = dev_sets[i % n_sets]
    harm.get_controls(d['amps'], d['harmonic_distribution'], d['f0_hz'])
    noise.get_controls(d['noise_magnitudes'])

  def kernel_ms(fn, steps=10, warmup=5, group=8):
    """Mean GPU duration of ONE call: event pairs around groups of `group`
    back-to-back launches (distinct input sets), divided by the group size."""
    for i in range(warmup):
      fn(i)
    torch.cuda.synchronize()
    pairs = []
    k = warmup
    for _ in range(steps):
      e0 = torch.cuda.Event(enable_timing=True)
      e1 = torch.cuda.Event(enable_timing=True)
      e0.record()
      for _ in range(group):
        fn(k)
        k += 1
      e1.record()
      pairs.append((e0, e1))
    torch.cuda.synchronize()
    return sum(a.elapsed_time(b) for a, b in pairs) / (steps * group)

  ms_harm = kernel_ms(harm_only)
  ms_noise = kernel_ms(noise_only)
  ms_ctl = kernel_ms(controls_only, group=2)
  clocks = sampler.stop() if rank == 0 else None
  del ctl, audio_bufs

  # -- the other configs, for context (rank 0, rank-local) ---------------------
  extra = {}
  if args.extra and rank == 0:
    try:
      # configs[1]: the same decoder at B=32
      B2 = 32
      h2 = make_host_inputs(B2, seed=77)
      sets2 = []
      for s in range(8):     # 8 x 37.8 MB > 2x L2
        d = {k: torch.from_numpy(v).to(dev) for k, v in h2.items()}
        d['amps'] = d['amps'] + 0.01 * s
        sets2.append(d)
      ms2 = timed(lambda i: group(sets2[i % 8]), 40, 8, collective=False) / 40
      extra['c2_batch32_samples_per_s'] = B2 * N_SAMPLES / (ms2 * 1e-3)
      extra['c2_ms_per_step'] = ms2
      extra['c2_decoder_fused_frac'] = (BYTES_DECODER_FUSED * B2 / (ms2 * 1e-3) / 1e9
                                        ) / _measured_peaks()[0]
      del sets2
    except Exception as e:  # pylint: disable=broad-except
      extra['c2_error'] = repr(e)
    try:
      # SURVEY 8(d)'s worst case for the compute bound: f0 = 60 Hz (+-3 % vibrato), so
      # all 100 harmonics stay below Nyquist in every frame - the same decoder, B=256
      from tests.util import synth_inputs as _si
      hw = _si(B, N_FRAMES, N_HARM, N_BANDS, N_SAMPLES, seed=91, f0_lo=60.0, f0_hi=60.0)
      setsw = []
      for s in range(2):     # 2 x 236 MB > 2x L2
        d = {k: torch.from_numpy(hw[k]).to(dev) for k in
             ('amps', 'harmonic_distribution', 'f0_hz', 'noise_magnitudes')}
        d['amps'] = d['amps'] + 0.01 * s
        setsw.append(d)
      msw = timed(lambda i: group(setsw[i % 2]), 20, 4, collective=False) / 20
      extra['worst_case_f0_60hz_all_harmonics_live_ms_per_step'] = msw
      extra['worst_case_samples_per_s'] = B * N_SAMPLES / (msw * 1e-3)
      del setsw, hw
    except Exception as e:  # pylint: disable=broad-except
      extra['worst_case_error'] = repr(e)
    try:
      # configs[0]: Harmonic only, B=1, 16000 samples, 64 harmonics, 250 frames
      from tests.util import synth_inputs
      c1 = synth_inputs(1, 250, 64, 65, 16000, seed=5)
      h1 = ddsp_b200.Harmonic(n_samples=16000, sample_rate=SAMPLE_RATE)
      a1 = [torch.from_numpy(c1[k]).to(dev) for k in
            ('amps', 'harmonic_distribution', 'f0_hz')]
      ms1 = timed(lambda i: h1(*a1), 50, 10, collective=False) / 50
      extra['c1_harmonic_b1_ms_per_step'] = ms1
      extra['c1_samples_per_s'] = 16000 / (ms1 * 1e-3)
      if not args.no_cpu_baseline and world == 1:
        extra['c1_cpu_port_samples_per_s'] = cpu_c1_throughput(c1)
    except Exception as e:  # pylint: disable=broad-except
      extra['c1_error'] = repr(e)
    try:
      # configs[3]: decoder forward + backward through the multi-scale
      # SpectralLoss (ae.gin:39-41), B=128 - context only, not the headline.
      from ddsp_b200 import autograd as ag
      from ddsp_b200 import losses
      B4 = 128
      h4 = make_host_inputs(B4, seed=55)
      d4 = {k: torch.from_numpy(v).to(dev) for k, v in h4.items()}
      for k in ('amps', 'harmonic_distribution', 'noise_magnitudes'):
        d4[k].requires_grad_(True)
      target = 0.1 * torch.randn(B4, N_SAMPLES, device=dev)
      loss_obj = losses.SpectralLoss(mag_weight=1.0, logmag_weight=1.0)

      def c4_step(i):
        for k in ('amps', 'harmonic_distribution', 'noise_magnitudes'):
          d4[k].grad = None
        audio = ag.decoder_train(d4['amps'], d4['harmonic_distribution'],
                                 d4['f0_hz'], d4['noise_magnitudes'],
                                 n_samples=N_SAMPLES, window_size=0, seed=1, offset=i)
        loss_obj(target, audio).backward()

      ms4 = timed(c4_step, 5, 2, collective=False) / 5
      extra['c4_fwd_bwd_spectral_loss_b128_ms_per_step'] = ms4
      extra['c4_samples_per_s'] = B4 * N_SAMPLES / (ms4 * 1e-3)
      del d4
    except Exception as e:  # pylint: disable=broad-except
      extra['c4_error'] = repr(e)

  if rank != 0:
    if world > 1:
      dist.barrier()
      dist.destroy_process_group()
    return None

  peak, peak_src = _measured_peaks()
  # DRAM traffic of the same kernels from one ncu --set full capture of this
  # workload (profiles/*traffic*.json; null for any other batch size)
  traffic = {}
  for name in ('r02_traffic_b256.json', 'r01_traffic_b32.json'):
    tpath = os.path.join(ROOT, 'profiles', name)
    if os.path.exists(tpath):
      with open(tpath) as f:
        traffic = {k: v for k, v in json.load(f).items() if v.get('batch') == B}
      if traffic:
        break
  dom_is_harm = ms_harm >= ms_noise
  dom_ms = ms_harm if dom_is_harm else ms_noise
  dom_bytes = (BYTES_HARMONIC if dom_is_harm else BYTES_NOISE + 4 * N_SAMPLES) * B
  achieved = dom_bytes / (dom_ms * 1e-3) / 1e9
  roofline = {
      'bound': 'hbm', 'kernel': 'harmonic_forward' if dom_is_harm else
               'filtered_noise_forward(accumulate)',
      'achieved': achieved, 'peak': peak, 'unit': 'GB/s',
      'frac': achieved / peak, 'peak_source': peak_src + ' (MEASURED_PEAKS.json hbm_gbs)',
      'traffic': (traffic.get('harmonic_forward' if dom_is_harm else
                              'filtered_noise_forward') or {}).get('traffic'),
      'traffic_source': (traffic.get('harmonic_forward' if dom_is_harm else
                                     'filtered_noise_forward') or {}).get('source'),
      'algorithmic_bytes_per_launch': dom_bytes,
      'kernel_ms': {'harmonic_forward': ms_harm,
                    'filtered_noise_forward': ms_noise,
                    'controls(2 kernels)': ms_ctl},
      'decoder_fused_frac': (BYTES_DECODER_FUSED * B / (ms_per_step * 1e-3) / 1e9) / peak,
  }

  # -- cpu baseline: bounded sample of the same workload on the host cores ----
  cpu = None
  if not args.no_cpu_baseline and world == 1:
    items = 8
    rate, dt, cores = cpu_reference_throughput(items, repeats=2)
    cpu = {'value': rate, 'unit': 'samples/s', 'cores': cores, 'kind': 'port',
           'sample': '%d of the %d batch items (torch-CPU op-by-op float32 port '
                     'of ddsp core/synths, validated against the unmodified '
                     'reference run on oracle/tf_shim; %.2f s)' % (items, B, dt)}

  cfg_name = ('configs[4]: decoder batch %d sharded over %d B200 (%d per GPU)'
              % (B * world, world, B)) if world > 1 else (
                  'configs[2]: decoder batch %d on one B200' % B)
  line = {
      'metric': 'audio samples/sec (Harmonic+FilteredNoise decoder)',
      'value': value, 'unit': 'samples/s', 'n_gpus': world,
      'steps': args.steps, 'warmup': args.warmup, 'ms_per_step': ms_per_step,
      'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None,
      'dtype': 'f32', 'data': 'synthetic',
      'config': {
          'workload': cfg_name + ' - ae.gin Harmonic(100)+FilteredNoise(65)+Add via '
                      'ProcessorGroup (get_controls + get_signal), N=64000 @16kHz, '
                      'F=1000',
          'batch_per_gpu': B, 'global_batch': B * world,
          'step': graph_note,
          'l2_policy': 'ring of %d distinct input/output sets (%.0f MB > 2x L2)'
                       % (n_sets, n_sets * set_bytes / 1e6),
          'noise': 'in-kernel Philox4x32-10', 'parallelism': 'batch-sharded replicas, no collective',
          'numa_node': numa_node,
      },
      'e2e': {'value': e2e_value, 'unit': 'samples/s', 'ms_per_step': ms_e2e,
              'h2d_bytes_per_step': h2d_bytes * world,
              'd2h_bytes_per_step': d2h_bytes * world,
              'api': 'ddsp_b200.HostDecoder(group)(pinned host inputs) -> pinned '
                     'host audio, %d chunks on 3 streams' % best_c,
              'ms_per_step_unpipelined': ms_e2e_serial,
              'ms_h2d_alone': ms_h2d_floor,
              'over_link_floor': ms_e2e / ms_h2d_floor},
      'gpu_launches': int(launches_timed),
      'clocks': clocks,
      'roofline': roofline,
      'cpu_baseline': cpu,
  }
  if all_gather is not None:
    line['all_gather'] = all_gather
  line.update(extra)
  if world > 1:
    dist.barrier()
    dist.destroy_process_group()
  return line


# ----------------------------------------------------------------------------
# configs[3]: decoder forward + backward through the multi-scale SpectralLoss
# ----------------------------------------------------------------------------
C4_BATCH = 128


def c4_cpu_throughput(items, repeats=1):
  """samples/s of oracle/ref_port_torch.train_step on `items` batch items."""
  import torch
  from oracle import ref_port_torch as rp
  torch.set_num_threads(_pick_cpu_threads(min(items, 8)))
  inp = make_host_inputs(items, seed=97)
  t = {k: torch.from_numpy(v) for k, v in inp.items()}
  target = 0.1 * torch.randn(items, N_SAMPLES)
  best = None
  for _ in range(repeats):
    t0 = time.perf_counter()
    rp.train_step(t['amps'], t['harmonic_distribution'], t['f0_hz'],
                  t['noise_magnitudes'], target, n_samples=N_SAMPLES)
    dt = time.perf_counter() - t0
    best = dt if best is None else min(best, dt)
  return items * N_SAMPLES / best, best, torch.get_num_threads()


def run_c4_reference(args):
  if int(os.environ.get('RANK', '0')) != 0:
    return None
  n_calls = args.warmup + args.steps
  items = max(1, min(4, int(150.0 / (2.5 * n_calls))))
  times = []
  cores = 0
  for i in range(n_calls):
    _, dt, cores = c4_cpu_throughput(items)
    if i >= args.warmup:
      times.append(dt)
  value = items * N_SAMPLES * len(times) / sum(times)
  return {
      'impl': 'reference', 'metric': 'audio samples/sec (decoder forward+backward '
      'through multi-scale SpectralLoss)', 'value': value, 'unit': 'samples/s',
      'n_gpus': args.gpus, 'steps': args.steps, 'warmup': args.warmup,
      'ms_per_step': 1e3 * sum(times) / len(times), 'higher_is_better': True,
      'scaling': 'weak', 'vs_baseline': None, 'dtype': 'f32', 'data': 'synthetic',
      'config': {'workload': 'configs[3]: decoder fwd+bwd through SpectralLoss (FFT '
                             '64-2048), N=64000; each step is a bounded sample of %d of '
                             'the 128 batch items' % items, 'batch_per_step': items},
      'cpu_baseline': {'value': value, 'unit': 'samples/s', 'cores': cores, 'kind': 'port',
                       'sample': '%d of the 128 batch items per step (torch-CPU port, '
                                 'torch autograd for the backward)' % items},
      'e2e': {'value': value, 'unit': 'samples/s', 'h2d_bytes_per_step': 0,
              'd2h_bytes_per_step': 0},
      'gpu_launches': 0}


def run_c4(args):
  """BASELINE.json configs[3] as its own bench line: `--config c4`."""
  import torch
  import torch.distributed as dist
  from ddsp_b200 import _lib, autograd as ag, host as host_mod, losses, spectral_ops
  world = int(os.environ.get('WORLD_SIZE', '1'))
  rank = int(os.environ.get('RANK', '0'))
  local_rank = int(os.environ.get('LOCAL_RANK', '0'))
  if not torch.cuda.is_available():
    raise SystemExit('bench.py (ours) needs a CUDA device; there is no CPU path.')
  torch.cuda.set_device(local_rank)
  dev = torch.device('cuda', local_rank)
  host_mod.bind_to_device_numa_node(dev)
  if world > 1:
    os.environ.setdefault('MASTER_ADDR', '127.0.0.1')
    import datetime
    dist.init_process_group('nccl', device_id=dev, timeout=datetime.timedelta(seconds=300))
  lib = _lib.load()
  B = C4_BATCH
  keys = ('amps', 'harmonic_distribution', 'f0_hz', 'noise_magnitudes')
  grad_keys = ('amps', 'harmonic_distribution', 'noise_magnitudes')
  host = make_host_inputs(B, seed=55 + rank)
  sets = []
  for s in range(3):                      # 3 x 151 MB of inputs + targets > 2x L2
    d = {k: torch.from_numpy(host[k]).to(dev) for k in keys}
    if s:
      d['amps'] = d['amps'] + 0.01 * s
    for k in grad_keys:
      d[k].requires_grad_(True)
    d['target'] = 0.1 * torch.randn(B, N_SAMPLES, device=dev)
    sets.append(d)
  pinned = {k: torch.from_numpy(host[k]).pin_memory() for k in keys}
  pinned['target'] = (0.1 * torch.randn(B, N_SAMPLES)).pin_memory()
  h2d_bytes = sum(v.numel() * 4 for v in pinned.values())
  loss_obj = losses.SpectralLoss(mag_weight=1.0, logmag_weight=1.0)
  last = {}

  def step(i, d=None):
    d = sets[i % len(sets)] if d is None else d
    for k in grad_keys:
      d[k].grad = None
    audio = ag.decoder_train(d['amps'], d['harmonic_distribution'], d['f0_hz'],
                             d['noise_magnitudes'], n_samples=N_SAMPLES, window_size=0,
                             seed=1 + rank, offset=i)
    loss = loss_obj(d['target'], audio)
    loss.backward()
    last['loss'] = loss
    return loss

  def barrier():
    torch.cuda.synchronize()
    if world > 1:
      dist.barrier()
      torch.cuda.synchronize()

  def timed(fn, steps, warmup):
    for i in range(warmup):
      fn(i)
    barrier()
    e0 = torch.cuda.Event(enable_timing=True)
    e1 = torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(steps):
      fn(warmup + i)
    e1.record()
    barrier()
    ms = e0.elapsed_time(e1)
    if world > 1:
      t = torch.tensor([ms], device=dev)
      dist.all_reduce(t, op=dist.ReduceOp.MAX)
      ms = float(t.item())
    return ms

  sampler = ClockSampler(local_rank)
  if rank == 0:
    sampler.start()
  c0 = lib.ddsp_b200_launch_count()
  sampler.mark_timed(0)
  ms_step = timed(step, args.steps, args.warmup) / args.steps
  sampler.mark_timed(1)
  if args.dump_outputs and rank == 0:
    # loss and input gradients of the last timed step (before the graph capture
    # below overwrites the gradients)
    d = sets[(args.warmup + args.steps - 1) % len(sets)]
    dump_outputs(args.dump_outputs, dict(
        loss=last['loss'], **{'grad_' + k: d[k].grad for k in grad_keys}))
  launches = (lib.ddsp_b200_launch_count() - c0) * args.steps // (args.steps + args.warmup)
  value = world * B * N_SAMPLES / (ms_step * 1e-3)

  # the same step replayed from CUDA graphs (whole forward + backward captured, one
  # graph per input set; each graph keeps the Philox offset it was captured with, so
  # the noise repeats every len(sets) steps - reported next to the eager number, not
  # instead of it): what is left when the 64 launches cost no host time
  ms_graph, graph_err = None, None
  try:
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
      for i in range(len(sets)):
        step(i)
    torch.cuda.current_stream().wait_stream(side)
    torch.cuda.synchronize()
    graphs = []
    for i, d in enumerate(sets):
      for k in grad_keys:
        d[k].grad = None
      g = torch.cuda.CUDAGraph()
      with torch.cuda.graph(g, stream=side):
        audio = ag.decoder_train(d['amps'], d['harmonic_distribution'], d['f0_hz'],
                                 d['noise_magnitudes'], n_samples=N_SAMPLES,
                                 window_size=0, seed=1 + rank, offset=1000 + i)
        loss_obj(d['target'], audio).backward()
      graphs.append(g)
    torch.cuda.synchronize()
    ms_graph = timed(lambda i: graphs[i % len(graphs)].replay(), args.steps,
                     args.warmup) / args.steps
    del graphs
  except Exception as e:  # pylint: disable=broad-except
    graph_err = repr(e)[:300]
    torch.cuda.synchronize()

  # e2e: host network outputs + target in, loss value out (gradients stay on the GPU)
  loss_host = torch.empty((), dtype=torch.float32).pin_memory()

  def step_e2e(i):
    d = {k: pinned[k].to(dev, non_blocking=True) for k in pinned}
    for k in grad_keys:
      d[k].requires_grad_(True)
    loss = step(i, d)
    loss_host.copy_(loss.detach(), non_blocking=True)
    torch.cuda.current_stream().synchronize()

  e2e_steps = max(5, min(args.steps, 20))
  ms_e2e = timed(step_e2e, e2e_steps, 3) / e2e_steps

  # dominant kernel of the step: the one-pass L1 magnitude / log-magnitude kernel
  # (18 launches per step, the largest share of the GPU time); timed alone on the
  # 2048-point STFTs, algorithmic bytes = two complex spectra in, one out
  size = 2048
  xt = spectral_ops.stft_cuda(sets[0]['target'], size).contiguous()
  xvs = [spectral_ops.stft_cuda(sets[i]['target'] * (1.0 + i), size).contiguous()
         for i in range(3)]
  sums = torch.zeros(2, dtype=torch.float64, device=dev)
  m = xt.numel()
  st_ptr = torch.cuda.current_stream().cuda_stream

  def l1_only(i):
    x = xvs[i % 3]
    _lib.check(lib.ddsp_b200_spectral_l1(xt.data_ptr(), x.data_ptr(), x.data_ptr(),
                                         sums.data_ptr(), m, 1.0, 1.0, xt.shape[-1],
                                         size, st_ptr))
  for i in range(5):
    l1_only(i)
  torch.cuda.synchronize()
  e0 = torch.cuda.Event(enable_timing=True)
  e1 = torch.cuda.Event(enable_timing=True)
  e0.record()
  for i in range(24):
    l1_only(i)
  e1.record()
  torch.cuda.synchronize()
  ms_l1 = e0.elapsed_time(e1) / 24
  clocks = sampler.stop() if rank == 0 else None
  if rank != 0:
    if world > 1:
      dist.barrier()
      dist.destroy_process_group()
    return None
  peak, peak_src = _measured_peaks()
  l1_bytes = 3 * 8 * m
  cpu = None
  if not args.no_cpu_baseline and world == 1:
    rate, dt, cores = c4_cpu_throughput(2)
    cpu = {'value': rate, 'unit': 'samples/s', 'cores': cores, 'kind': 'port',
           'sample': '2 of the %d batch items, forward + backward (torch-CPU port of '
                     'ddsp core/synths/losses, torch autograd; %.2f s)' % (B, dt)}
  line = {
      'metric': 'audio samples/sec (decoder forward+backward through multi-scale '
                'SpectralLoss)',
      'value': value, 'unit': 'samples/s', 'n_gpus': world, 'steps': args.steps,
      'warmup': args.warmup, 'ms_per_step': ms_step, 'higher_is_better': True,
      'scaling': 'weak', 'vs_baseline': None, 'dtype': 'f32', 'data': 'synthetic',
      'config': {'workload': 'configs[3]: ae.gin decoder forward + backward through '
                             'SpectralLoss (L1 mag + log-mag, FFT 2048..64), batch %d per '
                             'GPU, N=64000 @16kHz; gradients to amps, '
                             'harmonic_distribution, noise_magnitudes' % B,
                 'batch_per_gpu': B, 'global_batch': B * world,
                 'step': 'ddsp_b200.autograd.decoder_train (DecoderFn) + '
                         'losses.SpectralLoss (SpectralLossFn), eager autograd',
                 'l2_policy': 'ring of 3 distinct input / target sets',
                 'ffts': 'cuFFT through torch.fft (library call, not a hand kernel)'},
      'e2e': {'value': world * B * N_SAMPLES / (ms_e2e * 1e-3), 'unit': 'samples/s',
              'ms_per_step': ms_e2e, 'h2d_bytes_per_step': h2d_bytes * world,
              'd2h_bytes_per_step': 4 * world,
              'api': 'pinned host network outputs + target -> device, decoder_train, '
                     'SpectralLoss, backward; the loss value is read back'},
      'gpu_launches': int(launches), 'clocks': clocks,
      'roofline': {'bound': 'hbm', 'kernel': 'spectral_l1 (2048-point STFTs)',
                   'achieved': l1_bytes / (ms_l1 * 1e-3) / 1e9, 'peak': peak,
                   'unit': 'GB/s', 'frac': l1_bytes / (ms_l1 * 1e-3) / 1e9 / peak,
                   'peak_source': peak_src + ' (MEASURED_PEAKS.json hbm_gbs)',
                   'traffic': None, 'algorithmic_bytes_per_launch': l1_bytes,
                   'kernel_ms': {'spectral_l1': ms_l1}},
      'cpu_baseline': cpu,
      'loss': float(last['loss'].detach()),
      'ms_per_step_graph_replay': ms_graph,
      'graph_replay_note': graph_err or ('whole fwd+bwd step captured per input set; '
                                         'Philox offset fixed per graph'),
  }
  if world > 1:
    dist.barrier()
    dist.destroy_process_group()
  return line


def main():
  # Keep stdout clean for the ONE JSON line: NCCL (and anything else native)
  # writes its banners to fd 1, so run with fd 1 pointed at stderr and restore
  # it only for the final print.
  sys.stdout.flush()
  saved_stdout = os.dup(1)
  os.dup2(2, 1)
  try:
    line = _main()
  finally:
    sys.stdout.flush()
    os.dup2(saved_stdout, 1)
    os.close(saved_stdout)
  if line is not None:
    print(json.dumps(line), flush=True)


def _main():
  ap = argparse.ArgumentParser()
  ap.add_argument('--gpus', type=int, default=1)
  ap.add_argument('--steps', type=int, default=None,
                  help='timed steps (default 50; 10 with --config c4)')
  ap.add_argument('--warmup', type=int, default=10)
  ap.add_argument('--impl', default='ours', choices=['ours', 'reference'])
  ap.add_argument('--batch', type=int, default=BATCH_PER_GPU,
                  help='batch items per GPU (configs[2] / configs[4] = 256)')
  ap.add_argument('--no-cpu-baseline', action='store_true')
  ap.add_argument('--chunks', type=int, default=0,
                  help='chunks of the host-buffer (e2e) pipeline; 0 = pick among 2/3/4')
  ap.add_argument('--extra', type=int, default=1,
                  help='also time configs[1] / [0] / [3] on rank 0')
  ap.add_argument('--graph', type=int, default=1,
                  help='replay the step from a CUDA graph (0 = eager call)')
  ap.add_argument('--config', default='decoder', choices=['decoder', 'c4'],
                  help="'decoder' (default): configs[2] / configs[4]; 'c4': configs[3], "
                       'forward + backward through SpectralLoss, batch 128 per GPU')
  ap.add_argument('--dump-outputs', metavar='DIR', default=None,
                  help='after the timed steps, write what the last one computed as '
                       'DIR/<name>.npy (decoder: audio; c4: loss and input gradients)')
  args = ap.parse_args()
  if args.steps is None:
    args.steps = 10 if args.config == 'c4' else 50
  if args.steps < 1:
    ap.error('--steps must be at least 1')
  if args.dump_outputs and args.impl != 'ours':
    ap.error('--dump-outputs writes the outputs of --impl ours')
  args.warmup = max(args.warmup, 3)
  if args.config == 'c4':
    return run_c4_reference(args) if args.impl == 'reference' else run_c4(args)
  if args.impl == 'reference':
    return run_reference(args)
  return run_ours(args)


if __name__ == '__main__':
  main()
