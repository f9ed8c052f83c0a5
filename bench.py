#!/usr/bin/env python3
"""Headline benchmark: GCell/s of a SODA stencil program on B200s.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference]
                    [--dump-outputs DIR]

Workload (BASELINE.json configs[1]): jacobi2d, float32, 16384 x 16384,
iterate 64.  One "step" is one complete run of the program: 64 iterations
over the whole grid = 1.718e10 cell updates.  With N > 1 GPUs (launched by
torch.distributed.run, one process per GPU) every rank owns a 16384-row slab
of a 16384 x (16384 N) grid; after every temporally blocked launch its face
rows are copied into the neighbours' ghost rows (peer-mapped memory over
NVLink, copy engine + stream flags; soda/cuda_slab.py) while the interior is
computed: weak scaling, value = all ranks' cell updates / s.

What is timed
  value     inputs resident in HBM, CUDA events around K steps on the launch
            stream, max over ranks.
  e2e       the same workload through the reference-facing C ABI entry
            (soda_cuda_run, the generic form of `<app>(buffer_t*...)`) with
            pinned HOST buffers: H2D of the input and D2H of the output are
            inside the timed region.  With N > 1 it is ONE call on the global
            16384 x (16384 N) grid with "devices=0,..,N-1": the runtime cuts
            the host arrays into one slab per device (rank 0 makes the call,
            the other ranks wait).  `copy_ceiling` is the same bytes moved by
            plain cudaMemcpyAsync in both directions at once with no compute:
            what this machine's host<->device path allows at N devices.
  extra     BASELINE configs 1, 3, 4 and 5, device-resident, outside
            ms_per_step: blur 2000 x 1000 (launch-bound: one 12 us kernel),
            sobel2d / denoise2d 32768^2 (N = 1), heat3d /
            jacobi3d 1024^3 x 32 and denoise3d 768^3 x 16 applications cut
            into N slabs (STRONG scaling), each with its recomputed roofline
            fraction; with N > 1 also a small sharded run compared bit for
            bit with the same run on one GPU.
  roofline  the streaming kernel: algorithmic bytes per launch (8 B x cells:
            each input cell read once, each output cell written once;
            SURVEY.md 8d) / mean launch time, against the measured HBM copy
            bandwidth in MEASURED_PEAKS.json.
  cpu_baseline  the CPU oracle (a port of the reference's golden loop, built
            with the pinned flags) on the host's cores, on a bounded sample.

--impl reference times that CPU port alone with all host threads (the
reference has no executable of its own for this path: SURVEY.md 0.1).
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path[:0] = [os.path.join(ROOT, 'soda-compiler_b200')]

WORKLOAD = dict(program='jacobi2d', iterate=64, dims=(16384, 16384))
BYTES_PER_CELL = 8          # float32 in + float32 out (SURVEY.md 8d)
CPU_SAMPLE_ITERATE = 64     # iterations timed on the CPU: the whole workload
CPU_SINGLE_THREAD_ITERATE = 4   # ... and on one thread (SURVEY.md 8d asks for both)
HBM_FALLBACK_GBS = 6650.0   # B200_PROFILING.md, if MEASURED_PEAKS.json absent


def measured_hbm_gbs():
  try:
    with open(os.path.join(ROOT, 'MEASURED_PEAKS.json')) as handle:
      return float(json.load(handle)['hbm_gbs']), 'measured'
  except (OSError, KeyError, ValueError):
    return HBM_FALLBACK_GBS, 'fallback'


def load_stencil(iterate=None):
  from soda import core
  path = os.path.join(ROOT, 'benchmarks', WORKLOAD['program'] + '.soda')
  return core.Stencil.from_file(
      path, iterate=WORKLOAD['iterate'] if iterate is None else iterate)


class ClockSampler:
  """SM clock and throttle reasons sampled WHILE the timed region runs: NVML
  polled every 2 ms from a thread (nvidia-smi's fastest loop is slower than
  the whole timed region); `nvidia-smi` once as a fallback."""
  REASONS = (('hw_slowdown', 0x8), ('hw_thermal_slowdown', 0x40),
             ('sw_thermal_slowdown', 0x20), ('sw_power_cap', 0x4))

  def __init__(self, index):
    self.index = index
    self.clocks, self.masks, self.max_mhz = [], 0, None
    self._stop = threading.Event()
    self._thread = None
    try:
      import pynvml
      pynvml.nvmlInit()
      visible = os.environ.get('CUDA_VISIBLE_DEVICES')
      if visible:
        index = int(visible.split(',')[index])
      self._nvml = pynvml
      self._handle = pynvml.nvmlDeviceGetHandleByIndex(index)
      self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(
          self._handle, pynvml.NVML_CLOCK_SM)
      self._thread = threading.Thread(target=self._poll, daemon=True)
      self._thread.start()
    except Exception:   # pylint: disable=broad-except
      self._nvml = None

  def begin(self):
    """Start of the timed region: forget what was sampled before."""
    self.clocks, self.masks = [], 0

  def _poll(self):
    nv = self._nvml
    while not self._stop.is_set():
      try:
        clock = nv.nvmlDeviceGetClockInfo(self._handle, nv.NVML_CLOCK_SM)
        mask = nv.nvmlDeviceGetCurrentClocksEventReasons(self._handle)
        self.clocks.append(clock)
        self.masks |= mask
      except Exception:   # pylint: disable=broad-except
        break
      time.sleep(float(os.environ.get('SODA_BENCH_CLOCK_PERIOD', '0.002')))

  def _smi_once(self):
    query = ('clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,'
             'clocks_event_reasons.hw_thermal_slowdown,'
             'clocks_event_reasons.sw_thermal_slowdown,'
             'clocks_event_reasons.sw_power_cap')
    try:
      out = subprocess.run(
          ['nvidia-smi', '-i', str(self.index), '--query-gpu=' + query,
           '--format=csv,noheader,nounits'], stdout=subprocess.PIPE,
          stderr=subprocess.DEVNULL, text=True, timeout=20).stdout
      row = [c.strip() for c in out.strip().split(',')]
      return {'sm_mhz': int(row[0]), 'sm_max_mhz': int(row[1]),
              'reasons': [n for (n, _), c in zip(self.REASONS, row[2:6])
                          if c.lower().startswith('active')],
              'samples': 1, 'source': 'nvidia-smi after the timed region'}
    except Exception:   # pylint: disable=broad-except
      return {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': ['unavailable'],
              'samples': 0}

  def stop(self):
    self._stop.set()
    if self._thread is not None:
      self._thread.join(timeout=2)
    if not self.clocks:
      return self._smi_once()
    clocks = sorted(self.clocks)
    return {'sm_mhz': clocks[len(clocks) // 2], 'sm_max_mhz': self.max_mhz,
            'reasons': [n for n, bit in self.REASONS if self.masks & bit],
            'samples': len(clocks), 'source': 'NVML polled during the timed '
            'region'}


def cpu_port_gcells(iterate, threads=None):
  """GCell/s of the CPU oracle on the workload grid, `iterate` iterations."""
  sys.path.insert(0, os.path.join(ROOT, 'oracle'))
  import golden
  if threads:
    os.environ['OMP_NUM_THREADS'] = str(threads)
  oracle = golden.Oracle(load_stencil(iterate))
  if threads:
    # the environment only counts before libgomp starts; afterwards ask it
    try:
      import ctypes
      ctypes.CDLL('libgomp.so.1').omp_set_num_threads(int(threads))
    except OSError:
      pass
  inputs = oracle.reference_inputs(WORKLOAD['dims'])
  _, seconds = oracle.run(inputs, with_seconds=True)
  cells = WORKLOAD['dims'][0] * WORKLOAD['dims'][1]
  return cells * iterate / seconds / 1e9, seconds


def run_reference(args, rank):
  """--impl reference: the golden-loop port on the host cores."""
  if rank != 0:
    return
  cores = os.cpu_count() or 1
  for _ in range(min(args.warmup, 1)):
    cpu_port_gcells(CPU_SAMPLE_ITERATE, cores)
  values, total = [], 0.0
  for _ in range(args.steps):
    value, seconds = cpu_port_gcells(CPU_SAMPLE_ITERATE, cores)
    values.append(value)
    total += seconds
  value = sum(values) / len(values)
  sample = '%dx%d float32, %d of %d iterations per step' % (
      WORKLOAD['dims'] + (CPU_SAMPLE_ITERATE, WORKLOAD['iterate']))
  print(json.dumps({
      'impl': 'reference', 'metric': 'stencil_cell_updates_per_second',
      'value': value, 'unit': 'GCell/s', 'n_gpus': args.gpus,
      'steps': args.steps, 'warmup': args.warmup,
      'ms_per_step': total / args.steps * 1e3, 'higher_is_better': True,
      'scaling': 'weak', 'vs_baseline': None, 'dtype': 'f32',
      'data': 'synthetic (reference initialiser, host.py:1033-1051)',
      'config': workload_config(args.gpus),
      'cpu_baseline': {'value': value, 'unit': 'GCell/s', 'cores': cores,
                       'kind': 'port', 'sample': sample},
      'e2e': {'value': value, 'unit': 'GCell/s', 'h2d_bytes_per_step': 0,
              'd2h_bytes_per_step': 0},
      'gpu_launches': 0}))


def workload_config(n_gpus):
  d0, d1 = WORKLOAD['dims']
  return {'workload': 'jacobi2d.soda float32 %dx%d iterate %d (BASELINE '
                      'configs[1]); per GPU' % (d0, d1, WORKLOAD['iterate']),
          'global_grid': [d0, d1 * n_gpus], 'iterate': WORKLOAD['iterate'],
          'partition': 'single GPU' if n_gpus == 1 else
                       '%d slabs along the streamed dimension; per launch '
                       'the face rows go to the neighbours\' ghost rows by '
                       'copy engine over NVLink (peer-mapped memory + '
                       'stream flags)' % n_gpus,
          'l2': 'inputs (1.07 GB per GPU) exceed the 126 MB L2; no flush'}


# BASELINE configs 3, 4, 5: (program, iterate, global dims, bytes per cell
# update at T = 1 (SURVEY.md 8d), runs at N > 1, build).  The `fast` build of
# the two denoise programs (FMA contraction, approximate division, refined
# rsqrt: within 1e-6 relative / 2 ulp of the reference, the north star's bar
# for non-exact float builds) is listed NEXT TO the bit-exact one, which is
# bound by FP32 instruction issue in reference operation order.
EXTRA_CASES = (
    ('blur', 1, (2000, 1000), 4, False, 'exact'),      # BASELINE configs[0]
    ('sobel2d', 1, (32768, 32768), 4, False, 'exact'),
    ('denoise2d', 1, (32768, 32768), 12, False, 'exact'),
    ('denoise2d', 1, (32768, 32768), 12, False, 'fast'),
    ('heat3d', 32, (1024, 1024, 1024), 8, True, 'exact'),
    ('jacobi3d', 32, (1024, 1024, 1024), 8, True, 'exact'),
    ('denoise3d', 16, (768, 768, 768), 12, True, 'exact'),
    ('denoise3d', 16, (768, 768, 768), 12, False, 'fast'),
)


def extra_stencil(name, iterate):
  """The program compiled for `iterate` iterations, or for one when the
  reference refuses to iterate it (denoise: inputs != outputs, reference
  core.py:228-233) — then it is applied `iterate` times with u <- output."""
  from soda import core
  path = os.path.join(ROOT, 'benchmarks', name + '.soda')
  try:
    return core.Stencil.from_file(path, iterate=iterate)
  except Exception:   # pylint: disable=broad-except
    return core.Stencil.from_file(path, iterate=1)


def run_extra(rank, world, barrier, max_over_ranks, peak, reps=3):
  """Configs 3-5, device-resident, CUDA events, max over ranks; the global
  grid is fixed and cut into `world` slabs (strong scaling)."""
  import numpy as np
  import torch
  from soda import cuda as soda_cuda, cuda_slab
  results = []
  for name, iterate, dims, bytes_per_cell, sharded, build in EXTRA_CASES:
    if world > 1 and not sharded:
      continue
    entry = {'workload': '%s.soda %s iterate %d' % (
        name, 'x'.join(map(str, dims)), iterate), 'n_gpus': world,
             'scaling': 'strong' if world > 1 else 'single GPU',
             'build': 'bit-exact (default)' if build == 'exact' else
                      'fast (-DSODA_CUDA_FAST_MATH: within 1e-6 relative / 2 '
                      'ulp, tests/test_fastmath_gpu.py)'}
    try:
      library = soda_cuda.compile_stencil(extra_stencil(name, iterate),
                                          fast_math=build == 'fast')
      feedback = None
      if len(library.inputs) != len(library.outputs):
        feedback = {1: 0}        # denoise: u <- output, f stays
        entry['host_level_applications'] = iterate
      runner = cuda_slab.SlabRunner(library, dims, rank, world,
                                    feedback=feedback)
      # one GPU, the program's own iterate: the C ABI's device entry, as a
      # caller with device arrays makes it (the slab runner adds ~15 us of
      # Python per run, which is more than blur 2000 x 1000 takes)
      direct = world == 1 and feedback is None
      owned = []
      generator = torch.Generator(device='cuda').manual_seed(1 + rank)
      for local_in in runner.inputs:
        shape = runner.owned(local_in).shape
        if local_in.dtype.is_floating_point:
          owned.append(torch.rand(shape, device='cuda', generator=generator)
                       .to(local_in.dtype))
        else:
          owned.append(torch.randint(0, 30000, shape, device='cuda',
                                     generator=generator).to(local_in.dtype))
      runner.load_local(owned)
      del owned
      if direct:
        outs = [torch.empty_like(t) for t in runner.buffers[0]]
        stream = torch.cuda.current_stream().cuda_stream
        run_once = lambda: library.run_device(runner.inputs, outs, dims,
                                              iterate, stream)
      else:
        run_once = lambda: runner.run(iterate)
      for _ in range(2):
        run_once()
      times = []
      cells = float(np.prod(dims))
      inner = 50 if cells < 1e7 else 1     # microsecond kernels: time a batch
      for _ in range(reps):
        barrier()
        start, stop = torch.cuda.Event(True), torch.cuda.Event(True)
        start.record()
        for _ in range(inner):
          run_once()
        stop.record()
        torch.cuda.synchronize()
        times.append(max_over_ranks(start.elapsed_time(stop)) / inner)
      ms = float(np.median(times))
      passes = len(runner.plan(iterate))
      achieved = cells * bytes_per_cell * passes / (ms * 1e6)   # GB/s, all GPUs
      entry.update({
          'ms': ms, 'value': cells * iterate / (ms * 1e6), 'unit': 'GCell/s',
          'temporal_depth': runner.plan(iterate)[0], 'passes': passes,
          'launches_rank0': runner.launches_per_run(iterate),
          'runs_per_timing': inner,
          'entry': 'soda_cuda_run_device' if direct else
                   'soda_cuda_launch per slab (soda/cuda_slab.py)',
          'roofline': {
              'bound': 'hbm', 'achieved': achieved, 'peak': peak * world,
              'unit': 'GB/s', 'frac': achieved / (peak * world),
              'algorithmic_bytes_per_pass': cells * bytes_per_cell,
              'traffic': None,
              'traffic_source': 'not measured in this run; ncu captures of '
                                'these kernels are under profiles/'}})
      del runner
      library.release()
      torch.cuda.empty_cache()
    except Exception as e:   # pylint: disable=broad-except
      entry['error'] = '%s: %s' % (type(e).__name__, str(e)[:300])
    results.append(entry)
  return results


def sharded_parity(rank, world, barrier):
  """N > 1: a small heat3d run cut into `world` slabs (halo exchange per
  launch, soda/cuda_slab.py) against the SAME run on one GPU (rank 0, whole
  grid), bit for bit — SURVEY.md 8e "result invariance"."""
  import numpy as np
  import torch
  import torch.distributed as dist
  from soda import cuda as soda_cuda, cuda_slab
  name, iterate, dims = 'heat3d', 6, (256, 128, 32 * world)
  library = soda_cuda.compile_stencil(extra_stencil(name, 32))
  shape = tuple(reversed(dims))
  full = torch.rand(shape, device='cuda',
                    generator=torch.Generator(device='cuda').manual_seed(7))
  runner = cuda_slab.SlabRunner(library, dims, rank, world)
  runner.load_local([full[runner.begin:runner.end].clone()])
  mine = runner.run(iterate)[0].contiguous()
  torch.cuda.synchronize()
  rows = [e - b for b, e in cuda_slab.partition(dims[-1], world)]
  if rank == 0:
    whole = torch.empty(shape, dtype=torch.float32, device='cuda')
    library.run_device([full], [whole], dims, iterate,
                       torch.cuda.current_stream().cuda_stream)
    torch.cuda.synchronize()
  parts = [torch.empty((r,) + shape[1:], dtype=torch.float32, device='cuda')
           for r in rows] if rank == 0 else None
  # gather the slabs on rank 0 (NCCL send/recv; sizes differ by at most one)
  if rank == 0:
    parts[0].copy_(mine)
    for src in range(1, world):
      dist.recv(parts[src], src=src)
  else:
    dist.send(mine, dst=0)
  barrier()
  del runner
  if rank != 0:
    return None
  sharded = torch.cat(parts)
  same = bool(torch.equal(sharded.view(torch.int32), whole.view(torch.int32)))
  return {'case': '%s %s x%d, %d slabs vs one GPU' % (
      name, 'x'.join(map(str, dims)), iterate, world),
          'bit_identical': same,
          'cells_differing': int((sharded.view(torch.int32) !=
                                  whole.view(torch.int32)).sum().item())}


DUMP_CELLS = 1 << 22    # cells --dump-outputs samples in all: <= 32 MB


def dump_outputs(directory, library, outputs, regions, row_begin, suffix=''):
  """--dump-outputs: what the timed path's last step computed, as
  ``directory/<output name><suffix>.npy``.  Per output, the values (float32,
  or float64 for other types) of a fixed, seeded sample of the cells of its
  valid region, in row-major order: the same arguments give the same inputs
  and the same cells, so two builds compare output for output.  ``regions``
  are in global coordinates; ``outputs`` hold the global rows
  ``[row_begin, row_begin + rows)`` and keep the sampled cells among them."""
  import numpy as np
  import torch
  os.makedirs(directory, exist_ok=True)
  cells = DUMP_CELLS // len(outputs)
  for (name, _), out, region in zip(library.outputs, outputs, regions):
    box = [hi - lo for lo, hi in reversed(region)]      # numpy order
    count = int(np.prod(box))
    picks = np.arange(count) if count <= cells else np.unique(
        np.random.default_rng(0).integers(0, count, size=cells))
    coords = [c + lo for c, (lo, _) in zip(np.unravel_index(picks, box),
                                           reversed(region))]
    coords[0] -= row_begin
    mine = (coords[0] >= 0) & (coords[0] < out.shape[0])
    flat = np.ravel_multi_index([c[mine] for c in coords], tuple(out.shape))
    values = out.reshape(-1)[torch.from_numpy(flat).to(out.device)]
    values = values.cpu().numpy()
    if values.dtype not in (np.float32, np.float64):
      values = values.astype(np.float64)
    np.save(os.path.join(directory, name + suffix + '.npy'), values)


def copy_ceiling(world, slab_bytes, reps=3):
  """ms to move `slab_bytes` to each of `world` devices and as many back, both
  directions at once, with plain cudaMemcpyAsync from pinned memory and no
  compute: what the host<->device path of this machine allows."""
  import torch
  host_in, host_out, dev, streams = [], [], [], []
  for d in range(world):
    with torch.cuda.device(d):
      host_in.append(torch.empty(slab_bytes, dtype=torch.uint8,
                                 pin_memory=True))
      host_out.append(torch.empty(slab_bytes, dtype=torch.uint8,
                                  pin_memory=True))
      dev.append((torch.empty(slab_bytes, dtype=torch.uint8, device='cuda'),
                  torch.empty(slab_bytes, dtype=torch.uint8, device='cuda')))
      streams.append((torch.cuda.Stream(), torch.cuda.Stream()))
  times = []
  for _ in range(reps + 1):
    for d in range(world):
      torch.cuda.synchronize(d)
    t0 = time.perf_counter()
    for d in range(world):
      with torch.cuda.device(d):
        with torch.cuda.stream(streams[d][0]):
          dev[d][0].copy_(host_in[d], non_blocking=True)
        with torch.cuda.stream(streams[d][1]):
          host_out[d].copy_(dev[d][1], non_blocking=True)
    for d in range(world):
      torch.cuda.synchronize(d)
    times.append((time.perf_counter() - t0) * 1e3)
  return sorted(times[1:])[len(times[1:]) // 2]


def main():
  parser = argparse.ArgumentParser()
  parser.add_argument('--gpus', type=int, default=1)
  parser.add_argument('--steps', type=int, default=10)
  parser.add_argument('--warmup', type=int, default=3)
  parser.add_argument('--impl', default='b200', choices=['b200', 'reference'])
  parser.add_argument('--no-cpu-baseline', action='store_true')
  parser.add_argument('--no-extra', action='store_true',
                      help='skip BASELINE configs 3-5 (the `extra` block)')
  parser.add_argument('--dump-outputs', metavar='DIR',
                      help='after the timed steps, write a fixed sample of '
                           'what the last one computed to DIR/<output>.npy')
  args = parser.parse_args()
  if args.steps < 1:
    parser.error('--steps must be at least 1')
  if args.dump_outputs and args.impl != 'b200':
    parser.error('--dump-outputs dumps the b200 implementation\'s outputs')
  # the tree may be read-only; nothing is written into it
  sys.dont_write_bytecode = True
  rank = int(os.environ.get('RANK', '0'))
  world = int(os.environ.get('WORLD_SIZE', '1'))
  if args.impl == 'reference':
    run_reference(args, rank)
    return
  args.warmup = max(args.warmup, 3)

  import numpy as np
  import torch
  from soda import cuda as soda_cuda
  if not torch.cuda.is_available():
    sys.exit('bench.py: no CUDA device; this backend has no CPU path')
  local_rank = int(os.environ.get('LOCAL_RANK', '0'))
  distributed = world > 1
  # one process per GPU: keep each on its GPU's NUMA node where the machine
  # exposes one (the pool's KVM guests report a single node: nothing to bind)
  numa_node = soda_cuda.bind_host_to_gpu(local_rank) if distributed else None
  torch.cuda.set_device(local_rank)
  if distributed:
    import torch.distributed as dist
    dist.init_process_group('nccl', device_id=torch.device('cuda', local_rank))

  stencil = load_stencil()
  library = soda_cuda.compile_stencil(stencil)
  dims = WORKLOAD['dims']
  cells = dims[0] * dims[1]
  iterate = WORKLOAD['iterate']
  shape = (dims[1], dims[0])

  def barrier():
    torch.cuda.synchronize()
    if distributed:
      dist.barrier()
    torch.cuda.synchronize()

  def max_over_ranks(value):
    if not distributed:
      return value
    t = torch.tensor([value], dtype=torch.float64, device='cuda')
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t.item())

  # synthetic input: the reference initialiser's pattern (host.py:1033-1051)
  p = torch.arange(dims[0], device='cuda', dtype=torch.float32)
  q = torch.arange(dims[1], device='cuda', dtype=torch.float32) + (
      rank * dims[1] if distributed else 0)
  total = float(dims[0] + dims[1] * world)
  dev_in = ((q[:, None] + p[None, :]) / torch.tensor(
      total, dtype=torch.float32, device='cuda')).contiguous()
  stream = torch.cuda.current_stream().cuda_stream

  if distributed:
    from soda import cuda_slab
    runner = cuda_slab.SlabRunner(library, (dims[0], dims[1] * world), rank,
                                  world)
    runner.load_local([dev_in])
    step = lambda: runner.run(iterate)
    launches_per_step = runner.launches_per_run(iterate)
    passes_per_step = len(runner.plan(iterate))
    depth_planned = runner.plan(iterate)[0]
  else:
    dev_out = torch.empty(shape, dtype=torch.float32, device='cuda')
    step = lambda: library.run_device([dev_in], [dev_out], dims, iterate,
                                      stream)
    launches_per_step = passes_per_step = depth_planned = None

  # ---- device-resident timing ------------------------------------------------
  for _ in range(args.warmup):
    step()
  # NVML is initialised BEFORE the barrier: it takes milliseconds, and a rank
  # that enters the timed region late holds its neighbours up by as much
  sampler = ClockSampler(local_rank) if rank == 0 else None
  barrier()
  if sampler:
    sampler.begin()
  start, stop = torch.cuda.Event(True), torch.cuda.Event(True)
  start.record()
  for _ in range(args.steps):
    last = step()
  stop.record()
  barrier()
  clocks = sampler.stop() if sampler else None
  if args.dump_outputs and distributed:
    dump_outputs(args.dump_outputs, library, last,
                 runner.valid_regions(iterate), runner.begin, '.rank%d' % rank)
  elif args.dump_outputs:
    dump_outputs(args.dump_outputs, library, [dev_out],
                 library.valid_regions(dims, iterate), 0)
  ms_total = max_over_ranks(start.elapsed_time(stop))
  ms_per_step = ms_total / args.steps
  value = cells * world * iterate / (ms_per_step * 1e6)     # GCell/s
  stats = library.stats
  if launches_per_step is None:
    launches_per_step = passes_per_step = stats['launches']
  # slab runs launch faces and interior separately: a "pass" is one sweep of
  # the whole slab by the depth-T kernel, however many launches it took
  depth = depth_planned or stats['depth']
  if distributed:
    del runner
  torch.cuda.empty_cache()

  # ---- end to end through the C ABI with host buffers ------------------------
  # One call on the global grid.  N > 1: rank 0 makes it with
  # "devices=0,..,N-1" (the runtime cuts the host arrays into one slab per
  # device, soda_cuda_runtime.cu run_sharded); the other ranks wait.
  e2e = None
  barrier()
  if rank == 0:
    global_shape = (dims[1] * world, dims[0])
    host_in = torch.empty(global_shape, dtype=torch.float32, pin_memory=True)
    host_out = torch.empty(global_shape, dtype=torch.float32, pin_memory=True)
    columns = torch.arange(dims[0], dtype=torch.float32)[None, :]
    for r0 in range(0, global_shape[0], 4096):      # block-wise: no 8 GiB temps
      block = torch.arange(r0, min(r0 + 4096, global_shape[0]),
                           dtype=torch.float32)[:, None] + columns
      host_in[r0:r0 + 4096] = block / torch.tensor(total, dtype=torch.float32)
    np_in, np_out = host_in.numpy(), host_out.numpy()
    devices = list(range(world)) if distributed else None
    e2e_steps = max(2, min(args.steps, 5))
    for _ in range(2):
      library.run([np_in], [np_out], devices=devices)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
      # H2D + all launches + D2H, synchronous
      library.run([np_in], [np_out], devices=devices)
    e2e_ms = (time.perf_counter() - t0) * 1e3 / e2e_steps
    e2e_stats = library.stats
    slabs = library.slab_stats
    # the result of the timed call against the device-resident run's: a
    # checksum over the valid region (not a parity test, a did-it-run test)
    e2e_value = cells * world * iterate / (e2e_ms * 1e6)
    pageable = None
    if not distributed:
      # the same call on ordinary (pageable) numpy arrays, as a caller that
      # does not pin its memory makes it: through the runtime's bounce buffers
      page_in = np.array(np_in)          # a pageable copy
      page_out = np.empty_like(page_in)
      library.run([page_in], [page_out])
      t0 = time.perf_counter()
      for _ in range(2):
        library.run([page_in], [page_out])
      page_ms = (time.perf_counter() - t0) * 1e3 / 2
      pageable = {'ms_per_step': page_ms,
                  'value': cells * iterate / (page_ms * 1e6),
                  'unit': 'GCell/s',
                  'bit_identical_to_pinned': bool(
                      np.array_equal(page_out.view(np.uint32),
                                     np_out.view(np.uint32)))}
      del page_in, page_out
    del host_in, host_out, np_in, np_out
    ceiling_ms = copy_ceiling(world, cells * 4)
    e2e = {'value': e2e_value, 'unit': 'GCell/s', 'ms_per_step': e2e_ms,
           'h2d_bytes_per_step': cells * world * 4,
           'd2h_bytes_per_step': cells * world * 4,
           'h2d_ms': e2e_stats['h2d_ms'], 'd2h_ms': e2e_stats['d2h_ms'],
           'kernel_ms': e2e_stats['kernel_ms'], 'steps': e2e_steps,
           'launches_per_step': e2e_stats['launches'],
           'api': 'soda_cuda_run (C ABI form of jacobi2d(buffer_t*, '
                  'buffer_t*, const char*)), pinned host buffers, ONE call '
                  'on the global %d x %d grid%s' % (
                      dims[0], dims[1] * world,
                      ', config "devices=%s": one slab per device' % ','.join(
                          map(str, devices)) if devices else ''),
           'per_slab': [{k: s[k] for k in ('h2d_ms', 'd2h_ms', 'kernel_ms',
                                           'launches')} for s in slabs],
           'copy_ceiling': {
               'ms': ceiling_ms,
               'gb_per_s_each_direction': cells * world * 4 / (ceiling_ms * 1e6),
               'e2e_fraction_of_ceiling': ceiling_ms / e2e_ms,
               'what': 'the same %d x %.2f GB to the devices and as much '
                       'back at once, cudaMemcpyAsync from pinned memory, no '
                       'compute: the host<->device capacity of this machine '
                       'at %d device(s)' % (world, cells * 4 / 1e9, world)},
           'pageable_host_buffers': pageable,
           'numa_node_rank0': numa_node}
  barrier()

  peak, peak_kind = measured_hbm_gbs()
  # ---- BASELINE configs 3-5 and the multi-GPU parity check (not timed in
  # ms_per_step) ---------------------------------------------------------------
  parity = sharded_parity(rank, world, barrier) if distributed else None
  extra = None if args.no_extra else run_extra(rank, world, barrier,
                                               max_over_ranks, peak)

  if rank != 0:
    if distributed:
      dist.destroy_process_group()
    return

  launch_ms = ms_per_step / passes_per_step
  achieved = cells * BYTES_PER_CELL / (launch_ms * 1e6)        # GB/s
  traffic = None
  try:
    with open(os.path.join(ROOT, 'profiles', 'traffic.json')) as handle:
      traffic = json.load(handle).get('jacobi2d_d%d' % depth)
  except (OSError, ValueError):
    pass
  result = {
      'metric': 'stencil_cell_updates_per_second', 'value': value,
      'unit': 'GCell/s', 'n_gpus': world, 'steps': args.steps,
      'warmup': args.warmup, 'ms_per_step': ms_per_step,
      'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None,
      'dtype': 'f32',
      'data': 'synthetic (reference initialiser pattern, host.py:1033-1051)',
      'config': workload_config(world),
      'kernel': dict(temporal_depth=depth, launches_per_step=launches_per_step,
                     passes_per_step=passes_per_step,
                     threads=stats['threads'], smem_bytes=stats['smem_bytes'],
                     tma=bool(stats['used_tma'])),
      'e2e': e2e,
      'gpu_launches': launches_per_step * args.steps,
      'roofline': {
          'bound': 'hbm', 'achieved': achieved, 'peak': peak, 'unit': 'GB/s',
          'frac': achieved / peak, 'traffic': traffic,
          'traffic_source': 'profiles/traffic.json: dram__bytes_read.sum + '
                            'dram__bytes_write.sum of one launch of this '
                            'kernel from an `ncu --set full` capture of this '
                            'command (not measured in this run)',
          'peak_source': peak_kind + ' (MEASURED_PEAKS.json hbm_gbs)',
          'kernel': 'soda_jacobi2d_d%d<true>' % depth,
          'algorithmic_bytes_per_launch': cells * BYTES_PER_CELL,
          'launch_ms': launch_ms,
          'note': 'one launch advances %d iterations; the streaming-'
                  'equivalent rate (8 B x cells x iterate / time) is '
                  '%.0f GB/s' % (depth, cells * 8 * iterate /
                                 (ms_per_step * 1e6))},
      'clocks': clocks,
  }
  if parity is not None:
    result['multi_gpu_parity'] = parity
  if extra is not None:
    result['extra'] = extra
  if not args.no_cpu_baseline and world == 1:
    cores = os.cpu_count() or 1
    cpu_value, cpu_seconds = cpu_port_gcells(CPU_SAMPLE_ITERATE, cores)
    result['cpu_baseline'] = {
        'value': cpu_value, 'unit': 'GCell/s', 'cores': cores, 'kind': 'port',
        'seconds': cpu_seconds,
        'sample': '%dx%d float32, %d of %d iterations (same grid, ping-pong '
                  'golden loop, g++ -O3 -fopenmp)' % (
                      dims + (CPU_SAMPLE_ITERATE, iterate))}
    one_value, one_seconds = cpu_port_gcells(CPU_SINGLE_THREAD_ITERATE, 1)
    result['cpu_baseline']['single_thread'] = {
        'value': one_value, 'unit': 'GCell/s', 'cores': 1,
        'seconds': one_seconds,
        'sample': '%d of %d iterations' % (CPU_SINGLE_THREAD_ITERATE,
                                           iterate)}
  print(json.dumps(result))
  if distributed:
    dist.destroy_process_group()


if __name__ == '__main__':
  main()
