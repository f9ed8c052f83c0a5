#!/usr/bin/env python3
"""Strided device arrays against dense ones on one GPU (developer tool; needs
a CUDA device).

For every workload it times, with CUDA events on warmed device-resident
arrays larger than the 126 MB L2:
  (a) dense arrays, `run_device`,
  (b) views of pitched parents (+64 cells per row), `run_strided`,
  (c) interior views with an unaligned base (parents 2 cells larger per axis,
      the view 1 cell in), `run_strided`,
  (d) the copy route: the input view copied to a dense array, `run_device`,
      the dense result copied into the output view,
and prints GCell/s (cell updates: cells x iterations per second) and whether
the launches used TMA.  The odd-width workload has rows of 16383 floats
(dense: no TMA) against the same grid in rows of 16384.

  python tools/strided_bench.py [--only NAME] [--out FILE.json]
"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [os.path.join(ROOT, 'soda-compiler_b200')]

import numpy as np   # noqa: E402
import torch         # noqa: E402

from soda import core, cuda as soda_cuda   # noqa: E402

# label, program, iterate, dims, layouts timed
WORKLOADS = [
    ('jacobi2d-x1', 'jacobi2d', 1, (16384, 16384), 'abcd'),
    ('jacobi2d-x64', 'jacobi2d', 64, (16384, 16384), 'abcd'),
    ('sobel2d-u16', 'sobel2d', 1, (32768, 32768), 'abcd'),
    ('heat3d-x1', 'heat3d', 1, (1024, 1024, 1024), 'abcd'),
    ('heat3d-x32', 'heat3d', 32, (1024, 1024, 1024), 'abcd'),
    ('odd-width', 'jacobi2d', 1, (16383, 16384), 'ab'),
]


def _gpu():
  """Card name and power limit, read where the numbers are measured."""
  try:
    return subprocess.run(
        ['nvidia-smi', '--query-gpu=name,power.limit', '--format=csv,noheader'],
        stdout=subprocess.PIPE, text=True, check=True).stdout.strip()
  except (OSError, subprocess.CalledProcessError):
    return torch.cuda.get_device_name(0) + ', power limit not readable'


def _dtype(haoda_type):
  return torch.from_numpy(np.empty(0, soda_cuda.NUMPY_TYPES[haoda_type])).dtype


def _time(run, min_ms=200.0):
  """Milliseconds per call of ``run`` (enqueues work), CUDA events."""
  for _ in range(3):
    run()
  start, stop = torch.cuda.Event(True), torch.cuda.Event(True)
  torch.cuda.synchronize()
  start.record()
  run()
  stop.record()
  stop.synchronize()
  reps = int(min(100, max(3, min_ms / max(start.elapsed_time(stop), 1e-3))))
  start.record()
  for _ in range(reps):
    run()
  stop.record()
  stop.synchronize()
  return start.elapsed_time(stop) / reps


def _views(shape, dtype, layout, width):
  """A tensor of `shape` laid out as `layout` ('a' dense, 'b' pitched,
  'c' interior with an unaligned base); `width`: row length of 'b'."""
  if layout == 'b':
    parent = torch.empty(shape[:-1] + (width,), dtype=dtype, device='cuda')
    return parent[..., :shape[-1]]
  if layout == 'c':
    parent = torch.empty(tuple(n + 2 for n in shape), dtype=dtype,
                         device='cuda')
    return parent[tuple(slice(1, 1 + n) for n in shape)]
  return torch.empty(shape, dtype=dtype, device='cuda')


def main():
  parser = argparse.ArgumentParser(description=__doc__.split('\n')[0])
  parser.add_argument('--only', default=None)
  parser.add_argument('--out', default=None)
  args = parser.parse_args()
  gpu = _gpu()
  print('GPU: %s' % gpu, flush=True)
  stream = torch.cuda.current_stream().cuda_stream
  rows = []
  for label, name, iterate, dims, layouts in WORKLOADS:
    if args.only and args.only != label:
      continue
    stencil = core.Stencil.from_file(
        os.path.join(ROOT, 'benchmarks', name + '.soda'), iterate=iterate)
    library = soda_cuda.compile_stencil(stencil)
    shape = tuple(reversed(dims))
    cells = int(np.prod(dims))
    width = dims[0] + 64 if label != 'odd-width' else 16384
    gen = torch.Generator(device='cuda').manual_seed(1)
    row = {'workload': label, 'program': name, 'iterate': iterate,
           'dims': list(dims), 'ms': {}, 'gcells': {}, 'used_tma': {}}
    for layout in layouts:
      ins = [_views(shape, _dtype(t), layout, width)
             for _, t in library.inputs]
      for tensor in ins:
        if tensor.dtype.is_floating_point:
          tensor.copy_(torch.rand(shape, generator=gen, device='cuda'))
        else:
          tensor.copy_(torch.randint(0, 1 << 12, shape, generator=gen,
                                     device='cuda', dtype=torch.int32))
      outs = [_views(shape, _dtype(t), layout if layout != 'd' else 'b', width)
              for _, t in library.outputs]
      if layout == 'a':
        run = lambda: library.run_device(ins, outs, dims, 0, stream)
      elif layout in 'bc':
        run = lambda: library.run_strided(ins, outs, stream=stream)
      else:
        # the copy route from pitched views: copy in, dense run, copy out
        ins = [_views(shape, t.dtype, 'b', width).copy_(t) for t in ins]
        dense_in = [torch.empty(shape, dtype=t.dtype, device='cuda')
                    for t in ins]
        dense_out = [torch.empty(shape, dtype=t.dtype, device='cuda')
                     for t in outs]

        def run():
          for d, v in zip(dense_in, ins):
            d.copy_(v)
          library.run_device(dense_in, dense_out, dims, 0, stream)
          for v, d in zip(outs, dense_out):
            v.copy_(d)
      ms = _time(run)
      row['ms'][layout] = ms
      row['gcells'][layout] = cells * iterate / (ms * 1e6)
      row['used_tma'][layout] = library.stats['used_tma']
      del ins, outs, run
      torch.cuda.empty_cache()
    rows.append(row)
    print('%-13s %-17s GCell/s: %s' % (
        label, 'x'.join(map(str, dims)), '  '.join(
            '(%s) %8.1f%s' % (k, v, '' if row['used_tma'][k] else ' plain')
            for k, v in row['gcells'].items())), flush=True)
  if args.out:
    with open(args.out, 'w') as handle:
      json.dump({'gpu': gpu, 'workloads': rows}, handle, indent=1)


if __name__ == '__main__':
  main()
