#!/usr/bin/env python3
"""Batches of small grids on one GPU (developer tool; needs a CUDA device).

For every case it times, with CUDA events on warmed, device-resident arrays:
  (a) a loop of B `run_device` calls, one per item,
  (b) one `run_device_batch` over the B items,
  (c) one `run_device` on a single grid of the same cells (the items stacked
      along the streamed dimension: the streaming-rate reference; its results
      differ from (b) near the seams, where (b) reads zeros),
and prints GCell/s (cell updates: cells x iterations per second) of each, with
(b)/(a) and (b)/(c).  Working sets above the 126 MB L2 (B x cells >= 16 Mi
for one float32 input and output, 32 Mi for uint16) stream from HBM;
smaller ones are read from L2 after the first pass.

  python tools/batch_bench.py [--batches 1,16,256,1024] [--out FILE.json]
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

CASES = ([(name, 1, (n, n)) for name in ('blur', 'sobel2d', 'jacobi2d',
                                         'denoise2d') for n in (256, 512)] +
         [('heat3d', 2, (64, 64, 64))])


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


def _random(shape, haoda_type, gen):
  dtype = _dtype(haoda_type)
  if dtype.is_floating_point:
    return torch.rand(shape, generator=gen, device='cuda').to(dtype)
  return torch.randint(0, 1 << 12, shape, generator=gen, device='cuda',
                       dtype=torch.int32).to(dtype)


def _time(run, min_ms=50.0):
  """Milliseconds per call of ``run`` (enqueues work), CUDA events."""
  for _ in range(3):
    run()
  start, stop = torch.cuda.Event(True), torch.cuda.Event(True)
  torch.cuda.synchronize()
  start.record()
  run()
  stop.record()
  stop.synchronize()
  reps = int(min(200, max(3, min_ms / max(start.elapsed_time(stop), 1e-3))))
  start.record()
  for _ in range(reps):
    run()
  stop.record()
  stop.synchronize()
  return start.elapsed_time(stop) / reps


def main():
  parser = argparse.ArgumentParser(description=__doc__.split('\n')[0])
  parser.add_argument('--batches', default='1,16,256,1024')
  parser.add_argument('--out', default=None)
  args = parser.parse_args()
  batches = [int(b) for b in args.batches.split(',')]
  gpu = _gpu()
  print('GPU: %s' % gpu, flush=True)
  stream = torch.cuda.current_stream().cuda_stream
  rows = []
  for name, iterate, dims in CASES:
    stencil = core.Stencil.from_file(
        os.path.join(ROOT, 'benchmarks', name + '.soda'), iterate=iterate)
    library = soda_cuda.compile_stencil(stencil)
    cells = int(np.prod(dims))
    for batch in batches:
      shape = (batch,) + tuple(reversed(dims))
      gen = torch.Generator(device='cuda').manual_seed(batch)
      ins = [_random(shape, haoda_type, gen)
             for _, haoda_type in library.inputs]
      outs = [torch.empty(shape, dtype=_dtype(haoda_type), device='cuda')
              for _, haoda_type in library.outputs]

      def loop():
        for b in range(batch):
          library.run_device([t[b] for t in ins], [t[b] for t in outs], dims,
                             0, stream)

      def batched():
        library.run_device_batch(ins, outs, dims, batch, 0, stream)
      stacked_dims = tuple(dims[:-1]) + (dims[-1] * batch,)

      def stacked():
        library.run_device(ins, outs, stacked_dims, 0, stream)
      ms = {key: _time(fn) for key, fn in (('a', loop), ('b', batched),
                                             ('c', stacked))}
      updates = batch * cells * iterate
      rate = {key: updates / (t * 1e6) for key, t in ms.items()}
      row = {'program': name, 'iterate': iterate, 'dims': list(dims),
             'batch': batch, 'cells': batch * cells,
             'ms': ms, 'gcells': rate,
             'b_over_a': rate['b'] / rate['a'],
             'b_over_c': rate['b'] / rate['c']}
      rows.append(row)
      print('%-9s x%d %-9s B=%-5d %9d cells  GCell/s: (a) loop %7.1f  (b) '
            'batch %7.1f  (c) stacked %7.1f   (b)/(a) %6.2f  (b)/(c) %5.2f' % (
                name, iterate, 'x'.join(map(str, dims)), batch, batch * cells,
                rate['a'], rate['b'], rate['c'], row['b_over_a'],
                row['b_over_c']), flush=True)
      del ins, outs
  if args.out:
    with open(args.out, 'w') as handle:
      json.dump({'gpu': gpu, 'cases': rows}, handle, indent=1)


if __name__ == '__main__':
  main()
