"""Shared helpers of the test-suite."""
import functools
import os

import numpy as np

import golden   # oracle/golden.py (the CPU oracle; tests may use it)
from soda import core

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BENCH_DIR = os.path.join(ROOT, 'benchmarks')
GOLDEN_DIR = os.path.join(ROOT, 'tests', 'golden')
REFERENCE_DIR = '/root/reference'
BENCHMARKS = ('blur', 'sobel2d', 'jacobi2d', 'seidel2d', 'denoise2d',
              'jacobi3d', 'heat3d', 'denoise3d')


def have_reference():
  return os.path.isdir(os.path.join(REFERENCE_DIR, 'src', 'soda'))


def bench_path(name):
  return os.path.join(BENCH_DIR, name + '.soda')


def bench_text(name):
  with open(bench_path(name)) as handle:
    return handle.read()


def golden_output_case(path):
  """``(program, iterate, dims)`` of ``tests/golden/outputs/<app>_it<N>_<dims>.npz``."""
  name, it, dims = os.path.basename(path)[:-4].rsplit('_', 2)
  return name, int(it[2:]), tuple(int(x) for x in dims.split('x'))


@functools.lru_cache(maxsize=None)
def stencil(name, iterate=None):
  return core.Stencil.from_text(bench_text(name), iterate=iterate)


@functools.lru_cache(maxsize=None)
def oracle(name, iterate=None):
  return golden.Oracle(stencil(name, iterate))


def random_inputs(orc, dims, seed=0):
  """Second input distribution (not a reference fixture): uniform noise."""
  rng = np.random.default_rng(seed)
  shape = tuple(reversed(dims))
  arrays = []
  for dtype in orc.input_dtypes:
    if np.dtype(dtype).kind == 'f':
      arrays.append(rng.random(shape, dtype=np.float32).astype(dtype))
    else:
      info = np.iinfo(dtype)
      arrays.append(rng.integers(info.min, int(info.max) + 1, size=shape,
                                 dtype=np.int64).astype(dtype))
  return arrays


def bits(array):
  """View for bit-exact comparison (NaN-safe)."""
  array = np.ascontiguousarray(array)
  return array.view({1: np.uint8, 2: np.uint16, 4: np.uint32,
                     8: np.uint64}[array.dtype.itemsize])


def assert_bit_exact(got, want, what='', any_nan=False):
  """``any_nan``: a NaN matches a NaN of any sign/payload.  The default NaN
  an invalid operation produces is a property of the machine (x86 SSE:
  0xFFC00000, NVIDIA: 0x7FFFFFFF), not of the program; everything else, the
  infinities included, still compares bit for bit."""
  assert got.shape == want.shape and got.dtype == want.dtype, what
  same = bits(got) == bits(want)
  if any_nan and got.dtype.kind == 'f':
    same |= np.isnan(got) & np.isnan(want)
  if not same.all():
    bad = np.argwhere(~same)
    first = tuple(bad[0])
    raise AssertionError(
        '%s: %d of %d cells differ; first at %s (dims reversed): got %r, '
        'want %r' % (what, len(bad), same.size, first, got[first],
                     want[first]))
