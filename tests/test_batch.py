"""Batched runs without a GPU: every kernel family compiles with the batch
grid dimension, and ``run_batch`` checks its arrays before it calls the
library (tests/test_batch_gpu.py runs the batches)."""
import concurrent.futures
import re
import subprocess

import numpy as np
import pytest

import common
import dim4_programs
from soda import cuda as soda_cuda
from soda.codegen import cuda as codegen

STENCILS = ([(name, lambda name=name: common.stencil(name))
             for name in common.BENCHMARKS] +
            [(name, lambda name=name: dim4_programs.stencil_of(name))
             for name, _ in dim4_programs.CASES])


def _kernels(path):
  """Names of the __global__ functions in a library's sm_100a code."""
  sass = subprocess.run(['cuobjdump', '-sass', path], stdout=subprocess.PIPE,
                        text=True, check=True).stdout
  return re.findall(r'Function : (\S+)', sass)


def test_every_kernel_compiles_with_the_batch_dimension():
  """Benchmarks and 4-D programs, register and ring family, both input
  paths (kTma true and false): 2-D maps become rank 3, 3-D rank 4 and 4-D
  rank 5."""
  jobs = [(name, make, style) for name, make in STENCILS
          for style in ('reg', 'ring')]

  def build(job):
    _, make, style = job
    return soda_cuda.build(make(), options=codegen.Options(style=style))
  with concurrent.futures.ThreadPoolExecutor(max_workers=8) as pool:
    paths = list(pool.map(build, jobs))
  for (name, _, style), path in zip(jobs, paths):
    kernels = _kernels(path)
    for instance in ('ILb1', 'ILb0'):
      assert any(instance in k for k in kernels), (name, style, kernels)
    source = open(re.sub(r'libsoda_(\w+)\.so$', r'\1_kernel.cu', path)).read()
    assert 'a.item_begin + blockIdx.z' in source, (name, style)


@pytest.fixture(scope='module')
def library():
  return soda_cuda.compile_stencil(common.stencil('jacobi2d', 3))


@pytest.fixture(scope='module')
def multi():
  """Two inputs, one output."""
  return soda_cuda.compile_stencil(common.stencil('denoise2d'))


def _fail_on_call(library, monkeypatch):
  def refuse(*_):
    raise AssertionError('soda_cuda_run_batch was called')
  monkeypatch.setattr(library, '_lib', _Guard(library._lib, refuse))


class _Guard:
  """The library with soda_cuda_run_batch replaced."""

  def __init__(self, lib, refuse):
    self._wrapped = lib
    self.soda_cuda_run_batch = refuse

  def __getattr__(self, name):
    return getattr(self._wrapped, name)


def test_run_batch_checks_arrays_before_calling(library, multi, monkeypatch):
  for lib in (library, multi):
    _fail_on_call(lib, monkeypatch)
  f32 = np.float32
  good = np.zeros((3, 40, 64), dtype=f32)
  with pytest.raises(ValueError, match='3-dimensional'):      # wrong rank
    library.run_batch([np.zeros((40, 64), dtype=f32)])
  with pytest.raises(ValueError, match='3-dimensional'):
    library.run_batch([np.zeros((2, 3, 40, 64), dtype=f32)])
  with pytest.raises(TypeError):                               # wrong dtype
    library.run_batch([good.astype(np.float64)])
  with pytest.raises(ValueError, match='contiguous'):
    library.run_batch([np.zeros((3, 40, 128), dtype=f32)[:, :, ::2]])
  with pytest.raises(ValueError, match='contiguous'):
    library.run_batch([np.zeros((40, 3, 64), dtype=f32).transpose(1, 0, 2)])
  with pytest.raises(ValueError, match='expected'):            # B differs
    library.run_batch([good], [np.zeros((2, 40, 64), dtype=f32)])
  with pytest.raises(ValueError, match='expected'):            # extents
    library.run_batch([good], [np.zeros((3, 40, 65), dtype=f32)])
  with pytest.raises(TypeError):
    library.run_batch([good], [np.zeros((3, 40, 64), dtype=np.int32)])
  with pytest.raises(ValueError):
    library.run_batch([good, good])                            # input count
  a = np.zeros((4, 30, 50), dtype=f32)
  with pytest.raises(ValueError, match='expected'):            # between inputs
    multi.run_batch([a, np.zeros((5, 30, 50), dtype=f32)])
  with pytest.raises(ValueError, match='expected'):
    multi.run_batch([a, np.zeros((4, 31, 50), dtype=f32)])
  with pytest.raises(ValueError, match='expected'):
    multi.run_batch([a, a], [np.zeros((4, 30, 51), dtype=f32)])


def test_one_grid_run_still_refuses_a_batch(library):
  with pytest.raises(ValueError, match='2-dimensional'):
    library.run([np.zeros((3, 40, 64), dtype=np.float32)])


def _no_gpu():
  import torch
  if torch.cuda.is_available():
    pytest.skip('a GPU is present')


def test_no_cpu_fallback(library):
  _no_gpu()
  with pytest.raises(soda_cuda.CudaError) as info:
    library.run_batch([np.zeros((2, 40, 64), dtype=np.float32)])
  assert info.value.code == -19       # no_device_interface
  with pytest.raises(soda_cuda.CudaError) as info:
    soda_cuda.run_batch(common.stencil('jacobi2d', 3),
                        {'t1': np.zeros((2, 40, 64), dtype=np.float32)})
  assert info.value.code == -19


def test_bad_batch_and_bounds_query_are_refused(library):
  """batch < 1: access_out_of_bounds; host == NULL && dev == 0 (a bounds
  query for soda_cuda_run): buffer_argument_is_null.  Neither needs a
  device."""
  import ctypes
  BufferT = soda_cuda.BufferT
  buf = BufferT()
  buf.extent[0], buf.extent[1] = 64, 40
  buf.stride[0], buf.stride[1] = 1, 64
  buf.elem_size = 4
  data = np.zeros((2, 40, 64), dtype=np.float32)
  buf.host = data.ctypes.data
  query = BufferT()
  query.extent[0], query.extent[1] = 64, 40

  def ptrs(b):
    return (ctypes.POINTER(BufferT) * 1)(ctypes.pointer(b))
  run = library._lib.soda_cuda_run_batch
  assert run(ptrs(buf), ptrs(buf), None, 0) == -4
  assert run(ptrs(buf), ptrs(buf), None, -3) == -4
  assert run(ptrs(buf), ptrs(query), None, 2) == -12
  assert run(ptrs(query), ptrs(buf), None, 2) == -12
  dims = (ctypes.c_int32 * 4)(64, 40, 1, 1)
  assert library._lib.soda_cuda_run_device_batch(
      (ctypes.c_void_p * 1)(data.ctypes.data),
      (ctypes.c_void_p * 1)(data.ctypes.data), dims, 0, 0, None) == -4
