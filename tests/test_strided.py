"""Strided device arrays without a GPU: every kernel family compiles with
per-tensor strides, ``run_strided`` checks its tensors before it calls the
library, and the C entry point refuses NULL pointers (-12) and layouts
outside the rule (-4) before it looks for a device (tests/test_strided_gpu.py
runs them)."""
import concurrent.futures
import ctypes
import re

import numpy as np
import pytest

import common
import strided_programs
from soda import cuda as soda_cuda
from soda.codegen import cuda as codegen


def test_every_kernel_compiles_with_per_tensor_strides():
  """Benchmarks and the strided-test programs, register and ring family:
  the kernels address HBM through each tensor's own strides."""
  jobs = [(name, lambda name=name: common.stencil(name), style)
          for name in common.BENCHMARKS for style in ('reg', 'ring')]
  jobs += [(name, lambda k=kind, n=name, i=it: strided_programs.stencil_of(
      k, n, i), options.get('style', 'reg'))
           for kind, name, it, options in strided_programs.BUILDS
           if kind != 'bench']

  def build(job):
    _, make, style = job
    return soda_cuda.build(make(), options=codegen.Options(style=style))
  with concurrent.futures.ThreadPoolExecutor(max_workers=8) as pool:
    paths = list(pool.map(build, jobs))
  for (name, _, style), path in zip(jobs, paths):
    source = open(re.sub(r'libsoda_(\w+)\.so$', r'\1_kernel.cu', path)).read()
    assert 'a.out_stride[0]' in source, (name, style)
    assert 'a.stride[' not in source and 'goff' not in source, (name, style)


@pytest.fixture(scope='module')
def library():
  return soda_cuda.compile_stencil(common.stencil('jacobi2d', 3))


@pytest.fixture(scope='module')
def multi():
  """Two inputs, one output."""
  return soda_cuda.compile_stencil(common.stencil('denoise2d'))


class _Guard:
  """The library with the strided entry point replaced."""

  def __init__(self, lib, refuse):
    self._wrapped = lib
    self.soda_cuda_run_device_strided = refuse

  def __getattr__(self, name):
    return getattr(self._wrapped, name)


class _FakeCuda:
  """Stands in for a torch CUDA tensor on a machine without a device: the
  attributes run_strided reads, over a CPU tensor."""

  def __init__(self, tensor):
    self._t = tensor
    self.is_cuda = True
    self.device = 'cuda:0'
    self.dtype = tensor.dtype
    self.shape = tensor.shape

  def dim(self):
    return self._t.dim()

  def stride(self):
    return self._t.stride()

  def numel(self):
    return self._t.numel()


def test_run_strided_checks_tensors_before_calling(library, multi,
                                                   monkeypatch):
  torch = pytest.importorskip('torch')

  def refuse(*_):
    raise AssertionError('soda_cuda_run_device_strided was called')
  for lib in (library, multi):
    monkeypatch.setattr(lib, '_lib', _Guard(lib._lib, refuse))
  monkeypatch.setattr(torch, 'Tensor', _FakeCuda)
  f32 = torch.float32
  cuda = lambda t: _FakeCuda(t)
  good = cuda(torch.zeros(40, 64, dtype=f32))
  with pytest.raises(ValueError, match='2-dimensional'):          # rank
    library.run_strided([cuda(torch.zeros(3, 40, 64, dtype=f32))])
  with pytest.raises(ValueError, match='3-dimensional'):
    library.run_strided([good], batched=True)
  with pytest.raises(TypeError, match='must be'):                 # dtype
    library.run_strided([cuda(torch.zeros(40, 64, dtype=torch.float64))])
  with pytest.raises(TypeError, match='run / run_batch'):         # host arrays
    library.run_strided([np.zeros((40, 64), dtype=np.float32)])
  with pytest.raises(TypeError, match='run / run_batch'):
    library.run_strided([torch.zeros(40, 64, dtype=f32)])
  with pytest.raises(ValueError, match='stride 1'):               # stride(-1)
    library.run_strided([cuda(torch.zeros(40, 128, dtype=f32)[:, ::2])])
  with pytest.raises(ValueError, match='stride 1'):               # transposed
    library.run_strided([cuda(torch.zeros(64, 40, dtype=f32).t())])
  with pytest.raises(ValueError, match='layout'):   # items inside a row
    library.run_strided([cuda(torch.zeros(40, 3, 64, dtype=f32)
                              .permute(1, 0, 2))], batched=True)
  with pytest.raises(ValueError, match='layout'):                 # overlapping
    library.run_strided([cuda(torch.zeros(64 * 40, dtype=f32)
                              .as_strided((40, 64), (32, 1)))])
  with pytest.raises(ValueError, match='layout'):                 # broadcast
    library.run_strided([cuda(torch.zeros(1, 64, dtype=f32)
                              .expand(40, 64))])
  with pytest.raises(ValueError, match='expected'):               # out extents
    library.run_strided([good], [cuda(torch.zeros(40, 65, dtype=f32))])
  with pytest.raises(ValueError, match='expected'):
    library.run_strided([cuda(torch.zeros(3, 40, 64, dtype=f32))],
                        [cuda(torch.zeros(2, 40, 64, dtype=f32))],
                        batched=True)
  with pytest.raises(ValueError, match='expected'):               # between ins
    multi.run_strided([good, cuda(torch.zeros(40, 63, dtype=f32))])
  with pytest.raises(ValueError):
    library.run_strided([good, good])                             # input count


def _strides(rows):
  flat = [v for row in rows for v in row]
  return (ctypes.c_int64 * len(flat))(*flat)


def _call(library, ins, outs, in_strides, out_strides, dims, batch):
  return library._lib.soda_cuda_run_device_strided(
      ins, _strides(in_strides), outs, _strides(out_strides),
      (ctypes.c_int32 * 4)(*dims), batch, 0, None)


def test_entry_point_refuses_before_looking_for_a_device(library):
  """NULL pointers: -12; every broken rule: -4; absurd spans: -6.  None of
  them needs a device."""
  data = np.zeros(1 << 16, dtype=np.float32)
  ptr = (ctypes.c_void_p * 1)(data.ctypes.data)
  dims = (64, 40, 1, 1)
  dense = [(1, 64, 0, 0, 0)]
  lib = library._lib
  i64 = lambda rows: _strides(rows)
  i32 = (ctypes.c_int32 * 4)(*dims)
  assert lib.soda_cuda_run_device_strided(None, i64(dense), ptr, i64(dense),
                                          i32, 1, 0, None) == -12
  assert lib.soda_cuda_run_device_strided(ptr, None, ptr, i64(dense), i32, 1,
                                          0, None) == -12
  assert lib.soda_cuda_run_device_strided(ptr, i64(dense), ptr, None, i32, 1,
                                          0, None) == -12
  assert lib.soda_cuda_run_device_strided(ptr, i64(dense), ptr, i64(dense),
                                          None, 1, 0, None) == -12
  null = (ctypes.c_void_p * 1)(None)
  assert _call(library, null, ptr, dense, dense, dims, 1) == -12
  assert _call(library, ptr, null, dense, dense, dims, 1) == -12
  refused = [
      [(2, 64, 0, 0, 0)],            # stride[0] != 1
      [(1, 0, 0, 0, 0)],             # broadcast rows
      [(1, -64, 0, 0, 0)],           # negative
      [(1, 63, 0, 0, 0)],            # rows overlap
      [(1, 1, 0, 0, 0)],             # transposed-like: rows one cell apart
  ]
  for rows in refused:
    assert _call(library, ptr, ptr, rows, dense, dims, 1) == -4, rows
    assert _call(library, ptr, ptr, dense, rows, dims, 1) == -4, rows
  # items: the item stride must clear the last dimension's span
  assert _call(library, ptr, ptr, [(1, 64, 0, 0, 2559)], dense, dims, 2) == -4
  assert _call(library, ptr, ptr, [(1, 64, 0, 0, 0)], dense, dims, 2) == -4
  assert _call(library, ptr, ptr, [(1, 64, 0, 0, -2560)], dense, dims, 2) == -4
  assert _call(library, ptr, ptr, dense, dense, dims, 0) == -4   # batch < 1
  assert _call(library, ptr, ptr, dense, dense, (0, 40, 1, 1), 1) == -4
  assert _call(library, ptr, ptr, [(1, 1 << 42, 0, 0, 0)], dense, dims,
               1) == -6
  assert _call(library, ptr, ptr, [(1, 1 << 31, 0, 0, 0)], dense, dims,
               1) == -6


def test_valid_layouts_reach_the_device_lookup(library):
  """Pitched rows, a view's interior and channel-slice batches pass the
  checks: a machine without a device then answers -19."""
  import torch
  if torch.cuda.is_available():
    pytest.skip('a GPU is present')
  data = np.zeros(1 << 16, dtype=np.float32)
  ptr = (ctypes.c_void_p * 1)(data.ctypes.data)
  dims = (64, 40, 1, 1)
  for rows, batch in (([(1, 64, 0, 0, 0)], 1),
                      ([(1, 80, 0, 0, 0)], 1),
                      ([(1, 64, 7, 7, -5)], 1),     # ignored entries
                      ([(1, 100, 0, 0, 4000)], 3),
                      ([(1, 64, 0, 0, 2560)], 2)):
    assert _call(library, ptr, ptr, rows, rows, dims, batch) == -19, rows
  with pytest.raises(soda_cuda.CudaError) as info:
    library.run_device_strided([data.ctypes.data], [data.ctypes.data],
                               (64, 40), 1, [(1, 80)], [(1, 64)])
  assert info.value.code == -19
