"""Strided device arrays on the GPU: a run on views, pitched rows and channel
slices equals, bit for bit, ``run_device_batch`` on ``.contiguous()`` copies
of the same views (those dense runs are pinned to the oracle by the other
GPU tests).  Every parent array is filled with a sentinel outside its view
(NaN, or bytes of 0x5A): none may reach a result, and every cell of an output
parent outside its view must be left as it was."""
import numpy as np
import pytest

import common
import strided_programs
from soda import cuda as soda_cuda
from soda.codegen import cuda as codegen

pytestmark = pytest.mark.gpu


def _library(kind, name, iterate=None, **options):
  return soda_cuda.compile_stencil(
      strided_programs.stencil_of(kind, name, iterate),
      options=codegen.Options(**options))


# ---- layouts: shape -> (parent shape, index of the view in the parent) -----

def dense(shape):
  return shape, tuple(slice(None) for _ in shape)


def pitched(*pads):
  """Each of the last len(pads) axes padded by that many cells."""
  def layout(shape):
    lead = len(shape) - len(pads)
    parent = shape[:lead] + tuple(n + p for n, p in zip(shape[lead:], pads))
    return parent, tuple(slice(0, n) for n in shape)
  return layout


def interior(offset, pad):
  """The view starts `offset` cells into every non-item axis of a parent
  `pad` cells larger."""
  def layout(shape):
    lead = len(shape) - len(offset)
    parent = shape[:lead] + tuple(n + pad for n in shape[lead:])
    return parent, tuple(slice(None) for _ in range(lead)) + tuple(
        slice(o, o + n) for o, n in zip(offset, shape[lead:]))
  return layout


def channel(channels, c):
  """x[:, c] of a (B, channels, ...) parent: a batch of items
  channels x prod(dims) apart."""
  def layout(shape):
    return (shape[0], channels) + shape[1:], (slice(None), c)
  return layout


# ---- one run -----------------------------------------------------------------

def _torch_dtype(haoda_type):
  import torch
  return torch.from_numpy(np.empty(0, soda_cuda.NUMPY_TYPES[haoda_type])).dtype


def _bits(tensor):
  import torch
  return tensor.view({1: torch.uint8, 2: torch.int16, 4: torch.int32,
                      8: torch.int64}[tensor.element_size()])


def _place(shape, haoda_type, layout):
  import torch
  parent_shape, index = layout(shape)
  parent = torch.empty(parent_shape, dtype=_torch_dtype(haoda_type),
                       device='cuda')
  if parent.dtype.is_floating_point:
    parent.fill_(float('nan'))
  else:
    parent.view(torch.uint8).fill_(0x5A)
  return parent, parent[index], index


def _random(haoda_type, shape, rng):
  dtype = soda_cuda.NUMPY_TYPES[haoda_type]
  if np.dtype(dtype).kind == 'f':
    return rng.random(shape, dtype=np.float32).astype(dtype)
  info = np.iinfo(dtype)
  return rng.integers(info.min, int(info.max) + 1, size=shape,
                      dtype=np.int64).astype(dtype)


def run_and_check(library, dims, in_layout, out_layout=None, batch=None,
                  iterate=0, stream=None, seed=0):
  """Runs `library` on views laid out by `in_layout` / `out_layout` (batch
  None: one grid) and checks it against the dense run; returns the stats."""
  import torch
  out_layout = out_layout or in_layout
  shape = ((batch,) if batch else ()) + tuple(reversed(dims))
  rng = np.random.default_rng(seed)
  ins, in_parents = [], []
  for _, haoda_type in library.inputs:
    parent, view, _ = _place(shape, haoda_type, in_layout)
    view.copy_(torch.from_numpy(_random(haoda_type, shape, rng)))
    ins.append(view)
    in_parents.append((parent, parent.clone()))
  outs, out_parents = [], []
  for _, haoda_type in library.outputs:
    parent, view, index = _place(shape, haoda_type, out_layout)
    outs.append(view)
    out_parents.append((parent, parent.clone(), index))
  want = [torch.empty(shape, dtype=o.dtype, device='cuda') for o in outs]
  library.run_device_batch([v.contiguous() for v in ins], want, dims,
                           batch or 1, iterate)
  torch.cuda.synchronize()
  got = library.run_strided(ins, outs, batched=bool(batch), iterate=iterate,
                            stream=stream)
  assert all(g is o for g, o in zip(got, outs))
  torch.cuda.synchronize()
  stats = library.stats
  for k, (parent, before, index) in enumerate(out_parents):
    expected = before.clone()
    expected[index] = want[k]
    same = _bits(parent) == _bits(expected)
    if not bool(same.all()):
      bad = same.logical_not().nonzero()
      raise AssertionError('%s output %d: %d cells differ, first at %s' % (
          library.app_name, k, bad.shape[0], tuple(bad[0].tolist())))
  for parent, before in in_parents:
    assert torch.equal(_bits(parent), _bits(before)), 'inputs were modified'
  return stats


DIMS = {2: (1024, 200), 3: (128, 40, 36)}


@pytest.mark.parametrize('name', common.BENCHMARKS)
def test_benchmarks_on_pitched_rows(name):
  """Rows padded by 16 cells (a multiple of 16 B: TMA) and by 3 cells
  (plain loads); 3-D planes padded too."""
  library = _library('bench', name)
  dims = DIMS[library.dim]
  pads = (16,) if library.dim == 2 else (3, 16)
  stats = run_and_check(library, dims, pitched(*pads))
  assert stats['used_tma'] == 1
  odd = (3,) if library.dim == 2 else (1, 3)
  stats = run_and_check(library, dims, pitched(*odd), seed=1)
  assert stats['used_tma'] == 0


@pytest.mark.parametrize('name', ('jacobi2d', 'sobel2d', 'denoise2d',
                                  'heat3d', 'denoise3d'))
def test_interior_views_with_an_unaligned_base(name):
  library = _library('bench', name)
  dims = DIMS[library.dim]
  offset = (2, 1) if library.dim == 2 else (2, 3, 1)
  stats = run_and_check(library, dims, interior(offset, 5))
  assert stats['used_tma'] == 0
  # a strided input with a dense output, and the reverse
  run_and_check(library, dims, interior(offset, 5), dense, seed=1)
  run_and_check(library, dims, dense, pitched(*(3,) * (library.dim - 1)),
                seed=2)


def test_odd_widths_in_a_pitched_parent_get_tma():
  """Rows of 1021 float cells are not 16 B multiples: a dense grid takes
  plain loads, the same grid in rows 512 B apart takes TMA."""
  library = _library('bench', 'jacobi2d')
  assert run_and_check(library, (1021, 300), dense)['used_tma'] == 0
  assert run_and_check(library, (1021, 300), pitched(3))['used_tma'] == 1
  library = _library('bench', 'heat3d')
  assert run_and_check(library, (131, 20, 18), dense)['used_tma'] == 0
  assert run_and_check(library, (131, 20, 18),
                       pitched(0, 125))['used_tma'] == 1


def test_channel_slices_as_batches():
  library = _library('bench', 'jacobi2d')
  run_and_check(library, (512, 96), channel(4, 2), batch=3)
  library = _library('bench', 'heat3d')
  run_and_check(library, (64, 20, 18), channel(3, 1), batch=2)
  run_and_check(library, (64, 20, 18), channel(3, 0), dense, batch=2)


def test_a_batch_beyond_the_grid_limit():
  """65535 + 7 small pitched items take two launches (item_begin)."""
  library = _library('bench', 'blur', 1)
  stats = run_and_check(library, (32, 16), pitched(8), batch=65535 + 7)
  assert stats['launches'] == 2


@pytest.mark.parametrize('iterate,options', [(11, {'depth': 4}), (64, {})])
def test_several_launches_alternate_dense_scratch_and_strided_outputs(
    iterate, options):
  library = _library('bench', 'jacobi2d', iterate, **options)
  run_and_check(library, (1024, 260), pitched(16))
  run_and_check(library, (1024, 260), interior((3, 1), 4), pitched(5),
                seed=1)
  run_and_check(library, (512, 96), channel(3, 1), batch=2, seed=2)


def test_ring_family_and_the_plain_load_switch(monkeypatch):
  blur = _library('bench', 'blur', 1, style='ring')
  assert run_and_check(blur, (1024, 128), pitched(16))['used_tma'] == 1
  run_and_check(blur, (1024, 128), interior((1, 2), 4), seed=1)
  heat = _library('bench', 'heat3d', 2, style='ring')
  run_and_check(heat, (192, 48, 33), pitched(1, 16))
  run_and_check(heat, (192, 48, 33), interior((1, 2, 3), 4), seed=1)
  jacobi = _library('bench', 'jacobi2d')
  monkeypatch.setenv('SODA_CUDA_NO_TMA', '1')
  assert run_and_check(jacobi, (1024, 200), pitched(16))['used_tma'] == 0
  assert run_and_check(heat, (192, 48, 33), pitched(1, 16))['used_tma'] == 0


@pytest.mark.parametrize('kind,name,dims', [
    ('dim4', 'heat4d', (140, 21, 10, 9)),
    ('multi', 100, None),
    ('half', 'halfblur', (1024, 120)),
    ('int', 'u8grad', (1000, 77)),
    ('bench', 'sobel2d', (1000, 77)),
])
def test_other_programs_and_types(kind, name, dims):
  """4-D; outputs with different valid regions; half; uint8 -> int16 and
  uint16 grids."""
  import random_programs
  library = _library(kind, name)
  if dims is None:
    dims = random_programs.multi_dims(
        strided_programs.stencil_of(kind, name), name)
  pads = (16,) * (library.dim - 1)
  run_and_check(library, dims, pitched(*pads))
  run_and_check(library, dims, interior((1,) * library.dim, 3), seed=1)
  run_and_check(library, dims, pitched(*pads), batch=2, seed=2)


def test_side_stream_and_the_module_shortcut():
  import torch
  library = _library('bench', 'jacobi2d')
  stream = torch.cuda.Stream()
  torch.cuda.synchronize()
  run_and_check(library, (1024, 200), pitched(16), stream=stream)
  with torch.cuda.stream(stream):       # the current stream is used
    run_and_check(library, (1024, 200), interior((2, 1), 5), seed=1)
  parent = torch.rand(200, 1040, device='cuda')
  view = parent[:, :1024]
  got = soda_cuda.run_strided(common.stencil('jacobi2d'), {'t1': view})
  name = library.outputs[0][0]
  assert got[name].is_contiguous() and got[name].shape == view.shape
  want = torch.empty_like(got[name])
  library.run_device([view.contiguous()], [want], (1024, 200))
  torch.cuda.synchronize()
  assert torch.equal(_bits(got[name]), _bits(want))
