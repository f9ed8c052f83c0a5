"""Batched runs on the GPU: every item of a batch equals, bit for bit over the
whole array, the one-grid run of that item alone (and the CPU oracle), and no
item reads another's cells."""
import numpy as np
import pytest

import common
import dim4_programs
import golden
import half_programs
import param_programs
import random_programs
import wide_type_programs
from soda import cuda as soda_cuda
from soda.codegen import cuda as codegen

pytestmark = pytest.mark.gpu

# kind, name, iterate (benchmarks) or None, dims, backend options, batch sizes
CASES = [
    # unaligned: plain loads, partial tiles; aligned: TMA and 128-bit stores
    ('bench', 'blur', 1, (1037, 211), {}, (1, 3, 5)),
    ('bench', 'sobel2d', 1, (2048, 96), {}, (1, 3, 5)),
    ('bench', 'heat3d', 2, (131, 35, 52), {}, (1, 3)),
    ('bench', 'heat3d', 1, (256, 128, 64), {}, (1, 3)),
    ('bench', 'denoise2d', 1, (777, 141), {}, (1, 3)),
    # several launches: depth 8 twice; depth 4 and a remainder of 3
    ('bench', 'jacobi2d', 16, (2048, 260), {'depth': 8}, (1, 3)),
    ('bench', 'jacobi2d', 7, (1024, 300), {'depth': 4}, (1, 3, 5)),
    ('bench', 'heat3d', 3, (192, 48, 33), {'depth': 2}, (1, 3)),
    ('bench', 'jacobi2d', 4, (1024, 128), {'vec': 2}, (1, 3, 5)),
    ('bench', 'blur', 1, (2048, 128), {'style': 'ring'}, (1, 3, 5)),
    ('bench', 'heat3d', 2, (192, 48, 33), {'style': 'ring'}, (1, 3)),
    ('dim4', 'heat4d', None, (140, 21, 10, 9), {}, (1, 3)),
    ('dim4', 'box4d', None, (256, 16, 12, 11), {}, (1, 3)),
    # outputs defined on different boxes (2-D; 3-D over three launches)
    ('multi', 100, None, None, {}, (1, 3)),
    ('multi', 105, None, None, {}, (1, 3)),
    ('param', 'conv3', None, (1061, 97), {}, (1, 3)),
    ('half', 'halfblur', None, (1024, 120), {}, (1, 3, 5)),
    # the configuration in which ptxas once dropped stores (DESIGN.md §7)
    ('wide', 'dbl3d', None, (131, 35, 29), {'tile': [64, 48], 'threads': 768},
     (1, 3)),
]


def _stencil(kind, name, iterate):
  if kind == 'bench':
    return common.stencil(name, iterate)
  return {'dim4': dim4_programs.stencil_of,
          'multi': random_programs.multi_stencil,
          'param': param_programs.stencil_of,
          'half': half_programs.stencil_of,
          'wide': wide_type_programs.stencil_of}[kind](name)


def _dims(case):
  kind, name, _, dims, _, _ = case
  if kind == 'multi':
    return random_programs.multi_dims(_stencil(kind, name, None), name)
  return dims


def _ids(case):
  kind, name, iterate, _, options, _ = case
  return '%s%s-%s%s' % (name, '-it%d' % iterate if iterate else '',
                        'x'.join(map(str, _dims(case))),
                        ''.join('-%s%s' % kv for kv in options.items()))


def _library(case):
  kind, name, iterate, _, options, _ = case
  return soda_cuda.compile_stencil(_stencil(kind, name, iterate),
                                   options=codegen.Options(**options))


def _params(orc, seed=5):
  rng = np.random.default_rng(seed)
  return [rng.random(size, dtype=np.float32).astype(dtype)
          for _, dtype, size in orc.params] or None


def _extremes(orc, dims, seed):
  """Inputs of NaN and infinities (floats) or the type's limits (integers)."""
  rng = np.random.default_rng(seed)
  shape = tuple(reversed(dims))
  arrays = []
  for dtype in orc.input_dtypes:
    if np.dtype(dtype).kind == 'f':
      values = np.array([np.nan, np.inf, -np.inf, 0.0,
                         np.finfo(dtype).max, -np.finfo(dtype).max], dtype)
    else:
      info = np.iinfo(dtype)
      values = np.array([info.min, info.max, 0, -1 if info.min else 1], dtype)
    arrays.append(rng.choice(values, size=shape))
  return arrays


def _check_items(library, orc, items, params, got, what, oracle=True):
  for b, inputs in enumerate(items):
    alone = library.run(inputs, params=params)
    want = orc.run(inputs, params=params) if oracle else alone
    for k, (g, a, w) in enumerate(zip(got, alone, want)):
      tag = '%s item %d of %d output %d' % (what, b, len(items), k)
      common.assert_bit_exact(g[b], a, tag + ' vs its one-grid run')
      common.assert_bit_exact(g[b], w, tag + ' vs the oracle', any_nan=True)


@pytest.mark.parametrize('case', CASES, ids=_ids)
def test_every_item_equals_its_one_grid_run(case):
  kind, name, iterate, _, _, batches = case
  dims = _dims(case)
  library = _library(case)
  orc = golden.Oracle(_stencil(kind, name, iterate))
  params = _params(orc) if library.params else None
  cells = int(np.prod(dims))
  for batch in batches:
    items = [common.random_inputs(orc, dims, seed=10 * batch + b)
             for b in range(batch)]
    stacked = [np.stack(arrays) for arrays in zip(*items)]
    got = library.run_batch(stacked, params=params)
    assert library.stats['cells'] == batch * cells
    _check_items(library, orc, items, params, got, _ids(case),
                 oracle=cells * batch <= (1 << 21))


@pytest.mark.parametrize('case', [c for c in CASES if c[1] in (
    'sobel2d', 'jacobi2d', 'box4d')], ids=_ids)
def test_plain_load_path_batches(case, monkeypatch):
  """The same batches with the TMA path switched off."""
  kind, name, iterate, _, _, _ = case
  dims = _dims(case)
  library = _library(case)
  orc = golden.Oracle(_stencil(kind, name, iterate))
  items = [common.random_inputs(orc, dims, seed=b) for b in range(3)]
  stacked = [np.stack(arrays) for arrays in zip(*items)]
  with_tma = library.run_batch(stacked)
  assert library.stats['used_tma'] == 1
  monkeypatch.setenv('SODA_CUDA_NO_TMA', '1')
  got = library.run_batch(stacked)
  assert library.stats['used_tma'] == 0
  for g, w in zip(got, with_tma):
    common.assert_bit_exact(g, w, _ids(case) + ' without TMA')
  _check_items(library, orc, items, None, got, _ids(case) + ' without TMA',
               oracle=False)


EXTREME_CASES = [CASES[i] for i in (0, 1, 3, 6, 9, 12, 14, 16)] + [
    ('wide', 'i64vol', None, (131, 35, 29), {}, ())]


@pytest.mark.parametrize('case', EXTREME_CASES, ids=_ids)
def test_an_item_of_extremes_does_not_leak(case):
  """The middle item of three holds NaN and infinities (integers: the type's
  limits); its neighbours stay bit-identical to their one-grid runs."""
  kind, name, iterate, _, _, _ = case
  dims = _dims(case)
  library = _library(case)
  orc = golden.Oracle(_stencil(kind, name, iterate))
  params = _params(orc) if library.params else None
  items = [common.random_inputs(orc, dims, seed=1),
           _extremes(orc, dims, seed=2),
           common.random_inputs(orc, dims, seed=3)]
  stacked = [np.stack(arrays) for arrays in zip(*items)]
  got = library.run_batch(stacked, params=params)
  for b in (0, 2):
    for k, (g, a) in enumerate(zip(got, library.run(items[b], params=params))):
      common.assert_bit_exact(g[b], a, '%s item %d output %d' % (
          _ids(case), b, k))


def test_batches_beyond_the_grid_limit():
  """65535 + 7 items of a tiny grid take two launches (gridDim.z <= 65535);
  item b is pattern b % 7, across the split too."""
  library = soda_cuda.compile_stencil(common.stencil('blur', 1))
  orc = common.oracle('blur', 1)
  dims, batch = (32, 16), 65535 + 7
  patterns = [common.random_inputs(orc, dims, seed=s)[0] for s in range(7)]
  wants = np.stack([library.run([p])[0] for p in patterns])
  which = np.arange(batch) % 7
  got, = library.run_batch([np.stack(patterns)[which]])
  assert library.stats['launches'] == 2
  same = common.bits(got) == common.bits(wants[which])
  bad = np.argwhere(~same.reshape(batch, -1).all(axis=1)).ravel()
  assert bad.size == 0, 'items differ: %s' % bad[:20]
  for b in range(65534, 65542):
    common.assert_bit_exact(got[b], wants[b % 7], 'item %d' % b)


def test_torch_tensors_zero_copy_and_device_entry_on_a_stream():
  import torch
  case = CASES[6]          # jacobi2d, depth 4 + 3: scratch of the whole batch
  dims, batch = _dims(case), 3
  library = _library(case)
  orc = golden.Oracle(_stencil(*case[:3]))
  items = [common.random_inputs(orc, dims, seed=40 + b)[0]
           for b in range(batch)]
  host = np.stack(items)
  want, = library.run_batch([host])
  dev_in = torch.from_numpy(host).cuda()
  keep = dev_in.clone()
  dev_out, = library.run_batch([dev_in])
  assert dev_out.is_cuda and dev_out.shape == dev_in.shape
  common.assert_bit_exact(dev_out.cpu().numpy(), want, 'run_batch on torch')
  stream = torch.cuda.Stream()
  out = torch.full_like(dev_in, 7.0)
  torch.cuda.synchronize()
  with torch.cuda.stream(stream):
    library.run_device_batch([dev_in], [out], dims, batch, 0,
                             stream.cuda_stream)
  stream.synchronize()
  common.assert_bit_exact(out.cpu().numpy(), want, 'run_device_batch')
  assert torch.equal(dev_in, keep), 'inputs must not be modified'


def test_single_item_batch_equals_run():
  stencil = common.stencil('sobel2d', 1)
  library = soda_cuda.compile_stencil(stencil)
  arrays = dict(zip([name for name, _ in library.inputs], common.random_inputs(
      common.oracle('sobel2d', 1), (1101, 157), seed=9)))
  alone = soda_cuda.run(stencil, arrays)
  batched = soda_cuda.run_batch(stencil, {k: v[None] for k, v in
                                          arrays.items()})
  assert alone.keys() == batched.keys()
  for name in alone:
    common.assert_bit_exact(batched[name][0], alone[name], name)
