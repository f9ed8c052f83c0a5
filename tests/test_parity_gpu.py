"""Parity of the CUDA path with the CPU oracle, through the C ABI (needs a GPU).

Bar (BASELINE.json north_star): bit-exact for integer stencils and — in the
default exact build (-fmad=false, reference operation order, double sqrt) —
for float stencils too.  Every comparison below is bitwise over the WHOLE
array: the valid region must match the oracle and the border must be 0.
"""
import glob
import os

import numpy as np
import pytest

import common
from soda import cuda as soda_cuda
from soda.codegen import cuda as codegen

pytestmark = pytest.mark.gpu

# name, iterate, dims, backend options
CASES = [
    # BASELINE config 1, the reference's own CPU-runnable case
    ('blur', 1, (2000, 1000), {}),
    # one per benchmark, dims not multiples of anything (plain-load path,
    # scalar stores, partial tiles, several tiles and chunks)
    ('blur', 1, (1037, 211), {}),
    ('sobel2d', 1, (1101, 157), {}),
    ('jacobi2d', 1, (1203, 95), {}),
    ('seidel2d', 2, (999, 130), {}),
    ('denoise2d', 1, (777, 141), {}),
    ('jacobi3d', 2, (101, 67, 45), {}),
    ('heat3d', 2, (131, 35, 52), {}),
    ('denoise3d', 1, (93, 41, 37), {}),
    # aligned dims: TMA path + 128-bit stores
    ('sobel2d', 1, (2048, 96), {}),
    ('jacobi2d', 2, (1536, 200), {}),
    ('jacobi2d', 7, (1024, 300), {'depth': 4}),      # 4 + 3 remainder
    ('jacobi2d', 16, (2048, 260), {'depth': 8}),
    ('seidel2d', 4, (1280, 160), {'depth': 2}),
    ('denoise2d', 1, (1024, 128), {}),
    ('jacobi3d', 4, (128, 64, 40), {'depth': 2}),
    ('heat3d', 3, (192, 48, 33), {'depth': 2}),      # 2 + 1 remainder
    ('heat3d', 1, (256, 128, 64), {}),
    ('denoise3d', 1, (128, 48, 24), {}),
    # millions of `1.0f / sqrt(x)` cells: the float-arithmetic rounding decision
    # (soda::RecipSqrtF32) and its FP64 fallback both occur
    ('denoise2d', 1, (4096, 1536), {}),
    ('denoise3d', 1, (256, 192, 96), {}),
    # every tuning knob of the backend (sodac --cuda-*): narrower vectors
    # (TMA boxes of 256 bytes), other block sizes, queue geometries, the
    # shared-memory ring family
    ('jacobi2d', 4, (1024, 128), {'vec': 2}),
    ('blur', 1, (2048, 128), {'vec': 4}),
    ('denoise2d', 1, (1024, 128), {'vec': 2}),
    ('sobel2d', 1, (2048, 200), {'threads': 64, 'groups': 8}),
    ('sobel2d', 1, (2048, 200), {'threads': 256, 'prefetch': 2}),
    ('jacobi2d', 8, (2048, 260), {'depth': 8, 'prefetch': 12, 'paired': 0}),
    ('jacobi2d', 6, (2048, 260), {'depth': 6, 'prefetch': 24}),
    ('blur', 1, (2048, 128), {'style': 'ring'}),
    ('heat3d', 2, (192, 48, 33), {'style': 'ring'}),
    ('heat3d', 2, (256, 64, 40), {'tile': [128, 16], 'threads': 256}),
    # the tuned 3-D tile of the 1024^3 runs: 48 rows, 24 warps
    ('heat3d', 4, (256, 100, 40), {'depth': 2, 'tile': [128, 48],
                                   'threads': 768}),
    ('jacobi3d', 2, (131, 97, 33), {'tile': [128, 48], 'threads': 768}),
    # a three-box input queue (one box in flight: less shared memory, more
    # resident warps — the tuned choice of denoise2d)
    ('jacobi2d', 8, (2048, 260), {'depth': 8, 'groups': 3}),
    ('sobel2d', 1, (1101, 157), {'groups': 3}),
    ('denoise2d', 1, (1024, 128), {'groups': 3, 'threads': 64}),
    # single-use locals spliced into their readers (--cuda-inline 1)
    ('denoise2d', 1, (777, 141), {'inline': 1}),
    ('denoise3d', 1, (93, 41, 37), {'inline': 1}),
    ('denoise3d', 1, (128, 48, 24), {'inline': 1, 'tile': [128, 32],
                                     'threads': 512, 'prefetch': 1}),
    ('sobel2d', 1, (1101, 157), {'inline': 1}),
]


def _library(name, iterate, options):
  return soda_cuda.compile_stencil(common.stencil(name, iterate),
                                   options=codegen.Options(**options))


def _ids(case):
  name, iterate, dims, options = case
  return '%s-it%d-%s%s' % (name, iterate, 'x'.join(map(str, dims)),
                           ''.join('-%s%s' % kv for kv in options.items()))


@pytest.mark.parametrize('case', CASES, ids=_ids)
def test_matches_oracle_on_reference_inputs(case):
  name, iterate, dims, options = case
  orc = common.oracle(name, iterate)
  inputs = orc.reference_inputs(dims)
  want = orc.run(inputs)
  got = _library(name, iterate, options).run(inputs)
  for k, (g, w) in enumerate(zip(got, want)):
    common.assert_bit_exact(g, w, '%s output %d' % (_ids(case), k))


@pytest.mark.parametrize('case', CASES[1:], ids=_ids)
def test_matches_oracle_on_random_inputs(case):
  name, iterate, dims, options = case
  orc = common.oracle(name, iterate)
  inputs = common.random_inputs(orc, dims, seed=len(name) + iterate)
  want = orc.run(inputs)
  got = _library(name, iterate, options).run(inputs)
  for k, (g, w) in enumerate(zip(got, want)):
    common.assert_bit_exact(g, w, '%s output %d' % (_ids(case), k))


@pytest.mark.parametrize('name,iterate,dims', [
    ('jacobi2d', 2, (1536, 200)), ('heat3d', 1, (256, 128, 64)),
    ('sobel2d', 1, (2048, 96))])
def test_plain_load_path_equals_tma_path(name, iterate, dims, monkeypatch):
  """Same aligned problem through both input paths gives identical bits."""
  orc = common.oracle(name, iterate)
  inputs = common.random_inputs(orc, dims, seed=7)
  library = _library(name, iterate, {})
  with_tma = library.run(inputs)
  assert library.stats['used_tma'] == 1
  monkeypatch.setenv('SODA_CUDA_NO_TMA', '1')
  without = library.run(inputs)
  assert library.stats['used_tma'] == 0
  for a, b in zip(with_tma, without):
    common.assert_bit_exact(a, b, name)


def test_device_buffers_zero_copy():
  """torch CUDA tensors go through buffer_t.dev without host copies."""
  import torch
  name, iterate, dims = 'jacobi2d', 3, (1024, 128)
  orc = common.oracle(name, iterate)
  inputs = common.random_inputs(orc, dims, seed=3)
  want = orc.run(inputs)
  library = _library(name, iterate, {})
  dev_in = [torch.from_numpy(a).cuda() for a in inputs]
  keep = [t.clone() for t in dev_in]
  dev_out = library.run(dev_in)
  torch.cuda.synchronize()
  assert library.stats['h2d_ms'] == 0 or library.stats['h2d_ms'] < 1.0
  common.assert_bit_exact(dev_out[0].cpu().numpy(), want[0], 'device run')
  assert torch.equal(dev_in[0], keep[0]), 'inputs must not be modified'


def test_chunking_does_not_change_results(monkeypatch):
  """Any split of the streamed dimension gives the same bits."""
  name, iterate, dims = 'seidel2d', 2, (640, 333)
  orc = common.oracle(name, iterate)
  inputs = common.random_inputs(orc, dims, seed=11)
  want = orc.run(inputs)
  library = _library(name, iterate, {})
  for chunks in ('1', '2', '7', '333'):
    monkeypatch.setenv('SODA_CUDA_CHUNKS', chunks)
    got = library.run(inputs)
    common.assert_bit_exact(got[0], want[0], 'chunks=' + chunks)


@pytest.mark.parametrize('name,iterate,dims', [
    ('heat3d', 2, (128, 64, 90)), ('jacobi2d', 8, (2048, 700))])
def test_a_run_cut_at_block_boundaries_is_the_same_run(name, iterate, dims):
  """soda_cuda_chunk_rows + soda_cuda_launch_chunked (what the multi-GPU
  slab runner builds its face and interior launches from): first block,
  last block and the rest, on three streams, equal the one-launch run."""
  import torch
  library = _library(name, iterate, {'depth': iterate})
  orc = common.oracle(name, iterate)
  inputs = common.random_inputs(orc, dims, seed=13)
  want = orc.run(inputs)
  dev_in = [torch.from_numpy(a).cuda() for a in inputs]
  dev_out = [torch.full_like(dev_in[0], 123.0)]
  rows = dims[-1]
  chunk = library.chunk_rows(iterate, dims, rows)
  assert 1 <= chunk <= rows and library.lead_rows(iterate) > 0
  if 2 * chunk >= rows:
    chunk = max(1, rows // 4)      # any cut works; keep three pieces
  region = library.valid_region(dims, iterate)
  lo, hi = [r[0] for r in region], [r[1] for r in region]
  torch.cuda.synchronize()
  streams = [torch.cuda.Stream() for _ in range(3)]
  pieces = [(0, chunk), (rows - chunk, rows), (chunk, rows - chunk)]
  for stream, (r0, r1) in zip(streams, pieces):
    library.launch(iterate, dev_in, dev_out, dims, r0, r1, lo, hi,
                   stream.cuda_stream, chunk)
  torch.cuda.synchronize()
  common.assert_bit_exact(dev_out[0].cpu().numpy(), want[0], name)


REFERENCE_ACCEPTED = sorted(glob.glob(os.path.join(common.GOLDEN_DIR,
                                                   'outputs', '*.npz')))


@pytest.mark.parametrize('path', REFERENCE_ACCEPTED, ids=os.path.basename)
def test_matches_outputs_the_reference_harness_accepted(path):
  """tests/golden/outputs/: what the reference's own `<app>_test` accepted
  with zero mismatches on its initialiser's inputs (oracle/make_golden.py).
  The CUDA path reproduces them bit for bit, whole arrays, without the
  reference at hand."""
  name, iterate, dims = common.golden_output_case(path)
  inputs = common.oracle(name, iterate).reference_inputs(dims)
  got = _library(name, iterate, {}).run(inputs)
  with np.load(path) as want:
    for k, g in enumerate(got):
      common.assert_bit_exact(g, want['out%d' % k], os.path.basename(path))


REF_CASES = [('blur', 1, (2000, 1000)), ('sobel2d', 1, (1101, 157)),
             ('jacobi2d', 3, (1536, 200)), ('seidel2d', 2, (999, 130)),
             ('denoise2d', 1, (1024, 128)), ('jacobi3d', 2, (128, 64, 40)),
             ('heat3d', 2, (131, 35, 52)), ('denoise3d', 1, (128, 48, 24))]


@pytest.mark.parametrize('name,iterate,dims', REF_CASES)
def test_reference_harness_accepts_the_cuda_path(name, iterate, dims):
  """The reference's own generated `<app>_test` (host.print_test, compiled
  unmodified under oracle/_ref/ in the build container) calls the CUDA
  library where the FPGA would run and counts mismatches against its golden
  loop: integers exact, floats within its 1e-5 relative tolerance."""
  import os
  import ref_harness
  lib = ref_harness.lib_path(name, iterate)
  if not os.path.exists(lib):
    pytest.skip('oracle/_ref was not built (needs /root/reference)')
  stencil = common.stencil(name, iterate)
  harness = ref_harness.RefHarness(lib, stencil)
  library = _library(name, iterate, {})
  assert harness.test(dims, library.run) == 0

  orc = common.oracle(name, iterate)

  def on_random_inputs(inputs):
    for array, fresh in zip(inputs, common.random_inputs(orc, dims, seed=8)):
      array[...] = fresh
    return library.run(inputs)
  assert harness.test(dims, on_random_inputs) == 0


@pytest.mark.parametrize('case', [
    ('blur', 1, (1037, 211), {}), ('jacobi2d', 7, (1024, 300), {'depth': 4}),
    ('jacobi2d', 16, (2048, 260), {'depth': 8}),
    ('seidel2d', 4, (1280, 160), {'depth': 2}),
    ('denoise2d', 1, (777, 141), {}), ('heat3d', 3, (192, 48, 33), {'depth': 2}),
    ('denoise3d', 1, (93, 41, 37), {})], ids=_ids)
def test_pipelined_host_path_is_bit_identical(case, monkeypatch):
  """Host buffers are processed in pieces of the streamed dimension with the
  copies overlapping the launches; any number of pieces gives the bits of the
  one-shot run."""
  name, iterate, dims, options = case
  orc = common.oracle(name, iterate)
  inputs = common.random_inputs(orc, dims, seed=21)
  want = orc.run(inputs)
  library = _library(name, iterate, options)
  for pieces in ('1', '2', '5', '13'):
    monkeypatch.setenv('SODA_CUDA_PIECES', pieces)
    got = library.run(inputs)
    for g, w in zip(got, want):
      common.assert_bit_exact(g, w, '%s pieces=%s' % (_ids(case), pieces))


def test_bad_elem_size_is_rejected():
  library = _library('jacobi2d', 2, {})
  wrong = [np.zeros((64, 64), dtype=np.float64)]
  with pytest.raises(TypeError):
    library.run(wrong)


@pytest.mark.parametrize('case', [
    ('jacobi2d', 7, (1024, 300), {'depth': 4}),
    ('denoise2d', 1, (777, 141), {}), ('heat3d', 3, (192, 48, 33), {'depth': 2}),
    ('sobel2d', 1, (2048, 96), {})], ids=_ids)
def test_pageable_and_pinned_host_buffers_give_the_same_bits(case, monkeypatch):
  """Pageable caller memory (numpy arrays, the reference harness' `new`ed
  arrays) goes through the runtime's pinned bounce buffers, a few host
  threads copying; pinned memory is handed to the copy engine as it is.  Tiny
  slots make every piece rotate through all of them, in and out."""
  import torch
  name, iterate, dims, options = case
  orc = common.oracle(name, iterate)
  inputs = common.random_inputs(orc, dims, seed=31)
  want = orc.run(inputs)
  library = _library(name, iterate, options)
  monkeypatch.setenv('SODA_CUDA_STAGE_KB', '64')
  for pieces, devices in (('1', None), ('3', None), ('2', '0,0')):
    monkeypatch.setenv('SODA_CUDA_PIECES', pieces)
    got = library.run(inputs, devices=devices)
    for g, w in zip(got, want):
      common.assert_bit_exact(g, w, '%s pageable, %s piece(s), devices %s' % (
          name, pieces, devices), any_nan=name == 'denoise2d')
  pinned_in = [torch.from_numpy(a).pin_memory() for a in inputs]
  pinned_out = [torch.empty(w.shape, dtype=t.dtype).pin_memory()
                for w, t in zip(want, [torch.from_numpy(w) for w in want])]
  library.run([t.numpy() for t in pinned_in], [t.numpy() for t in pinned_out])
  for g, w in zip(pinned_out, want):
    common.assert_bit_exact(g.numpy(), w, '%s pinned' % name,
                            any_nan=name == 'denoise2d')
  monkeypatch.setenv('SODA_CUDA_STAGING', '0')      # the driver's own staging
  got = library.run(inputs)
  for g, w in zip(got, want):
    common.assert_bit_exact(g, w, '%s unstaged' % name,
                            any_nan=name == 'denoise2d')
