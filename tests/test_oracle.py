"""Pinning the CPU oracle (oracle/golden.py) — the checker of every GPU test.

1. Against committed golden vectors (tests/golden/outputs/*.npz): outputs that
   the reference's own generated ``<app>_test`` harness accepted with zero
   mismatches when they were made (oracle/make_golden.py).
2. Where /root/reference is present: against that unmodified harness directly,
   on the reference's ramp inputs AND on random inputs (the hook overwrites the
   harness' input arrays before the golden loop reads them), with a negative
   control proving the harness notices a single wrong cell.
3. Independently of any C code: a numpy restatement for the float stencils
   whose lowered expression is simple enough to transcribe by hand.
"""
import glob
import os

import numpy as np
import pytest

import common
import golden

VECTORS = sorted(glob.glob(os.path.join(common.GOLDEN_DIR, 'outputs',
                                        '*.npz')))


@pytest.mark.parametrize('path', VECTORS, ids=os.path.basename)
def test_oracle_reproduces_reference_accepted_outputs(path):
  name, iterate, dims = common.golden_output_case(path)
  orc = common.oracle(name, iterate)
  got = orc.run(orc.reference_inputs(dims))
  with np.load(path) as want:
    for k, g in enumerate(got):
      common.assert_bit_exact(g, want['out%d' % k], os.path.basename(path))


REF_CASES = [('blur', 1, (72, 33)), ('sobel2d', 1, (40, 37)),
             ('jacobi2d', 3, (50, 41)), ('seidel2d', 2, (45, 38)),
             ('denoise2d', 1, (36, 31)), ('jacobi3d', 2, (17, 15, 14)),
             ('heat3d', 2, (18, 14, 13)), ('denoise3d', 1, (15, 14, 13))]


@pytest.mark.skipif(not common.have_reference(),
                    reason='needs /root/reference')
@pytest.mark.parametrize('name,iterate,dims', REF_CASES)
def test_unmodified_reference_harness_accepts_the_oracle(name, iterate, dims):
  import ref_harness
  soda_file = os.path.join(common.REFERENCE_DIR, 'tests', 'src',
                           name + '.soda')
  stencil = golden.stencil_from_file(soda_file, iterate)
  harness = ref_harness.RefHarness(ref_harness.build_ref(soda_file, iterate),
                                   stencil)
  orc = common.oracle(name, iterate)
  assert harness.test(dims, orc.run) == 0

  def on_random_inputs(inputs):
    for array, fresh in zip(inputs, common.random_inputs(orc, dims, seed=5)):
      array[...] = fresh          # the harness' golden loop reads these too
    return orc.run(inputs)
  assert harness.test(dims, on_random_inputs) == 0

  def one_wrong_cell(inputs):
    outputs = orc.run(inputs)
    middle = tuple(n // 2 for n in outputs[0].shape)
    outputs[0][middle] = 7 if outputs[0][middle] != 7 else 9
    return outputs
  assert harness.test(dims, one_wrong_cell) == 1


def test_numpy_restatement_jacobi2d():
  orc = common.oracle('jacobi2d', 2)
  (a,) = common.random_inputs(orc, (37, 29), seed=1)
  want = orc.run([a])[0]
  f = np.float32

  def sweep(t):    # (t1(0,1) + t1(1,0) + t1(0,0) + t1(0,-1) + t1(-1,0)) * 0.2f
    out = np.zeros_like(t)
    out[1:-1, 1:-1] = ((((t[2:, 1:-1] + t[1:-1, 2:]) + t[1:-1, 1:-1]) +
                        t[:-2, 1:-1]) + t[1:-1, :-2]) * f(0.2)
    return out
  got = sweep(sweep(a))
  valid = np.zeros_like(got)
  valid[2:-2, 2:-2] = got[2:-2, 2:-2]
  common.assert_bit_exact(valid, want, 'numpy jacobi2d')


def test_numpy_restatement_blur_integer_semantics():
  orc = common.oracle('blur', 1)
  (a,) = common.random_inputs(orc, (33, 21), seed=2)
  want = orc.run([a])[0]
  wide = a.astype(np.int32)       # uint16 operands promote to int
  bx = np.zeros_like(wide)
  bx[:-2, :] = (wide[:-2, :] + wide[1:-1, :] + wide[2:, :]) // 3
  bx = bx.astype(np.uint16).astype(np.int32)     # stored as uint16
  by = np.zeros_like(wide)
  by[:, :-2] = (bx[:, :-2] + bx[:, 1:-1] + bx[:, 2:]) // 3
  got = np.zeros_like(a)
  got[:-2, :-2] = by[:-2, :-2].astype(np.uint16)
  common.assert_bit_exact(got, want, 'numpy blur')


def test_sobel_follows_the_reference_lowering_not_the_dsl_text():
  """65535 - (mx*mx + my*my) is lowered to 65535 - (mx*mx) + (my*my)
  (SURVEY.md 0.4); the oracle must follow the lowered form."""
  orc = common.oracle('sobel2d', 1)
  (a,) = common.random_inputs(orc, (20, 17), seed=4)
  want = orc.run([a])[0]
  w = a.astype(np.int64)
  c = lambda dy, dx: w[1 + dy:w.shape[0] - 1 + dy, 1 + dx:w.shape[1] - 1 + dx]
  mx = ((c(-1, 1) - c(-1, -1)) + (c(0, 1) - c(0, -1)) * 3 +
        (c(1, 1) - c(1, -1))).astype(np.uint16).astype(np.int64)
  my = ((c(1, -1) - c(-1, -1)) + (c(1, 0) - c(-1, 0)) * 3 +
        (c(1, 1) - c(-1, 1))).astype(np.uint16).astype(np.int64)
  lowered = (65535 - mx * mx + my * my).astype(np.uint16)
  common.assert_bit_exact(want[1:-1, 1:-1], lowered, 'sobel lowered form')
  as_written = (65535 - (mx * mx + my * my)).astype(np.uint16)
  assert not np.array_equal(want[1:-1, 1:-1], as_written)


def test_partial_iterations_and_border():
  orc = common.oracle('jacobi2d', 5)
  (a,) = common.random_inputs(orc, (40, 30), seed=9)
  three = orc.run([a], iterate=3)[0]
  direct = common.oracle('jacobi2d', 3).run([a])[0]
  common.assert_bit_exact(three, direct, 'iterate override')
  assert not three[:3].any() and not three[:, :3].any()
  assert three[3:-3, 3:-3].all()


@pytest.mark.skipif(not common.have_reference(),
                    reason='needs /root/reference')
@pytest.mark.parametrize('name', ['chain2', 'chain3d'])
def test_reference_harness_accepts_the_oracle_on_chained_outputs(name,
                                                                 tmp_path):
  """Two outputs, the second reading the first, iterated (the Stencil IR's
  `<input>_iter1` alias): the unmodified reference's generated harness judges
  the oracle's outputs — ramp and random inputs — and notices one wrong
  cell."""
  import random_programs as rp
  import ref_harness
  soda_file = tmp_path / (name + '.soda')
  soda_file.write_text(rp.EXTRA[name][0])
  stencil = golden.stencil_from_file(str(soda_file))
  harness = ref_harness.RefHarness(
      ref_harness.build_ref(str(soda_file), None, force=True), stencil)
  orc = golden.Oracle(stencil)
  dims = (60, 40) if stencil.dim == 2 else (24, 20, 18)
  assert harness.test(dims, orc.run) == 0

  def on_random_inputs(inputs):
    for array, fresh in zip(inputs, common.random_inputs(orc, dims, seed=5)):
      array[...] = fresh
    return orc.run(inputs)
  assert harness.test(dims, on_random_inputs) == 0

  def one_wrong_cell(inputs):
    outputs = orc.run(inputs)
    outputs[1][tuple(n // 2 for n in outputs[1].shape)] += 1
    return outputs
  assert harness.test(dims, one_wrong_cell) == 1


@pytest.mark.skipif(not common.have_reference(),
                    reason='needs /root/reference')
@pytest.mark.parametrize('seed', [0, 1, 5, 7, 13])
def test_reference_harness_accepts_the_oracle_on_random_programs(seed,
                                                                 tmp_path):
  """Beyond the benchmarks: seeded random programs (integer and float types,
  a stage of another width, 2-D / 3-D, up to 4 iterations) — the unmodified
  reference parses them, generates its golden harness, and that harness
  accepts the oracle's outputs (integers compare exactly, host.py:1118-1146)."""
  import random_programs as rp
  import ref_harness
  soda_file = tmp_path / ('rnd%d.soda' % seed)
  soda_file.write_text(rp.program_text(seed))
  stencil = golden.stencil_from_file(str(soda_file))
  harness = ref_harness.RefHarness(
      ref_harness.build_ref(str(soda_file), None, force=True), stencil)
  orc = golden.Oracle(stencil)
  dims = (60, 40) if stencil.dim == 2 else (24, 20, 18)
  assert harness.test(dims, orc.run) == 0

  def on_random_inputs(inputs):
    for array, fresh in zip(inputs, common.random_inputs(orc, dims, seed=5)):
      array[...] = fresh
    return orc.run(inputs)
  assert harness.test(dims, on_random_inputs) == 0
