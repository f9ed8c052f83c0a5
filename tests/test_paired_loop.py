"""The steady-state loop of the paired 2-D kernel that bench.py times
(jacobi2d, 64 iterations, 8 per launch), read from its SASS (no GPU).

One trip is 9 rows x 4 cells x 8 iterations: the additions are 576 FADD2
(iterations k and k + 4 in one instruction), the products 288 scalar FMUL
(exact mode: nothing may be contracted into FFMA / FFMA2).  The trip carries
no store-path control flow and builds its register pairs without moves, so
the loop stays at or below 1250 instructions, and at or below 168 registers
the kernel keeps 3 blocks of 128 threads per SM.
"""
import os
import shutil
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, 'tools'))

pytestmark = pytest.mark.skipif(
    shutil.which('nvcc') is None or shutil.which('cuobjdump') is None,
    reason='needs nvcc and cuobjdump')


def test_jacobi2d_x64_steady_loop():
  import sass_count
  count, cells, _, ops, regs = sass_count.measure('jacobi2d:64')
  assert cells == 288
  assert ops['FADD2'] == 576
  assert ops['FMUL'] == 288
  assert not ops['FFMA'] and not ops['FFMA2'] and not ops['FMUL2']
  assert count <= 1250, ops
  assert regs is not None and regs <= 168
