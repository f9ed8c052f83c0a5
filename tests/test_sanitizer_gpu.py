"""compute-sanitizer over the kernels (needs a GPU): memcheck (out-of-bounds
and misaligned accesses, also of the TMA boxes at grid edges) and racecheck
(shared-memory hazards: the 3-D kernels share planes between warps with ONE
block barrier per step; the 2-D kernels read rows a TMA request deposited).

Cases: one 2-D program with fused iterations (register kernel, per-warp TMA
queue, paired f32x2), one 3-D program (shared plane rings), one multi-stage
3-D program, and a run sharded over two slabs (two host threads, two lanes).
Small ragged grids: the sanitizer slows a kernel down 10-100x.
"""
import os
import shutil
import subprocess
import sys

import pytest

import common

pytestmark = pytest.mark.gpu

CASES = [
    ('jacobi2d', 8, '531x60', None),
    ('heat3d', 4, '140x37x14', None),
    ('denoise3d', 1, '131x21x12', None),
    ('jacobi2d', 5, '300x90', '0,0'),
]
SANITIZER = shutil.which('compute-sanitizer') or \
    '/usr/local/cuda/bin/compute-sanitizer'


def _sanitizer_runs():
  """An installation may lack the tool or not let this user execute it."""
  try:
    return subprocess.run([SANITIZER, '--version'], stdout=subprocess.DEVNULL,
                          stderr=subprocess.DEVNULL, timeout=120,
                          check=False).returncode == 0
  except (OSError, subprocess.SubprocessError):
    return False


SANITIZER_RUNS = _sanitizer_runs()


def _run(tool, case, extra=()):
  name, iterate, dims, devices = case
  command = [SANITIZER, '--tool', tool, '--error-exitcode', '86',
             '--print-limit', '5'] + list(extra) + [
                 sys.executable, os.path.join(common.ROOT, 'tests',
                                              'sanitizer_case.py'),
                 name, str(iterate), dims] + ([devices] if devices else [])
  env = dict(os.environ)
  return subprocess.run(command, stdout=subprocess.PIPE,
                        stderr=subprocess.STDOUT, text=True, env=env,
                        timeout=900)


@pytest.mark.skipif(not SANITIZER_RUNS,
                    reason='compute-sanitizer not installed or not executable')
@pytest.mark.parametrize('case', CASES, ids=['%s-x%d-%s' % c[:3] for c in CASES])
def test_memcheck_is_clean(case):
  done = _run('memcheck', case)
  assert 'SANITIZER_CASE_OK' in done.stdout, done.stdout[-3000:]
  assert done.returncode == 0 and 'ERROR SUMMARY: 0 errors' in done.stdout, \
      done.stdout[-3000:]


@pytest.mark.skipif(not SANITIZER_RUNS,
                    reason='compute-sanitizer not installed or not executable')
@pytest.mark.parametrize('case', CASES[:3],
                         ids=['%s-x%d-%s' % c[:3] for c in CASES[:3]])
def test_racecheck_is_clean(case):
  done = _run('racecheck', case)
  assert 'SANITIZER_CASE_OK' in done.stdout, done.stdout[-3000:]
  assert done.returncode == 0 and 'RACECHECK SUMMARY: 0 hazards' in \
      done.stdout, done.stdout[-3000:]
