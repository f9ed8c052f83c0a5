#!/usr/bin/env python3
"""Compile, here (no GPU needed), every library the GPU tests and benchmarks
load, so that GPU-box time is not spent in nvcc.  Builds are cached in-tree
under soda-compiler_b200/_build/ and travel with the repository snapshot.

  python tools/prebuild.py [--clean] [case ...]     case = quick_bench syntax
"""
import concurrent.futures
import os
import shutil
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for sub in ('', 'tests', 'oracle', 'soda-compiler_b200', 'tools'):
  sys.path.insert(0, os.path.join(ROOT, sub))

from soda import core, cuda as soda_cuda          # noqa: E402
from soda.codegen import cuda as codegen          # noqa: E402


def build(job):
  """job: (benchmark name, iterate, options) or (label, stencil, options)."""
  name, iterate, options = job
  options = dict(options)
  fast = bool(options.pop('fast', 0))
  stencil = iterate if hasattr(iterate, 'app_name') else core.Stencil.from_file(
      os.path.join(ROOT, 'benchmarks', name + '.soda'), iterate=iterate)
  return soda_cuda.build(stencil, fast_math=fast,
                         options=codegen.Options(**options))


def main():
  args = sys.argv[1:]
  if '--clean' in args:
    args.remove('--clean')
    shutil.rmtree(soda_cuda.DEFAULT_BUILD_DIR, ignore_errors=True)
  jobs, untuned = [], []
  if args:
    import quick_bench
    for text in args:
      name, iterate, _, options = quick_bench.parse_case(text)
      for key in ('e2e', 'weak', 'feed', 'exchange'):
        options.pop(key, None)
      try:
        core.Stencil.from_file(os.path.join(
            ROOT, 'benchmarks', name + '.soda'), iterate=iterate)
      except Exception:   # pylint: disable=broad-except
        iterate = 1       # applied `iterate` times by the caller (denoise)
      jobs.append((name, iterate, options))
  else:
    import test_parity_gpu
    import test_slab_gpu
    import test_rsqrt_exact
    print('%-40s %s' % ('rsqrt check', os.path.relpath(
        test_rsqrt_exact.build_check(), ROOT)))
    import __graft_entry__ as entry
    for name, iterate, _, options in test_parity_gpu.CASES:
      jobs.append((name, iterate, options))
    for name, iterate, _ in test_parity_gpu.REF_CASES:
      jobs.append((name, iterate, {}))
    import common
    for path in test_parity_gpu.REFERENCE_ACCEPTED:
      jobs.append(common.golden_output_case(path)[:2] + ({},))
    marks = [m for m in
             test_parity_gpu.test_a_run_cut_at_block_boundaries_is_the_same_run
             .pytestmark if m.name == 'parametrize']
    for name, iterate, _ in marks[0].args[1]:
      jobs.append((name, iterate, {'depth': iterate}))
    for name, iterate, options, *_ in test_slab_gpu.CASES:
      jobs.append((name, iterate, options))
    import test_types_gpu
    for name, _, options in test_types_gpu.CASES:
      jobs.append((name, test_types_gpu.stencil_of(name), options))
    import param_programs
    for name, _, options in param_programs.CASES:
      jobs.append((name, param_programs.stencil_of(name), options))
    import random_programs
    for seed in random_programs.SEEDS:
      jobs.append(('rnd%d' % seed, random_programs.stencil_of(seed), {}))
    for name in random_programs.EXTRA:
      jobs.append((name, random_programs.extra_stencil(name), {}))
    import test_zz_random_programs_gpu as zz
    for seed in zz.MULTI_GPU_SEEDS:
      jobs.append(('multi%d' % seed, random_programs.multi_stencil(seed), {}))
    import test_math_calls
    jobs.append(('calls', core.Stencil.from_text(test_math_calls.TEXT), {}))
    import test_sharded_run_gpu
    for name, iterate, _ in test_sharded_run_gpu.CASES:
      jobs.append((name, iterate, {}))
    import test_sanitizer_gpu
    for name, iterate, _, _ in test_sanitizer_gpu.CASES:
      jobs.append((name, iterate, {}))
    import dim4_programs
    for name, _ in dim4_programs.CASES:
      jobs.append((name, dim4_programs.stencil_of(name), {}))
    import half_programs
    for name, _, options in half_programs.CASES:
      jobs.append((name, half_programs.stencil_of(name), options))
    import wide_type_programs
    for name, _, options in wide_type_programs.CASES:
      jobs.append((name, wide_type_programs.stencil_of(name), options))
    import test_quotients_gpu
    for name, (body, _) in test_quotients_gpu.PROGRAMS.items():
      stencil = core.Stencil.from_text(test_quotients_gpu.HEADER % name + body)
      jobs += [(name, stencil, {}), (name, stencil, {'style': 'ring'})]
    import test_fastmath_gpu
    for name, iterate, _ in test_fastmath_gpu.CASES:
      jobs.append((name, iterate, {'fast': 1}))
    import test_fullsize_gpu
    for name, iterate, _, _ in test_fullsize_gpu.CONFIGS:
      jobs.append((name, iterate, {}))
    import test_batch
    for name, make in test_batch.STENCILS:
      for style in ('reg', 'ring'):
        jobs.append((name, make(), {'style': style}))
    import test_batch_gpu
    for case in test_batch_gpu.CASES + test_batch_gpu.EXTREME_CASES:
      kind, name, iterate, _, options, _ = case
      jobs.append((str(name), test_batch_gpu._stencil(kind, name, iterate),
                   options))
    # the autotuner test times the planner's own choices, not tuned.json's
    import test_tune_gpu
    marks = [m for m in test_tune_gpu.test_tune_times_every_candidate
             .pytestmark if m.name == 'parametrize']
    for name, iterate, _, option_sets in marks[0].args[1]:
      untuned += [(name, iterate, options) for options in option_sets]
    jobs += [(n, None, {}) for n in entry.BENCHMARKS]
    jobs += [(n, it, {}) for n, it in entry.EXTRA_BUILDS]

  def label(job):
    stencil = job[1] if hasattr(job[1], 'app_name') else None
    return (job[0], stencil.iterate if stencil else job[1],
            sorted(job[2].items()))
  from soda import fpga_layout
  kept = {os.path.dirname(os.path.abspath(fpga_layout.build()))}
  for group, env in ((jobs, None), (untuned, '0')):
    unique = []
    for job in group:
      if label(job) not in [label(j) for j in unique]:
        unique.append(job)
    if env is not None:
      os.environ['SODA_CUDA_TUNED'] = env
    with concurrent.futures.ThreadPoolExecutor(max_workers=8) as pool:
      for job, path in zip(unique, pool.map(build, unique)):
        print('%-40s %s' % (label(job), os.path.relpath(path, ROOT)))
        kept.add(os.path.dirname(os.path.abspath(path)))
    os.environ.pop('SODA_CUDA_TUNED', None)
  if not args:
    # a full prebuild names every library the tests and benches load: builds
    # of earlier source states (other hashes) only fatten the GPU snapshot
    import re
    stale = [os.path.join(soda_cuda.DEFAULT_BUILD_DIR, name)
             for name in os.listdir(soda_cuda.DEFAULT_BUILD_DIR)
             if re.fullmatch(r'\w+-[0-9a-f]{12}', name)]
    stale = [path for path in stale if path not in kept and any(
        f.startswith('libsoda_') for f in os.listdir(path))]
    for path in stale:
      shutil.rmtree(path, ignore_errors=True)
    print('removed %d stale build(s)' % len(stale))


if __name__ == '__main__':
  main()
