#!/usr/bin/env python3
"""Static instruction count of the streaming loop of compiled SODA kernels
(no GPU needed): a proxy for issue-bound kernels while tuning the emitter.

  python tools/sass_count.py sobel2d:1 blur:1 jacobi2d:64:depth=8

Per kernel (kTma = true instance): SASS instructions in the streamed loop
(largest backward branch span), the cells one trip produces, instructions per
cell update, and the mix by issue pipe (IMAD/FFMA.. = fma, IADD3/LOP3/PRMT.. =
alu).  Paired 2-D kernels run their steady-state trips in a loop of their own,
without the tile-edge store path, and that loop is the one counted.  In the
other kernels the loop span includes the tile-edge store path, which
steady-state rows skip, so the per-cell figure is an upper bound.
"""
import collections
import os
import re
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [os.path.join(ROOT, 'soda-compiler_b200')]

from soda import core, cuda as soda_cuda          # noqa: E402
from soda.codegen import cuda as codegen          # noqa: E402
from soda.codegen.cuda import plan                # noqa: E402

LINE = re.compile(r'/\*([0-9a-f]{4,})\*/\s+(?:@!?U?P\w+\s+)?([A-Z][A-Z0-9_]*)'
                  r'([.\w]*)\s*(.*?);')
FMA = {'IMAD', 'FFMA', 'FMUL', 'FADD', 'FFMA2', 'FMUL2', 'FADD2', 'HFMA2',
       'IDP', 'DFMA', 'DMUL', 'DADD'}
MEM = {'LDS', 'STS', 'LDG', 'STG', 'LDSM', 'SHFL', 'UTMALDG', 'SYNCS', 'LDC',
       'LDCU', 'ATOMS', 'BAR'}
CTL = {'BRA', 'EXIT', 'BSSY', 'BSYNC', 'WARPSYNC', 'NOP', 'ENDCOLLECTIVE',
       'CALL', 'RET', 'YIELD', 'BREAK'}


def loop_stats(sass):
  insts = [(int(m.group(1), 16), m.group(2), m.group(4))
           for m in map(LINE.search, sass.splitlines()) if m]
  best = None
  exits = [addr for addr, op, _ in insts if op == 'EXIT']
  for addr, op, rest in insts:
    if op == 'BRA':
      target = re.search(r'0x([0-9a-f]+)', rest)
      if target and int(target.group(1), 16) < addr:
        span = (int(target.group(1), 16), addr)
        # ptxas parks cold blocks (the unconverged-warp form of every
        # shuffle) after the kernel's EXIT and branches back from there:
        # those are not loops
        if any(span[0] <= e <= span[1] for e in exits):
          continue
        if best is None or span[1] - span[0] > best[1] - best[0]:
          best = span
  if best is None:
    return len(insts), collections.Counter(), collections.Counter()
  body = [op for addr, op, _ in insts if best[0] <= addr <= best[1]]
  mix = collections.Counter(
      'fma' if op in FMA else 'mem' if op in MEM else 'ctl' if op in CTL
      else 'mufu' if op == 'MUFU' else 'alu' for op in body)
  return len(body), mix, collections.Counter(body)


def measure(text):
  """Compile ``name:iterate[:option=value..]``; returns (loop instructions,
  cell updates per trip, pipe mix, opcode counts, registers or None)."""
  parts = text.split(':')
  name, iterate = parts[0], int(parts[1])
  options = {}
  for item in parts[2:]:
    key, value = item.split('=')
    options[key] = ([int(v) for v in value.split('x')] if key == 'tile'
                    else value if key == 'style' else int(value))
  stencil = core.Stencil.from_file(
      os.path.join(ROOT, 'benchmarks', name + '.soda'), iterate=iterate)
  opts = codegen.Options(**options)
  path = soda_cuda.build(stencil, options=opts)
  sched = codegen.make_schedules(plan.extract_program(stencil), opts)[0]
  sass = subprocess.run(['cuobjdump', '-sass', path], stdout=subprocess.PIPE,
                        text=True, check=True).stdout
  chunks = re.split(r'\n\s*Function : ', sass)
  want = 'd%dILb1' % sched.depth
  body = next(c for c in chunks[1:] if want in c.split('\n')[0])
  regs = re.search(r'REG:(\d+)', subprocess.run(
      ['cuobjdump', '-res-usage', path], stdout=subprocess.PIPE, text=True,
      check=False).stdout.split(want)[1])
  count, mix, ops = loop_stats(body)
  period = (getattr(sched, 'flat_box', 0) or getattr(sched, 'trip', 0) or
            getattr(sched, 'period', 1))
  cells = period * sched.vec * sched.vecs_per_thread * sched.depth
  return count, cells, mix, ops, int(regs.group(1)) if regs else None


def main():
  for text in sys.argv[1:]:
    count, cells, mix, _, regs = measure(text)
    print('%-34s loop %5d inst / %4d cell updates = %6.2f per update  '
          '(fma %d alu %d mem %d ctl %d mufu %d)  regs %s' % (
              text, count, cells, count / cells, mix['fma'], mix['alu'],
              mix['mem'], mix['ctl'], mix['mufu'],
              regs if regs is not None else '?'))


if __name__ == '__main__':
  main()
