"""Programs and cases of the strided-array tests (shared by the CPU and GPU
tests and the prebuild tool)."""
from soda import core

import common
import dim4_programs
import half_programs
import random_programs

HEADER = 'kernel: %s\nburst width: 64\nunroll factor: 1\niterate: 1\n'
PROGRAMS = {
    # narrow integers: 8-bit in, 16-bit out
    'u8grad': HEADER % 'u8grad' + (
        'input uint8: a(64, *)\n'
        'output int16: o(0, 0) = a(1, 0) - a(-1, 0) + a(0, 1) - a(0, -1)\n'),
}


def stencil_of(kind, name, iterate=None):
  if kind == 'bench':
    return common.stencil(name, iterate)
  return {'dim4': dim4_programs.stencil_of,
          'multi': random_programs.multi_stencil,
          'half': half_programs.stencil_of,
          'int': lambda n: core.Stencil.from_text(PROGRAMS[n])}[kind](name)


# kind, name, iterate (benchmarks) or None, backend options
BUILDS = ([('bench', name, None, {}) for name in common.BENCHMARKS] + [
    ('bench', 'jacobi2d', 64, {}),
    ('bench', 'jacobi2d', 11, {'depth': 4}),
    ('bench', 'blur', 1, {'style': 'ring'}),
    ('bench', 'heat3d', 2, {'style': 'ring'}),
    ('dim4', 'heat4d', None, {}),
    ('multi', 100, None, {}),
    ('half', 'halfblur', None, {}),
    ('int', 'u8grad', None, {}),
])
