"""Emit the register-streaming sm_100a kernel of a SODA program.

The kernel realises a ``plan.RegSchedule``: every thread walks the streamed
dimension with ``vec`` cells of its own, keeps the last few planes of every
tensor of the fused chain it needs again in **registers**, takes dimension-0
neighbours from the adjacent lanes with **warp shuffles**, and goes through
shared memory only for neighbours in the other tiled dimensions (3-D: y +- 1).
Per stage the reference-lowered expression (``Node.c_expr`` with Refs swapped
for storage, the recipe of the golden loop's ``mutate_load_for_host``,
reference src/soda/codegen/xilinx/host.py:1093-1117; FPGA counterpart
src/soda/codegen/xilinx/hls_kernel.py:487-489) is spliced in once per cell of
the thread's vector.

2-D programs  no block barrier.  A block is ``warps`` independent strips of
              32 x vec cells.  Each warp owns a shared-memory ring of input
              rows: one elected lane requests row i + prefetch by TMA
              (cp.async.bulk.tensor.2d, out-of-grid cells arrive as 0) on the
              slot's mbarrier, every lane takes its cells of row i with one
              128-bit shared load.  Rows in flight cost no registers, so the
              queue is as deep as the HBM latency needs.  Outputs leave with
              128-bit streaming stores.  Shapes TMA cannot describe take
              element-wise loads one row ahead instead (kTma = false).
3-D programs  input planes arrive by TMA (cp.async.bulk.tensor + mbarrier) in
              a shared ring as in kernel.py; each thread copies its own cells
              of the newest plane into its history; stages whose results are
              read at y +- 1 also write a shared plane; one __syncthreads()
              per step.

The streamed loop is unrolled ``period`` times so that history slots are
compile-time register names: the row computed k steps ago sits in slot
``(phase - k) mod period``.
"""
import collections
import re

from haoda import util
from soda.codegen.cuda import kernel as kernel_mod
from soda.codegen.cuda import plan as plan_mod

_TMA_MAX_BOX = 256


def kernel_name(sched):
  return 'soda_%s_d%d' % (sched.program.app_name, sched.depth)


class Layout:
  """Dynamic shared memory of a register-streaming kernel (3-D only)."""

  def __init__(self, sched):
    self.sched = sched
    self.guard = -(-sched.guard_elems * 8 // 128) * 128
    self.ring_depth = {}
    self.ring_offset = {}
    loaded = [n for n in sched.inputs if n.ring_depth]
    self.in_depth = max([n.ring_depth for n in loaded] + [1])
    offset = self.guard
    for node in sched.nodes:
      if not node.ring_depth:
        continue
      depth = self.in_depth if node.is_input else node.ring_depth
      self.ring_depth[node.index] = depth
      self.ring_offset[node.index] = offset
      ring = depth * sched.ring_pitch * node.elem_size
      offset += -(-ring // 128) * 128
    offset += self.guard
    self.bar_offset = offset
    if loaded:
      offset += -(-8 * self.in_depth // 128) * 128
    self.total = offset if self.ring_offset else 0
    self.loaded_inputs = loaded
    if sched.sdim == 1:
      # per-warp input queue: `slots` rows of every input that is read, then
      # one mbarrier per slot
      self.slots = sched.flat_slots
      self.box_rows = sched.flat_box
      self.groups = self.slots // self.box_rows
      loaded = self.loaded_inputs = [n for n in sched.inputs
                                     if n.hist_oldest is not None]
      self.row_bytes = {n.index: sched.tile[0] * n.elem_size for n in loaded}
      self.queue_offset, offset = {}, 0
      for node in loaded:
        self.queue_offset[node.index] = offset
        offset += -(-self.slots * self.row_bytes[node.index] // 128) * 128
      self.warp_bytes = offset
      self.bar_offset = offset * sched.warps
      self.total = self.bar_offset + -(-8 * self.groups * sched.warps // 128) * 128
    self.plane_bytes = {n.index: sched.plane_elems * n.elem_size
                        for n in loaded}
    self.box0 = sched.tile[0]
    self.boxes_per_row = 1
    if loaded:
      if sched.tile[0] > _TMA_MAX_BOX:
        raise util.SemanticError('tile width %d exceeds the TMA box limit' %
                                 sched.tile[0])
      for extent in sched.tile[1:]:
        if extent > _TMA_MAX_BOX:
          raise util.SemanticError('tile extent %d exceeds the TMA box limit'
                                   % extent)


def _log2(n):
  return n.bit_length() - 1


def _render(stage, ref_code, k, split_top=False):
  """``(let lines, expression)`` of cell ``k`` of the thread's vector."""
  return stage.render(lambda load: ref_code(load, k), call_prefix='soda_fn_',
                      let_prefix='let_', split_top=split_top)


def batches_rare_paths(stage):
  """Float statements that are a quotient at their top (`g = 1.0f / sqrt(..)`,
  `r1 = (..) / (..)`): an IEEE float division and the exact ``a / sqrt(x)``
  each end in a rarely taken branch (operands outside the quick sequence's
  range; an undecided rounding), and a branch per cell keeps the compiler from
  interleaving the cells' dependent chains — the exact denoise kernels waited
  two cycles per instruction on them.  Such a statement is emitted as: the
  numerators and denominators of all cells of the vector; ``soda::div_try`` on
  each pair — the quick sequence, unconditionally, raising ``rare`` where it
  does not apply; then, if ``rare``, the plain quotient of every pair.  One
  branch per vector, and what it guards needs only the pairs.

  (A quotient spliced into another statement keeps the compiler's division:
  computing it ahead of its reader the same way, one variable per cell, cost
  denoise3d 4 % at its 73 registers per thread — 122.7 vs 128.3 GCell/s,
  capture r3n.)"""
  return stage.c_type == 'float' and stage.top_division()


_INT_TYPES = {'uint8', 'uint16', 'uint32', 'uint64', 'int8', 'int16', 'int32',
              'int64'}
# + - * on tensor cells and plain integer literals: the low w bits of such an
# expression depend only on the low w bits of its operands
_RING_TOKEN = re.compile(r'\s+|[-+*()]|@|(?:0[xX][0-9a-fA-F]+|\d+)[uU]?(?![.\w])')


def ring_expression(stage, program):
  """Is the stage's lowered C expression a polynomial (+ - *) in integer
  tensor cells and integer literals?  Judged on the emitted text, which is
  what the reference evaluates (its parenthesisation is not the tree's)."""
  if stage.lets or program.types[stage.name] not in _INT_TYPES:
    return False
  for load in stage.loads:
    if program.types.get(load.parent) not in _INT_TYPES:
      return False
  _, text = stage.render(lambda load: '@')
  pos = 0
  while pos < len(text):
    match = _RING_TOKEN.match(text, pos)
    if not match:
      return False
    pos = match.end()
  return True


class _Emitter:

  def __init__(self, p, sched):
    self.p = p
    self.sched = sched
    # Lazy truncation.  An 8- or 16-bit integer tensor is kept in 32-bit
    # registers whose upper bits are unspecified ("loose"): an input cell is
    # the loaded word shifted down, a stage result is not narrowed.  A stage
    # that is a polynomial in its operands and no wider than them reads loose
    # values as they are (arithmetic modulo 2^32 agrees with the reference's
    # int arithmetic on the bits that are kept); any other stage reads them
    # through a cast to the declared type.  Stores narrow once, when packing.
    program = sched.program
    self.loose = {
        node.index: (not sched.paired and node.elem_size < 4 and
                     program.types[node.name] in _INT_TYPES)
        for node in sched.nodes}
    self.ring = {node.index: ring_expression(node.stage, program)
                 for node in sched.stage_nodes}
    self.lay = Layout(sched)
    self.s = sched.sdim
    self.V = sched.vec
    self.NT = sched.threads
    self.VPT = sched.vecs_per_thread
    self.U = sched.period
    self.P = sched.prefetch
    self.PLANE = sched.plane_elems
    # ring slots are `ring_pitch` elements apart: a plane plus a gap no one
    # writes, where neighbour reads that leave the plane land (see plan)
    self.PITCH = sched.ring_pitch
    self.flat = sched.sdim == 1          # 2-D program: registers only
    # paired 2-D kernels peel their trips: the steady-state trips, whose rows
    # every lane stores whole or not at all, are a copy of the trip without
    # the masked store path; rows are addressed from a pointer per trip
    self.peel = self.flat and sched.paired
    assert not self.peel or self.VPT == 1
    self.steady = False                  # emitting the steady-state trip
    self.DIN = self.lay.in_depth

  # ---- naming ---------------------------------------------------------------
  def hist(self, node, phase, age):
    """Register array holding the row of ``node`` that is ``age`` steps old."""
    return 'h_%s_%d' % (node.ident, (phase - age) % self.U)

  def ctype(self, node):
    """Type of a cell of ``node`` in registers: a pair of float32 (iteration
    k, iteration k + depth/2) when the schedule pairs iterations."""
    if self.loose[node.index]:
      return 'uint32_t'
    return 'soda::f32x2' if self.sched.paired else node.c_type

  def ring_slot(self, node, age, phase):
    """Slot of the plane that is ``age`` steps old at step ``phase`` of a
    trip: ring depths divide the trip, so this is a constant."""
    return (phase - age) % self.lay.ring_depth[node.index]

  # ---- pieces ----------------------------------------------------------------
  def emit(self):
    p, sched, lay, s, V = self.p, self.sched, self.lay, self.s, self.V
    name = kernel_name(sched)
    p.println('// %s' % sched.describe().replace('\n', '\n// '))
    p.println('template <bool kTma>')
    p.println('__global__ void __launch_bounds__(%d, %d) %s(' % (
        self.NT, sched.min_blocks, name))
    p.println('    const __grid_constant__ soda::StreamArgs a)')
    p.do_scope()
    if lay.total:
      p.println('extern __shared__ __align__(1024) unsigned char smem_raw[];')
    if self.flat:
      p.println('// input queue of this warp: %d boxes of %d rows per input, '
                'one mbarrier per box' % (lay.groups, lay.box_rows))
      p.println('unsigned char* const queue = smem_raw + (threadIdx.x >> 5) * '
                '%d;' % lay.warp_bytes)
      p.println('uint64_t* const bars = reinterpret_cast<uint64_t*>(smem_raw + '
                '%d) + (threadIdx.x >> 5) * %d;' % (lay.bar_offset, lay.groups))
      p.println('(void)queue; (void)bars;')
    elif lay.total:
      for node in sched.nodes:
        if node.index in lay.ring_offset:
          p.println('%s* const ring_%s = reinterpret_cast<%s*>(smem_raw + %d);'
                    '  // %d planes' % (node.c_type, node.ident, node.c_type,
                                        lay.ring_offset[node.index],
                                        lay.ring_depth[node.index]))
      if lay.loaded_inputs:
        p.println('uint64_t* const bars = reinterpret_cast<uint64_t*>('
                  'smem_raw + %d);' % lay.bar_offset)
    p.println('const int tid = threadIdx.x;')
    p.println('const int lane = tid & 31;')
    p.println('(void)lane;')
    plan_mod.emit_param_pointers(p, sched.program)
    p.println()
    self.emit_geometry()
    self.emit_histories()
    if self.flat:
      self.emit_flat_prologue()
    else:
      self.emit_tma_prologue()
    self.emit_output_windows()
    # `steps` is a whole number of trips: the surplus steps compute rows no
    # block stores (beyond mine_hi) from rows that read as 0 or as real data
    trip = lay.box_rows if self.flat else sched.trip
    if self.peel:
      self.emit_steady_window(trip)
    if self.flat:
      p.println('for (int i = 0, box = 0; i < steps; i += %d, ++box)' % trip)
    else:
      p.println('for (int i = 0; i < steps; i += %d)' % trip)
    p.do_scope()
    if self.peel:
      p.println('for (; static_cast<unsigned>(i - steady_lo) < steady_n; '
                'i += %d, ++box)' % trip)
      p.do_scope()
      self.steady = True
      self.emit_trip(trip)
      self.steady = False
      p.un_scope()
      p.println('if (i >= steps) break;')
    self.emit_trip(trip)
    p.un_scope()
    p.un_scope()
    p.println()
    return lay

  def emit_trip(self, trip):
    p, sched = self.p, self.sched
    if self.flat:
      self.emit_flat_box()
    for phase in range(trip):
      p.println('// ---- step %d of %d' % (phase, trip))
      p.do_scope()
      p.println('const int ii = i + %d;' % phase)
      self.emit_step(phase)
      p.un_scope()
    if self.peel:
      # the row pointers move to the next trip
      for node in self.lay.loaded_inputs:
        p.println('lp%d += ipitch%d * %dll;' % (node.input_index,
                                              node.input_index, trip))
      for node in sched.outputs:
        p.println('op%d[0] += opitch%d * %dll;' % (node.output_index,
                                                 node.output_index, trip))

  def emit_steady_window(self, trip):
    """Trips ``i`` in [steady_lo, steady_lo + steady_n) store every row of
    every output with one 128-bit store per lane, or not at all: all their
    rows lie in each output's valid rows, and no lane of the warp owns only
    part of its vector or has cells outside the valid columns."""
    p, sched = self.p, self.sched
    outs = [node.output_index for node in sched.outputs]
    p.println('// steady-state trips: the whole trip lies in every output\'s '
              'valid rows and every lane')
    p.println('// of the warp stores its whole vector (one 128-bit store) or '
              'nothing')
    p.println('const bool whole = own[0] == 0u || (%s);' % ' && '.join(
        'fast%d[0]' % n for n in outs))
    lo, hi = 'ok_lo%d' % outs[0], 'ok_lo%d + static_cast<int>(ok_n%d)' % (
        outs[0], outs[0])
    for n in outs[1:]:
      lo = 'max(%s, ok_lo%d)' % (lo, n)
      hi = 'min(%s, ok_lo%d + static_cast<int>(ok_n%d))' % (hi, n, n)
    p.println('const int steady_lo = %s;' % lo)
    p.println('const int steady_hi = %s - %d;' % (hi, trip - 1))
    p.println('const unsigned steady_n = __all_sync(0xffffffffu, whole) && '
              'steady_hi > steady_lo ? static_cast<unsigned>(steady_hi - '
              'steady_lo) : 0u;')
    p.println()

  def emit_geometry(self):
    p, sched, s, V, VPT = self.p, self.sched, self.s, self.V, self.VPT
    if self.flat:
      p.println('// this warp: one strip of dimension 0, one chunk of the '
                'streamed dimension')
      p.println('const int strip = blockIdx.x * %d + (tid >> 5);' %
                sched.tiles_per_block)
      p.println('if (strip >= a.tiles[0]) return;   // whole warps; no block '
                'barrier in this kernel')
      p.println('const int org0 = strip * %d - %d;' % (
          sched.own[0], sched.tile_halo_lo[0]))
    else:
      p.println('// this block: one tile of the non-streamed dims, one chunk '
                'of the streamed dim')
      p.println('int tile_rest = blockIdx.x;')
      for d in range(s):
        p.println('const int org%d = (tile_rest %% a.tiles[%d]) * %d - %d;' % (
            d, d, sched.own[d], sched.tile_halo_lo[d]))
        if d + 1 < s:
          p.println('tile_rest /= a.tiles[%d];' % d)
    p.println('const int r0 = a.row_begin + blockIdx.y * a.chunk_rows;')
    p.println('const int r1 = min(a.row_end, r0 + a.chunk_rows);')
    p.println('const int base = r0 - %d;   // streamed coordinate of step 0' %
              sched.lead)
    trip = sched.flat_box if self.flat else sched.trip
    p.println('// steps to run: (r1 - r0) + %d, rounded up to whole trips of '
              'the streamed loop' % (sched.lead + sched.out_delay))
    p.println('const int steps = ((r1 - r0) + %d) / %d * %d;' % (
        sched.lead + sched.out_delay + trip - 1, trip, trip))
    kernel_mod.emit_item(p)
    p.println()
    p.println('// per-thread vectors: position in the plane, offset in HBM, '
              'cells this tile')
    p.println('// owns (store) and cells in the valid region (else 0)')
    p.println('int pos[%d];' % VPT)
    kernel_mod.emit_offset_arrays(p, self.lay.loaded_inputs, sched.outputs,
                                  VPT)
    p.println('unsigned own[%d];' % VPT)
    for n in range(len(sched.outputs)):
      p.println('unsigned val%d[%d];   // output %d: cells in ITS valid region'
                % (n, VPT, n))
      p.println('bool fast%d[%d];   // whole vector owned and valid: one '
                '128-bit store' % (n, VPT))
    p.println('bool xin[%d];   // the vector lies inside the grid in the tiled '
              'dims' % VPT)
    p.println('int gx[%d];' % VPT)
    for d in range(1, s):
      p.println('int gc%d[%d];' % (d, VPT))
    p.println('#pragma unroll')
    p.println('for (int j = 0; j < %d; ++j)' % VPT)
    p.do_scope()
    if self.flat:
      p.println('const int q = lane;')
    else:
      p.println('const int q = tid + j * %d;' % self.NT)
    p.println('pos[j] = q * %d;' % V)
    p.println('const int c0 = (q & 31) * %d;' % V)
    p.println('int rest = q >> 5;')
    for d in range(1, s):
      p.println('const int c%d = rest %% %d;' % (d, sched.tile[d]))
      if d + 1 < s:
        p.println('rest /= %d;' % sched.tile[d])
    p.println('(void)rest;')
    p.println('gx[j] = org0 + c0;')
    p.println('bool mine = true, inside = true;')
    for n in range(len(sched.outputs)):
      p.println('bool ok%d = true;' % n)
    for d in range(1, s):
      p.println('gc%d[j] = org%d + c%d;' % (d, d, d))
      p.println('mine = mine && c%d >= %d && c%d < %d && gc%d[j] < a.dims[%d];'
                % (d, sched.tile_halo_lo[d], d,
                   sched.tile[d] - sched.tile_halo_hi[d], d, d))
      for n in range(len(sched.outputs)):
        p.println('ok%d = ok%d && gc%d[j] >= a.valid_lo[%d][%d] && gc%d[j] < '
                  'a.valid_hi[%d][%d];' % (n, n, d, n, d, d, n, d))
      p.println('inside = inside && gc%d[j] >= 0 && gc%d[j] < a.dims[%d];' % (
          d, d, d))
    kernel_mod.emit_offsets(p, self.lay.loaded_inputs, sched.outputs, s)
    p.println('xin[j] = inside && gx[j] >= 0 && gx[j] + %d <= a.dims[0];' % V)
    p.println('unsigned m = 0;')
    for n in range(len(sched.outputs)):
      p.println('unsigned v%d = 0;' % n)
    p.println('#pragma unroll')
    p.println('for (int k = 0; k < %d; ++k)' % V)
    p.do_scope()
    p.println('const int x = gx[j] + k;')
    p.println('if (mine && c0 + k >= %d && c0 + k < %d && x < a.dims[0]) '
              'm |= 1u << k;' % (sched.tile_halo_lo[0],
                                 sched.tile[0] - sched.tile_halo_hi[0]))
    for n in range(len(sched.outputs)):
      p.println('if (ok%d && x >= a.valid_lo[%d][0] && x < a.valid_hi[%d][0]) '
                'v%d |= 1u << k;' % (n, n, n, n))
    p.un_scope()
    p.println('own[j] = m;')
    for n in range(len(sched.outputs)):
      p.println('val%d[j] = v%d;' % (n, n))
      p.println('fast%d[j] = m == %du && v%d == %du && a.vec_store[%d];' % (
          n, (1 << V) - 1, n, (1 << V) - 1, n))
    p.un_scope()
    p.println()

  def out_lag(self, node):
    """An output row leaves ``out_lag`` steps after its input row arrived."""
    return node.delay + (self.sched.pair_lag if self.sched.paired else 0)

  def emit_output_windows(self):
    """Per output: the steps whose row this block stores ([mine_lo, mine_hi))
    and, inside, the steps whose row lies in the valid region ([ok_lo, ok_lo +
    ok_n)); plus the output pointers, which walk down the rows with the steps."""
    p, sched, s = self.p, self.sched, self.s
    for node in sched.outputs:
      n, lag = node.output_index, self.out_lag(node)
      p.println('const int mine_lo%d = %d, mine_hi%d = (r1 - r0) + %d;' % (
          n, sched.lead + lag, n, sched.lead + lag))
      p.println('const int ok_lo%d = max(mine_lo%d, a.valid_lo[%d][%d] - base '
                '+ %d);' % (n, n, n, s, lag))
      p.println('const unsigned ok_n%d = static_cast<unsigned>(max(0, min('
                'mine_hi%d, a.valid_hi[%d][%d] - base + %d) - ok_lo%d));' % (
                    n, n, n, s, lag, n))
      p.println('// steps whose row this thread stores with one 128-bit store: '
                'the valid steps if')
      p.println('// its whole vector is owned and valid, none otherwise (one '
                'compare per step)')
      p.println('unsigned fast_n%d[%d];' % (n, self.VPT))
      p.println('#pragma unroll')
      p.println('for (int j = 0; j < %d; ++j) fast_n%d[j] = fast%d[j] ? ok_n%d '
                ': 0u;' % (self.VPT, n, n, n))
      if self.V == 2:
        # likewise the steps it stores cell by cell (see emit_stage)
        p.println('unsigned slow_n%d[%d];' % (n, self.VPT))
        p.println('#pragma unroll')
        p.println('for (int j = 0; j < %d; ++j) slow_n%d[j] = own[j] ? '
                  'static_cast<unsigned>(mine_hi%d - mine_lo%d) : 0u;' % (
                      self.VPT, n, n, n))
      p.println('%s* op%d[%d];   // row of step 0 (dereferenced only inside '
                'the window)' % (node.c_type, n, self.VPT))
      p.println('#pragma unroll')
      p.println('for (int j = 0; j < %d; ++j)' % self.VPT)
      p.println('  op%d[j] = static_cast<%s*>(a.out_ptr[%d]) + (base - %d) * '
                'a.out_stride[%d][%d] + ooff%d[j];' % (n, node.c_type, n, lag,
                                                       n, s, n))
    p.println()

  def emit_histories(self):
    p, sched = self.p, self.sched
    p.println('// register histories: slot (phase - age) mod %d holds the row '
              'computed `age` steps ago' % self.U)
    for node in sched.nodes:
      if node.hist_oldest is None:
        continue
      for slot in range(self.U):
        p.println('%s h_%s_%d[%d][%d] = {};' % (
            self.ctype(node), node.ident, slot, self.VPT, self.V))
      if sched.paired and node.is_input:
        p.println('%s fb_%s[%d][%d] = {};   // newest output row of lane A, '
                  'input of lane B' % (node.c_type, node.ident, self.VPT,
                                       self.V))
    p.println()

  # ---- 2-D input path: per-warp TMA queue in shared memory --------------------
  def flat_issue(self, box_code):
    """Lane 0 requests box ``box_code`` (rows box * B .. box * B + B - 1 of
    this chunk) of every input into its slots."""
    p, lay = self.p, self.lay
    G, B = lay.groups, lay.box_rows
    p.println('uint64_t* const bar = &bars[(%s) %% %d];' % (box_code, G))
    p.println('soda::mbar_expect_tx(bar, %d);' % (
        B * sum(lay.row_bytes.values())))
    for node in lay.loaded_inputs:
      p.println('soda::tma_load(queue + %d + ((%s) %% %d) * %d, &a.in_map[%d], '
                'bar, org0, base + (%s) * %d, item);' % (
                    lay.queue_offset[node.index], box_code, G,
                    B * lay.row_bytes[node.index], node.input_index, box_code,
                    B))

  def flat_plain_load(self, rel_code, row=None):
    """kTma = false: row ``base + rel`` of every input, cell by cell, into the
    ``nx_`` registers; cells outside the grid read as 0.  Peeled kernels read
    it ``row`` rows after the trip's row pointer, the others advance the
    pointer by a row."""
    p, lay, V = self.p, self.lay, self.V
    p.println('const bool lrow_in = static_cast<unsigned>(base + (%s)) < '
              'static_cast<unsigned>(a.dims[%d]);' % (rel_code, self.s))
    for node in lay.loaded_inputs:
      k = node.input_index
      src = 'lp%d' % k
      if row:
        src = '(lp%d + ipitch%d * %dll)' % (k, k, row)
      p.println('#pragma unroll')
      p.println('for (int k = 0; k < %d; ++k)' % V)
      p.println('  nx_%s[k] = (lrow_in && gx[0] + k >= 0 && gx[0] + k < '
                'a.dims[0]) ? %s[k] : %s(0);' % (node.ident, src, node.c_type))
      if row is None:
        p.println('lp%d += a.in_stride[%d][%d];' % (k, k, self.s))

  def emit_flat_prologue(self):
    p, lay = self.p, self.lay
    G, B = lay.groups, lay.box_rows
    if self.peel:
      p.println('// rows of each tensor are its `pitch` elements apart (the '
                'runtime keeps 2-D row')
      p.println('// strides below 2^31)')
      for node in lay.loaded_inputs:
        p.println('const int ipitch%d = static_cast<int>(a.in_stride[%d][%d]);'
                  % (node.input_index, node.input_index, self.s))
      for node in self.sched.outputs:
        p.println('const int opitch%d = static_cast<int>(a.out_stride[%d][%d]);'
                  % (node.output_index, node.output_index, self.s))
    for node in lay.loaded_inputs:
      k = node.input_index
      p.println('%s nx_%s[%d] = {};   // kTma = false: the next row' % (
          node.c_type, node.ident, self.V))
      p.println('const %s* lp%d = static_cast<const %s*>(a.in_ptr[%d]) + '
                'base * a.in_stride[%d][%d] + ioff%d[0];' % (
                    node.c_type, k, node.c_type, k, k, self.s, k))
    p.println('if (kTma)')
    p.do_scope()
    p.println('if (lane == 0)')
    p.do_scope()
    for node in lay.loaded_inputs:
      p.println('soda::tma_prefetch_desc(&a.in_map[%d]);' % node.input_index)
    p.println('for (int n = 0; n < %d; ++n) soda::mbar_init(&bars[n], 1);' % G)
    p.println('soda::mbar_fence_init();')
    p.println('soda::fence_proxy_async();')
    p.println('// the first %d boxes are in flight before the loop starts' %
              (G - 2))
    p.println('for (int n = 0; n < %d && n * %d < steps; ++n)' % (G - 2, B))
    p.do_scope()
    self.flat_issue('n')
    p.un_scope()
    p.un_scope()
    p.println('__syncwarp();')
    p.un_scope()
    p.println('else')
    p.do_scope()
    self.flat_plain_load('0', 0 if self.peel else None)
    p.un_scope()
    p.println()

  def emit_flat_box(self):
    """Start of a trip: request the box G - 2 ahead, wait for this one."""
    p, lay = self.p, self.lay
    G, B = lay.groups, lay.box_rows
    p.println('if (kTma)')
    p.do_scope()
    p.println('// rows i .. i + %d are box `box`; the box requested now '
              'replaces the one read %d .. %d steps ago' % (B - 1, B + 1, 2 * B))
    p.println('__syncwarp();')
    p.println('if (lane == 0 && (box + %d) * %d < steps)' % (G - 2, B))
    p.do_scope()
    self.flat_issue('box + %d' % (G - 2))
    p.un_scope()
    # (the queue holds G boxes, 3 or a power of two: constants, so the
    # compiler turns these into masks and shifts where it can)
    p.println('soda::mbar_wait(&bars[box %% %d], (box / %d) & 1);' % (G, G))
    p.un_scope()
    for node in lay.loaded_inputs:
      p.println('const unsigned char* const rows_%s = queue + %d + (box %% %d) * '
                '%d + lane * %d;' % (
                    node.ident, lay.queue_offset[node.index], G,
                    B * lay.row_bytes[node.index], self.V * node.elem_size))

  def emit_flat_input(self, phase):
    """Start of a step: take row ii (row `phase` of the current box)."""
    p, sched, lay, V = self.p, self.sched, self.lay, self.V
    for node in lay.loaded_inputs:
      dst = '%s[0]' % self.hist(node, phase, 0)
      p.do_scope()
      loose = self.loose[node.index] and V * node.elem_size % 4 == 0
      if loose:
        # whole words; a cell is its word shifted down, upper bits loose
        per = 4 // node.elem_size
        p.println('uint32_t t[%d];' % V)
        p.println('if (kTma)')
        p.do_scope()
        p.println('uint32_t words[%d];' % (V // per))
        p.println('soda::ld_pack<uint32_t, %d>(words, reinterpret_cast<const '
                  'uint32_t*>(rows_%s + %d));' % (
                      V // per, node.ident,
                      phase * lay.row_bytes[node.index]))
        p.println('#pragma unroll')
        p.println('for (int k = 0; k < %d; ++k) t[k] = words[k / %d] >> '
                  '(%d * (k %% %d));' % (V, per, 8 * node.elem_size, per))
        p.un_scope()
      else:
        p.println('%s t[%d];' % (node.c_type, V))
        p.println('if (kTma)')
        if sched.paired:
          p.println('  for (int k = 0; k < %d; ++k) t[k] = soda::lds_f32('
                    'rows_%s + %d + 4 * k);' % (
                        V, node.ident, phase * lay.row_bytes[node.index]))
        else:
          p.println('  soda::ld_pack<%s, %d>(t, reinterpret_cast<const %s*>('
                    'rows_%s + %d));' % (
                        node.c_type, V, node.c_type, node.ident,
                        phase * lay.row_bytes[node.index]))
      p.println('else')
      p.do_scope()
      p.println('#pragma unroll')
      p.println('for (int k = 0; k < %d; ++k) t[k] = nx_%s[k];' % (
          V, node.ident))
      p.un_scope()
      p.println('#pragma unroll')
      p.println('for (int k = 0; k < %d; ++k)' % V)
      if sched.paired:
        # lane A reads the input, lane B the newest output row of lane A
        p.println('  %s[k] = soda::make_f32x2(t[k], fb_%s[0][k]);' % (
            dst, node.ident))
      else:
        p.println('  %s[k] = t[k];' % dst)
      p.un_scope()
    p.println('if (!kTma)')
    p.do_scope()
    self.flat_plain_load('ii + 1', phase + 1 if self.peel else None)
    p.un_scope()

  # ---- 3-D input path: TMA into a shared ring --------------------------------
  def tma_issue(self, rel_code, slot):
    """Request plane ``base + rel`` of every input into ring slot ``slot``."""
    p, lay, s = self.p, self.lay, self.s
    p.println('uint64_t* const bar = &bars[%d];' % slot)
    p.println('soda::mbar_expect_tx(bar, %d);' % sum(lay.plane_bytes.values()))
    for node in lay.loaded_inputs:
      coords = ['org%d' % d for d in range(s)] + ['base + (%s)' % rel_code,
                                                  'item']
      p.println('soda::tma_load(ring_%s + %d, &a.in_map[%d], bar, %s);' % (
          node.ident, slot * self.PITCH, node.input_index, ', '.join(coords)))

  def plain_load(self, rel_code, slot):
    p, lay, s, V = self.p, self.lay, self.s, self.V
    p.println('const int lrow = base + (%s);' % rel_code)
    p.println('const bool lrow_in = lrow >= 0 && lrow < a.dims[%d];' % s)
    for node in lay.loaded_inputs:
      p.println('#pragma unroll')
      p.println('for (int j = 0; j < %d; ++j)' % self.VPT)
      p.do_scope()
      p.println('%s t[%d];' % (node.c_type, V))
      cond = ' && '.join(['lrow_in'] + [
          'gc%d[j] >= 0 && gc%d[j] < a.dims[%d]' % (d, d, d)
          for d in range(1, s)])
      p.println('const bool in = %s;' % cond)
      k = node.input_index
      p.println('const %s* src = static_cast<const %s*>(a.in_ptr[%d]) + '
                'lrow * a.in_stride[%d][%d] + ioff%d[j];' % (
                    node.c_type, node.c_type, k, k, s, k))
      p.println('if (in && a.vec_load[%d] && gx[j] >= 0 && gx[j] + %d <= '
                'a.dims[0])' % (k, V))
      p.do_scope()
      p.println('soda::ld_pack<%s, %d>(t, src);' % (node.c_type, V))
      p.un_scope()
      p.println('else')
      p.do_scope()
      p.println('#pragma unroll')
      p.println('for (int k = 0; k < %d; ++k)' % V)
      p.println('  t[k] = (in && gx[j] + k >= 0 && gx[j] + k < a.dims[0]) ? '
                'src[k] : %s(0);' % node.c_type)
      p.un_scope()
      p.println('soda::st_pack<%s, %d>(ring_%s + %d + pos[j], t);' % (
          node.c_type, V, node.ident, slot * self.PITCH))
      p.un_scope()

  def emit_tma_prologue(self):
    p, lay = self.p, self.lay
    if not lay.loaded_inputs:
      return
    p.println('if (kTma)')
    p.do_scope()
    p.println('if (tid == 0)')
    p.do_scope()
    for node in lay.loaded_inputs:
      p.println('soda::tma_prefetch_desc(&a.in_map[%d]);' % node.input_index)
    p.println('for (int n = 0; n < %d; ++n) soda::mbar_init(&bars[n], 1);' %
              self.DIN)
    p.println('soda::mbar_fence_init();')
    p.un_scope()
    p.println('__syncthreads();')
    p.println('if (tid == 0)')
    p.do_scope()
    for rel in range(self.P):
      p.println('if (%d < steps)' % rel)
      p.do_scope()
      self.tma_issue(str(rel), rel % self.DIN)
      p.un_scope()
    p.un_scope()
    p.un_scope()
    p.println('else')
    p.do_scope()
    p.do_scope()
    self.plain_load('0', 0)
    p.un_scope()
    p.println('__syncthreads();')
    p.un_scope()
    p.println()

  # ---- one step ---------------------------------------------------------------
  def emit_step(self, phase):
    p, sched, lay, V = self.p, self.sched, self.lay, self.V
    if self.flat:
      self.emit_flat_input(phase)
    elif lay.loaded_inputs:
      p.println('if (kTma)')
      p.do_scope()
      p.println('if (tid == 0 && ii + %d < steps)' % self.P)
      p.do_scope()
      self.tma_issue('ii + %d' % self.P, (phase + self.P) % self.DIN)
      p.un_scope()
      # slot `phase mod DIN` is on its (i / DIN + phase / DIN)-th plane
      p.println('soda::mbar_wait(&bars[%d], (i / %d + %d) & 1);' % (
          phase % self.DIN, self.DIN, phase // self.DIN))
      p.un_scope()
      for node in lay.loaded_inputs:
        if node.hist_oldest is None:
          continue
        p.println('#pragma unroll')
        p.println('for (int j = 0; j < %d; ++j)' % self.VPT)
        if self.loose[node.index]:
          p.do_scope()
          p.println('%s t[%d];' % (node.c_type, V))
          p.println('soda::ld_pack<%s, %d>(t, ring_%s + %d + pos[j]);' % (
              node.c_type, V, node.ident,
              self.ring_slot(node, 0, phase) * self.PITCH))
          p.println('#pragma unroll')
          p.println('for (int k = 0; k < %d; ++k) %s[j][k] = t[k];' % (
              V, self.hist(node, phase, 0)))
          p.un_scope()
        else:
          p.println('  soda::ld_pack<%s, %d>(%s[j], ring_%s + %d + pos[j]);'
                    % (node.c_type, V, self.hist(node, phase, 0), node.ident,
                       self.ring_slot(node, 0, phase) * self.PITCH))
    self.shuffled = {}     # (node index, age, element) -> variable, this step
    for node in sched.stage_nodes:
      self.emit_stage(node, phase)
    if not self.flat:
      if lay.loaded_inputs:
        p.println('if (!kTma && ii + 1 < steps)')
        p.do_scope()
        self.plain_load('ii + 1', (phase + 1) % self.DIN)
        p.un_scope()
      p.println('__syncthreads();')

  def emit_stage(self, node, phase):
    p, sched, lay, s, V = self.p, self.sched, self.lay, self.s, self.V
    stage = node.stage
    p.println('// %s: plane ii - %d' % (node.ident, node.delay))
    # shuffle variables live at step scope so later stages can reuse them
    reg_loads = [(parent, off) for parent, off in node.loads
                 if not sched.via_smem(off)]
    fresh = []
    for parent, off in reg_loads:
      age = node.delay - off[s]
      for c in sorted({k + off[0] for k in range(V)}):
        if 0 <= c < V:
          continue
        key = (parent.index, age, c)
        if key in self.shuffled:
          continue
        var = 'x_%s_a%s_%s' % (parent.ident, str(age).replace('-', 'm'),
                               ('m%d' % -c) if c < 0 else ('p%d' % c))
        self.shuffled[key] = var
        fresh.append((parent, age, c, var))
        p.println('%s %s[%d];' % (self.ctype(parent), var, self.VPT))
    p.do_scope()
    # A block runs its lead-in steps and the surplus steps that fill its last
    # trip with every stage; the rows the LAST stage would produce there are
    # not this block's to store, and when nothing reads that stage (a final
    # output, no history, no shared plane) the whole stage is skipped for the
    # step — a branch the block takes as one.  3-D kernels only: their blocks
    # are tens of rows long (4-8 such steps in 30-70), the 2-D strips
    # thousands.
    skips = (node.output_index is not None and not sched.paired and
             not self.flat and node is sched.stage_nodes[-1] and
             node.hist_oldest is None and node.index not in lay.ring_offset)
    if node.output_index is not None and not self.steady:
      n = node.output_index
      p.println('const bool row_ok = static_cast<unsigned>(ii - ok_lo%d) < '
                'ok_n%d;' % (n, n))
      if V != 2 or skips:
        p.println('const bool row_mine = ii >= mine_lo%d && ii < mine_hi%d;'
                  % (n, n))
    if skips:
      p.println('if (!row_mine)')
      p.do_scope()
      p.println('#pragma unroll')
      p.println('for (int j = 0; j < %d; ++j) op%d[j] += a.out_stride[%d][%d];'
                % (self.VPT, node.output_index, node.output_index, s))
      p.un_scope()
      p.println('else')
    p.println('#pragma unroll')
    p.println('for (int j = 0; j < %d; ++j)' % self.VPT)
    p.do_scope()
    for parent, age, c, var in fresh:
      lanes, elem = divmod(c, V)      # c < 0: lanes < 0 (from the left)
      src = '%s[j][%d]' % (self.hist(parent, phase, age), elem)
      if lanes < 0:
        p.println('%s[j] = soda::shfl_up<%s>(%s, %d);' % (
            var, self.ctype(parent), src, -lanes))
      else:
        p.println('%s[j] = soda::shfl_down<%s>(%s, %d);' % (
            var, self.ctype(parent), src, lanes))

    # operands read through shared memory: one window per (parent, offsets in
    # dims 1..), as in kernel.py
    groups = collections.OrderedDict()
    parent_of = {}
    for parent, off in node.loads:
      if not sched.via_smem(off):
        continue
      key = (parent.index, off[1:])
      groups.setdefault(key, set()).add(off[0])
      parent_of[parent.index] = parent
    window_of = {}
    for g, ((pindex, rest), dxs) in enumerate(groups.items()):
      parent = parent_of[pindex]
      xlo, xhi = min(dxs), max(dxs)
      used = sorted({k + dx for dx in dxs for k in range(V)})
      inplane = sum(rest[d - 1] * sched.plane_pitch(d) for d in range(1, s))
      age = node.delay - rest[s - 1]
      p.println('const %s* const s%d = ring_%s + pos[j] + (%d);' % (
          parent.c_type, g, parent.ident,
          self.ring_slot(parent, age, phase) * self.PITCH + inplane))
      p.println('%s w%d[%d];' % (parent.c_type, g, V + xhi - xlo))
      inside = [c for c in used if 0 <= c < V]
      if len(inside) >= 2 and xlo <= 0 <= xhi:
        p.println('soda::ld_pack<%s, %d>(w%d + %d, s%d);' % (
            parent.c_type, V, g, -xlo, g))
        outside = [c for c in used if not 0 <= c < V]
      else:
        outside = used
      for c in outside:
        p.println('w%d[%d] = s%d[%d];' % (g, c - xlo, g, c))
      window_of[(pindex, rest)] = (g, xlo)

    resolved = dict(zip(
        [l for l in stage.loads if l.parent not in sched.program.params],
        node.loads))

    def ref_code(load, k):
      if load.parent in sched.program.params:
        return plan_mod.param_code(sched.program, load)
      parent, off = resolved[load]
      if sched.via_smem(off):
        g, xlo = window_of[(parent.index, off[1:])]
        return 'w%d[%d]' % (g, k + off[0] - xlo)
      age = node.delay - off[s]
      c = k + off[0]
      code = ('%s[j][%d]' % (self.hist(parent, phase, age), c)
              if 0 <= c < V else
              '%s[j]' % self.shuffled[(parent.index, age, c)])
      if self.loose[parent.index] and not (
          self.ring[node.index] and node.elem_size <= parent.elem_size):
        code = 'static_cast<%s>(%s)' % (parent.c_type, code)
      return code

    keeps = node.hist_oldest is not None
    target = ('%s[j]' % self.hist(node, phase, node.delay)) if keeps else 'r'
    if not keeps:
      p.println('%s r[%d];' % (self.ctype(node), V))
    batched = (not sched.paired and batches_rare_paths(stage) and
               not (self.loose[node.index] and self.ring[node.index]))
    rendered = [_render(stage, ref_code, k, batched) for k in range(V)]
    if batched:
      for k in range(V):
        numerator, denominator = rendered[k][1]
        p.println('const auto num%d = %s;' % (k, numerator))
        p.println('const auto den%d = %s;' % (k, denominator))
      p.println('bool rare = false;')
      for k in range(V):
        p.println('%s[%d] = soda::store_cast<%s>(soda::div_try(num%d, den%d, '
                  'rare));' % (target, k, node.c_type, k, k))
      p.println('if (rare)')
      p.do_scope()
      for k in range(V):
        p.println('%s[%d] = soda::store_cast<%s>(num%d / den%d);' % (
            target, k, node.c_type, k, k))
      p.un_scope()
    else:
      for k in range(V):
        lets, expr = rendered[k]
        if lets:
          p.do_scope()
          for let in lets:
            p.println(let)
        if sched.paired:
          p.println('%s[%d] = %s;' % (target, k, expr))
        elif self.loose[node.index] and self.ring[node.index]:
          p.println('%s[%d] = static_cast<uint32_t>(%s);' % (target, k, expr))
        else:
          p.println('%s[%d] = soda::store_cast<%s>(%s);' % (
              target, k, node.c_type, expr))
        if lets:
          p.un_scope()
    if node.index in lay.ring_offset:
      plane = target
      if self.loose[node.index]:
        plane = 'narrow'
        p.println('%s narrow[%d];' % (node.c_type, V))
        p.println('#pragma unroll')
        p.println('for (int k = 0; k < %d; ++k) narrow[k] = static_cast<%s>('
                  '%s[k]);' % (V, node.c_type, target))
      p.println('soda::st_pack<%s, %d>(ring_%s + %d + pos[j], %s);' % (
          node.c_type, V, node.ident,
          self.ring_slot(node, node.delay, phase) * self.PITCH, plane))
    if node.output_index is not None and sched.paired:
      # lane A's result (iteration depth/2 - 1) feeds lane B one step later
      feeds = sched.inputs[node.output_index]
      p.println('#pragma unroll')
      p.println('for (int k = 0; k < %d; ++k)' % V)
      p.println('  fb_%s[j][k] = %s[k].v.x;' % (feeds.ident, target))
    if node.output_index is not None:
      n = node.output_index
      half = '.v.y' if sched.paired else ''
      out = 'op%d[j]' % n
      if self.peel:
        out = 'orow'
        p.println('%s* const orow = op%d[j] + opitch%d * %dll;' % (
            node.c_type, n, n, phase))
      if self.steady:
        p.println('if (fast%d[j])' % n)
      else:
        p.println('if (static_cast<unsigned>(ii - ok_lo%d) < fast_n%d[j])' % (
            n, n))
      p.do_scope()
      p.println('%s o[%d];' % (node.c_type, V))
      p.println('#pragma unroll')
      p.println('for (int k = 0; k < %d; ++k) o[k] = static_cast<%s>(%s[k]%s);'
                % (V, node.c_type, target, half))
      p.println('soda::st_pack_global<%s, %d>(%s, o);' % (node.c_type, V, out))
      p.un_scope()
    if node.output_index is not None and not self.steady:
      # two-cell vectors: ptxas 12.9 keeps the two `own` bits in predicates and
      # was seen to fold `row_mine && own[j]` into the wrong 3-input LUT
      # (fully owned vectors skipped in two steps of a trip: dbl3d, 64x48
      # tile, -O3 only; DESIGN.md §7) -- one unsigned compare against a
      # per-thread count, like the fast test, leaves it nothing to fold
      p.println('else if (static_cast<unsigned>(ii - mine_lo%d) < slow_n%d[j])'
                % (n, n) if V == 2 else 'else if (row_mine && own[j])')
      p.do_scope()
      p.println('// tile or grid edge: cells outside the valid region are '
                'stored as 0')
      p.println('const unsigned keep = row_ok ? val%d[j] : 0u;' % n)
      p.println('%s o[%d];' % (node.c_type, V))
      p.println('#pragma unroll')
      p.println('for (int k = 0; k < %d; ++k)' % V)
      p.println('  o[k] = ((keep >> k) & 1u) ? static_cast<%s>(%s[k]%s) : '
                '%s(0);' % (node.c_type, target, half, node.c_type))
      p.println('if (own[j] == %du && a.vec_store[%d])' % ((1 << V) - 1, n))
      p.do_scope()
      p.println('soda::st_pack_global<%s, %d>(%s, o);' % (node.c_type, V, out))
      p.un_scope()
      p.println('else')
      p.do_scope()
      p.println('#pragma unroll')
      p.println('for (int k = 0; k < %d; ++k)' % V)
      p.println('  if ((own[j] >> k) & 1u) %s[k] = o[k];' % out)
      p.un_scope()
      p.un_scope()
      if not self.peel:
        p.println('op%d[j] += a.out_stride[%d][%d];' % (n, n, s))
    p.un_scope()
    p.un_scope()


def emit_kernel(p, sched):
  """Write the kernel for ``sched`` through Printer ``p``; returns its Layout."""
  return _Emitter(p, sched).emit()
