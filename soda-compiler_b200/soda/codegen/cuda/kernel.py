"""Emit the sm_100a streaming kernel of a SODA program (``--cuda-kernel``).

For every ``plan.Schedule`` (one per temporal depth compiled in) this writes
one ``template <bool kTma> __global__`` function built from the hand-written
pieces in csrc/soda_cuda_device.cuh, with each stage's reference-lowered
expression spliced into the per-cell loop.  The counterpart on the FPGA side is
the reference's HLS kernel emitter (src/soda/codegen/xilinx/hls_kernel.py:
12-103 top level, :209-498 per-module bodies, :487-489 the spliced ``c_expr``).

Shape of an emitted kernel (see plan.py for the schedule it realises):

    prologue   carve shared memory into one plane ring per tensor, locate this
               block's tile / chunk, precompute per-thread store masks,
               init mbarriers, request the first `prefetch` input planes (TMA)
    per step   thread 0 requests input plane i+prefetch; everyone waits for
               plane i; every stage computes its plane (i - delay) from ring
               planes finished in earlier steps and writes its own ring slot;
               final outputs go to HBM with 128-bit stores; __syncthreads()
"""
import collections

from haoda import util
from soda.codegen.cuda import plan as plan_mod

_TMA_MAX_BOX = 256


def kernel_name(sched):
  return 'soda_%s_d%d' % (sched.program.app_name, sched.depth)


class Layout:
  """Byte offsets of rings, guards and barriers in dynamic shared memory."""

  def __init__(self, sched):
    self.sched = sched
    self.guard = -(-sched.guard_elems * 8 // 128) * 128
    loaded = [n for n in sched.inputs if n.ring_depth]
    self.in_depth = max([n.ring_depth for n in loaded] + [1])
    self.ring_depth = {}
    self.ring_offset = {}
    offset = self.guard
    for node in sched.nodes:
      depth = self.in_depth if node.is_input else node.ring_depth
      if not node.ring_depth:
        continue
      self.ring_depth[node.index] = depth
      self.ring_offset[node.index] = offset
      ring = depth * sched.plane_elems * node.elem_size
      offset += -(-ring // 128) * 128
    offset += self.guard
    self.bar_offset = offset
    offset += -(-8 * self.in_depth // 128) * 128
    self.total = offset
    # TMA boxes: dim 0 split so no box edge exceeds 256 elements
    tile0 = sched.tile[0]
    self.boxes_per_row = -(-tile0 // _TMA_MAX_BOX)
    if tile0 % self.boxes_per_row:
      raise util.SemanticError('tile width %d cannot be split into equal TMA '
                               'boxes' % tile0)
    self.box0 = tile0 // self.boxes_per_row
    if self.boxes_per_row > 1 and sched.sdim > 1:
      # a box is dense in shared memory, so a split row only matches the
      # plane layout when the plane is a single row
      raise util.SemanticError('tiles wider than %d elements need a 2-D '
                               'program' % _TMA_MAX_BOX)
    for extent in sched.tile[1:]:
      if extent > _TMA_MAX_BOX:
        raise util.SemanticError('tile extent %d exceeds the TMA box limit' %
                                 extent)
    self.plane_bytes = {n.index: sched.plane_elems * n.elem_size
                        for n in loaded}
    self.loaded_inputs = loaded


def _log2(n):
  return n.bit_length() - 1


def emit_item(p):
  """The grid item of a batch this block works on: plain loads and stores
  reach it through the per-tensor offsets (``emit_offsets``), TMA loads
  through the item coordinate of the tensor maps."""
  p.println('const int item = a.item_begin + blockIdx.z;   // of the batch')


def emit_offset_arrays(p, inputs, outputs, vpt):
  """Declare the per-thread HBM offsets of every loaded input and output."""
  for node in inputs:
    p.println('long long ioff%d[%d];   // input %d' % (
        node.input_index, vpt, node.input_index))
  for node in outputs:
    p.println('long long ooff%d[%d];   // output %d' % (
        node.output_index, vpt, node.output_index))


def emit_offsets(p, inputs, outputs, sdim):
  """Inside the per-vector loop over ``j``: where vector ``j`` of the item
  lies in each tensor, in elements from its base, for plane 0 of the streamed
  dimension.  Every tensor has strides of its own (a view, a pitched
  allocation); in the TMA instance the inputs' offsets are dead code."""
  def offset(which, k):
    terms = ['gx[j]', 'item * a.%s_stride[%d][soda::kMaxDim]' % (which, k)]
    terms += ['gc%d[j] * a.%s_stride[%d][%d]' % (d, which, k, d)
              for d in range(1, sdim)]
    return ' + '.join(terms)
  for node in inputs:
    p.println('ioff%d[j] = %s;' % (node.input_index,
                                   offset('in', node.input_index)))
  for node in outputs:
    p.println('ooff%d[j] = %s;' % (node.output_index,
                                   offset('out', node.output_index)))


def _render_stage(stage, ref_code):
  """``Stage.render`` for device code: DSL calls go through the soda_fn_*
  wrappers and let variables get a prefix that cannot clash with the
  kernel's own identifiers."""
  return stage.render(ref_code, call_prefix='soda_fn_', let_prefix='let_')


def emit_kernel(p, sched):
  """Write the kernel for ``sched`` through Printer ``p``; returns its Layout."""
  prog = sched.program
  lay = Layout(sched)
  s = sched.sdim
  V = sched.vec
  NT = sched.threads
  VPT = sched.vecs_per_thread
  PLANE = sched.plane_elems
  XV = sched.tile[0] // V
  name = kernel_name(sched)
  P = sched.prefetch
  DIN = lay.in_depth

  p.println('// %s' % sched.describe().replace('\n', '\n// '))
  p.println('template <bool kTma>')
  p.println('__global__ void __launch_bounds__(%d) %s(' % (NT, name))
  p.println('    const __grid_constant__ soda::StreamArgs a)')
  p.do_scope()
  p.println('extern __shared__ __align__(1024) unsigned char smem_raw[];')
  for node in sched.nodes:
    if node.index in lay.ring_offset:
      p.println('%s* const ring_%s = reinterpret_cast<%s*>(smem_raw + %d);'
                '  // %d planes' % (node.c_type, node.ident, node.c_type,
                                    lay.ring_offset[node.index],
                                    lay.ring_depth[node.index]))
  p.println('uint64_t* const bars = reinterpret_cast<uint64_t*>(smem_raw + %d);'
            % lay.bar_offset)
  p.println('const int tid = threadIdx.x;')
  plan_mod.emit_param_pointers(p, sched.program)
  p.println()
  p.println('// this block: one tile of the non-streamed dims, one chunk of '
            'the streamed dim')
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
  p.println('const int steps = (r1 - r0) + %d;' %
            (sched.lead + sched.out_delay))
  emit_item(p)
  p.println()
  p.println('// per-thread vectors: linear position in the plane, where they '
            'land in HBM,')
  p.println('// which cells this tile owns (store) and which are in the '
            'valid region (else 0)')
  p.println('int pos[%d];' % VPT)
  emit_offset_arrays(p, lay.loaded_inputs, sched.outputs, VPT)
  p.println('unsigned own[%d];' % VPT)
  for n in range(len(sched.outputs)):
    p.println('unsigned val%d[%d];   // output %d: cells in ITS valid region' %
              (n, VPT, n))
  p.println('int gx[%d];' % VPT)
  for d in range(1, s):
    p.println('int gc%d[%d];' % (d, VPT))
  p.println('#pragma unroll')
  p.println('for (int j = 0; j < %d; ++j)' % VPT)
  p.do_scope()
  p.println('const int q = tid + j * %d;' % NT)
  p.println('pos[j] = q * %d;' % V)
  p.println('const int c0 = (q %% %d) * %d;' % (XV, V))
  p.println('int rest = q / %d;' % XV)
  for d in range(1, s):
    p.println('const int c%d = rest %% %d;' % (d, sched.tile[d]))
    if d + 1 < s:
      p.println('rest /= %d;' % sched.tile[d])
  p.println('(void)rest;')
  p.println('gx[j] = org0 + c0;')
  p.println('bool mine = true;')
  for n in range(len(sched.outputs)):
    p.println('bool ok%d = true;' % n)
  for d in range(1, s):
    p.println('gc%d[j] = org%d + c%d;' % (d, d, d))
    p.println('mine = mine && c%d >= %d && c%d < %d && gc%d[j] < a.dims[%d];' %
              (d, sched.tile_halo_lo[d], d,
               sched.tile[d] - sched.tile_halo_hi[d], d, d))
    for n in range(len(sched.outputs)):
      p.println('ok%d = ok%d && gc%d[j] >= a.valid_lo[%d][%d] && gc%d[j] < '
                'a.valid_hi[%d][%d];' % (n, n, d, n, d, d, n, d))
  emit_offsets(p, lay.loaded_inputs, sched.outputs, s)
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
  p.un_scope()
  p.println()

  # --- input plane requests ---------------------------------------------------
  def tma_issue(rel_code):
    """Code for thread 0: request every input's plane `rel`."""
    p.println('uint64_t* const bar = &bars[(%s) & %d];' % (rel_code, DIN - 1))
    total = sum(lay.plane_bytes.values())
    p.println('soda::mbar_expect_tx(bar, %d);' % total)
    for node in lay.loaded_inputs:
      for b in range(lay.boxes_per_row):
        coords = ['org0 + %d' % (b * lay.box0)] + [
            'org%d' % d for d in range(1, s)] + ['base + (%s)' % rel_code,
                                                 'item']
        p.println('soda::tma_load(ring_%s + ((%s) & %d) * %d + %d, '
                  '&a.in_map[%d], bar, %s);' % (
                      node.ident, rel_code, DIN - 1, PLANE, b * lay.box0,
                      node.input_index, ', '.join(coords)))

  def plain_load(rel_code, into_smem):
    """Fallback: every thread fetches its own vectors of plane `rel`."""
    p.println('const int lrow = base + (%s);' % rel_code)
    p.println('const bool lrow_in = lrow >= 0 && lrow < a.dims[%d];' % s)
    for node in lay.loaded_inputs:
      p.println('#pragma unroll')
      p.println('for (int j = 0; j < %d; ++j)' % VPT)
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
      p.println('soda::st_pack<%s, %d>(ring_%s + ((%s) & %d) * %d + pos[j], '
                't);' % (node.c_type, V, node.ident, rel_code, DIN - 1, PLANE))
      p.un_scope()
    del into_smem

  p.println('if (kTma)')
  p.do_scope()
  p.println('if (tid == 0)')
  p.do_scope()
  for node in lay.loaded_inputs:
    p.println('soda::tma_prefetch_desc(&a.in_map[%d]);' % node.input_index)
  p.println('for (int n = 0; n < %d; ++n) soda::mbar_init(&bars[n], 1);' % DIN)
  p.println('soda::mbar_fence_init();')
  p.un_scope()
  p.println('__syncthreads();')
  p.println('if (tid == 0)')
  p.do_scope()
  p.println('for (int rel = 0; rel < %d && rel < steps; ++rel)' % P)
  p.do_scope()
  tma_issue('rel')
  p.un_scope()
  p.un_scope()
  p.un_scope()
  p.println('else')
  p.do_scope()
  p.do_scope()
  plain_load('0', True)
  p.un_scope()
  p.println('__syncthreads();')
  p.un_scope()
  p.println()

  # --- the streamed loop ------------------------------------------------------
  p.println('for (int i = 0; i < steps; ++i)')
  p.do_scope()
  p.println('if (kTma)')
  p.do_scope()
  p.println('if (tid == 0 && i + %d < steps)' % P)
  p.do_scope()
  tma_issue('i + %d' % P)
  p.un_scope()
  p.println('soda::mbar_wait(&bars[i & %d], (i >> %d) & 1);' % (
      DIN - 1, _log2(DIN)))
  p.un_scope()

  for node in sched.stage_nodes:
    _emit_stage(p, sched, lay, node)

  p.println('if (!kTma && i + 1 < steps)')
  p.do_scope()
  plain_load('i + 1', True)
  p.un_scope()
  p.println('__syncthreads();')
  p.un_scope()
  p.un_scope()
  p.println()
  del prog
  return lay


def _emit_stage(p, sched, lay, node):
  s = sched.sdim
  V = sched.vec
  VPT = sched.vecs_per_thread
  PLANE = sched.plane_elems
  stage = node.stage
  p.println('// %s: plane i - %d' % (node.ident, node.delay))
  p.do_scope()
  if node.output_index is not None:
    p.println('const int row = base + i - %d;' % node.delay)
    p.println('const bool row_mine = row >= r0 && row < r1;')
    p.println('const bool row_ok = row >= a.valid_lo[%d][%d] && row < '
              'a.valid_hi[%d][%d];' % (node.output_index, s,
                                       node.output_index, s))
  p.println('#pragma unroll')
  p.println('for (int j = 0; j < %d; ++j)' % VPT)
  p.do_scope()

  # operand windows, one per (parent, offsets in dims 1..)
  groups = collections.OrderedDict()
  parent_of = {}
  for parent, off in node.loads:
    key = (parent.index, off[1:])
    groups.setdefault(key, set()).add(off[0])
    parent_of[parent.index] = parent
  window_of = {}
  for g, ((pindex, rest), dxs) in enumerate(groups.items()):
    parent = parent_of[pindex]
    depth = lay.ring_depth[pindex]
    xlo, xhi = min(dxs), max(dxs)
    used = sorted({k + dx for dx in dxs for k in range(V)})
    inplane = sum(rest[d - 1] * sched.plane_pitch(d) for d in range(1, s))
    slot = '((i + (%d)) & %d)' % (rest[s - 1] - node.delay, depth - 1)
    p.println('const %s* const s%d = ring_%s + %s * %d + pos[j] + (%d);' % (
        parent.c_type, g, parent.ident, slot, PLANE, inplane))
    p.println('%s w%d[%d];' % (parent.c_type, g, V + xhi - xlo))
    inside = [c for c in used if 0 <= c < V]
    if len(inside) >= 2 and xlo <= 0 <= xhi:   # the aligned vector fits in w
      p.println('soda::ld_pack<%s, %d>(w%d + %d, s%d);' % (
          parent.c_type, V, g, -xlo, g))
      outside = [c for c in used if not 0 <= c < V]
    else:
      outside = used
    for c in outside:
      p.println('w%d[%d] = s%d[%d];' % (g, c - xlo, g, c))
    window_of[(pindex, rest)] = (g, xlo)

  # a stage's Load names the program tensor; node.loads holds, in the same
  # order, the chain tensor it resolves to in this fused iteration
  resolved = dict(zip(
      [l for l in stage.loads if l.parent not in sched.program.params],
      node.loads))

  def ref_code(load):
    if load.parent in sched.program.params:
      return plan_mod.param_code(sched.program, load)
    parent, off = resolved[load]
    g, xlo = window_of[(parent.index, off[1:])]
    return 'w%d[k + %d]' % (g, off[0] - xlo)

  lets, expr = _render_stage(stage, ref_code)
  p.println('%s r[%d];' % (node.c_type, V))
  p.println('#pragma unroll')
  p.println('for (int k = 0; k < %d; ++k)' % V)
  p.do_scope()
  for let in lets:
    p.println(let)
  p.println('r[k] = soda::store_cast<%s>(%s);' % (node.c_type, expr))
  p.un_scope()
  if node.index in lay.ring_offset:
    p.println('soda::st_pack<%s, %d>(ring_%s + ((i + (%d)) & %d) * %d + pos[j],'
              ' r);' % (node.c_type, V, node.ident, -node.delay,
                        lay.ring_depth[node.index] - 1, PLANE))
  if node.output_index is not None:
    full = (1 << V) - 1
    p.println('if (row_mine && own[j])')
    p.do_scope()
    n = node.output_index
    p.println('%s* const dst = static_cast<%s*>(a.out_ptr[%d]) + row * '
              'a.out_stride[%d][%d] + ooff%d[j];' % (node.c_type, node.c_type,
                                                     n, n, s, n))
    p.println('const unsigned keep = row_ok ? val%d[j] : 0u;' % node.output_index)
    p.println('if (keep != %du)' % full)
    p.do_scope()
    p.println('#pragma unroll')
    p.println('for (int k = 0; k < %d; ++k)' % V)
    p.println('  if (!((keep >> k) & 1u)) r[k] = %s(0);' % node.c_type)
    p.un_scope()
    p.println('if (own[j] == %du && a.vec_store[%d])' % (full, n))
    p.do_scope()
    p.println('soda::st_pack_global<%s, %d>(dst, r);' % (node.c_type, V))
    p.un_scope()
    p.println('else')
    p.do_scope()
    p.println('#pragma unroll')
    p.println('for (int k = 0; k < %d; ++k)' % V)
    p.println('  if ((own[j] >> k) & 1u) dst[k] = r[k];')
    p.un_scope()
    p.un_scope()
  p.un_scope()
  p.un_scope()
