"""Build, load and run SODA programs on a B200: ``soda.cuda.run(stencil, arrays)``.

The thin Python side of the CUDA backend: it drives ``soda.codegen.cuda`` to emit
the kernel and host files of a ``soda.core.Stencil``, compiles them offline with
``nvcc -gencode arch=compute_100a,code=sm_100a`` into one shared library per
program, and calls that library through the C ABI of include/soda_cuda.h with
ctypes.  There is no CPU fallback and no other backend: without nvcc the build
raises, without a CUDA device the library returns ``no_device_interface``
(-19) and ``run`` raises.

Arrays follow the reference harness' layout (reference
src/soda/codegen/xilinx/host.py:1011-1020): dense, dimension 0 fastest — a numpy
array of shape ``(dims[n-1], ..., dims[0])``, C-contiguous.  numpy arrays are
host buffers (copied to and from the device inside the call); torch CUDA
tensors are passed zero-copy through ``buffer_t.dev``.
"""
import ctypes
import hashlib
import io
import os
import shutil
import subprocess
import threading

import numpy as np

from haoda import util
from soda.codegen import cuda as codegen
from soda.codegen.cuda import host as host_gen
from soda.codegen.cuda import plan as plan_mod

_PKG_ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC_DIR = os.path.join(_PKG_ROOT, 'csrc')
INCLUDE_DIR = os.path.join(os.path.dirname(_PKG_ROOT), 'include')
DEFAULT_BUILD_DIR = os.path.join(_PKG_ROOT, '_build')
ARCH_FLAGS = ['-gencode', 'arch=compute_100a,code=sm_100a']

NUMPY_TYPES = {
    'uint8': np.uint8, 'uint16': np.uint16, 'uint32': np.uint32,
    'uint64': np.uint64, 'int8': np.int8, 'int16': np.int16,
    'int32': np.int32, 'int64': np.int64, 'float': np.float32,
    'float32': np.float32, 'double': np.float64, 'float64': np.float64,
    'half': np.float16}

ERROR_NAMES = {
    -1: 'generic_error', -3: 'bad_elem_size', -4: 'access_out_of_bounds',
    -6: 'buffer_extents_too_large', -11: 'out_of_memory',
    -12: 'buffer_argument_is_null', -14: 'copy_to_host_failed',
    -15: 'copy_to_device_failed', -16: 'device_malloc_failed',
    -17: 'device_sync_failed', -19: 'no_device_interface',
    -22: 'internal_error', -23: 'device_run_failed'}


class CudaError(RuntimeError):
  """A call into a compiled SODA library failed (code: Halide numbering)."""

  def __init__(self, what, code):
    super().__init__('%s failed: %d (%s)' % (
        what, code, ERROR_NAMES.get(code, 'unknown')))
    self.code = code


class BufferT(ctypes.Structure):
  """Legacy Halide buffer_t (reference header.py:36-48); sizeof == 72."""
  _fields_ = [('dev', ctypes.c_uint64), ('host', ctypes.c_void_p),
              ('extent', ctypes.c_int32 * 4), ('stride', ctypes.c_int32 * 4),
              ('min', ctypes.c_int32 * 4), ('elem_size', ctypes.c_int32),
              ('host_dirty', ctypes.c_bool), ('dev_dirty', ctypes.c_bool),
              ('_padding', ctypes.c_uint8 * 2)]


class Stats(ctypes.Structure):
  _fields_ = [('kernel_ms', ctypes.c_double), ('h2d_ms', ctypes.c_double),
              ('d2h_ms', ctypes.c_double), ('cells', ctypes.c_int64),
              ('iterate', ctypes.c_int32), ('launches', ctypes.c_int32),
              ('depth', ctypes.c_int32), ('used_tma', ctypes.c_int32),
              ('blocks', ctypes.c_int32), ('threads', ctypes.c_int32),
              ('smem_bytes', ctypes.c_int32), ('reserved', ctypes.c_int32)]

  def as_dict(self):
    return {name: getattr(self, name) for name, _ in self._fields_
            if name != 'reserved'}


# --- build --------------------------------------------------------------------

def generate_sources(stencil, options=None, fast_math=False):
  """``(program, kernel source, host source)`` for a Stencil."""
  program = plan_mod.extract_program(stencil)
  schedules = codegen.make_schedules(program, options, fast_math)
  kernel, host = io.StringIO(), io.StringIO()
  codegen.print_kernel(program, schedules, kernel, fast_math)
  host_gen.print_code(program, host)
  return program, kernel.getvalue(), host.getvalue()


def nvcc_command(sources, output, fast_math=False, extra=()):
  flags = ['-O3', '-std=c++17', '-lineinfo', '-Xcompiler', '-fPIC', '-shared',
           '-I', CSRC_DIR, '-I', INCLUDE_DIR]
  # exact mode: no FMA contraction, so float results match the reference's
  # x86-64 golden loop bit for bit (SURVEY.md §0.5)
  # fast mode (tolerance-tested only): FMA contraction, approximate division
  # (div.approx: 2 ulp) and square root, a / sqrt(x) as a refined MUFU.RSQ
  flags += (['-DSODA_CUDA_FAST_MATH', '-prec-div=false', '-prec-sqrt=false']
            if fast_math else ['-fmad=false'])
  return (['nvcc'] + ARCH_FLAGS + flags + list(extra) + list(sources) +
          ['-o', output])


def build(stencil, build_dir=None, options=None, fast_math=False,
          force=False, verbose=False):
  """Emit and compile ``stencil``; returns the path of ``libsoda_<app>.so``.

  Builds are cached by a hash of the generated and hand-written sources and
  the flags, under ``<package>/_build/<app>-<hash>/`` (in-tree on purpose: the
  libraries travel with the repository snapshot to GPU machines).
  """
  if shutil.which('nvcc') is None:
    raise RuntimeError('nvcc not found: the SODA CUDA backend compiles its '
                       'kernels offline and has no other execution path')
  program, kernel_src, host_src = generate_sources(stencil, options,
                                                   fast_math)
  runtime = os.path.join(CSRC_DIR, 'soda_cuda_runtime.cu')
  digest = hashlib.sha256()
  for text in (kernel_src, host_src, str(fast_math)):
    digest.update(text.encode())
  # what a program library is compiled from besides its generated files (the
  # wire-format kernels in csrc/ are a library of their own)
  for name in ('soda_cuda_device.cuh', 'soda_cuda_runtime.cu',
               'soda_cuda_runtime.h', '../../include/soda_cuda.h'):
    with open(os.path.join(CSRC_DIR, name), 'rb') as handle:
      digest.update(handle.read())
  out_dir = os.path.join(build_dir or DEFAULT_BUILD_DIR, '%s-%s' % (
      program.app_name, digest.hexdigest()[:12]))
  lib = os.path.join(out_dir, 'libsoda_%s.so' % program.app_name)
  if os.path.exists(lib) and not force:
    return lib
  os.makedirs(out_dir, exist_ok=True)
  kernel_path = os.path.join(out_dir, '%s_kernel.cu' % program.app_name)
  host_path = os.path.join(out_dir, '%s_host.cpp' % program.app_name)
  with open(kernel_path, 'w') as handle:
    handle.write(kernel_src)
  with open(host_path, 'w') as handle:
    handle.write(host_src)
  # concurrent builders (processes or threads) do not collide
  tmp = '%s.%d.%d.tmp' % (lib, os.getpid(), threading.get_ident())
  command = nvcc_command([kernel_path, host_path, runtime], tmp,
                         fast_math, ['-Xptxas', '-v'] if verbose else [])
  done = subprocess.run(command, stdout=subprocess.PIPE,
                        stderr=subprocess.STDOUT, text=True, check=False)
  if verbose:
    print(done.stdout)
  if done.returncode != 0:
    raise RuntimeError('nvcc failed for %s:\n%s\n%s' % (
        program.app_name, ' '.join(command), done.stdout))
  os.replace(tmp, lib)
  return lib


# --- load ---------------------------------------------------------------------

class Library:
  """A compiled SODA program, bound through the C ABI (include/soda_cuda.h)."""

  def __init__(self, path):
    self.path = path
    lib = self._lib = ctypes.CDLL(path)
    c_int, c_void_p, c_char_p = ctypes.c_int, ctypes.c_void_p, ctypes.c_char_p
    i32p = ctypes.POINTER(ctypes.c_int32)
    bufpp = ctypes.POINTER(ctypes.POINTER(BufferT))
    voidpp = ctypes.POINTER(c_void_p)
    for name, restype, argtypes in (
        ('soda_cuda_app_name', c_char_p, []),
        ('soda_cuda_dim', c_int, []),
        ('soda_cuda_iterate', c_int, []),
        ('soda_cuda_num_inputs', c_int, []),
        ('soda_cuda_num_outputs', c_int, []),
        ('soda_cuda_tensor_name', c_char_p, [c_int, c_int]),
        ('soda_cuda_tensor_type', c_char_p, [c_int, c_int]),
        ('soda_cuda_tensor_elem_size', c_int, [c_int, c_int]),
        ('soda_cuda_window', c_int, [c_int, i32p, i32p]),
        ('soda_cuda_window_of', c_int, [c_int, c_int, i32p, i32p]),
        ('soda_cuda_run', c_int, [bufpp, bufpp, c_char_p]),
        ('soda_cuda_run_params', c_int, [bufpp, bufpp, bufpp, c_char_p]),
        ('soda_cuda_num_params', c_int, []),
        ('soda_cuda_param_name', c_char_p, [c_int]),
        ('soda_cuda_param_type', c_char_p, [c_int]),
        ('soda_cuda_param_size', c_int, [c_int, i32p]),
        ('soda_cuda_set_params', c_int, [voidpp]),
        ('soda_cuda_run_device', c_int,
         [voidpp, voidpp, i32p, c_int, c_void_p]),
        ('soda_cuda_run_batch', c_int, [bufpp, bufpp, bufpp, c_int]),
        ('soda_cuda_run_device_batch', c_int,
         [voidpp, voidpp, i32p, c_int, c_int, c_void_p]),
        ('soda_cuda_launch', c_int,
         [c_int, voidpp, voidpp, i32p, c_int, c_int, i32p, i32p, c_void_p]),
        ('soda_cuda_launch_chunked', c_int,
         [c_int, voidpp, voidpp, i32p, c_int, c_int, i32p, i32p, c_int,
          c_void_p]),
        ('soda_cuda_chunk_rows', c_int, [c_int, i32p, c_int]),
        ('soda_cuda_lead_rows', c_int, [c_int]),
        ('soda_cuda_depths', c_int, [i32p, c_int]),
        ('soda_cuda_flag_write', c_int, [c_void_p, ctypes.c_uint32, c_void_p]),
        ('soda_cuda_flag_wait_geq', c_int,
         [c_void_p, ctypes.c_uint32, c_void_p]),
        ('soda_cuda_ipc_export', c_int,
         [c_void_p, ctypes.c_char_p, ctypes.POINTER(ctypes.c_uint64)]),
        ('soda_cuda_ipc_open', c_int, [ctypes.c_char_p, voidpp]),
        ('soda_cuda_ipc_close', c_int, [c_void_p]),
        ('soda_cuda_copy_async', c_int,
         [c_void_p, c_void_p, ctypes.c_uint64, c_void_p]),
        ('soda_cuda_last_stats', ctypes.POINTER(Stats), []),
        ('soda_cuda_shard_plan', c_int,
         [i32p, c_int, i32p, i32p, i32p, i32p]),
        ('soda_cuda_slab_stats', c_int, [c_int, ctypes.POINTER(Stats)]),
        ('soda_cuda_release', None, []),
    ):
      fn = getattr(lib, name)
      fn.restype, fn.argtypes = restype, argtypes
    self.app_name = lib.soda_cuda_app_name().decode()
    self.dim = lib.soda_cuda_dim()
    self.iterate = lib.soda_cuda_iterate()
    self.inputs = [(lib.soda_cuda_tensor_name(0, k).decode(),
                    lib.soda_cuda_tensor_type(0, k).decode())
                   for k in range(lib.soda_cuda_num_inputs())]
    self.outputs = [(lib.soda_cuda_tensor_name(1, k).decode(),
                     lib.soda_cuda_tensor_type(1, k).decode())
                    for k in range(lib.soda_cuda_num_outputs())]
    depths = (ctypes.c_int32 * 16)()
    self.depths = list(depths[:lib.soda_cuda_depths(depths, 16)])
    self.params = []            # [(name, haoda type, size tuple)]
    for k in range(lib.soda_cuda_num_params()):
      size = (ctypes.c_int32 * 4)()
      rank = lib.soda_cuda_param_size(k, size)
      self.params.append((lib.soda_cuda_param_name(k).decode(),
                          lib.soda_cuda_param_type(k).decode(),
                          tuple(size[:rank])))

  def window(self, iterate=None):
    """``(lo, hi)`` offsets per dim read by the cells of any output after
    ``iterate`` iterations (the union over the outputs: sizes halos)."""
    lo, hi = (ctypes.c_int32 * 4)(), (ctypes.c_int32 * 4)()
    code = self._lib.soda_cuda_window(
        self.iterate if iterate is None else iterate, lo, hi)
    if code:
      raise CudaError('soda_cuda_window', code)
    return tuple(lo[:self.dim]), tuple(hi[:self.dim])

  def window_of(self, output, iterate=None):
    """The window of output number ``output`` alone: bounds where THAT output
    is defined (reference host.py:1082-1091)."""
    lo, hi = (ctypes.c_int32 * 4)(), (ctypes.c_int32 * 4)()
    code = self._lib.soda_cuda_window_of(
        output, self.iterate if iterate is None else iterate, lo, hi)
    if code:
      raise CudaError('soda_cuda_window_of', code)
    return tuple(lo[:self.dim]), tuple(hi[:self.dim])

  def valid_region(self, dims, iterate=None, output=0):
    """``[(lo, hi)]`` per dimension where output ``output`` is defined."""
    lo, hi = self.window_of(output, iterate)
    return [(max(0, -l), n - max(0, h)) for l, h, n in zip(lo, hi, dims)]

  def valid_regions(self, dims, iterate=None):
    return [self.valid_region(dims, iterate, k)
            for k in range(len(self.outputs))]

  @property
  def stats(self):
    return self._lib.soda_cuda_last_stats().contents.as_dict()

  def release(self):
    self._lib.soda_cuda_release()

  def shard_plan(self, dims, n_slabs):
    """How ``run(..., devices=[..])`` cuts a grid: per slab ``(local_begin,
    local_end, own_begin, own_end)`` rows of the streamed dimension."""
    arrays = [(ctypes.c_int32 * n_slabs)() for _ in range(4)]
    used = self._lib.soda_cuda_shard_plan(
        (ctypes.c_int32 * 4)(*(list(dims) + [1] * (4 - len(dims)))), n_slabs,
        *arrays)
    if used < 0:
      raise CudaError('soda_cuda_shard_plan', used)
    return [tuple(a[r] for a in arrays) for r in range(used)]

  @property
  def slab_stats(self):
    """Per slab of the last sharded run (empty if it was not sharded)."""
    count = self._lib.soda_cuda_slab_stats(-1, None)
    result = []
    for index in range(count):
      stats = Stats()
      self._lib.soda_cuda_slab_stats(index, ctypes.byref(stats))
      result.append(stats.as_dict())
    return result

  # ---- buffers ----
  def _describe(self, array, haoda_type, what, batched=False):
    """array -> (BufferT, dims); numpy = host memory, torch CUDA = device.

    ``batched``: the array holds a batch, shape ``(B, dims[n-1], .., dims[0])``;
    the buffer describes item 0 and ``dims`` ends with ``B``."""
    elem = util.get_width_in_bytes(haoda_type)
    buf = BufferT()
    if isinstance(array, np.ndarray):
      if array.dtype != NUMPY_TYPES[haoda_type]:
        raise TypeError('%s must be %s, got %s' % (what, haoda_type,
                                                   array.dtype))
      if not array.flags['C_CONTIGUOUS']:
        raise ValueError('%s must be C-contiguous' % what)
      buf.host = array.ctypes.data
      shape = array.shape
    elif hasattr(array, 'data_ptr'):    # torch tensor
      if not array.is_contiguous():
        raise ValueError('%s must be contiguous' % what)
      if array.element_size() != elem:
        raise TypeError('%s must have %d-byte elements' % (what, elem))
      if array.is_cuda:
        buf.dev = array.data_ptr()
      else:
        buf.host = array.data_ptr()
      shape = tuple(array.shape)
    else:
      raise TypeError('%s: expected a numpy array or a torch tensor' % what)
    rank = self.dim + (1 if batched else 0)
    if len(shape) != rank:
      raise ValueError('%s must be %d-dimensional%s' % (
          what, rank, ' (a leading batch dimension)' if batched else ''))
    dims = tuple(reversed(shape))
    stride = 1
    for d, extent in enumerate(dims[:self.dim]):
      buf.extent[d], buf.stride[d] = extent, stride
      stride *= extent
    buf.elem_size = elem
    return buf, dims

  def _param_arrays(self, params):
    """The param arrays as C-contiguous numpy arrays of the declared type
    and shape (``T name[s0][s1]``: numpy shape ``(s0, s1)``)."""
    if isinstance(params, dict):
      params = [params[name] for name, _, _ in self.params]
    if params is None or len(params) != len(self.params):
      raise ValueError('%s takes %d param array(s): %s' % (
          self.app_name, len(self.params),
          ', '.join(name for name, _, _ in self.params)))
    arrays = []
    for array, (name, haoda_type, size) in zip(params, self.params):
      array = np.ascontiguousarray(array, dtype=NUMPY_TYPES[haoda_type])
      if array.shape != size:
        raise ValueError('param `%s` must have shape %s, got %s' % (
            name, size, array.shape))
      arrays.append(array)
    return arrays

  def set_params(self, params):
    """Upload the param arrays for the device-level entry points
    (run_device, launch); they stay in effect until set again."""
    arrays = self._param_arrays(params)
    pointers = (ctypes.c_void_p * len(arrays))(
        *[a.ctypes.data for a in arrays])
    code = self._lib.soda_cuda_set_params(pointers)
    if code:
      raise CudaError('soda_cuda_set_params(%s)' % self.app_name, code)

  def run(self, inputs, outputs=None, params=None, devices=None):
    """Run the whole program (all ``iterate`` iterations); returns outputs.

    ``devices``: CUDA ordinals (or ``'all'``) to spread a run on HOST arrays
    over — one slab of the streamed dimension per entry, bit-identical to
    the one-device run (soda_cuda_run's "devices=" config).

    ``inputs`` in program order.  ``outputs``: arrays to fill, or None to
    allocate them like the first input (numpy -> numpy, torch -> torch).
    ``params``: the program's param arrays (list in program order or dict by
    name), required if it declares any.
    """
    if len(inputs) != len(self.inputs):
      raise ValueError('%s takes %d input(s)' % (self.app_name,
                                                 len(self.inputs)))
    in_bufs = []
    dims = None
    for array, (name, haoda_type) in zip(inputs, self.inputs):
      buf, got = self._describe(array, haoda_type, 'input `%s`' % name)
      if dims is not None and got != dims:
        raise ValueError('input `%s` has extent %s, expected %s' %
                         (name, got, dims))
      dims = got
      in_bufs.append(buf)
    if outputs is None:
      outputs = [self._allocate_like(inputs[0], haoda_type, dims)
                 for _, haoda_type in self.outputs]
    out_bufs = []
    for array, (name, haoda_type) in zip(outputs, self.outputs):
      buf, got = self._describe(array, haoda_type, 'output `%s`' % name)
      if got != dims:
        raise ValueError('output `%s` has extent %s, expected %s' %
                         (name, got, dims))
      out_bufs.append(buf)
    in_ptrs = (ctypes.POINTER(BufferT) * len(in_bufs))(
        *[ctypes.pointer(b) for b in in_bufs])
    out_ptrs = (ctypes.POINTER(BufferT) * len(out_bufs))(
        *[ctypes.pointer(b) for b in out_bufs])
    config = None
    if devices is not None:
      config = ('devices=%s' % (devices if isinstance(devices, str) else
                                ','.join(str(d) for d in devices))).encode()
    if self.params:
      param_ptrs, keep_alive = self._param_buffers(params)
      code = self._lib.soda_cuda_run_params(in_ptrs, out_ptrs, param_ptrs,
                                            config)
    else:
      code = self._lib.soda_cuda_run(in_ptrs, out_ptrs, config)
    if code:
      raise CudaError('soda_cuda_run(%s)' % self.app_name, code)
    return list(outputs)

  def _param_buffers(self, params):
    """``(buffer_t* array, the arrays it points into)`` of the params."""
    arrays = self._param_arrays(params)
    param_bufs = []
    for array, (_, haoda_type, size) in zip(arrays, self.params):
      buf = BufferT()
      buf.host = array.ctypes.data
      buf.elem_size = util.get_width_in_bytes(haoda_type)
      stride = 1
      for d, extent in enumerate(size):
        # the reference harness' descriptor of a param (host.py:1022-1030)
        buf.extent[d], buf.stride[d] = extent, stride
        stride *= extent
      param_bufs.append(buf)
    pointers = (ctypes.POINTER(BufferT) * len(param_bufs))(
        *[ctypes.pointer(b) for b in param_bufs])
    return pointers, (arrays, param_bufs)

  def run_batch(self, inputs, outputs=None, params=None):
    """Run the whole program on a batch of independent grids; returns the
    outputs.

    Every array has shape ``(B, dims[n-1], .., dims[0])``: ``B`` grids of the
    same extents, each computed exactly as ``run`` computes it alone.  numpy
    arrays are host memory, torch CUDA tensors are used in place.
    ``outputs``: arrays to fill, or None to allocate them like the first
    input.  ``params`` (as for ``run``) are shared by all items.
    """
    if len(inputs) != len(self.inputs):
      raise ValueError('%s takes %d input(s)' % (self.app_name,
                                                 len(self.inputs)))
    if outputs is not None and len(outputs) != len(self.outputs):
      raise ValueError('%s has %d output(s)' % (self.app_name,
                                                len(self.outputs)))
    in_bufs, extents = [], None
    for array, (name, haoda_type) in zip(inputs, self.inputs):
      buf, got = self._describe(array, haoda_type, 'input `%s`' % name, True)
      if extents is not None and got != extents:
        raise ValueError('input `%s` has extent %s (items last), expected %s'
                         % (name, got, extents))
      extents = got
      in_bufs.append(buf)
    if outputs is None:
      outputs = [self._allocate_like(inputs[0], haoda_type, extents)
                 for _, haoda_type in self.outputs]
    out_bufs = []
    for array, (name, haoda_type) in zip(outputs, self.outputs):
      buf, got = self._describe(array, haoda_type, 'output `%s`' % name, True)
      if got != extents:
        raise ValueError('output `%s` has extent %s (items last), expected %s'
                         % (name, got, extents))
      out_bufs.append(buf)
    in_ptrs = (ctypes.POINTER(BufferT) * len(in_bufs))(
        *[ctypes.pointer(b) for b in in_bufs])
    out_ptrs = (ctypes.POINTER(BufferT) * len(out_bufs))(
        *[ctypes.pointer(b) for b in out_bufs])
    param_ptrs = None
    if self.params:
      param_ptrs, keep_alive = self._param_buffers(params)
    code = self._lib.soda_cuda_run_batch(in_ptrs, out_ptrs, param_ptrs,
                                         extents[-1])
    if code:
      raise CudaError('soda_cuda_run_batch(%s)' % self.app_name, code)
    return list(outputs)

  @staticmethod
  def _allocate_like(like, haoda_type, dims):
    shape = tuple(reversed(dims))
    if isinstance(like, np.ndarray):
      return np.empty(shape, dtype=NUMPY_TYPES[haoda_type])
    import torch
    dtype = torch.from_numpy(np.empty(0, NUMPY_TYPES[haoda_type])).dtype
    return torch.empty(shape, dtype=dtype, device=like.device)

  # ---- device-resident entry points (torch CUDA tensors or raw pointers) ----
  @staticmethod
  def _pointers(items):
    values = [item.data_ptr() if hasattr(item, 'data_ptr') else int(item)
              for item in items]
    return (ctypes.c_void_p * len(values))(*values)

  def run_device(self, inputs, outputs, dims, iterate=0, stream=None):
    """Enqueue all iterations on device arrays (asynchronous)."""
    code = self._lib.soda_cuda_run_device(
        self._pointers(inputs), self._pointers(outputs),
        (ctypes.c_int32 * 4)(*dims), iterate, stream)
    if code:
      raise CudaError('soda_cuda_run_device(%s)' % self.app_name, code)

  def run_device_batch(self, inputs, outputs, dims, batch, iterate=0,
                       stream=None):
    """``run_device`` on ``batch`` grids of extents ``dims`` stored one after
    the other in each array (asynchronous)."""
    code = self._lib.soda_cuda_run_device_batch(
        self._pointers(inputs), self._pointers(outputs),
        (ctypes.c_int32 * 4)(*dims), batch, iterate, stream)
    if code:
      raise CudaError('soda_cuda_run_device_batch(%s)' % self.app_name, code)

  def ipc_export(self, address):
    """``(handle bytes, offset)`` of the device allocation holding
    ``address``, for another process to map (see soda_cuda_ipc_export)."""
    handle = ctypes.create_string_buffer(64)
    offset = ctypes.c_uint64()
    code = self._lib.soda_cuda_ipc_export(address, handle,
                                          ctypes.byref(offset))
    if code:
      raise CudaError('soda_cuda_ipc_export', code)
    return handle.raw, offset.value

  def ipc_open(self, handle):
    """Base address, in this process, of a neighbour's exported allocation."""
    base = ctypes.c_void_p()
    code = self._lib.soda_cuda_ipc_open(handle, ctypes.byref(base))
    if code:
      raise CudaError('soda_cuda_ipc_open', code)
    return base.value

  def copy_async(self, dst, src, nbytes, stream=None):
    code = self._lib.soda_cuda_copy_async(dst, src, nbytes, stream)
    if code:
      raise CudaError('soda_cuda_copy_async', code)

  def flag_write(self, address, value, stream=None):
    """Stream-ordered store of a 32-bit flag (see soda_cuda_flag_write)."""
    code = self._lib.soda_cuda_flag_write(address, value, stream)
    if code:
      raise CudaError('soda_cuda_flag_write', code)

  def flag_wait_geq(self, address, value, stream=None):
    """The stream waits until the 32-bit flag is >= ``value``."""
    code = self._lib.soda_cuda_flag_wait_geq(address, value, stream)
    if code:
      raise CudaError('soda_cuda_flag_wait_geq', code)

  def launch(self, depth, inputs, outputs, dims, row_begin, row_end,
             valid_lo, valid_hi, stream=None, chunk_rows=0):
    """Enqueue one kernel launch (see soda_cuda_launch[_chunked]).

    ``valid_lo`` / ``valid_hi``: one box per output (a list of per-dimension
    lists), or a single box that applies to every output."""
    pad = lambda xs, fill: (ctypes.c_int32 * 4)(
        *(list(xs) + [fill] * (4 - len(xs))))

    def boxes(box, fill):
      per_output = (list(box) if box and hasattr(box[0], '__len__')
                    else [box] * len(self.outputs))
      if len(per_output) != len(self.outputs):
        raise ValueError('one valid box per output')
      flat = []
      for one in per_output:
        flat += list(one) + [fill] * (4 - len(one))
      return (ctypes.c_int32 * len(flat))(*flat)
    code = self._lib.soda_cuda_launch_chunked(
        depth, self._pointers(inputs), self._pointers(outputs), pad(dims, 1),
        row_begin, row_end, boxes(valid_lo, 0), boxes(valid_hi, 1),
        chunk_rows or 0, stream)
    if code:
      raise CudaError('soda_cuda_launch(%s)' % self.app_name, code)

  def lead_rows(self, depth):
    """Rows a block streams besides the rows it owns (lead-in + drain)."""
    value = self._lib.soda_cuda_lead_rows(depth)
    if value < 0:
      raise CudaError('soda_cuda_lead_rows(%s)' % self.app_name, value)
    return value

  def chunk_rows(self, depth, dims, rows):
    """Rows per block a launch over ``rows`` streamed rows would use."""
    value = self._lib.soda_cuda_chunk_rows(
        depth, (ctypes.c_int32 * 4)(*(list(dims) + [1] * (4 - len(dims)))),
        rows)
    if value <= 0:
      raise CudaError('soda_cuda_chunk_rows(%s)' % self.app_name, value)
    return value


def bind_host_to_gpu(device_index):
  """Run this process on the CPUs of the NUMA node GPU ``device_index``
  hangs off, so that host buffers allocated from now on (first touch, pinned
  or not) sit on that node and host<->device copies do not cross the socket
  interconnect.  Matters with one process per GPU on a two-socket box, where
  an unbound process may land on the far socket.  Returns the node, or None
  when the topology is not exposed (virtualised PCI) — then nothing changes.
  """
  try:
    import pynvml
    pynvml.nvmlInit()
    visible = os.environ.get('CUDA_VISIBLE_DEVICES')
    index = device_index
    if visible:
      entry = visible.split(',')[device_index].strip()
      if entry.isdigit():
        index = int(entry)
    bus = pynvml.nvmlDeviceGetPciInfo(
        pynvml.nvmlDeviceGetHandleByIndex(index)).busId
    bus = bus.decode() if isinstance(bus, bytes) else bus
    bus = bus.lower()
    if len(bus.split(':')[0]) == 8:      # NVML pads the domain to 8 digits
      bus = bus[4:]
    with open('/sys/bus/pci/devices/%s/numa_node' % bus) as handle:
      node = int(handle.read())
    if node < 0:
      return None
    with open('/sys/devices/system/node/node%d/cpulist' % node) as handle:
      text = handle.read().strip()
    cpus = set()
    for part in text.split(','):
      first, _, last = part.partition('-')
      cpus.update(range(int(first), int(last or first) + 1))
    cpus &= os.sched_getaffinity(0)
    if not cpus:
      return None
    os.sched_setaffinity(0, cpus)
    return node
  except Exception:   # pylint: disable=broad-except
    return None


_loaded = {}


def load(path):
  path = os.path.abspath(path)
  if path not in _loaded:
    _loaded[path] = Library(path)
  return _loaded[path]


def compile_stencil(stencil, **kwargs):
  """Build (cached) and load the library of ``stencil``."""
  return load(build(stencil, **kwargs))


def run(stencil, arrays, params=None, devices=None, **kwargs):
  """Run ``stencil`` on ``arrays`` on the current CUDA device (or, for host
  arrays, sharded over ``devices``).

  ``arrays``: the inputs in program order, or a dict by input name (which may
  also hold the param arrays by name).  Returns the outputs in program order
  (a dict by name if ``arrays`` was a dict).
  """
  library = compile_stencil(stencil, **kwargs)
  if isinstance(arrays, dict):
    inputs = [arrays[name] for name, _ in library.inputs]
    if params is None and library.params:
      params = [arrays[name] for name, _, _ in library.params]
    outputs = library.run(inputs, params=params, devices=devices)
    return {name: out for (name, _), out in zip(library.outputs, outputs)}
  return library.run(list(arrays), params=params, devices=devices)


def run_batch(stencil, arrays, params=None, **kwargs):
  """Run ``stencil`` on a batch of independent grids on the current CUDA
  device: every array has a leading batch dimension (see
  ``Library.run_batch``).  ``arrays`` and the result take the forms of
  ``run``."""
  library = compile_stencil(stencil, **kwargs)
  if isinstance(arrays, dict):
    inputs = [arrays[name] for name, _ in library.inputs]
    if params is None and library.params:
      params = [arrays[name] for name, _, _ in library.params]
    outputs = library.run_batch(inputs, params=params)
    return {name: out for (name, _), out in zip(library.outputs, outputs)}
  return library.run_batch(list(arrays), params=params)
