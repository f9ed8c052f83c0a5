/* C ABI of a compiled SODA stencil program on B200 (one shared library per
 * .soda program, built by `sodac --cuda-kernel K.cu --cuda-host H.cu` + nvcc).
 *
 * The library exports two faces:
 *
 * 1. The reference's own entry point, unchanged, with C++ linkage exactly as
 *    the reference's generated header declares it
 *    (reference src/soda/codegen/xilinx/header.py:57-60, defined for the FPGA
 *    by host.print_entrance, src/soda/codegen/xilinx/host.py:931-945):
 *
 *        int <app>(buffer_t *var_<in0>_buffer, ..., buffer_t *var_<out0>_buffer,
 *                  ..., const char *xclbin);
 *
 *    so the reference's generated test harness `<app>_test`
 *    (host.py:984-1167) links against it unmodified.  `xclbin` is an opaque
 *    string for the FPGA flow; here NULL or "" are fine, and "devices=0,1"
 *    spreads a run on host buffers over several GPUs (see soda_cuda_run).
 *
 * 2. The `extern "C"` functions below, which are what a foreign-function
 *    binding (ctypes: soda/cuda.py; cgo/JNI stubs: INTEGRATION.md) loads.
 *    Symbol names are fixed; the program identity is queried at run time.
 *
 * All arrays are dense with dimension 0 fastest: stride[0] = 1,
 * stride[d] = extent[0] * ... * extent[d-1], as the reference harness sets
 * them up (host.py:1011-1020).  Return value 0 is success; negative values
 * follow the Halide numbering the reference host uses (host.py:118-133),
 * e.g. -3 = bad_elem_size, -12 = buffer_argument_is_null, -23 =
 * device_run_failed.  Nothing here falls back to the CPU: without a CUDA
 * device every compute entry returns -19 (no_device_interface).
 */
#ifndef SODA_CUDA_H_
#define SODA_CUDA_H_

#include <stdbool.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

/* Legacy Halide buffer_t, byte-for-byte the struct the reference emits
 * (header.py:32-49): sizeof 72; offsets dev 0, host 8, extent 16, stride 32,
 * min 48, elem_size 64.  `host` is caller-owned memory; `dev`, unused by the
 * reference host, may carry a CUDA device pointer (then host may be NULL and
 * no copies are made).  host == NULL && dev == 0 requests bounds-query mode
 * (host.py:204-252): extents/strides are filled in and nothing is computed. */
#ifndef BUFFER_T_DEFINED
#define BUFFER_T_DEFINED
typedef struct buffer_t {
  uint64_t dev;
  uint8_t* host;
  int32_t extent[4];
  int32_t stride[4];
  int32_t min[4];
  int32_t elem_size;
  bool host_dirty;
  bool dev_dirty;
  uint8_t _padding[10 - sizeof(void*)];
} buffer_t;
#endif /* BUFFER_T_DEFINED */

/* What the last soda_cuda_run / soda_cuda_run_device call did. */
typedef struct soda_cuda_stats_t {
  double kernel_ms;      /* device time of all launches (CUDA events) */
  double h2d_ms;         /* host->device copies, 0 for device buffers */
  double d2h_ms;
  int64_t cells;         /* prod(dims), times the items of a batch */
  int32_t iterate;
  int32_t launches;      /* kernels launched */
  int32_t depth;         /* iterations fused by the main launches */
  int32_t used_tma;      /* 1: TMA input path, 0: plain-load path */
  int32_t blocks;        /* thread blocks of the last launch (x * y * z, all
                            items of a batch) */
  int32_t threads;
  int32_t smem_bytes;
  int32_t reserved;
} soda_cuda_stats_t;

/* ---- program identity (what `sodac` compiled into this library) ---------- */
const char* soda_cuda_app_name(void);
int soda_cuda_dim(void);
int soda_cuda_iterate(void);        /* the program's `iterate` */
int soda_cuda_num_inputs(void);
int soda_cuda_num_outputs(void);
/* kind 0: input, 1: output.  Type is the haoda name, e.g. "float", "uint16". */
const char* soda_cuda_tensor_name(int kind, int index);
const char* soda_cuda_tensor_type(int kind, int index);
int soda_cuda_tensor_elem_size(int kind, int index);
/* Offsets of the inputs read by the cells of ANY output after `iterate`
 * iterations: lo[d] <= offset <= hi[d] (the union over the outputs: what a
 * caller needs to size halos and ghost planes). */
int soda_cuda_window(int iterate, int32_t lo[4], int32_t hi[4]);
/* The same box for output number `output` alone: that output is defined on
 * [-lo, dims - hi) — the loop bounds of the reference's golden loop for that
 * tensor (window from all inputs to it, reference
 * src/soda/codegen/xilinx/host.py:1082-1091, src/soda/core.py:793-835).
 * Outputs of one program may have different windows. */
int soda_cuda_window_of(int output, int iterate, int32_t lo[4], int32_t hi[4]);

/* ---- running ---------------------------------------------------------------
 * soda_cuda_run: the generic form of `<app>()` — n_in input and n_out output
 * buffer_t pointers in program order.  Synchronous: outputs are complete (in
 * `host`, or in `dev` for device buffers) on return.  Cells outside the
 * valid region are written as 0. */
int soda_cuda_run(buffer_t* const* inputs, buffer_t* const* outputs,
                  const char* config);

/* Several GPUs behind the same call.  `config` — the `xclbin` string of
 * `<app>()`, opaque to the FPGA flow (the call site is the single
 * `<app>(...)` of the reference harness, host.py:1068-1070) — may contain
 * "devices=0,1,2,3" (ordinals, repeats allowed) or "devices=all"; the
 * environment variable SODA_CUDA_DEVICES means the same when the string does
 * not say.  HOST buffers are then cut into one slab per listed device along
 * the streamed (last) dimension; every device loads its slab plus ghost rows
 * of the whole run's reach over its own PCIe link, runs all iterations
 * without talking to the others, and writes its own rows back: the result is
 * bit-identical to the one-device run.  (Device buffers live on one device;
 * for them the list is ignored.  Device-resident multi-GPU runs with a halo
 * exchange per launch are soda/cuda_slab.py.)
 * soda_cuda_shard_plan reports that cut for a grid of extents `dims` (no
 * device needed): slab r owns rows [own_begin[r], own_end[r]) and holds
 * [local_begin[r], local_end[r]); returns the number of slabs used (<=
 * n_slabs).  soda_cuda_slab_stats: how many slabs the last run had (0: not
 * sharded) and, for 0 <= index < that, what slab `index` did. */
int soda_cuda_shard_plan(const int32_t* dims, int n_slabs,
                         int32_t* local_begin, int32_t* local_end,
                         int32_t* own_begin, int32_t* own_end);
int soda_cuda_slab_stats(int index, soda_cuda_stats_t* out);

/* `param` statements (small constant arrays; reference grammar.py:38, passed
 * after the outputs by the reference entry, header.py:57-60).  A param is a
 * C array `T name[s0][s1]..` (first index slowest, reference
 * host.py:1004-1008) in host memory.  soda_cuda_run_params is soda_cuda_run
 * with the param buffers (extent[d] = size[d], elem_size checked);
 * soda_cuda_set_params uploads raw host arrays for callers of the
 * device-level entry points — the values stay in effect until set again.
 * Programs with params refuse to launch (-12) before they are set. */
int soda_cuda_num_params(void);
const char* soda_cuda_param_name(int index);
const char* soda_cuda_param_type(int index);
/* Fills size[0..rank) and returns the rank; < 0: no such param. */
int soda_cuda_param_size(int index, int32_t size[4]);
int soda_cuda_run_params(buffer_t* const* inputs, buffer_t* const* outputs,
                         buffer_t* const* params, const char* config);
int soda_cuda_set_params(const void* const* host_arrays);

/* Device-resident dense arrays, `iterate` iterations (0: the program's own),
 * enqueued on `stream` (a cudaStream_t; NULL = default stream), asynchronous.
 * Inputs are not modified. */
int soda_cuda_run_device(const void* const* inputs, void* const* outputs,
                         const int32_t* dims, int iterate, void* stream);

/* Batches: `batch` >= 1 independent grids ("items") of the same extents, each
 * computed exactly as one soda_cuda_run of that item alone would (valid
 * region and zero border; no item reads another's cells).  Every buffer_t /
 * pointer describes item 0; items follow at stride prod(extent) elements
 * (numpy/torch shape (batch, dims[n-1], .., dims[0])).  Param arrays are
 * shared by all items.
 * soda_cuda_run_batch: host (copied in and out) or dev (zero copy) buffers,
 * as soda_cuda_run; params: NULL for programs without params.  Synchronous.
 * There is no bounds-query mode (such buffers are refused with -12) and no
 * device list: SODA_CUDA_DEVICES is ignored and the batch runs on the
 * current device.
 * soda_cuda_run_device_batch: soda_cuda_run_device on `batch` items.
 * batch < 1 returns -4 (access_out_of_bounds). */
int soda_cuda_run_batch(buffer_t* const* inputs, buffer_t* const* outputs,
                        buffer_t* const* params, int batch);
int soda_cuda_run_device_batch(const void* const* inputs, void* const* outputs,
                               const int32_t* dims, int batch, int iterate,
                               void* stream);

/* One kernel launch: `depth` fused iterations (must be a compiled depth, see
 * soda_cuda_depths) producing streamed planes [row_begin, row_end) of the
 * outputs from the full input arrays.  `valid_lo` / `valid_hi` hold one box of
 * 4 ints per output (output k: valid_lo[4k .. 4k+3]); cells of output k
 * outside its box are stored as 0.  For slab-partitioned multi-GPU runs
 * (soda/cuda_slab.py). */
int soda_cuda_launch(int depth, const void* const* inputs,
                     void* const* outputs, const int32_t* dims, int row_begin,
                     int row_end, const int32_t* valid_lo,
                     const int32_t* valid_hi, void* stream);
/* The same launch with the rows per thread block along the streamed
 * dimension given (`chunk_rows` > 0) instead of chosen.  A caller that splits
 * a slab into several launches (faces first, see soda/cuda_slab.py) passes the
 * value soda_cuda_chunk_rows returns for the whole slab, so that the pieces
 * together are exactly the blocks of the one-launch decomposition: no row is
 * led into twice. */
int soda_cuda_launch_chunked(int depth, const void* const* inputs,
                             void* const* outputs, const int32_t* dims,
                             int row_begin, int row_end,
                             const int32_t* valid_lo, const int32_t* valid_hi,
                             int chunk_rows, void* stream);
/* Rows per block soda_cuda_launch picks for `rows` streamed rows of a grid of
 * extents `dims` (whole waves of resident blocks on this device); < 0: error. */
int soda_cuda_chunk_rows(int depth, const int32_t* dims, int rows);
/* Streamed rows a block of the depth-`depth` kernel runs through besides the
 * rows it owns (lead-in + drain): the price of one more launch over a row
 * range.  < 0: error. */
int soda_cuda_lead_rows(int depth);
/* Fills up to `max` compiled depths (decreasing); returns how many exist. */
int soda_cuda_depths(int32_t* depths, int max);

/* Stream-ordered 32-bit flags in device memory (cuStreamWriteValue32 /
 * cuStreamWaitValue32 with CU_STREAM_WAIT_VALUE_GEQ): executed by the GPU's
 * front end, no SM needed, so a neighbour's halo planes can be announced and
 * awaited while a launch occupies every SM.  `flag` is a 4-byte aligned
 * device address, local or peer-mapped (CUDA IPC).  Used by the multi-GPU
 * slab runner (soda/cuda_slab.py); no counterpart in the reference, which has
 * no multi-device support (SURVEY.md 8e). */
int soda_cuda_flag_write(void* flag, uint32_t value, void* stream);
int soda_cuda_flag_wait_geq(void* flag, uint32_t value, void* stream);

/* Peer mapping of another process's device arrays (one process per GPU).
 * soda_cuda_ipc_export: CUDA IPC handle (64 bytes) of the allocation that
 * holds `ptr`, and the offset of `ptr` in it.  soda_cuda_ipc_open: maps that
 * allocation into the CALLER's context on its own current device (peer access
 * over NVLink) and returns its base address there; this process never creates
 * a context on the neighbour's GPU, which would time-slice with the
 * neighbour's kernels.  soda_cuda_copy_async: copy-engine transfer between
 * any two device addresses, enqueued on `stream`. */
int soda_cuda_ipc_export(const void* ptr, unsigned char handle[64],
                         uint64_t* offset);
int soda_cuda_ipc_open(const unsigned char handle[64], void** base);
int soda_cuda_ipc_close(void* base);
int soda_cuda_copy_async(void* dst, const void* src, uint64_t bytes,
                         void* stream);

const soda_cuda_stats_t* soda_cuda_last_stats(void);
/* Releases cached device buffers and streams. */
void soda_cuda_release(void);

#ifdef __cplusplus
}
#endif

#endif /* SODA_CUDA_H_ */
