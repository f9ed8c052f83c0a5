// Host runtime behind the generated `<app>()` entry point and the C ABI in
// include/soda_cuda.h.  Hand-written; one copy is linked into every
// per-program library next to the generated kernel and host files.
//
// It replaces, for the GPU, what the reference's generated OpenCL host does
// between receiving `buffer_t`s and returning results
// (reference src/soda/codegen/xilinx/host.py:186-929 `<app>_wrapped`): argument
// checks and bounds-query mode (:204-252), device setup (:350-561), moving
// data to the device in the kernel's layout (:629-686 — here a plain dense
// copy, no tiling/burst/bank packing), launching and timing (:775-804), and
// copying the valid region back (:823-901).
#pragma once

#include <cuda.h>
#include <cuda_runtime.h>
#include <stdint.h>

#include "soda_cuda.h"

namespace soda {

constexpr int kRtMaxDim = 4;
constexpr int kRtMaxTensors = 8;

// One compiled streaming kernel: `depth` iterations fused (plan.Schedule).
struct KernelVariant {
  int depth;
  int threads;
  int vec;
  int tile[kRtMaxDim - 1];      // block tile in the non-streamed dims
  int own[kRtMaxDim - 1];       // cells of the tile this block stores
  int halo_lo[kRtMaxDim - 1];   // tile origin = tile index * own - halo_lo
  int lead;                     // steps before the first owned plane
  int out_delay;                // steps after the last owned plane
  int smem_bytes;
  int box0;                     // TMA box extent along dim 0
  int boxes_per_row;
  int box_rows;                 // TMA box extent along the streamed dim
  int tiles_per_block;          // 2-D register kernels: strips (warps) per block
  int uses_tma;                 // the first kernel below needs tensor maps
  int trip;                     // steps per trip of the streamed loop: a block
                                // runs a whole number of trips
  const void* kernel_tma;       // __global__ void(StreamArgs): TMA / aligned
                                // 128-bit input path
  const void* kernel_plain;     // same, any alignment
};

struct ProgramDesc {
  const char* app_name;
  int dim;
  int iterate;
  int n_in, n_out;
  const char* in_name[kRtMaxTensors];
  const char* out_name[kRtMaxTensors];
  const char* in_type[kRtMaxTensors];    // haoda type names
  const char* out_type[kRtMaxTensors];
  int in_elem[kRtMaxTensors];            // bytes per element
  int out_elem[kRtMaxTensors];
  // window[(n * 2 + side) * kRtMaxDim + d]: bounding box (side 0: min offset,
  // side 1: max offset) of the inputs read by outputs after n iterations,
  // n = 0..iterate.  Defines the valid region [-min, dims - max).
  const int* window;
  // out_window[((n * n_out + k) * 2 + side) * kRtMaxDim + d]: the same box for
  // output k alone.  Every output is defined on [-min, dims - max) of ITS OWN
  // window (the reference bounds each tensor's golden loop separately,
  // host.py:1082-1091); `window` above is the union and sizes halos.
  const int* out_window;
  // STENCIL_DIM_d of the reference host (host.py:1188-1189): window extents.
  int stencil_dim[kRtMaxDim];
  int n_variants;
  const KernelVariant* variants;         // sorted by decreasing depth
  // `param` statements: small constant arrays passed after the outputs
  // (reference header.py:57-60); C arrays `T name[s0][s1]..`, first index
  // slowest (host.py:1004-1008).
  int n_param;
  const char* param_name[kRtMaxTensors];
  const char* param_type[kRtMaxTensors];
  int param_elem[kRtMaxTensors];         // bytes per element
  int param_rank[kRtMaxTensors];
  int param_size[kRtMaxTensors][kRtMaxDim];
};

// Result codes: the Halide error numbering the reference host uses
// (host.py:118-133).
enum {
  kSuccess = 0,
  kGenericError = -1,
  kBadElemSize = -3,
  kAccessOutOfBounds = -4,
  kBufferExtentsTooLarge = -6,
  kOutOfMemory = -11,
  kBufferArgumentIsNull = -12,
  kCopyToHostFailed = -14,
  kCopyToDeviceFailed = -15,
  kDeviceMallocFailed = -16,
  kDeviceSyncFailed = -17,
  kNoDeviceInterface = -19,
  kInternalError = -22,
  kDeviceRunFailed = -23,
};

// `<app>(buffer_t*..., const char*)`: host or device buffers, bounds query.
// `config` (the reference's opaque `xclbin` argument) may hold
// "devices=0,1,..": host buffers are then cut into one slab per listed device
// along the streamed dimension (SODA_CUDA_DEVICES does the same from the
// environment; "all" = every visible device).
int run_buffers(const ProgramDesc& prog, buffer_t* const* inputs,
                buffer_t* const* outputs, const char* config,
                buffer_t* const* params = nullptr);

// Copies the program's param arrays (host memory, one pointer per param, in
// program order) to the device; every later launch of this library reads
// them.  `run_buffers` calls this when it is given params.
int set_params(const ProgramDesc& prog, const void* const* host_arrays);

// `batch` independent grids of extents `dims` in each buffer (item b starts
// b * prod(dims) elements in), host or device memory, params as in
// run_buffers: copied in, run, copied out.  No bounds query (-12) and no
// device list.
int run_batch(const ProgramDesc& prog, buffer_t* const* inputs,
              buffer_t* const* outputs, buffer_t* const* params, int batch);

// All `iterate` iterations on device-resident dense arrays of `batch` items
// (as in run_batch), asynchronously on `stream`.  Inputs are not modified.
int run_device(const ProgramDesc& prog, const void* const* inputs,
               void* const* outputs, const int32_t* dims, int iterate,
               cudaStream_t stream, int batch = 1);

// run_device on arrays of any layout check_layout accepts: kRtMaxDim + 1
// element strides per tensor (along dimensions 0 .. dim-1, entries beyond
// ignored, then the item stride, ignored when batch == 1).  NULL pointers give
// -12 and refused layouts -4 / -6, both before any device is looked up.
// Outputs must not overlap the inputs or each other (not checked).
int run_device_strided(const ProgramDesc& prog, const void* const* inputs,
                       const int64_t* in_strides, void* const* outputs,
                       const int64_t* out_strides, const int32_t* dims,
                       int batch, int iterate, cudaStream_t stream);

// The layouts the kernels address, where no two cells of a tensor share an
// address: stride[0] == 1, stride[d] >= stride[d-1] * dims[d-1], and for
// batch > 1 item stride >= stride[dim-1] * dims[dim-1].  Anything else
// (transposed, broadcast, negative, overlapping), batch < 1 and empty extents
// give -4; a tensor spanning 2^48 elements or more, or 2-D rows 2^31 or more
// elements apart, -6.  Needs no device.
int check_layout(const ProgramDesc& prog, const int32_t* dims, int batch,
                 const int64_t* in_strides, const int64_t* out_strides);

// One launch of the variant with `depth` fused iterations producing streamed
// planes [row_begin, row_end) of the outputs; cells of output k outside
// [valid_lo[4k..], valid_hi[4k..]) are stored as 0 (one box of kRtMaxDim ints
// per output).  Building block for slab-partitioned
// multi-GPU runs, where the caller owns ping-pong buffers and halo exchange.
int launch(const ProgramDesc& prog, int depth, const void* const* inputs,
           void* const* outputs, const int32_t* dims, int row_begin,
           int row_end, const int32_t* valid_lo, const int32_t* valid_hi,
           cudaStream_t stream, int forced_chunk_rows = 0);

// Rows per block along the streamed dimension that `launch` picks for a range
// of `rows` rows (whole waves of resident blocks); negative = error code.
int chunk_rows(const ProgramDesc& prog, int depth, const int32_t* dims,
               int rows);

// Streamed rows a block runs through before and after the rows it owns (its
// lead-in and drain): what every extra launch over a row range costs.
int lead_rows(const ProgramDesc& prog, int depth);

// Stream-ordered flag in device memory (local or peer-mapped): written and
// awaited by the GPU front end, not by a kernel.
int flag_write(void* flag, uint32_t value, cudaStream_t stream);
int flag_wait_geq(void* flag, uint32_t value, cudaStream_t stream);

// CUDA IPC: export the allocation holding `ptr`; map a neighbour's allocation
// into this process's context on its own device; copy-engine transfers.
int ipc_export(const void* ptr, unsigned char handle[64], uint64_t* offset);
int ipc_open(const unsigned char handle[64], void** base);
int ipc_close(void* base);
int copy_async(void* dst, const void* src, uint64_t bytes, cudaStream_t stream);

// How a run on host buffers over `n_slabs` devices cuts the streamed
// dimension: slab r owns rows [own_begin[r], own_end[r]) and holds rows
// [local_begin[r], local_end[r]) — its own plus ghost rows of the whole run's
// reach on the sides where the grid continues.  Returns the slab count
// actually used (thin grids use fewer).  Needs no device.
int shard_plan(const ProgramDesc& prog, const int32_t* dims, int n_slabs,
               int32_t* local_begin, int32_t* local_end, int32_t* own_begin,
               int32_t* own_end);

const soda_cuda_stats_t* last_stats();

// Slabs of the last sharded run (0 if it was not sharded); `out`, if given
// and `index` is in range, receives what that slab's device did.
int slab_stats(int index, soda_cuda_stats_t* out);

// Frees the cached device buffers.
void release_all();

}  // namespace soda
