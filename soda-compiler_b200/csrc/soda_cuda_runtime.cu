// Host runtime of the SODA CUDA backend: see soda_cuda_runtime.h.
#include "soda_cuda_runtime.h"

#include <algorithm>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <memory>
#include <mutex>
#include <string>
#include <thread>
#include <vector>

#include "soda_cuda_device.cuh"

namespace soda {
namespace {

#define SODA_CHECK(call, code)                                              \
  do {                                                                      \
    cudaError_t err_ = (call);                                              \
    if (err_ != cudaSuccess) {                                              \
      fprintf(stderr, "ERROR: %s failed: %s (%s:%d)\n", #call,              \
              cudaGetErrorString(err_), __FILE__, __LINE__);                \
      return (code);                                                        \
    }                                                                       \
  } while (0)

using EncodeTiledFn = CUresult (*)(
    CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
    const cuuint64_t*, const cuuint32_t*, const cuuint32_t*,
    CUtensorMapInterleave, CUtensorMapSwizzle, CUtensorMapL2promotion,
    CUtensorMapFloatOOBfill);

using StreamValueFn = CUresult (*)(CUstream, CUdeviceptr, cuuint32_t,
                                   unsigned int);
using AddressRangeFn = CUresult (*)(CUdeviceptr*, size_t*, CUdeviceptr);

// Driver entry points, process wide.
struct DriverApi {
  bool ready = false;
  EncodeTiledFn encode = nullptr;
  StreamValueFn write_value = nullptr;
  StreamValueFn wait_value = nullptr;
  AddressRangeFn address_range = nullptr;
};

struct PoolEntry {
  void* ptr;
  size_t bytes;
  bool busy;
};

// What a launch needs to know about a kernel on a device, found out once:
// the shared-memory attribute is set, the resident blocks per SM measured.
struct FnInfo {
  const void* fn;
  int per_sm;
};

// Rows per block chosen for (kernel, tile grid, items, rows): the search walks
// every chunk count, so its answer is kept.
struct ChunkEntry {
  const void* fn;
  long long grid_x;
  int batch;
  int rows;
  int chunk_rows;
};

// A tensor map depends on the address, the extents (the batch's included) and
// the box only.
struct MapEntry {
  const void* ptr;
  int elem, dim, batch;
  int32_t dims[kRtMaxDim];
  uint32_t box[kRtMaxDim];
  CUtensorMap map;
};

// Pinned bounce buffers for PAGEABLE caller memory.  cudaMemcpyAsync on
// pageable memory is staged by the driver on one thread (measured 5.8 GB/s
// each way on this pool's hosts against 50 GB/s from pinned memory, capture
// r2s) and pinning the caller's arrays for the call costs more than it saves
// (registering 2 x 1 GiB: 165-280 ms).  Instead the runtime copies through
// its own pinned slots with a few host threads: slot i + 1 is filled while
// slot i is on the wire.
struct Stager {
  static constexpr int kSlots = 3;
  size_t slot_bytes = 0;
  void* slot[kSlots] = {};
  cudaEvent_t done[kSlots] = {};
  bool busy[kSlots] = {};        // `done` has been recorded for this slot
  void* out_dst[kSlots] = {};    // copy-out pending: caller memory, bytes
  size_t out_bytes[kSlots] = {};
  int next = 0;
};

// One execution lane: a device with the streams, events, buffer pool and
// caches of one stream of calls.  Lane (d, 0) serves callers whose current
// device is d; a sharded run over devices "0,1,1" also uses lane (1, 1).
struct Lane {
  int ordinal = 0;
  int replica = 0;
  bool ready = false;
  int sm_count = 0;
  std::mutex run_mutex;    // one run at a time per lane
  std::mutex mutex;        // pool and caches
  std::vector<PoolEntry> pool;
  cudaStream_t streams[3] = {};   // h2d, compute, d2h
  bool streams_ready = false;
  cudaEvent_t ev[6] = {};  // kernel start/stop, h2d start/stop, d2h start/stop
  std::vector<cudaEvent_t> idle_events;   // recycled ordering events
  void* param_dev[kRtMaxTensors] = {};
  unsigned long long params_version = 0;
  soda_cuda_stats_t stats = {};
  bool stats_pending = false;
  std::vector<FnInfo> fns;
  std::vector<ChunkEntry> chunks;
  std::vector<MapEntry> maps;
  Stager stage_in, stage_out;
};

std::mutex g_mutex;            // lanes, params, last-run bookkeeping
DriverApi g_api;
std::vector<std::unique_ptr<Lane>> g_lanes;
thread_local Lane* t_lane = nullptr;   // set while a thread runs a slab
Lane* g_last_lane = nullptr;           // whose stats `last_stats` reports
soda_cuda_stats_t g_stats = {};        // aggregate of the last sharded run
bool g_stats_aggregate = false;
std::vector<soda_cuda_stats_t> g_lane_stats;   // per slab of the last run
// host copy of the param arrays: lanes upload it when theirs is older
std::vector<std::vector<unsigned char>> g_params_host;
unsigned long long g_params_version = 0;

bool env_flag(const char* name) {
  const char* v = getenv(name);
  return v != nullptr && v[0] != '\0' && v[0] != '0';
}

bool verbose() {
  static const bool on = env_flag("SODA_CUDA_VERBOSE");
  return on;
}

int ensure_api() {
  if (g_api.ready) return kSuccess;
  std::lock_guard<std::mutex> lock(g_mutex);
  if (g_api.ready) return kSuccess;
  int count = 0;
  if (cudaGetDeviceCount(&count) != cudaSuccess || count == 0) {
    cudaGetLastError();
    fprintf(stderr, "ERROR: no CUDA device; the SODA CUDA backend has no CPU "
                    "fallback\n");
    return kNoDeviceInterface;
  }
  void* fn = nullptr;
  cudaDriverEntryPointQueryResult qres;
  SODA_CHECK(cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn,
                                     cudaEnableDefault, &qres),
             kNoDeviceInterface);
  g_api.encode = reinterpret_cast<EncodeTiledFn>(fn);
  SODA_CHECK(cudaGetDriverEntryPoint("cuStreamWriteValue32", &fn,
                                     cudaEnableDefault, &qres),
             kNoDeviceInterface);
  g_api.write_value = reinterpret_cast<StreamValueFn>(fn);
  SODA_CHECK(cudaGetDriverEntryPoint("cuStreamWaitValue32", &fn,
                                     cudaEnableDefault, &qres),
             kNoDeviceInterface);
  g_api.wait_value = reinterpret_cast<StreamValueFn>(fn);
  SODA_CHECK(cudaGetDriverEntryPoint("cuMemGetAddressRange", &fn,
                                     cudaEnableDefault, &qres),
             kNoDeviceInterface);
  g_api.address_range = reinterpret_cast<AddressRangeFn>(fn);
  g_api.ready = true;
  return kSuccess;
}

// The lane (ordinal, replica), created on first use.  The caller's current
// device must be `ordinal`.
int lane_for(int ordinal, int replica, Lane** out) {
  int rc = ensure_api();
  if (rc != kSuccess) return rc;
  Lane* lane = nullptr;
  {
    std::lock_guard<std::mutex> lock(g_mutex);
    for (auto& l : g_lanes)
      if (l->ordinal == ordinal && l->replica == replica) lane = l.get();
    if (lane == nullptr) {
      g_lanes.emplace_back(new Lane);
      lane = g_lanes.back().get();
      lane->ordinal = ordinal;
      lane->replica = replica;
    }
  }
  std::lock_guard<std::mutex> lock(lane->mutex);
  if (!lane->ready) {
    SODA_CHECK(cudaDeviceGetAttribute(&lane->sm_count,
                                      cudaDevAttrMultiProcessorCount, ordinal),
               kNoDeviceInterface);
    for (auto& ev : lane->ev)
      SODA_CHECK(cudaEventCreate(&ev), kNoDeviceInterface);
    lane->ready = true;
  }
  *out = lane;
  return kSuccess;
}

// The lane of the calling thread: the slab it is running, else lane 0 of its
// current device.
int current_lane(Lane** out) {
  if (t_lane != nullptr) {
    *out = t_lane;
    return kSuccess;
  }
  int rc = ensure_api();
  if (rc != kSuccess) return rc;
  int dev = 0;
  SODA_CHECK(cudaGetDevice(&dev), kNoDeviceInterface);
  return lane_for(dev, 0, out);
}

int ensure_streams(Lane* lane) {
  std::lock_guard<std::mutex> lock(lane->mutex);
  if (lane->streams_ready) return kSuccess;
  for (auto& st : lane->streams)
    SODA_CHECK(cudaStreamCreateWithFlags(&st, cudaStreamNonBlocking),
               kDeviceRunFailed);
  lane->streams_ready = true;
  return kSuccess;
}

void* pool_acquire(Lane* lane, size_t bytes) {
  std::lock_guard<std::mutex> lock(lane->mutex);
  PoolEntry* best = nullptr;
  for (auto& e : lane->pool)
    if (!e.busy && e.bytes >= bytes && e.bytes <= 2 * bytes + 4096 &&
        (best == nullptr || e.bytes < best->bytes))
      best = &e;
  if (best != nullptr) {
    best->busy = true;
    return best->ptr;
  }
  void* ptr = nullptr;
  if (cudaMalloc(&ptr, bytes) != cudaSuccess) {
    cudaGetLastError();
    // drop idle buffers and retry once
    for (auto& e : lane->pool)
      if (!e.busy && e.ptr != nullptr) {
        cudaFree(e.ptr);
        e.ptr = nullptr;
        e.bytes = 0;
      }
    if (cudaMalloc(&ptr, bytes) != cudaSuccess) {
      cudaGetLastError();
      return nullptr;
    }
  }
  lane->pool.push_back({ptr, bytes, true});
  return ptr;
}

void pool_release(Lane* lane, void* ptr) {
  std::lock_guard<std::mutex> lock(lane->mutex);
  for (auto& e : lane->pool)
    if (e.ptr == ptr) e.busy = false;
}

// Hands buffers back to the pool when it goes out of scope.  When a run fails
// half way, copies and kernels may still be using them: unless the run says
// it completed (it synchronised its streams), the device is drained first.
struct PoolLease {
  Lane* lane;
  std::vector<void*> held;
  bool completed = false;
  explicit PoolLease(Lane* l) : lane(l) {}
  void* get(size_t bytes) {
    void* p = pool_acquire(lane, bytes);
    if (p != nullptr) held.push_back(p);
    return p;
  }
  ~PoolLease() {
    if (!completed && !held.empty()) {
      cudaDeviceSynchronize();
      cudaGetLastError();
    }
    for (void* p : held) pool_release(lane, p);
  }
};

// Ordering events of one run, recycled through the lane; returned on every
// exit path.
struct EventLease {
  Lane* lane;
  std::vector<cudaEvent_t> held;
  explicit EventLease(Lane* l) : lane(l) {}
  cudaEvent_t get() {
    cudaEvent_t ev = nullptr;
    {
      std::lock_guard<std::mutex> lock(lane->mutex);
      if (!lane->idle_events.empty()) {
        ev = lane->idle_events.back();
        lane->idle_events.pop_back();
      }
    }
    if (ev == nullptr &&
        cudaEventCreateWithFlags(&ev, cudaEventDisableTiming) != cudaSuccess) {
      cudaGetLastError();
      return nullptr;
    }
    held.push_back(ev);
    return ev;
  }
  ~EventLease() {
    std::lock_guard<std::mutex> lock(lane->mutex);
    for (cudaEvent_t ev : held) lane->idle_events.push_back(ev);
  }
};

// ---- pageable caller memory ---------------------------------------------------

bool staging_enabled() {
  const char* v = getenv("SODA_CUDA_STAGING");
  return v == nullptr || v[0] != '0';
}

// Is `ptr` ordinary (not pinned, not registered, not managed) host memory?
bool is_pageable(const void* ptr) {
  cudaPointerAttributes attr;
  if (cudaPointerGetAttributes(&attr, ptr) != cudaSuccess) {
    cudaGetLastError();
    return true;
  }
  return attr.type == cudaMemoryTypeUnregistered;
}

// memcpy by a few threads (SODA_CUDA_COPY_THREADS, default half the cores, at
// most 8): one thread does not saturate the host's memory system.
void parallel_memcpy(void* dst, const void* src, size_t bytes) {
  static const int wanted = [] {
    if (const char* v = getenv("SODA_CUDA_COPY_THREADS")) return atoi(v);
    const unsigned cores = std::thread::hardware_concurrency();
    return static_cast<int>(std::min(8u, std::max(1u, cores / 2)));
  }();
  const int parts = static_cast<int>(std::max<size_t>(
      1, std::min<size_t>(std::max(1, wanted), bytes >> 20)));
  if (parts == 1) {
    memcpy(dst, src, bytes);
    return;
  }
  const size_t each = ((bytes + parts - 1) / parts + 4095) & ~size_t(4095);
  std::vector<std::thread> helpers;
  for (int t = 1; t < parts; ++t) {
    const size_t begin = std::min(bytes, each * t);
    const size_t end = std::min(bytes, begin + each);
    if (end > begin)
      helpers.emplace_back([=] {
        memcpy(static_cast<char*>(dst) + begin,
               static_cast<const char*>(src) + begin, end - begin);
      });
  }
  memcpy(dst, src, std::min(bytes, each));
  for (auto& h : helpers) h.join();
}

int ensure_stager(Stager* st) {
  size_t want = size_t(32) << 20;
  if (const char* v = getenv("SODA_CUDA_STAGE_KB"))
    want = std::max<size_t>(4096, static_cast<size_t>(atol(v)) << 10);
  if (st->slot_bytes == want) return kSuccess;
  for (int k = 0; k < Stager::kSlots; ++k) {
    if (st->slot[k] != nullptr) {
      if (st->busy[k]) cudaEventSynchronize(st->done[k]);
      cudaFreeHost(st->slot[k]);
      st->slot[k] = nullptr;
    }
    st->busy[k] = false;
    st->out_bytes[k] = 0;
    if (st->done[k] == nullptr)
      SODA_CHECK(cudaEventCreateWithFlags(&st->done[k], cudaEventDisableTiming),
                 kDeviceRunFailed);
    SODA_CHECK(cudaHostAlloc(&st->slot[k], want, cudaHostAllocDefault),
               kOutOfMemory);
  }
  st->slot_bytes = want;
  st->next = 0;
  return kSuccess;
}

// A slot whose bytes have reached the device (copy-in) or the caller
// (copy-out) and may be refilled.
int drain_slot(Stager* st, int k) {
  if (st->busy[k]) {
    SODA_CHECK(cudaEventSynchronize(st->done[k]), kDeviceSyncFailed);
    st->busy[k] = false;
  }
  if (st->out_bytes[k] != 0) {
    parallel_memcpy(st->out_dst[k], st->slot[k], st->out_bytes[k]);
    st->out_bytes[k] = 0;
  }
  return kSuccess;
}

// Host -> device on `stream`; pageable sources go through the bounce slots.
int copy_in(Lane* lane, void* dst, const void* src, size_t bytes, bool staged,
            cudaStream_t stream) {
  if (!staged) {
    SODA_CHECK(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyHostToDevice, stream),
               kCopyToDeviceFailed);
    return kSuccess;
  }
  Stager* st = &lane->stage_in;
  int rc = ensure_stager(st);
  if (rc != kSuccess) return rc;
  for (size_t off = 0; off < bytes; off += st->slot_bytes) {
    const int k = st->next;
    st->next = (k + 1) % Stager::kSlots;
    rc = drain_slot(st, k);
    if (rc != kSuccess) return rc;
    const size_t n = std::min(st->slot_bytes, bytes - off);
    parallel_memcpy(st->slot[k], static_cast<const char*>(src) + off, n);
    SODA_CHECK(cudaMemcpyAsync(static_cast<char*>(dst) + off, st->slot[k], n,
                               cudaMemcpyHostToDevice, stream),
               kCopyToDeviceFailed);
    SODA_CHECK(cudaEventRecord(st->done[k], stream), kCopyToDeviceFailed);
    st->busy[k] = true;
  }
  return kSuccess;
}

// Device -> host on `stream`; pageable destinations receive their bytes when
// the slot is drained (at its next use, or by finish_copies).
int copy_out(Lane* lane, void* dst, const void* src, size_t bytes, bool staged,
             cudaStream_t stream) {
  if (!staged) {
    SODA_CHECK(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDeviceToHost, stream),
               kCopyToHostFailed);
    return kSuccess;
  }
  Stager* st = &lane->stage_out;
  int rc = ensure_stager(st);
  if (rc != kSuccess) return rc;
  for (size_t off = 0; off < bytes; off += st->slot_bytes) {
    const int k = st->next;
    st->next = (k + 1) % Stager::kSlots;
    rc = drain_slot(st, k);
    if (rc != kSuccess) return rc;
    const size_t n = std::min(st->slot_bytes, bytes - off);
    SODA_CHECK(cudaMemcpyAsync(st->slot[k], static_cast<const char*>(src) + off,
                               n, cudaMemcpyDeviceToHost, stream),
               kCopyToHostFailed);
    SODA_CHECK(cudaEventRecord(st->done[k], stream), kCopyToHostFailed);
    st->busy[k] = true;
    st->out_dst[k] = static_cast<char*>(dst) + off;
    st->out_bytes[k] = n;
  }
  return kSuccess;
}

// Everything still in a copy-out slot reaches the caller's memory, oldest
// first.
int finish_copies(Lane* lane) {
  Stager* st = &lane->stage_out;
  for (int step = 0; step < Stager::kSlots; ++step) {
    const int rc = drain_slot(st, (st->next + step) % Stager::kSlots);
    if (rc != kSuccess) return rc;
  }
  return kSuccess;
}

const KernelVariant* find_variant(const ProgramDesc& prog, int depth) {
  for (int i = 0; i < prog.n_variants; ++i)
    if (prog.variants[i].depth == depth) return &prog.variants[i];
  return nullptr;
}

CUtensorMapDataType tma_type(int elem) {
  switch (elem) {
    case 1: return CU_TENSOR_MAP_DATA_TYPE_UINT8;
    case 2: return CU_TENSOR_MAP_DATA_TYPE_UINT16;
    case 4: return CU_TENSOR_MAP_DATA_TYPE_UINT32;
    default: return CU_TENSOR_MAP_DATA_TYPE_UINT64;
  }
}

// One box of kRtMaxDim ints per output.
struct Boxes {
  int32_t lo[kRtMaxTensors * kRtMaxDim];
  int32_t hi[kRtMaxTensors * kRtMaxDim];
};

// Where each output is defined after `iterate` iterations: the bounds of the
// reference's golden loop for that tensor (host.py:1082-1091).
void valid_region(const ProgramDesc& prog, int iterate, const int32_t* dims,
                  Boxes* boxes) {
  for (int k = 0; k < kRtMaxTensors; ++k) {
    int32_t* lo = boxes->lo + k * kRtMaxDim;
    int32_t* hi = boxes->hi + k * kRtMaxDim;
    for (int d = 0; d < kRtMaxDim; ++d) {
      lo[d] = 0;
      hi[d] = 1;
    }
    if (k >= prog.n_out) continue;
    const int* w =
        prog.out_window + (iterate * prog.n_out + k) * 2 * kRtMaxDim;
    for (int d = 0; d < prog.dim; ++d) {
      lo[d] = std::max(0, -w[d]);
      hi[d] = dims[d] - std::max(0, w[kRtMaxDim + d]);
    }
  }
}

// Intermediate launches store every cell they own.
void full_region(const ProgramDesc& prog, const int32_t* dims, Boxes* boxes) {
  for (int k = 0; k < kRtMaxTensors; ++k)
    for (int d = 0; d < kRtMaxDim; ++d) {
      boxes->lo[k * kRtMaxDim + d] = 0;
      boxes->hi[k * kRtMaxDim + d] = d < prog.dim ? dims[d] : 1;
    }
}

// Blocks along the streamed dimension: minimise (waves x steps per block).
int pick_chunks(long long tile_blocks, long long resident, int rows,
                int overhead) {
  const int max_chunks = std::max(1, std::min(rows, 65535));
  long long best_cost = -1;
  int best = 1;
  for (int chunks = 1; chunks <= max_chunks; ++chunks) {
    const int chunk_rows = (rows + chunks - 1) / chunks;
    const int real_chunks = (rows + chunk_rows - 1) / chunk_rows;
    if (real_chunks != chunks) continue;
    const long long waves = (tile_blocks * chunks + resident - 1) / resident;
    // (a block runs whole trips of its streamed loop, up to trip - 1 surplus
    // steps; counting them here picks coarser chunks, which measured 2-7 %
    // slower on blur, sobel2d and denoise2d: the finer grid balances the tail)
    const long long cost = waves * (chunk_rows + overhead);
    if (best_cost < 0 || cost < best_cost) {
      best_cost = cost;
      best = chunks;
    }
    if (chunk_rows <= overhead) break;   // finer only adds lead-in work
  }
  return best;
}

// The launches of a run: greedily the deepest compiled variant that still
// fits the remaining iterations (SODA_CUDA_DEPTH caps the depth).
int plan_depths(const ProgramDesc& prog, int iterate, std::vector<int>* depths) {
  int forced = 0;
  if (const char* v = getenv("SODA_CUDA_DEPTH")) forced = atoi(v);
  for (int left = iterate; left > 0;) {
    int pick = 0;
    for (int i = 0; i < prog.n_variants; ++i) {
      const int d = prog.variants[i].depth;
      if (d <= left && (forced <= 0 || d <= forced) && d > pick) pick = d;
    }
    if (pick == 0) {
      fprintf(stderr, "ERROR: no compiled depth fits %d remaining iterations\n",
              left);
      return kInternalError;
    }
    depths->push_back(pick);
    left -= pick;
  }
  if (depths->size() > 1 && prog.n_in != prog.n_out) return kInternalError;
  return kSuccess;
}

// Resident blocks per SM of `fn` on this lane's device (and, once, the
// kernel's dynamic shared memory limit).
int fn_info(Lane* lane, const ProgramDesc& prog, const KernelVariant* kv,
            const void* fn, int* per_sm_out) {
  {
    std::lock_guard<std::mutex> lock(lane->mutex);
    for (const FnInfo& info : lane->fns)
      if (info.fn == fn) {
        *per_sm_out = info.per_sm;
        return kSuccess;
      }
  }
  SODA_CHECK(cudaFuncSetAttribute(fn,
                                  cudaFuncAttributeMaxDynamicSharedMemorySize,
                                  kv->smem_bytes),
             kDeviceRunFailed);
  int per_sm = 0;
  SODA_CHECK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(
                 &per_sm, fn, kv->threads, kv->smem_bytes),
             kDeviceRunFailed);
  if (per_sm < 1) {
    fprintf(stderr, "ERROR: kernel of %s does not fit on an SM (%d B smem)\n",
            prog.app_name, kv->smem_bytes);
    return kDeviceRunFailed;
  }
  std::lock_guard<std::mutex> lock(lane->mutex);
  lane->fns.push_back({fn, per_sm});
  *per_sm_out = per_sm;
  return kSuccess;
}

// Rows per block along the streamed dimension for a launch over `rows` rows
// of `batch` items (blockIdx.z).
int choose_chunk_rows(Lane* lane, const ProgramDesc& prog,
                      const KernelVariant* kv, const void* fn,
                      const int32_t* dims, int rows, int batch,
                      long long* grid_x_out, int* per_sm_out) {
  int per_sm = 0;
  const int rc = fn_info(lane, prog, kv, fn, &per_sm);
  if (rc != kSuccess) return rc;
  long long tile_blocks = 1;
  for (int d = 0; d + 1 < prog.dim; ++d)
    tile_blocks *= (dims[d] + kv->own[d] - 1) / kv->own[d];
  // 2-D register kernels pack `tiles_per_block` independent strips in a block
  const int per_block = std::max(1, kv->tiles_per_block);
  const long long grid_x = (tile_blocks + per_block - 1) / per_block;
  if (grid_x_out != nullptr) *grid_x_out = grid_x;
  if (per_sm_out != nullptr) *per_sm_out = per_sm;
  if (const char* forced = getenv("SODA_CUDA_CHUNKS")) {
    const int chunks = std::max(1, std::min(rows, atoi(forced)));
    return (rows + chunks - 1) / chunks;
  }
  {
    std::lock_guard<std::mutex> lock(lane->mutex);
    for (const ChunkEntry& e : lane->chunks)
      if (e.fn == fn && e.grid_x == grid_x && e.batch == batch &&
          e.rows == rows)
        return e.chunk_rows;
  }
  const long long resident = static_cast<long long>(per_sm) * lane->sm_count;
  const int chunks = pick_chunks(grid_x * batch, resident, rows,
                                 kv->lead + kv->out_delay);
  const int chunk_rows = (rows + chunks - 1) / chunks;
  std::lock_guard<std::mutex> lock(lane->mutex);
  if (lane->chunks.size() >= 256) lane->chunks.clear();
  lane->chunks.push_back({fn, grid_x, batch, rows, chunk_rows});
  return chunk_rows;
}

// The tensor map of input `ptr`, encoded once per (address, shape, box): rank
// dim + 1, the outermost dimension counting the `batch` items of the input.
bool tensor_map(Lane* lane, const void* ptr, int elem, int dim, int batch,
                const int32_t* dims, const long long* stride,
                const uint32_t* box, CUtensorMap* out) {
  {
    std::lock_guard<std::mutex> lock(lane->mutex);
    for (const MapEntry& e : lane->maps)
      if (e.ptr == ptr && e.elem == elem && e.dim == dim &&
          e.batch == batch && memcmp(e.dims, dims, sizeof(e.dims)) == 0 &&
          memcmp(e.box, box, sizeof(e.box)) == 0) {
        *out = e.map;
        return true;
      }
  }
  cuuint64_t gdim[kRtMaxDim + 1];
  cuuint64_t gstride[kRtMaxDim];
  cuuint32_t estr[kRtMaxDim + 1];
  cuuint32_t cbox[kRtMaxDim + 1];
  long long item_stride = 1;
  for (int d = 0; d < dim; ++d) {
    gdim[d] = static_cast<cuuint64_t>(dims[d]);
    estr[d] = 1;
    cbox[d] = box[d];
    if (d > 0) gstride[d - 1] = static_cast<cuuint64_t>(stride[d]) * elem;
    item_stride *= dims[d];
  }
  gdim[dim] = static_cast<cuuint64_t>(batch);
  estr[dim] = 1;
  cbox[dim] = 1;
  gstride[dim - 1] = static_cast<cuuint64_t>(item_stride) * elem;
  MapEntry entry;
  memset(&entry, 0, sizeof(entry));
  const CUresult res = g_api.encode(
      &entry.map, tma_type(elem), dim + 1, const_cast<void*>(ptr), gdim,
      gstride, cbox, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
      CU_TENSOR_MAP_SWIZZLE_NONE,
      CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (res != CUDA_SUCCESS) {
    if (verbose())
      fprintf(stderr, "INFO: tensor map rejected (%d); plain loads\n",
              static_cast<int>(res));
    return false;
  }
  entry.ptr = ptr;
  entry.elem = elem;
  entry.dim = dim;
  entry.batch = batch;
  memcpy(entry.dims, dims, sizeof(entry.dims));
  memcpy(entry.box, box, sizeof(entry.box));
  *out = entry.map;
  std::lock_guard<std::mutex> lock(lane->mutex);
  if (lane->maps.size() >= 64) lane->maps.erase(lane->maps.begin());
  lane->maps.push_back(entry);
  return true;
}

// Brings the lane's device copies of the param arrays up to date.
int sync_params(Lane* lane, const ProgramDesc& prog) {
  if (prog.n_param == 0) return kSuccess;
  std::lock_guard<std::mutex> lock(g_mutex);
  if (g_params_version == 0) {
    fprintf(stderr, "ERROR: params of %s have not been set "
                    "(soda_cuda_set_params)\n", prog.app_name);
    return kBufferArgumentIsNull;
  }
  if (lane->params_version == g_params_version) return kSuccess;
  // earlier launches may still be reading the previous values
  SODA_CHECK(cudaDeviceSynchronize(), kDeviceSyncFailed);
  for (int k = 0; k < prog.n_param; ++k) {
    const size_t bytes = g_params_host[k].size();
    if (lane->param_dev[k] == nullptr)
      SODA_CHECK(cudaMalloc(&lane->param_dev[k], std::max<size_t>(bytes, 16)),
                 kDeviceMallocFailed);
    SODA_CHECK(cudaMemcpy(lane->param_dev[k], g_params_host[k].data(), bytes,
                          cudaMemcpyHostToDevice),
               kCopyToDeviceFailed);
  }
  lane->params_version = g_params_version;
  return kSuccess;
}

// Launches of the variant with `depth` fused iterations over `batch` items
// of extents `dims` stored one after the other: one launch per kMaxItems
// items (gridDim.z), all with the same tile and chunk grid.
constexpr int kMaxItems = 65535;

int launch_on(Lane* lane, const ProgramDesc& prog, int depth,
              const void* const* inputs, void* const* outputs,
              const int32_t* dims, int batch, int row_begin, int row_end,
              const int32_t* valid_lo, const int32_t* valid_hi,
              cudaStream_t stream, int forced_chunk_rows) {
  const KernelVariant* kv = find_variant(prog, depth);
  if (kv == nullptr) {
    fprintf(stderr, "ERROR: %s was not compiled with temporal depth %d\n",
            prog.app_name, depth);
    return kInternalError;
  }
  const int s = prog.dim - 1;
  if (row_end <= row_begin) return kSuccess;

  StreamArgs args;
  memset(&args, 0, sizeof(args));
  long long stride = 1, cells = 1;
  int32_t dims4[kRtMaxDim];
  for (int d = 0; d < kRtMaxDim; ++d) {
    dims4[d] = args.dims[d] = d < prog.dim ? dims[d] : 1;
    args.stride[d] = stride;
    stride *= args.dims[d];
    args.tiles[d] = 1;
  }
  for (int k = 0; k < prog.n_out; ++k)
    for (int d = 0; d < kRtMaxDim; ++d) {
      args.valid_lo[k][d] = d < prog.dim ? valid_lo[k * kRtMaxDim + d] : 0;
      args.valid_hi[k][d] = d < prog.dim ? valid_hi[k * kRtMaxDim + d] : 1;
    }
  cells = stride;
  if (batch < 1) return kAccessOutOfBounds;
  if (cells * batch >= (1LL << 40)) return kBufferExtentsTooLarge;
  long long tile_blocks = 1;
  for (int d = 0; d < s; ++d) {
    args.tiles[d] = (dims[d] + kv->own[d] - 1) / kv->own[d];
    tile_blocks *= args.tiles[d];
  }
  if (tile_blocks * batch > 0x7fffffffLL) return kBufferExtentsTooLarge;
  args.row_begin = row_begin;
  args.row_end = row_end;
  args.item_stride = cells;

  bool aligned = (dims[0] % kv->vec) == 0;
  bool tma_ok = !env_flag("SODA_CUDA_NO_TMA");   // (tests flip it per call)
  for (int k = 0; k < prog.n_in; ++k) {
    args.in_ptr[k] = inputs[k];
    const uintptr_t p = reinterpret_cast<uintptr_t>(inputs[k]);
    if (p % 16 != 0) aligned = tma_ok = false;
    if ((static_cast<long long>(dims[0]) * prog.in_elem[k]) % 16 != 0)
      tma_ok = false;
  }
  for (int k = 0; k < prog.n_out; ++k) {
    args.out_ptr[k] = outputs[k];
    if (reinterpret_cast<uintptr_t>(outputs[k]) % 16 != 0) aligned = false;
  }
  args.vec_store = aligned ? 1 : 0;
  if (prog.n_param > 0) {
    const int rc = sync_params(lane, prog);
    if (rc != kSuccess) return rc;
    for (int k = 0; k < prog.n_param; ++k)
      args.param_ptr[k] = lane->param_dev[k];
  }

  if (tma_ok && kv->uses_tma) {
    uint32_t box[kRtMaxDim] = {1, 1, 1, 1};
    for (int d = 0; d < prog.dim; ++d)
      box[d] = d == 0 ? kv->box0 : (d < s ? kv->tile[d] : kv->box_rows);
    for (int k = 0; k < prog.n_in && tma_ok; ++k)
      tma_ok = tensor_map(lane, inputs[k], prog.in_elem[k], prog.dim, batch,
                          dims4, args.stride, box, &args.in_map[k]);
  }
  const void* fn = tma_ok ? kv->kernel_tma : kv->kernel_plain;
  const int rows = row_end - row_begin;
  long long grid_x = 0;
  int per_sm = 0;
  const int items = std::min(batch, kMaxItems);   // per launch
  const int chosen = choose_chunk_rows(lane, prog, kv, fn, dims, rows, items,
                                       &grid_x, &per_sm);
  if (chosen < 0) return chosen;
  args.chunk_rows = forced_chunk_rows > 0 ? std::min(forced_chunk_rows, rows)
                                          : chosen;
  const int chunks = (rows + args.chunk_rows - 1) / args.chunk_rows;
  if (chunks > 65535) return kBufferExtentsTooLarge;

  dim3 block(kv->threads);
  void* params[] = {&args};
  for (int begin = 0; begin < batch; begin += kMaxItems) {
    args.item_begin = begin;
    dim3 grid(static_cast<unsigned>(grid_x), static_cast<unsigned>(chunks),
              static_cast<unsigned>(std::min(kMaxItems, batch - begin)));
    SODA_CHECK(
        cudaLaunchKernel(fn, grid, block, params, kv->smem_bytes, stream),
        kDeviceRunFailed);
    lane->stats.launches += 1;
  }
  lane->stats.used_tma = tma_ok ? 1 : 0;
  lane->stats.blocks = static_cast<int32_t>(
      std::min<long long>(grid_x * chunks * batch, 0x7fffffffLL));
  lane->stats.threads = kv->threads;
  lane->stats.smem_bytes = kv->smem_bytes;
  if (verbose())
    fprintf(stderr,
            "INFO: %s depth %d on device %d: grid %lld x %d x %d items (%d "
            "blocks/SM resident), %d threads, %d B smem, %s, rows [%d, %d) in "
            "chunks of %d\n",
            prog.app_name, depth, lane->ordinal, grid_x, chunks, batch, per_sm,
            kv->threads, kv->smem_bytes,
            !tma_ok ? "plain loads" : kv->uses_tma ? "TMA" : "128-bit loads",
            row_begin, row_end, args.chunk_rows);
  return kSuccess;
}

void begin_stats(Lane* lane, long long cells, int iterate, int depth,
                 bool pending) {
  memset(&lane->stats, 0, sizeof(lane->stats));
  lane->stats.cells = cells;
  lane->stats.iterate = iterate;
  lane->stats.depth = depth;
  lane->stats_pending = pending;
  std::lock_guard<std::mutex> lock(g_mutex);
  if (t_lane == nullptr) {
    g_last_lane = lane;
    g_stats_aggregate = false;
  }
}

}  // namespace

int chunk_rows(const ProgramDesc& prog, int depth, const int32_t* dims,
               int rows) {
  Lane* lane = nullptr;
  int rc = current_lane(&lane);
  if (rc != kSuccess) return rc;
  const KernelVariant* kv = find_variant(prog, depth);
  if (kv == nullptr || rows < 1) return kInternalError;
  return choose_chunk_rows(lane, prog, kv, kv->kernel_tma, dims, rows, 1,
                           nullptr, nullptr);
}

int set_params(const ProgramDesc& prog, const void* const* host_arrays) {
  int rc = ensure_api();
  if (rc != kSuccess) return rc;
  for (int k = 0; k < prog.n_param; ++k)
    if (host_arrays == nullptr || host_arrays[k] == nullptr)
      return kBufferArgumentIsNull;
  std::lock_guard<std::mutex> lock(g_mutex);
  g_params_host.resize(prog.n_param);
  for (int k = 0; k < prog.n_param; ++k) {
    size_t bytes = static_cast<size_t>(prog.param_elem[k]);
    for (int d = 0; d < prog.param_rank[k]; ++d) bytes *= prog.param_size[k][d];
    const unsigned char* src =
        static_cast<const unsigned char*>(host_arrays[k]);
    g_params_host[k].assign(src, src + bytes);
  }
  g_params_version += 1;     // every lane uploads before its next launch
  return kSuccess;
}

int lead_rows(const ProgramDesc& prog, int depth) {
  const KernelVariant* kv = find_variant(prog, depth);
  if (kv == nullptr) return kInternalError;
  const int trip = std::max(1, kv->trip);
  return (kv->lead + kv->out_delay + trip - 1) / trip * trip;
}

int launch(const ProgramDesc& prog, int depth, const void* const* inputs,
           void* const* outputs, const int32_t* dims, int row_begin,
           int row_end, const int32_t* valid_lo, const int32_t* valid_hi,
           cudaStream_t stream, int forced_chunk_rows) {
  Lane* lane = nullptr;
  int rc = current_lane(&lane);
  if (rc != kSuccess) return rc;
  {
    // callers that drive single launches (the slab runner) read the kernel
    // configuration of their last launch from the same place as a run's
    std::lock_guard<std::mutex> lock(g_mutex);
    g_last_lane = lane;
    g_stats_aggregate = false;
  }
  return launch_on(lane, prog, depth, inputs, outputs, dims, 1, row_begin,
                   row_end, valid_lo, valid_hi, stream, forced_chunk_rows);
}

int run_device(const ProgramDesc& prog, const void* const* inputs,
               void* const* outputs, const int32_t* dims, int iterate,
               cudaStream_t stream, int batch) {
  if (batch < 1) return kAccessOutOfBounds;
  Lane* lane = nullptr;
  int rc = current_lane(&lane);
  if (rc != kSuccess) return rc;
  if (iterate <= 0) iterate = prog.iterate;
  if (iterate > prog.iterate) {
    fprintf(stderr, "ERROR: %s was compiled for at most %d iterations\n",
            prog.app_name, prog.iterate);
    return kInternalError;
  }
  std::vector<int> depths;
  rc = plan_depths(prog, iterate, &depths);
  if (rc != kSuccess) return rc;
  const int n_launch = static_cast<int>(depths.size());

  long long cells = batch;     // all items
  for (int d = 0; d < prog.dim; ++d) cells *= dims[d];
  if (cells >= (1LL << 40)) return kBufferExtentsTooLarge;
  // ping-pong between the caller's outputs and one scratch set, arranged so
  // the last launch lands in the outputs
  PoolLease lease(lane);
  void* scratch[kRtMaxTensors] = {};
  if (n_launch > 1)
    for (int k = 0; k < prog.n_out; ++k) {
      scratch[k] = lease.get(static_cast<size_t>(cells) * prog.out_elem[k]);
      if (scratch[k] == nullptr) return kDeviceMallocFailed;
    }
  Boxes full, fin;
  full_region(prog, dims, &full);
  valid_region(prog, iterate, dims, &fin);

  begin_stats(lane, cells, iterate, depths[0], true);
  SODA_CHECK(cudaEventRecord(lane->ev[0], stream), kDeviceRunFailed);
  const void* src[kRtMaxTensors];
  void* dst[kRtMaxTensors];
  for (int k = 0; k < prog.n_in; ++k) src[k] = inputs[k];
  for (int l = 0; l < n_launch; ++l) {
    const bool last = l + 1 == n_launch;
    const bool to_outputs = ((n_launch - 1 - l) % 2) == 0;
    for (int k = 0; k < prog.n_out; ++k)
      dst[k] = to_outputs ? outputs[k] : scratch[k];
    rc = launch_on(lane, prog, depths[l], src, dst, dims, batch, 0,
                   dims[prog.dim - 1], last ? fin.lo : full.lo,
                   last ? fin.hi : full.hi, stream, 0);
    if (rc != kSuccess) return rc;
    for (int k = 0; k < prog.n_out; ++k) src[k] = dst[k];
  }
  SODA_CHECK(cudaEventRecord(lane->ev[1], stream), kDeviceRunFailed);
  if (n_launch > 1) {
    // scratch goes back to the pool when the stream has drained past here
    SODA_CHECK(cudaStreamSynchronize(stream), kDeviceSyncFailed);
  }
  lease.completed = true;
  return kSuccess;
}

namespace {

bool is_query(const buffer_t* b) { return b->host == nullptr && b->dev == 0; }

void rewrite(buffer_t* b, int elem, int dim, const int32_t* min,
             const int32_t* extent) {
  int32_t stride = 1;
  for (int d = 0; d < 4; ++d) {
    b->min[d] = d < dim ? min[d] : 0;
    b->extent[d] = d < dim ? extent[d] : 0;
    b->stride[d] = d < dim ? stride : 0;
    if (d < dim) stride *= extent[d];
  }
  b->elem_size = elem;
}

// One slab of a run on host buffers: the rows [local_begin, local_end) of the
// global grid are this lane's local array; rows [own_begin, own_end) of the
// global grid are what it copies back.  A run on one device is the slab that
// covers everything.
struct Slab {
  int local_begin, local_end;
  int own_begin, own_end;
};

// Host buffers: cut the streamed dimension into pieces and overlap
//   H2D(piece k+1) | all launches on piece k | D2H(piece k-1).
//
// Every launch j keeps a frontier f_j: its output rows [need_lo_j, f_j) are
// done.  When input rows [0, avail) are on the device, launch 0 can extend
// its frontier to avail - reach_hi (to the end of what it needs once
// everything is loaded), launch 1 follows launch 0's frontier the same way,
// and so on; rows behind the last launch's frontier are final and go back to
// the host.  No cell is computed twice and every cell sees exactly the
// operands of the one-shot run, so the result is bit-identical.  The
// ping-pong buffers are shared between launches j and j-2; holding f_j back
// by max(reach_hi[j], reach_lo[j-1]) keeps launch j's writes below every row
// launch j-1 will still read.
//
// A slab of a sharded run carries ghost rows (the reach of ALL iterations) on
// the sides where the grid continues, instead of exchanging halos: launch j
// only computes the rows the later launches still need to produce the owned
// rows, [own_begin - reach of launches j+1.., own_end + ...), so the ghost
// work shrinks launch by launch.  Ghost cells next to the cut see zeros
// where the neighbour's rows would be — garbage that never reaches an owned
// row (the crop property the full-size tests rely on).
int run_pipelined(Lane* lane, const ProgramDesc& prog, buffer_t* const* inputs,
                  buffer_t* const* outputs, const int32_t* global_dims,
                  const Slab& slab, int pieces) {
  const int s = prog.dim - 1;
  const int rows = slab.local_end - slab.local_begin;     // local rows
  int32_t dims[kRtMaxDim] = {1, 1, 1, 1};
  long long row_cells = 1;
  for (int d = 0; d < prog.dim; ++d) {
    dims[d] = d == s ? rows : global_dims[d];
    if (d < s) row_cells *= global_dims[d];
  }
  const long long cells = row_cells * rows;
  std::vector<int> depths;
  int rc = plan_depths(prog, prog.iterate, &depths);
  if (rc != kSuccess) return rc;
  const int n_launch = static_cast<int>(depths.size());
  rc = ensure_streams(lane);
  if (rc != kSuccess) return rc;
  cudaStream_t s_in = lane->streams[0], s_run = lane->streams[1],
               s_out = lane->streams[2];

  PoolLease lease(lane);
  EventLease events(lane);
  void* in_dev[kRtMaxTensors];
  void* out_dev[kRtMaxTensors];
  void* scratch[kRtMaxTensors] = {};
  for (int k = 0; k < prog.n_in; ++k) {
    in_dev[k] = lease.get(static_cast<size_t>(cells) * prog.in_elem[k]);
    if (in_dev[k] == nullptr) return kDeviceMallocFailed;
  }
  for (int k = 0; k < prog.n_out; ++k) {
    out_dev[k] = lease.get(static_cast<size_t>(cells) * prog.out_elem[k]);
    if (out_dev[k] == nullptr) return kDeviceMallocFailed;
    if (n_launch > 1) {
      scratch[k] = lease.get(static_cast<size_t>(cells) * prog.out_elem[k]);
      if (scratch[k] == nullptr) return kDeviceMallocFailed;
    }
  }
  begin_stats(lane, cells, prog.iterate, depths[0], false);
  // pageable caller memory goes through pinned bounce buffers (Stager)
  bool stage_input[kRtMaxTensors] = {}, stage_output[kRtMaxTensors] = {};
  if (staging_enabled()) {
    for (int k = 0; k < prog.n_in; ++k)
      stage_input[k] = is_pageable(inputs[k]->host);
    for (int k = 0; k < prog.n_out; ++k)
      stage_output[k] = is_pageable(outputs[k]->host);
  }

  // streamed reach of every launch; rows (local) each launch must produce
  std::vector<int> reach_lo(n_launch), reach_hi(n_launch), hold(n_launch);
  std::vector<int> need_lo(n_launch), need_hi(n_launch);
  for (int j = 0; j < n_launch; ++j) {
    const int* w = prog.window + depths[j] * 2 * kRtMaxDim;
    reach_lo[j] = std::max(0, -w[s]);
    reach_hi[j] = std::max(0, w[kRtMaxDim + s]);
  }
  for (int j = 0; j < n_launch; ++j)
    hold[j] = std::max(reach_hi[j], j > 0 ? reach_lo[j - 1] : 0);
  const int copy_begin = slab.own_begin - slab.local_begin;
  const int copy_end = slab.own_end - slab.local_begin;
  for (int j = n_launch - 1, lo = copy_begin, hi = copy_end; j >= 0; --j) {
    need_lo[j] = std::max(0, lo);
    need_hi[j] = std::min(rows, hi);
    lo -= reach_lo[j];     // what launch j reads, launch j - 1 must produce
    hi += reach_hi[j];
  }
  // where the outputs are defined, in local coordinates
  Boxes full, fin;
  full_region(prog, dims, &full);
  valid_region(prog, prog.iterate, global_dims, &fin);
  for (int k = 0; k < prog.n_out; ++k) {
    int32_t& lo = fin.lo[k * kRtMaxDim + s];
    int32_t& hi = fin.hi[k * kRtMaxDim + s];
    lo = std::min(std::max(0, lo - slab.local_begin), rows);
    hi = std::min(std::max(0, hi - slab.local_begin), rows);
  }

  std::vector<int> frontier(need_lo);
  SODA_CHECK(cudaEventRecord(lane->ev[2], s_in), kCopyToDeviceFailed);
  SODA_CHECK(cudaEventRecord(lane->ev[0], s_run), kDeviceRunFailed);
  bool d2h_started = false;
  int loaded = 0;
  int copied = copy_begin;
  pieces = std::max(1, std::min(pieces, rows));
  // Piece boundaries: equal pieces, the last one cut again into 1/2, 1/4, 1/4.
  // The host-to-device copies are the critical resource; what follows the
  // last of them — its launches and the copy back of its rows — is exposed,
  // so the last piece is small.
  std::vector<int> bounds;
  for (int piece = 0; piece < pieces; ++piece)
    bounds.push_back(static_cast<int>(
        static_cast<long long>(rows) * (piece + 1) / pieces));
  if (pieces >= 4) {
    const int last_begin = bounds[pieces - 2], last = rows - last_begin;
    if (last >= 64) {
      bounds.back() = last_begin + last / 2;
      bounds.push_back(last_begin + last / 2 + last / 4);
      bounds.push_back(rows);
    }
  }
  pieces = static_cast<int>(bounds.size());
  for (int piece = 0; piece < pieces; ++piece) {
    const int upto = bounds[piece];
    if (upto <= loaded) continue;
    for (int k = 0; k < prog.n_in; ++k) {
      const size_t off =
          static_cast<size_t>(loaded) * row_cells * prog.in_elem[k];
      const size_t host_off = static_cast<size_t>(slab.local_begin + loaded) *
                              row_cells * prog.in_elem[k];
      const size_t bytes =
          static_cast<size_t>(upto - loaded) * row_cells * prog.in_elem[k];
      rc = copy_in(lane, static_cast<char*>(in_dev[k]) + off,
                   inputs[k]->host + host_off, bytes, stage_input[k], s_in);
      if (rc != kSuccess) return rc;
    }
    loaded = upto;
    cudaEvent_t arrived = events.get();
    if (arrived == nullptr) return kDeviceRunFailed;
    SODA_CHECK(cudaEventRecord(arrived, s_in), kCopyToDeviceFailed);
    SODA_CHECK(cudaStreamWaitEvent(s_run, arrived, 0), kDeviceRunFailed);
    if (piece + 1 == pieces)
      SODA_CHECK(cudaEventRecord(lane->ev[3], s_in), kCopyToDeviceFailed);

    int avail = loaded;              // rows of the source that exist
    bool source_complete = loaded >= rows;
    const void* src[kRtMaxTensors];
    void* dst[kRtMaxTensors];
    for (int j = 0; j < n_launch; ++j) {
      const int target =
          source_complete
              ? need_hi[j]
              : std::min(need_hi[j], std::max(frontier[j], avail - hold[j]));
      const bool last = j + 1 == n_launch;
      const bool to_outputs = ((n_launch - 1 - j) % 2) == 0;
      for (int k = 0; k < prog.n_in; ++k)
        src[k] = j == 0 ? in_dev[k]
                        : (to_outputs ? scratch[k] : out_dev[k]);
      for (int k = 0; k < prog.n_out; ++k)
        dst[k] = to_outputs ? out_dev[k] : scratch[k];
      if (target > frontier[j]) {
        rc = launch_on(lane, prog, depths[j], src, dst, dims, 1, frontier[j],
                       target, last ? fin.lo : full.lo,
                       last ? fin.hi : full.hi, s_run, 0);
        if (rc != kSuccess) return rc;
        frontier[j] = target;
      }
      avail = frontier[j];
      source_complete = frontier[j] >= need_hi[j];
    }
    const int done = std::min(frontier[n_launch - 1], copy_end);
    if (done > copied) {
      cudaEvent_t computed = events.get();
      if (computed == nullptr) return kDeviceRunFailed;
      SODA_CHECK(cudaEventRecord(computed, s_run), kDeviceRunFailed);
      SODA_CHECK(cudaStreamWaitEvent(s_out, computed, 0), kCopyToHostFailed);
      if (!d2h_started) {
        SODA_CHECK(cudaEventRecord(lane->ev[4], s_out), kCopyToHostFailed);
        d2h_started = true;
      }
      for (int k = 0; k < prog.n_out; ++k) {
        const size_t off =
            static_cast<size_t>(copied) * row_cells * prog.out_elem[k];
        const size_t host_off = static_cast<size_t>(slab.local_begin + copied) *
                                row_cells * prog.out_elem[k];
        const size_t bytes = static_cast<size_t>(done - copied) * row_cells *
                             prog.out_elem[k];
        rc = copy_out(lane, outputs[k]->host + host_off,
                      static_cast<char*>(out_dev[k]) + off, bytes,
                      stage_output[k], s_out);
        if (rc != kSuccess) return rc;
      }
      copied = done;
    }
  }
  if (!d2h_started)
    SODA_CHECK(cudaEventRecord(lane->ev[4], s_out), kCopyToHostFailed);
  SODA_CHECK(cudaEventRecord(lane->ev[1], s_run), kDeviceRunFailed);
  SODA_CHECK(cudaEventRecord(lane->ev[5], s_out), kCopyToHostFailed);
  SODA_CHECK(cudaStreamSynchronize(s_in), kDeviceSyncFailed);
  SODA_CHECK(cudaStreamSynchronize(s_run), kDeviceSyncFailed);
  SODA_CHECK(cudaStreamSynchronize(s_out), kDeviceSyncFailed);
  rc = finish_copies(lane);
  if (rc != kSuccess) return rc;
  lease.completed = true;
  if (copied != copy_end) {
    fprintf(stderr, "ERROR: pipeline finished at row %d of %d\n", copied,
            copy_end);
    return kInternalError;
  }
  float ms = 0;
  if (cudaEventElapsedTime(&ms, lane->ev[2], lane->ev[3]) == cudaSuccess)
    lane->stats.h2d_ms = ms;
  if (cudaEventElapsedTime(&ms, lane->ev[4], lane->ev[5]) == cudaSuccess)
    lane->stats.d2h_ms = ms;
  if (cudaEventElapsedTime(&ms, lane->ev[0], lane->ev[1]) == cudaSuccess)
    lane->stats.kernel_ms = ms;
  lane->stats.reserved = pieces;
  return kSuccess;
}

// "0,1,2", "all" or "" -> device ordinals; < 0: malformed.
int parse_devices(const char* text, std::vector<int>* out) {
  out->clear();
  if (text == nullptr) return 0;
  while (*text == ' ') ++text;
  if (*text == '\0') return 0;
  int count = 0;
  if (cudaGetDeviceCount(&count) != cudaSuccess) {
    cudaGetLastError();
    return kNoDeviceInterface;
  }
  if (strncmp(text, "all", 3) == 0) {
    for (int d = 0; d < count; ++d) out->push_back(d);
    return 0;
  }
  const char* p = text;
  while (*p != '\0') {
    char* end = nullptr;
    const long v = strtol(p, &end, 10);
    if (end == p || v < 0 || v >= count) {
      fprintf(stderr, "ERROR: bad device list `%s` (%d device(s) visible)\n",
              text, count);
      return kInternalError;
    }
    out->push_back(static_cast<int>(v));
    p = end;
    while (*p == ',' || *p == ' ') ++p;
  }
  return 0;
}

// The devices of a run: `devices=...` in the config string of the entry point
// (the reference's opaque `xclbin` argument), else SODA_CUDA_DEVICES.
int run_devices(const char* config, std::vector<int>* out) {
  out->clear();
  if (config != nullptr) {
    const char* at = strstr(config, "devices=");
    if (at != nullptr) {
      std::string list(at + 8);
      const size_t stop = list.find_first_of("; ");
      if (stop != std::string::npos) list.resize(stop);
      return parse_devices(list.c_str(), out);
    }
  }
  return parse_devices(getenv("SODA_CUDA_DEVICES"), out);
}

}  // namespace

int shard_plan(const ProgramDesc& prog, const int32_t* dims, int n_slabs,
               int32_t* local_begin, int32_t* local_end, int32_t* own_begin,
               int32_t* own_end) {
  const int s = prog.dim - 1;
  const int rows = dims[s];
  const int* w = prog.window + prog.iterate * 2 * kRtMaxDim;
  const int ghost_lo = std::max(0, -w[s]);
  const int ghost_hi = std::max(0, w[kRtMaxDim + s]);
  // a slab thinner than its ghost rows computes more ghost than grid
  int n = std::max(1, std::min(n_slabs, rows));
  while (n > 1 && rows / n < ghost_lo + ghost_hi) --n;
  for (int r = 0; r < n; ++r) {
    own_begin[r] = static_cast<int32_t>(static_cast<long long>(rows) * r / n);
    own_end[r] =
        static_cast<int32_t>(static_cast<long long>(rows) * (r + 1) / n);
    local_begin[r] = std::max(0, own_begin[r] - ghost_lo);
    local_end[r] = std::min(rows, own_end[r] + ghost_hi);
  }
  return n;
}

namespace {

// Host buffers on several devices: one slab per entry of `devices` along the
// streamed dimension, one host thread per slab, no exchange between devices
// (ghost rows of the whole run's reach are loaded and recomputed instead):
// every device moves its share of the arrays over its own PCIe link.
int run_sharded(const ProgramDesc& prog, buffer_t* const* inputs,
                buffer_t* const* outputs, const int32_t* dims,
                const std::vector<int>& devices) {
  const int wanted = static_cast<int>(devices.size());
  std::vector<int32_t> lb(wanted), le(wanted), ob(wanted), oe(wanted);
  const int n = shard_plan(prog, dims, wanted, lb.data(), le.data(), ob.data(),
                           oe.data());
  const int s = prog.dim - 1;
  long long row_cells = 1;
  for (int d = 0; d < s; ++d) row_cells *= dims[d];
  std::vector<int> codes(n, kSuccess);
  std::vector<Lane*> lanes(n, nullptr);
  std::vector<std::thread> threads;
  int caller_device = 0;
  SODA_CHECK(cudaGetDevice(&caller_device), kNoDeviceInterface);
  for (int r = 0; r < n; ++r) {
    int replica = 0;
    for (int q = 0; q < r; ++q)
      if (devices[q] == devices[r]) ++replica;
    threads.emplace_back([&, r, replica]() {
      if (cudaSetDevice(devices[r]) != cudaSuccess) {
        cudaGetLastError();
        codes[r] = kNoDeviceInterface;
        return;
      }
      Lane* lane = nullptr;
      codes[r] = lane_for(devices[r], replica, &lane);
      if (codes[r] != kSuccess) return;
      lanes[r] = lane;
      std::lock_guard<std::mutex> run_lock(lane->run_mutex);
      t_lane = lane;
      const Slab slab = {lb[r], le[r], ob[r], oe[r]};
      size_t moved = 0;
      for (int k = 0; k < prog.n_in; ++k)
        moved += static_cast<size_t>(le[r] - lb[r]) * row_cells *
                 prog.in_elem[k];
      for (int k = 0; k < prog.n_out; ++k)
        moved += static_cast<size_t>(oe[r] - ob[r]) * row_cells *
                 prog.out_elem[k];
      int pieces = static_cast<int>(std::min<size_t>(16, moved >> 26));
      if (const char* v = getenv("SODA_CUDA_PIECES")) pieces = atoi(v);
      codes[r] = run_pipelined(lane, prog, inputs, outputs, dims, slab,
                               std::max(1, pieces));
      t_lane = nullptr;
    });
  }
  for (auto& t : threads) t.join();
  cudaSetDevice(caller_device);
  for (int r = 0; r < n; ++r)
    if (codes[r] != kSuccess) return codes[r];
  // what the run did: times are the slowest slab's, launches are summed
  std::lock_guard<std::mutex> lock(g_mutex);
  g_lane_stats.clear();
  memset(&g_stats, 0, sizeof(g_stats));
  for (int r = 0; r < n; ++r) {
    const soda_cuda_stats_t& st = lanes[r]->stats;
    g_lane_stats.push_back(st);
    g_stats.kernel_ms = std::max(g_stats.kernel_ms, st.kernel_ms);
    g_stats.h2d_ms = std::max(g_stats.h2d_ms, st.h2d_ms);
    g_stats.d2h_ms = std::max(g_stats.d2h_ms, st.d2h_ms);
    g_stats.launches += st.launches;
    g_stats.depth = st.depth;
    g_stats.used_tma = st.used_tma;
    g_stats.blocks = st.blocks;
    g_stats.threads = st.threads;
    g_stats.smem_bytes = st.smem_bytes;
  }
  g_stats.cells = row_cells * dims[s];
  g_stats.iterate = prog.iterate;
  g_stats.reserved = n;
  g_stats_aggregate = true;
  if (verbose())
    fprintf(stderr, "INFO: %d slab(s): h2d %.3f ms, launches %.3f ms, d2h "
                    "%.3f ms (slowest slab, overlapped)\n", n, g_stats.h2d_ms,
            g_stats.kernel_ms, g_stats.d2h_ms);
  return kSuccess;
}

}  // namespace

namespace {

int check_present(const ProgramDesc& prog, buffer_t* const* inputs,
                  buffer_t* const* outputs) {
  for (int k = 0; k < prog.n_in; ++k)
    if (inputs == nullptr || inputs[k] == nullptr) return kBufferArgumentIsNull;
  for (int k = 0; k < prog.n_out; ++k)
    if (outputs == nullptr || outputs[k] == nullptr)
      return kBufferArgumentIsNull;
  return kSuccess;
}

// What every run on buffer_t's checks: element sizes, params (uploaded when
// given), dense arrays of one common extent, which `dims` receives.
int check_buffers(const ProgramDesc& prog, buffer_t* const* inputs,
                  buffer_t* const* outputs, buffer_t* const* params,
                  int32_t* dims) {
  for (int k = 0; k < prog.n_out; ++k)
    if (outputs[k]->elem_size != prog.out_elem[k]) {
      fprintf(stderr, "ERROR: Buffer %s has type %s but elem_size of the "
                      "buffer passed in is %d instead of %d\n",
              prog.out_name[k], prog.out_type[k], outputs[k]->elem_size,
              prog.out_elem[k]);
      return kBadElemSize;
    }
  for (int k = 0; k < prog.n_in; ++k)
    if (inputs[k]->elem_size != prog.in_elem[k]) {
      fprintf(stderr, "ERROR: Buffer %s has type %s but elem_size of the "
                      "buffer passed in is %d instead of %d\n",
              prog.in_name[k], prog.in_type[k], inputs[k]->elem_size,
              prog.in_elem[k]);
      return kBadElemSize;
    }

  if (prog.n_param > 0 && params != nullptr) {
    // param arrays: small, host memory, uploaded before the launches
    const void* host_arrays[kRtMaxTensors] = {};
    for (int k = 0; k < prog.n_param; ++k) {
      const buffer_t* b = params[k];
      if (b == nullptr || b->host == nullptr) return kBufferArgumentIsNull;
      if (b->elem_size != prog.param_elem[k]) {
        fprintf(stderr, "ERROR: Buffer %s has type %s but elem_size of the "
                        "buffer passed in is %d instead of %d\n",
                prog.param_name[k], prog.param_type[k], b->elem_size,
                prog.param_elem[k]);
        return kBadElemSize;
      }
      for (int d = 0; d < prog.param_rank[k]; ++d)
        if (b->extent[d] != prog.param_size[k][d]) return kAccessOutOfBounds;
      host_arrays[k] = b->host;
    }
    const int rc = set_params(prog, host_arrays);
    if (rc != kSuccess) return rc;
  }

  for (int d = 0; d < kRtMaxDim; ++d) dims[d] = 1;
  for (int d = 0; d < prog.dim; ++d) {
    dims[d] = inputs[0]->extent[d];
    if (dims[d] <= 0) return kAccessOutOfBounds;
  }
  auto dense = [&](const buffer_t* b) {
    int32_t stride = 1;
    for (int d = 0; d < prog.dim; ++d) {
      if (b->extent[d] != dims[d] || b->stride[d] != stride) return false;
      stride *= dims[d];
    }
    return true;
  };
  for (int k = 0; k < prog.n_in; ++k)
    if (!dense(inputs[k])) {
      fprintf(stderr, "ERROR: input %s is not a dense array of the common "
                      "extent\n", prog.in_name[k]);
      return kAccessOutOfBounds;
    }
  for (int k = 0; k < prog.n_out; ++k)
    if (!dense(outputs[k])) {
      fprintf(stderr, "ERROR: output %s is not a dense array of the common "
                      "extent\n", prog.out_name[k]);
      return kAccessOutOfBounds;
    }
  return kSuccess;
}

// `batch` items of extents `dims` in each buffer, one after the other: copy
// the host buffers in, run, copy back, on the default stream.  Device
// buffers are used in place.
int run_copied(Lane* lane, const ProgramDesc& prog, buffer_t* const* inputs,
               buffer_t* const* outputs, const int32_t* dims, int batch) {
  long long cells = batch;
  for (int d = 0; d < prog.dim; ++d) cells *= dims[d];
  cudaStream_t stream = nullptr;
  PoolLease lease(lane);
  const void* in_dev[kRtMaxTensors];
  void* out_dev[kRtMaxTensors];
  SODA_CHECK(cudaEventRecord(lane->ev[2], stream), kCopyToDeviceFailed);
  for (int k = 0; k < prog.n_in; ++k) {
    const size_t bytes = static_cast<size_t>(cells) * prog.in_elem[k];
    if (inputs[k]->dev != 0) {
      in_dev[k] = reinterpret_cast<const void*>(inputs[k]->dev);
      continue;
    }
    void* p = lease.get(bytes);
    if (p == nullptr) return kDeviceMallocFailed;
    SODA_CHECK(cudaMemcpyAsync(p, inputs[k]->host, bytes,
                               cudaMemcpyHostToDevice, stream),
               kCopyToDeviceFailed);
    in_dev[k] = p;
  }
  SODA_CHECK(cudaEventRecord(lane->ev[3], stream), kCopyToDeviceFailed);
  for (int k = 0; k < prog.n_out; ++k) {
    const size_t bytes = static_cast<size_t>(cells) * prog.out_elem[k];
    if (outputs[k]->dev != 0) {
      out_dev[k] = reinterpret_cast<void*>(outputs[k]->dev);
      continue;
    }
    out_dev[k] = lease.get(bytes);
    if (out_dev[k] == nullptr) return kDeviceMallocFailed;
  }
  const int rc = run_device(prog, in_dev, out_dev, dims, prog.iterate, stream,
                            batch);
  if (rc != kSuccess) return rc;
  SODA_CHECK(cudaEventRecord(lane->ev[4], stream), kCopyToHostFailed);
  for (int k = 0; k < prog.n_out; ++k) {
    if (outputs[k]->dev != 0) continue;
    const size_t bytes = static_cast<size_t>(cells) * prog.out_elem[k];
    SODA_CHECK(cudaMemcpyAsync(outputs[k]->host, out_dev[k], bytes,
                               cudaMemcpyDeviceToHost, stream),
               kCopyToHostFailed);
  }
  SODA_CHECK(cudaEventRecord(lane->ev[5], stream), kCopyToHostFailed);
  SODA_CHECK(cudaStreamSynchronize(stream), kDeviceSyncFailed);
  lease.completed = true;
  float ms = 0;
  if (cudaEventElapsedTime(&ms, lane->ev[2], lane->ev[3]) == cudaSuccess)
    lane->stats.h2d_ms = ms;
  if (cudaEventElapsedTime(&ms, lane->ev[4], lane->ev[5]) == cudaSuccess)
    lane->stats.d2h_ms = ms;
  const soda_cuda_stats_t* st = last_stats();
  if (verbose()) {
    // the two lines the reference host prints (host.py:796-800)
    fprintf(stderr, "INFO: Kernel execution time: %lf us\n",
            st->kernel_ms * 1e3);
    fprintf(stderr, "INFO: Kernel throughput: %lf pixel/ns\n",
            st->kernel_ms > 0 ? cells / (st->kernel_ms * 1e6) : 0.0);
  }
  return kSuccess;
}

}  // namespace

int run_buffers(const ProgramDesc& prog, buffer_t* const* inputs,
                buffer_t* const* outputs, const char* config,
                buffer_t* const* params) {
  int rc = check_present(prog, inputs, outputs);
  if (rc != kSuccess) return rc;

  // bounds-query mode (reference host.py:204-252): a buffer with neither host
  // nor device memory gets its shape filled in; nothing is computed.
  bool query = false;
  for (int k = 0; k < prog.n_out; ++k)
    if (is_query(outputs[k])) {
      query = true;
      rewrite(outputs[k], prog.out_elem[k], prog.dim, outputs[k]->min,
              outputs[k]->extent);
    }
  for (int k = 0; k < prog.n_in; ++k)
    if (is_query(inputs[k])) {
      query = true;
      int32_t extent[4] = {0, 0, 0, 0};
      for (int d = 0; d < prog.dim; ++d)
        extent[d] = outputs[0]->extent[d] + prog.stencil_dim[d] - 1;
      rewrite(inputs[k], prog.in_elem[k], prog.dim, outputs[0]->min, extent);
    }
  if (query) return kSuccess;

  int32_t dims[kRtMaxDim];
  rc = check_buffers(prog, inputs, outputs, params, dims);
  if (rc != kSuccess) return rc;

  Lane* lane = nullptr;
  rc = current_lane(&lane);
  if (rc != kSuccess) return rc;

  long long cells = 1;
  for (int d = 0; d < prog.dim; ++d) cells *= dims[d];
  bool all_host = true;
  size_t moved = 0;
  for (int k = 0; k < prog.n_in; ++k) {
    all_host = all_host && inputs[k]->dev == 0;
    moved += static_cast<size_t>(cells) * prog.in_elem[k];
  }
  for (int k = 0; k < prog.n_out; ++k) {
    all_host = all_host && outputs[k]->dev == 0;
    moved += static_cast<size_t>(cells) * prog.out_elem[k];
  }

  // several devices (config "devices=0,1,.." or SODA_CUDA_DEVICES): one slab
  // of the streamed dimension per device, each over its own PCIe link
  std::vector<int> devices;
  rc = run_devices(config, &devices);
  if (rc != kSuccess) return rc;
  if (devices.size() > 1) {
    if (all_host) return run_sharded(prog, inputs, outputs, dims, devices);
    if (verbose())
      fprintf(stderr, "INFO: device buffers live on one device; the device "
                      "list is ignored\n");
  }

  std::lock_guard<std::mutex> run_lock(lane->run_mutex);
  // large all-host problems: overlap the copies with the launches
  int pieces = static_cast<int>(std::min<size_t>(16, moved >> 27));  // 128 MiB
  if (const char* v = getenv("SODA_CUDA_PIECES")) pieces = atoi(v);
  pieces = std::min(pieces, dims[prog.dim - 1]);
  // pageable arrays of some size: one piece, but through the bounce buffers
  // (the driver's own staging of pageable copies runs at a ninth of the link)
  if (all_host && pieces <= 1 && moved >= (size_t(16) << 20) &&
      staging_enabled() && getenv("SODA_CUDA_PIECES") == nullptr) {
    bool pageable = false;
    for (int k = 0; k < prog.n_in; ++k)
      pageable = pageable || is_pageable(inputs[k]->host);
    for (int k = 0; k < prog.n_out; ++k)
      pageable = pageable || is_pageable(outputs[k]->host);
    if (pageable) pieces = 2;
  }
  if (all_host && pieces > 1) {
    const Slab whole = {0, dims[prog.dim - 1], 0, dims[prog.dim - 1]};
    rc = run_pipelined(lane, prog, inputs, outputs, dims, whole, pieces);
    if (rc == kSuccess && verbose())
      fprintf(stderr, "INFO: %d pieces: h2d %.3f ms, launches %.3f ms, d2h "
                      "%.3f ms (overlapped)\n", pieces, lane->stats.h2d_ms,
              lane->stats.kernel_ms, lane->stats.d2h_ms);
    return rc;
  }

  return run_copied(lane, prog, inputs, outputs, dims, 1);
}

int run_batch(const ProgramDesc& prog, buffer_t* const* inputs,
              buffer_t* const* outputs, buffer_t* const* params, int batch) {
  if (batch < 1) return kAccessOutOfBounds;
  int rc = check_present(prog, inputs, outputs);
  if (rc != kSuccess) return rc;
  for (int k = 0; k < prog.n_in; ++k)
    if (is_query(inputs[k])) return kBufferArgumentIsNull;
  for (int k = 0; k < prog.n_out; ++k)
    if (is_query(outputs[k])) return kBufferArgumentIsNull;
  int32_t dims[kRtMaxDim];
  rc = check_buffers(prog, inputs, outputs, params, dims);
  if (rc != kSuccess) return rc;
  Lane* lane = nullptr;
  rc = current_lane(&lane);
  if (rc != kSuccess) return rc;
  std::lock_guard<std::mutex> run_lock(lane->run_mutex);
  return run_copied(lane, prog, inputs, outputs, dims, batch);
}

int flag_write(void* flag, uint32_t value, cudaStream_t stream) {
  if (int code = ensure_api()) return code;
  const CUresult res = g_api.write_value(
      stream, reinterpret_cast<CUdeviceptr>(flag), value,
      CU_STREAM_WRITE_VALUE_DEFAULT);
  if (res != CUDA_SUCCESS) {
    fprintf(stderr, "ERROR: cuStreamWriteValue32 failed (%d)\n",
            static_cast<int>(res));
    return kDeviceRunFailed;
  }
  return kSuccess;
}

int flag_wait_geq(void* flag, uint32_t value, cudaStream_t stream) {
  if (int code = ensure_api()) return code;
  const CUresult res = g_api.wait_value(
      stream, reinterpret_cast<CUdeviceptr>(flag), value,
      CU_STREAM_WAIT_VALUE_GEQ);
  if (res != CUDA_SUCCESS) {
    fprintf(stderr, "ERROR: cuStreamWaitValue32 failed (%d)\n",
            static_cast<int>(res));
    return kDeviceRunFailed;
  }
  return kSuccess;
}

static_assert(sizeof(cudaIpcMemHandle_t) == 64, "IPC handles are 64 bytes");

int ipc_export(const void* ptr, unsigned char handle[64], uint64_t* offset) {
  if (int code = ensure_api()) return code;
  CUdeviceptr base = 0;
  size_t size = 0;
  if (g_api.address_range(&base, &size, reinterpret_cast<CUdeviceptr>(ptr)) !=
      CUDA_SUCCESS) {
    fprintf(stderr, "ERROR: %p is not a device allocation\n", ptr);
    return kDeviceRunFailed;
  }
  cudaIpcMemHandle_t h;
  SODA_CHECK(cudaIpcGetMemHandle(&h, reinterpret_cast<void*>(base)),
             kDeviceRunFailed);
  memcpy(handle, &h, 64);
  *offset = reinterpret_cast<CUdeviceptr>(ptr) - base;
  return kSuccess;
}

int ipc_open(const unsigned char handle[64], void** base) {
  if (int code = ensure_api()) return code;
  cudaIpcMemHandle_t h;
  memcpy(&h, handle, 64);
  SODA_CHECK(cudaIpcOpenMemHandle(base, h, cudaIpcMemLazyEnablePeerAccess),
             kDeviceRunFailed);
  return kSuccess;
}

int ipc_close(void* base) {
  SODA_CHECK(cudaIpcCloseMemHandle(base), kDeviceRunFailed);
  return kSuccess;
}

int copy_async(void* dst, const void* src, uint64_t bytes,
               cudaStream_t stream) {
  SODA_CHECK(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDefault, stream),
             kDeviceRunFailed);
  return kSuccess;
}

const soda_cuda_stats_t* last_stats() {
  std::lock_guard<std::mutex> lock(g_mutex);
  if (g_stats_aggregate) return &g_stats;
  Lane* lane = g_last_lane;
  if (lane == nullptr) return &g_stats;
  if (lane->stats_pending) {
    if (cudaEventSynchronize(lane->ev[1]) == cudaSuccess) {
      float ms = 0;
      if (cudaEventElapsedTime(&ms, lane->ev[0], lane->ev[1]) == cudaSuccess)
        lane->stats.kernel_ms = ms;
    }
    cudaGetLastError();
    lane->stats_pending = false;
  }
  return &lane->stats;
}

int slab_stats(int index, soda_cuda_stats_t* out) {
  std::lock_guard<std::mutex> lock(g_mutex);
  const int n = g_stats_aggregate ? static_cast<int>(g_lane_stats.size()) : 0;
  if (out != nullptr && index >= 0 && index < n) *out = g_lane_stats[index];
  return n;
}

void release_all() {
  std::lock_guard<std::mutex> lock(g_mutex);
  int caller_device = 0;
  if (cudaGetDevice(&caller_device) != cudaSuccess) {
    cudaGetLastError();
    return;
  }
  for (auto& lane : g_lanes) {
    std::lock_guard<std::mutex> lane_lock(lane->mutex);
    cudaSetDevice(lane->ordinal);
    for (auto& e : lane->pool)
      if (e.ptr != nullptr) cudaFree(e.ptr);
    lane->pool.clear();
    lane->maps.clear();
    for (void*& p : lane->param_dev) {
      if (p != nullptr) cudaFree(p);
      p = nullptr;
    }
    lane->params_version = 0;
    for (Stager* st : {&lane->stage_in, &lane->stage_out}) {
      for (int k = 0; k < Stager::kSlots; ++k) {
        if (st->slot[k] != nullptr) cudaFreeHost(st->slot[k]);
        st->slot[k] = nullptr;
        st->busy[k] = false;
        st->out_bytes[k] = 0;
      }
      st->slot_bytes = 0;
    }
  }
  g_params_host.clear();      // params must be set again before a launch
  g_params_version = 0;
  cudaSetDevice(caller_device);
}

}  // namespace soda
