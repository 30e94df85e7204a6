// libceres_b200.so — the precompiled, type-erased half of the evaluation engine.
//
// Implements the C ABI of include/ceres_b200.h: device buffers, the
// structure-of-arrays tables the kernels read, the per-rank Jacobian slices, the
// cost reduction, host<->device transfers and the NCCL all-reduce.  The templated
// kernels live in include/ceres/internal/evaluate_kernel.cuh and reach this file
// only as launch thunks.
//
// Replaces (reference): internal/ceres/registered_cuda_evaluators.cc:46-280,
// include/ceres/internal/autodiff_residual_block_cuda_evaluator.h:96-271,
// include/ceres/internal/cuda_buffer.h:52-182, internal/ceres/context_impl.cc:112-174.
//
// Differences from the reference that matter for speed:
//  * no memset of residuals / Jacobian values (every element is written exactly
//    once by the kernel; only the gradient accumulator is zeroed);
//  * no per-thread Jacobian scratch (reference: 2 x nRB x kRes x sum(Ns) doubles);
//  * one host synchronisation per Evaluate instead of two per residual type;
//  * the program POSITION of each residual block indexes the layouts, never
//    ResidualBlock::index() (stale after the Schur reordering, SURVEY.md hazard 1).
#include <cuda_runtime.h>
#include <dlfcn.h>
#include <sys/mman.h>

#include <algorithm>
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <nvtx3/nvToolsExt.h>  // header-only; ranges cost nothing unless a tool is attached
#include <cstring>
#include <mutex>
#include <string>
#include <utility>
#include <vector>

#include "ceres_b200.h"

namespace {

// ---- NCCL through dlopen: torch (when it hosts the process) already has
// libnccl.so.2 loaded and dlopen returns that same copy.
struct Uid {
  char internal[128];
};
struct NcclApi {
  void* handle = nullptr;
  int (*GetUniqueId)(void*) = nullptr;
  int (*CommInitRank)(void**, int, /* ncclUniqueId by value */ Uid, int) = nullptr;
  int (*AllReduce)(const void*, void*, size_t, int, int, void*, cudaStream_t) = nullptr;
  int (*Broadcast)(const void*, void*, size_t, int, int, void*, cudaStream_t) = nullptr;
  int (*AllGather)(const void*, void*, size_t, int, void*, cudaStream_t) = nullptr;
  int (*GroupStart)() = nullptr;
  int (*GroupEnd)() = nullptr;
  int (*CommDestroy)(void*) = nullptr;
  const char* (*GetErrorString)(int) = nullptr;
};
constexpr int kNcclFloat64 = 8;  // ncclDouble
constexpr int kNcclSum = 0;      // ncclSum

NcclApi* GetNccl() {
  static NcclApi api;
  static bool tried = false;
  if (!tried) {
    tried = true;
    const char* names[] = {"libnccl.so.2", "libnccl.so"};
    for (const char* n : names) {
      api.handle = dlopen(n, RTLD_NOW | RTLD_GLOBAL);
      if (api.handle) break;
    }
    if (api.handle) {
      api.GetUniqueId = reinterpret_cast<int (*)(void*)>(dlsym(api.handle, "ncclGetUniqueId"));
      api.CommInitRank = reinterpret_cast<int (*)(void**, int, Uid, int)>(
          dlsym(api.handle, "ncclCommInitRank"));
      api.AllReduce =
          reinterpret_cast<int (*)(const void*, void*, size_t, int, int, void*, cudaStream_t)>(
              dlsym(api.handle, "ncclAllReduce"));
      api.Broadcast =
          reinterpret_cast<int (*)(const void*, void*, size_t, int, int, void*, cudaStream_t)>(
              dlsym(api.handle, "ncclBroadcast"));
      api.AllGather =
          reinterpret_cast<int (*)(const void*, void*, size_t, int, void*, cudaStream_t)>(
              dlsym(api.handle, "ncclAllGather"));
      api.GroupStart = reinterpret_cast<int (*)()>(dlsym(api.handle, "ncclGroupStart"));
      api.GroupEnd = reinterpret_cast<int (*)()>(dlsym(api.handle, "ncclGroupEnd"));
      api.CommDestroy = reinterpret_cast<int (*)(void*)>(dlsym(api.handle, "ncclCommDestroy"));
      api.GetErrorString =
          reinterpret_cast<const char* (*)(int)>(dlsym(api.handle, "ncclGetErrorString"));
    }
  }
  return (api.handle && api.GetUniqueId && api.CommInitRank && api.AllReduce) ? &api : nullptr;
}

template <typename T>
struct DeviceBuffer {
  T* ptr = nullptr;
  size_t count = 0;
  cudaError_t Resize(size_t n) {
    if (n == count && ptr) return cudaSuccess;
    Free();
    if (n == 0) return cudaSuccess;
    cudaError_t e = cudaMalloc(reinterpret_cast<void**>(&ptr), n * sizeof(T));
    if (e == cudaSuccess) count = n;
    return e;
  }
  cudaError_t Upload(const std::vector<T>& v, cudaStream_t s) {
    cudaError_t e = Resize(v.size());
    if (e != cudaSuccess || v.empty()) return e;
    return cudaMemcpyAsync(ptr, v.data(), v.size() * sizeof(T), cudaMemcpyHostToDevice, s);
  }
  void Free() {
    if (ptr) cudaFree(ptr);
    ptr = nullptr;
    count = 0;
  }
};

struct Segment {
  int64_t global_begin, length, local_begin;
};

// One interval of the gradient in the exchange plan: owner >= 0 means only that rank's
// residual blocks touch these entries (its values are broadcast), owner < 0 means several
// ranks contribute (all-reduce).
struct GradientInterval {
  int64_t begin, length;
  int32_t owner;
};

struct ResidualType {
  cb200_residual_type desc;
  // Host copies as handed over (all residual blocks of the type, any rank).
  std::vector<int32_t> position;   // program position
  std::vector<int32_t> pb_ids;     // [n][nb]
  std::vector<char> functors;
  std::vector<char> loss_table;
  int32_t num_losses = 1;
  std::vector<int32_t> loss_index;
  // This rank's tables.
  int32_t n_local = 0;
  int32_t grid = 0;
  int32_t cost_partial_offset = 0;
  DeviceBuffer<char> d_functors, d_loss_table;
  DeviceBuffer<int32_t> d_loss_index, d_pb, d_soff, d_doff, d_jpos, d_jstride, d_respos;
  bool plain = true;
  // Tables that turned out to be arithmetic progressions (cb200_launch_args::affine).
  uint32_t affine = 0;
  int32_t residual_base = 0, row_stride = 0;
  int32_t jacobian_base[CB200_MAX_PARAMETER_BLOCKS] = {};
  int32_t jacobian_step[CB200_MAX_PARAMETER_BLOCKS] = {};
};

// Sums the per-thread-block cost partials in a fixed order (one block, tree in
// shared memory), adds the m per-chunk costs of a chunked launch, also in a fixed order, and
// writes the total next to the gradient.  Launched with kReduceCostThreads threads; the
// per-thread-block partials are summed by the first 256 of them.
// out[1] = the evaluation status as a double, so that it travels through the same sum over
// the ranks as the cost: every rank then returns the same verdict (a functor failing on one
// rank fails the whole Evaluate, like the CPU evaluator's all-or-nothing contract).
constexpr int kReduceCostThreads = 1024;
__global__ void __launch_bounds__(kReduceCostThreads)
ReduceCostKernel(const double* __restrict__ partials, int n, const double* __restrict__ chunk_costs,
                 int m, double* out, const int32_t* __restrict__ status) {
  __shared__ double sm[256];
  __shared__ double chunk_sm[kReduceCostThreads];
  const int tid = threadIdx.x;
  if (tid < 256) {
    double acc = 0.0;
    for (int i = tid; i < n; i += 256) acc += partials[i];
    sm[tid] = acc;
  }
  // ~30 k chunks on the largest problems: eight loads in flight per thread
  double acc = 0.0;
#pragma unroll 8
  for (int i = tid; i < m; i += kReduceCostThreads) acc += chunk_costs[i];
  chunk_sm[tid] = acc;
  __syncthreads();
  for (int s = kReduceCostThreads / 2; s > 0; s >>= 1) {
    if (tid < s) {
      chunk_sm[tid] += chunk_sm[tid + s];
      if (s < 256) sm[tid] += sm[tid + s];
    }
    __syncthreads();
  }
  if (tid == 0) {
    out[0] = m > 0 ? sm[0] + chunk_sm[0] : sm[0];
    out[1] = *status ? 1.0 : 0.0;
  }
}

// ---- gradient exchange over peer-mapped memory (several ranks on one NVLink domain).
// After a Schur ordering the residual blocks of a point are consecutive, so almost every
// gradient entry is touched by one rank only: the evaluation kernel itself copies those
// into the other ranks' buffers, chunk by chunk (kChunked in evaluate_kernel.cuh).  What is
// left - the entries several ranks add to (the cameras of a bundle adjustment problem, the
// points at rank boundaries), the cost and the status - is about 1 MB and is summed here:
// every rank writes its partial sums into its slot on every rank, raises a flag there, waits
// for the others' flags and adds the slots in rank order, so all ranks end up with the same
// bits.  Flags carry the evaluation's sequence number and are never reset.
constexpr int kMaxRanks = CB200_MAX_PEERS + 1;
constexpr int kMaxSharedIntervals = 32;
struct SharedExchange {
  int32_t world, rank;
  int32_t num_intervals;
  int32_t begin[kMaxSharedIntervals];   // gradient offset of each shared interval
  int32_t start[kMaxSharedIntervals];   // its first slot entry (prefix sum of the lengths)
  int32_t count;                        // slot entries: all intervals + cost + failed
  double* gradient;                     // this rank's [gradient | cost | failed]
  int32_t cost_offset;                  // num_effective
  double* slots[kMaxRanks];             // slots[q]: rank q's staging area [world][count]
  unsigned long long* flags[kMaxRanks]; // flags[q]: rank q's flag array [world]
  unsigned long long epoch;
  unsigned* arrivals;                   // this rank, zero between launches
};

// Copies this rank's exclusive gradient range into the other ranks' buffers (used when the
// evaluation kernel of the call has no chunked variant; otherwise the kernel does it).
struct PeerPush {
  int32_t num_peers;
  int64_t begin, length;
  const double* gradient;
  double* peer[CB200_MAX_PEERS];
};
__global__ void __launch_bounds__(256) PushExclusiveKernel(const PeerPush x) {
  for (int64_t i = blockIdx.x * static_cast<int64_t>(blockDim.x) + threadIdx.x; i < x.length;
       i += static_cast<int64_t>(gridDim.x) * blockDim.x) {
    const double v = __ldcg(x.gradient + x.begin + i);
    for (int q = 0; q < x.num_peers; ++q) __stcg(x.peer[q] + x.begin + i, v);
  }
}

__device__ __forceinline__ int SharedIndexToGradient(const SharedExchange& x, int i) {
  if (i >= x.count - 2) return x.cost_offset + (i - (x.count - 2));
  int k = 0;
  while (k + 1 < x.num_intervals && i >= x.start[k + 1]) ++k;
  return x.begin[k] + (i - x.start[k]);
}

__global__ void __launch_bounds__(256) ExchangeSharedKernel(const SharedExchange x) {
  const int tid = blockIdx.x * blockDim.x + threadIdx.x;
  const int threads = gridDim.x * blockDim.x;
  // (1) this rank's partial sums into its slot on every rank
  for (int i = tid; i < x.count; i += threads) {
    const double v = __ldcg(x.gradient + SharedIndexToGradient(x, i));
    for (int q = 0; q < x.world; ++q)
      __stcg(x.slots[q] + static_cast<size_t>(x.rank) * x.count + i, v);
  }
  // (2) once every thread block has written: raise this rank's flag on every rank
  __shared__ bool last;
  __threadfence_system();
  __syncthreads();
  if (threadIdx.x == 0) last = atomicAdd(x.arrivals, 1u) == gridDim.x - 1;
  __syncthreads();
  if (last) {
    __threadfence_system();
    if (threadIdx.x < x.world) {
      unsigned long long* flag = x.flags[threadIdx.x] + x.rank;
      asm volatile("st.release.sys.global.u64 [%0], %1;" ::"l"(flag), "l"(x.epoch) : "memory");
    }
    if (threadIdx.x == 0) *x.arrivals = 0;
  }
  // (3) wait for every rank's flag (their slots here, and every copy the evaluation kernels
  // of the other ranks made into this rank's gradient, are then complete) ...
  if (threadIdx.x < x.world) {
    const unsigned long long* flag = x.flags[x.rank] + threadIdx.x;
    unsigned long long seen;
    do {
      asm volatile("ld.acquire.sys.global.u64 %0, [%1];" : "=l"(seen) : "l"(flag) : "memory");
    } while (seen < x.epoch);
  }
  __syncthreads();
  // (4) ... and add the slots in rank order
  const double* mine = x.slots[x.rank];
  for (int i = tid; i < x.count; i += threads) {
    double sum = 0.0;
    for (int q = 0; q < x.world; ++q) sum += __ldcg(mine + static_cast<size_t>(q) * x.count + i);
    x.gradient[SharedIndexToGradient(x, i)] = sum;
  }
}

// ---- linear algebra on the device-resident Jacobian (SURVEY.md section 8(f) 1-2).
// The kernels walk the same per-type tables the evaluation kernel writes through:
// block (j, i) of a type is a dense num_residuals x tangent cell at jacobian_pos, row
// stride = tangent (block sparse) or the block's CRS row stride, columns starting at
// delta_offset.  They are bandwidth bound (one pass over the values), so sizes are
// runtime arguments and one instantiation serves every residual-block type.
struct JacobianWalk {
  int32_t n, nb, kres, crs, plain;
  int32_t sizes[CB200_MAX_PARAMETER_BLOCKS];
  const int32_t* doff;     // [nb][n]
  const int32_t* jpos;     // [nb][n]
  const int32_t* pb;       // [nb][n]
  const int32_t* jstride;  // [n]
  const int32_t* respos;   // [n]
  const int32_t* pb_table;
  double* values;
};

__device__ __forceinline__ void RedAddF64(double* address, double value) {
  asm volatile("red.global.add.f64 [%0], %1;" ::"l"(address), "d"(value) : "memory");
}

enum { kOpRight = 0, kOpLeft = 1, kOpColumnNorm = 2, kOpScale = 3, kOpNormal = 4,
       kOpScaleNorm = 5 };  // kOpScaleNorm: kOpScale with x, then kOpColumnNorm into y (one pass
                            // in the per-type kernel, two table walks otherwise)

// One thread per residual block.  x / y meaning per operation:
//   kOpRight:      y[rows] = sum_c J(r, c) x[c]        (y indexed by local residual)
//   kOpLeft:       y[c]   += sum_r J(r, c) x[r]        (atomic; x indexed by local residual)
//   kOpColumnNorm: y[c]   += sum_r J(r, c)^2           (atomic)
//   kOpScale:      J(r, c) *= x[c]
template <int kOp>
__global__ void __launch_bounds__(256) JacobianWalkKernel(const JacobianWalk w,
                                                          const double* __restrict__ x,
                                                          double* __restrict__ y) {
  // Columns are handled in chunks of kChunk with the loads of a chunk issued back to back:
  // a thread's row of a cell is contiguous, so its sectors are requested together and
  // used once, instead of being re-fetched after other warps evicted them.
  constexpr int kChunk = 8;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < w.n; i += gridDim.x * blockDim.x) {
    const int row0 = w.respos[i];
    if (kOp == kOpRight) {
      // rows in groups of kRows accumulators; x is loaded once per column and group
      constexpr int kRows = 8;
      for (int r0 = 0; r0 < w.kres; r0 += kRows) {
        double acc[kRows];
#pragma unroll
        for (int r = 0; r < kRows; ++r) acc[r] = 0.0;
        for (int j = 0; j < w.nb; ++j) {
          const size_t at = static_cast<size_t>(j) * w.n + i;
          const int jp = w.jpos[at];
          if (jp < 0) continue;
          const int col = w.doff[at];
          const int tan = w.plain ? w.sizes[j] : w.pb_table[8 * w.pb[at] + 2];
          const int rs = w.crs ? w.jstride[i] : tan;
          const double* __restrict__ v = w.values + jp + static_cast<size_t>(r0) * rs;
          const double* __restrict__ xs = x + col;
          for (int c0 = 0; c0 < tan; c0 += kChunk) {
            double b[kChunk];
#pragma unroll
            for (int k = 0; k < kChunk; ++k) b[k] = c0 + k < tan ? xs[c0 + k] : 0.0;
#pragma unroll
            for (int r = 0; r < kRows; ++r) {
              if (r0 + r < w.kres) {
                double a[kChunk];
#pragma unroll
                for (int k = 0; k < kChunk; ++k)
                  a[k] = c0 + k < tan ? v[static_cast<size_t>(r) * rs + c0 + k] : 0.0;
#pragma unroll
                for (int k = 0; k < kChunk; ++k) acc[r] = fma(a[k], b[k], acc[r]);
              }
            }
          }
        }
#pragma unroll
        for (int r = 0; r < kRows; ++r)
          if (r0 + r < w.kres) y[row0 + r0 + r] = acc[r];
      }
    } else {
      for (int j = 0; j < w.nb; ++j) {
        const size_t at = static_cast<size_t>(j) * w.n + i;
        const int jp = w.jpos[at];
        if (jp < 0) continue;
        const int col = w.doff[at];
        const int tan = w.plain ? w.sizes[j] : w.pb_table[8 * w.pb[at] + 2];
        const int rs = w.crs ? w.jstride[i] : tan;
        double* v = w.values + jp;
        for (int c0 = 0; c0 < tan; c0 += kChunk) {
          if (kOp == kOpScale) {
            double sc[kChunk];
#pragma unroll
            for (int k = 0; k < kChunk; ++k) sc[k] = c0 + k < tan ? x[col + c0 + k] : 1.0;
            for (int r = 0; r < w.kres; ++r) {
              double* row = v + static_cast<size_t>(r) * rs + c0;
#pragma unroll
              for (int k = 0; k < kChunk; ++k)
                if (c0 + k < tan) row[k] *= sc[k];
            }
          } else {
            double acc[kChunk];
#pragma unroll
            for (int k = 0; k < kChunk; ++k) acc[k] = 0.0;
            for (int r = 0; r < w.kres; ++r) {
              const double* row = v + static_cast<size_t>(r) * rs + c0;
              const double wr = kOp == kOpLeft ? x[row0 + r] : 0.0;
#pragma unroll
              for (int k = 0; k < kChunk; ++k) {
                const double a = c0 + k < tan ? row[k] : 0.0;
                acc[k] = fma(a, kOp == kOpLeft ? wr : a, acc[k]);
              }
            }
#pragma unroll
            for (int k = 0; k < kChunk; ++k)
              if (c0 + k < tan) RedAddF64(y + col + c0 + k, acc[k]);
          }
        }
      }
    }
  }
}


// y += J'(J x) with ONE pass over the values: a residual block's rows of J x stay in
// registers and are multiplied straight back through the same cells (second read from
// cache), so a conjugate-gradient iteration on the normal equations reads the Jacobian once
// instead of twice.  Needs num_residuals <= kNormalRows.
constexpr int kNormalRows = 8;
__global__ void __launch_bounds__(256) JacobianNormalKernel(const JacobianWalk w,
                                                            const double* __restrict__ x,
                                                            double* __restrict__ y) {
  constexpr int kChunk = 8;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < w.n; i += gridDim.x * blockDim.x) {
    double wr[kNormalRows];
#pragma unroll
    for (int r = 0; r < kNormalRows; ++r) wr[r] = 0.0;
    for (int j = 0; j < w.nb; ++j) {
      const size_t at = static_cast<size_t>(j) * w.n + i;
      const int jp = w.jpos[at];
      if (jp < 0) continue;
      const int tan = w.plain ? w.sizes[j] : w.pb_table[8 * w.pb[at] + 2];
      const int rs = w.crs ? w.jstride[i] : tan;
      const double* __restrict__ v = w.values + jp;
      const double* __restrict__ xs = x + w.doff[at];
      for (int c0 = 0; c0 < tan; c0 += kChunk) {
        double b[kChunk];
#pragma unroll
        for (int k = 0; k < kChunk; ++k) b[k] = c0 + k < tan ? xs[c0 + k] : 0.0;
#pragma unroll
        for (int r = 0; r < kNormalRows; ++r) {
          if (r < w.kres) {
            double a[kChunk];
#pragma unroll
            for (int k = 0; k < kChunk; ++k)
              a[k] = c0 + k < tan ? v[static_cast<size_t>(r) * rs + c0 + k] : 0.0;
#pragma unroll
            for (int k = 0; k < kChunk; ++k) wr[r] = fma(a[k], b[k], wr[r]);
          }
        }
      }
    }
    for (int j = 0; j < w.nb; ++j) {
      const size_t at = static_cast<size_t>(j) * w.n + i;
      const int jp = w.jpos[at];
      if (jp < 0) continue;
      const int col = w.doff[at];
      const int tan = w.plain ? w.sizes[j] : w.pb_table[8 * w.pb[at] + 2];
      const int rs = w.crs ? w.jstride[i] : tan;
      const double* __restrict__ v = w.values + jp;
      for (int c0 = 0; c0 < tan; c0 += kChunk) {
        double acc[kChunk];
#pragma unroll
        for (int k = 0; k < kChunk; ++k) acc[k] = 0.0;
#pragma unroll
        for (int r = 0; r < kNormalRows; ++r) {
          if (r < w.kres) {
#pragma unroll
            for (int k = 0; k < kChunk; ++k) {
              const double a = c0 + k < tan ? v[static_cast<size_t>(r) * rs + c0 + k] : 0.0;
              acc[k] = fma(a, wr[r], acc[k]);
            }
          }
        }
#pragma unroll
        for (int k = 0; k < kChunk; ++k)
          if (c0 + k < tan) RedAddF64(y + col + c0 + k, acc[k]);
      }
    }
  }
}

// Same operation with the values staged through shared memory.  In the block-sparse layout
// the cells of a warp's 32 consecutive residual blocks are one contiguous run per argument
// (block_jacobian_writer.cc:62-150), so the warp copies the run as it lies in memory with
// 16-byte cp.async (two cache lines per instruction instead of 32) and every thread then
// reads its own cell from shared memory, for both passes.  Arguments whose run is not
// contiguous / aligned (constant blocks, the ragged last tile) are read from global memory
// as in the kernel above.
constexpr int kNormalThreads = 128;
__device__ __forceinline__ void CopyAsync16(void* smem, const void* gmem) {
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(
                   static_cast<unsigned>(__cvta_generic_to_shared(smem))),
               "l"(gmem)
               : "memory");
}
__global__ void __launch_bounds__(kNormalThreads) JacobianNormalStagedKernel(
    const JacobianWalk w, const double* __restrict__ x, double* __restrict__ y,
    int cell_doubles_per_block) {
  extern __shared__ double2 normal_smem[];
  constexpr int kChunk = 8;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  double* const stage = reinterpret_cast<double*>(normal_smem) + warp * 32 * cell_doubles_per_block;
  for (int i0 = (blockIdx.x * (kNormalThreads / 32) + warp) * 32; i0 < w.n;
       i0 += gridDim.x * kNormalThreads) {
    const bool full = i0 + 32 <= w.n;
    const bool valid = i0 + lane < w.n;
    const int i = valid ? i0 + lane : w.n - 1;
    // ---- stage the contiguous runs
    unsigned staged = 0u;
    int offset = 0;  // doubles, per warp
    for (int j = 0; j < w.nb; ++j) {
      const size_t at = static_cast<size_t>(j) * w.n + i;
      const int jp = w.jpos[at];
      const int tan = w.plain ? w.sizes[j] : w.pb_table[8 * w.pb[at] + 2];
      const int jp0 = __shfl_sync(0xffffffffu, jp, 0);
      const int tan0 = __shfl_sync(0xffffffffu, tan, 0);
      const int cs = w.kres * tan0;
      const bool ok = full && jp0 >= 0 && (jp0 & 1) == 0 && tan == tan0 && jp == jp0 + lane * cs &&
                      tan0 <= w.sizes[j];
      if (__all_sync(0xffffffffu, ok)) {
        const double2* src = reinterpret_cast<const double2*>(w.values + jp0);
        double2* dst = reinterpret_cast<double2*>(stage + offset);
        for (int k = lane; k < 16 * cs; k += 32) CopyAsync16(dst + k, src + k);
        staged |= 1u << j;
      }
      offset += 32 * w.kres * w.sizes[j];
    }
    asm volatile("cp.async.wait_all;" ::: "memory");
    __syncwarp();

    double wr[kNormalRows];
#pragma unroll
    for (int r = 0; r < kNormalRows; ++r) wr[r] = 0.0;
    if (valid) {
      offset = 0;
      for (int j = 0; j < w.nb; ++j) {
        const size_t at = static_cast<size_t>(j) * w.n + i;
        const int jp = w.jpos[at];
        const int tan = w.plain ? w.sizes[j] : w.pb_table[8 * w.pb[at] + 2];
        const double* v =
            ((staged >> j) & 1u) ? stage + offset + lane * w.kres * tan : w.values + jp;
        offset += 32 * w.kres * w.sizes[j];
        if (jp < 0) continue;
        const double* __restrict__ xs = x + w.doff[at];
        for (int c0 = 0; c0 < tan; c0 += kChunk) {
          double b[kChunk];
#pragma unroll
          for (int k = 0; k < kChunk; ++k) b[k] = c0 + k < tan ? xs[c0 + k] : 0.0;
#pragma unroll
          for (int r = 0; r < kNormalRows; ++r) {
            if (r < w.kres) {
#pragma unroll
              for (int k = 0; k < kChunk; ++k)
                wr[r] = fma(c0 + k < tan ? v[r * tan + c0 + k] : 0.0, b[k], wr[r]);
            }
          }
        }
      }
      offset = 0;
      for (int j = 0; j < w.nb; ++j) {
        const size_t at = static_cast<size_t>(j) * w.n + i;
        const int jp = w.jpos[at];
        const int tan = w.plain ? w.sizes[j] : w.pb_table[8 * w.pb[at] + 2];
        const double* v =
            ((staged >> j) & 1u) ? stage + offset + lane * w.kres * tan : w.values + jp;
        offset += 32 * w.kres * w.sizes[j];
        if (jp < 0) continue;
        const int col = w.doff[at];
        const bool in_smem = (staged >> j) & 1u;
        double* sums = stage + (offset - 32 * w.kres * w.sizes[j]) + lane * w.kres * tan;
        for (int c0 = 0; c0 < tan; c0 += kChunk) {
          double acc[kChunk];
#pragma unroll
          for (int k = 0; k < kChunk; ++k) acc[k] = 0.0;
#pragma unroll
          for (int r = 0; r < kNormalRows; ++r) {
            if (r < w.kres) {
#pragma unroll
              for (int k = 0; k < kChunk; ++k)
                acc[k] = fma(c0 + k < tan ? v[r * tan + c0 + k] : 0.0, wr[r], acc[k]);
            }
          }
          if (in_smem) {
            // columns c0.. of the cell are not read again: its first row takes their sums
            // for the warp-wide scatter below
#pragma unroll
            for (int k = 0; k < kChunk; ++k)
              if (c0 + k < tan) sums[c0 + k] = acc[k];
          } else {
#pragma unroll
            for (int k = 0; k < kChunk; ++k)
              if (c0 + k < tan) RedAddF64(y + col + c0 + k, acc[k]);
          }
        }
      }
    }
    // ---- staged arguments: the sums leave by runs, consecutive
    // lanes adding to consecutive addresses of a parameter block (a red instruction then
    // touches a few sectors instead of 32)
    if (staged) {
      __syncwarp();
      int offset2 = 0;
      for (int j = 0; j < w.nb; ++j) {
        const size_t at = static_cast<size_t>(j) * w.n + i;
        const int tan = w.plain ? w.sizes[j] : w.pb_table[8 * w.pb[at] + 2];
        const int col = w.doff[at];
        const int base = offset2;
        offset2 += 32 * w.kres * w.sizes[j];
        if (!((staged >> j) & 1u)) continue;  // warp-uniform, and so is tan when staged
        const int cs = w.kres * tan;
        const unsigned magic = tan == 1 ? 0u : 0xffffffffu / static_cast<unsigned>(tan) + 1u;
        for (int k = 0; k < tan; ++k) {
          const int e = k * 32 + lane;
          const int owner = magic ? static_cast<int>(__umulhi(static_cast<unsigned>(e), magic)) : e;
          const int c = e - owner * tan;
          const int ocol = __shfl_sync(0xffffffffu, col, owner);
          RedAddF64(y + ocol + c, stage[base + owner * cs + c]);
        }
      }
    }
    __syncwarp();  // the next tile overwrites the staging area
  }
}

// Conjugate-gradient vector kernels.  S is a small array of device scalars:
enum { kSRho = 0, kSLastRho, kSPq, kSRnorm2, kSXbr, kSJyB, kSJy2, kSCount };

__device__ __forceinline__ double BlockSum(double v) {
  __shared__ double sm[8];
  for (int o = 16; o > 0; o >>= 1) v += __shfl_down_sync(0xffffffffu, v, o);
  __syncthreads();
  if ((threadIdx.x & 31) == 0) sm[threadIdx.x >> 5] = v;
  __syncthreads();
  v = threadIdx.x < 8 ? sm[threadIdx.x] : 0.0;
  if (threadIdx.x < 32)
    for (int o = 4; o > 0; o >>= 1) v += __shfl_down_sync(0xffffffffu, v, o);
  return v;  // valid in thread 0
}

// Reproducible grid-wide sums: every thread block writes its partial sums, the last block to
// arrive adds them in a fixed order.  The conjugate-gradient scalars are then bit-identical
// run to run and, because every rank holds identical vectors, rank to rank: all ranks take
// the same termination decision and issue the same number of collectives.
struct ScalarReduce {
  double* partials;    // [gridDim.x][3]
  unsigned* arrivals;  // zero between kernels
};
template <int kCount>
__device__ __forceinline__ void FinishScalars(const ScalarReduce red, const double (&v)[kCount],
                                              double* S, const int (&slot)[kCount]) {
  __shared__ bool last;
  if (threadIdx.x == 0) {
#pragma unroll
    for (int k = 0; k < kCount; ++k) red.partials[blockIdx.x * 3 + k] = v[k];
    __threadfence();
    last = atomicAdd(red.arrivals, 1u) == gridDim.x - 1;
  }
  __syncthreads();
  if (!last) return;
  __threadfence();
#pragma unroll
  for (int k = 0; k < kCount; ++k) {
    double acc = 0.0;
    for (int b = threadIdx.x; b < gridDim.x; b += blockDim.x)
      acc += __ldcg(red.partials + b * 3 + k);
    acc = BlockSum(acc);
    if (threadIdx.x == 0) S[slot[k]] = acc;
  }
  if (threadIdx.x == 0) *red.arrivals = 0;
}

// minv = 1 / (colnorm + d2);  r = b;  z = minv r;  p = z;  x = 0;  rho = r.z;  rnorm2 = r.r
__global__ void __launch_bounds__(256) CgInitKernel(int n, const double* __restrict__ colnorm,
                                                    const double* __restrict__ d2,
                                                    const double* __restrict__ b, double* minv,
                                                    double* r, double* p, double* x, double* S,
                                                    const ScalarReduce red) {
  double rho = 0.0, rr = 0.0;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
    const double m = 1.0 / (colnorm[i] + (d2 ? d2[i] : 0.0));
    const double ri = b[i], zi = (isfinite(m) ? m : 1.0) * ri;
    minv[i] = isfinite(m) ? m : 1.0;
    r[i] = ri;
    p[i] = zi;
    x[i] = 0.0;
    rho += ri * zi;
    rr += ri * ri;
  }
  const double v[2] = {BlockSum(rho), BlockSum(rr)};
  const int slot[2] = {kSRho, kSRnorm2};
  FinishScalars<2>(red, v, S, slot);
}

// pq = p.(q + d2 p)
__global__ void __launch_bounds__(256) CgDotKernel(int n, const double* __restrict__ p,
                                                   const double* __restrict__ q,
                                                   const double* __restrict__ d2, double* S,
                                                   const ScalarReduce red) {
  double acc = 0.0;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x)
    acc += p[i] * (q[i] + (d2 ? d2[i] : 0.0) * p[i]);
  const double v[1] = {BlockSum(acc)};
  const int slot[1] = {kSPq};
  FinishScalars<1>(red, v, S, slot);
}

// alpha = rho / pq;  x += alpha p;  r -= alpha (q + d2 p);  accumulates the next rho = r.(minv r),
// |r|^2 and x.(b + r) into Snext
__global__ void __launch_bounds__(256) CgUpdateKernel(int n, const double* __restrict__ p,
                                                      const double* __restrict__ q,
                                                      const double* __restrict__ d2,
                                                      const double* __restrict__ minv,
                                                      const double* __restrict__ b, double* x,
                                                      double* r, const double* S, double* Snext,
                                                      const ScalarReduce red) {
  const double alpha = S[kSRho] / S[kSPq];
  double rho = 0.0, rr = 0.0, xbr = 0.0;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
    const double pi = p[i];
    const double xi = x[i] + alpha * pi;
    const double ri = r[i] - alpha * (q[i] + (d2 ? d2[i] : 0.0) * pi);
    x[i] = xi;
    r[i] = ri;
    rho += ri * ri * minv[i];
    rr += ri * ri;
    xbr += xi * (b[i] + ri);
  }
  const double v[3] = {BlockSum(rho), BlockSum(rr), BlockSum(xbr)};
  const int slot[3] = {kSRho, kSRnorm2, kSXbr};
  FinishScalars<3>(red, v, Snext, slot);
}

// p = minv r + (rho_next / rho) p
__global__ void __launch_bounds__(256) CgDirectionKernel(int n, const double* __restrict__ r,
                                                         const double* __restrict__ minv,
                                                         double* p, const double* S,
                                                         const double* Snext) {
  const double beta = Snext[kSRho] / S[kSRho];
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x)
    p[i] = minv[i] * r[i] + beta * p[i];
}

// jy.b and |jy|^2 over this rank's residuals
__global__ void __launch_bounds__(256) CgModelKernel(int n, const double* __restrict__ jy,
                                                     const double* __restrict__ b, double* S,
                                                     const ScalarReduce red) {
  double d = 0.0, s = 0.0;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
    d += jy[i] * b[i];
    s += jy[i] * jy[i];
  }
  const double v[2] = {BlockSum(d), BlockSum(s)};
  const int slot[2] = {kSJyB, kSJy2};
  FinishScalars<2>(red, v, S, slot);
}

// ---- trust-region vector kernels (state, step and diagonals resident in HBM)
__global__ void __launch_bounds__(256) JacobiScaleKernel(int n, const double* __restrict__ colnorm,
                                                         double* __restrict__ scale) {
  // trust_region_minimizer.cc:259-275: 1 / (1 + sqrt(column norm^2))
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x)
    scale[i] = 1.0 / (1.0 + sqrt(colnorm[i]));
}
__global__ void __launch_bounds__(256) ClampKernel(int n, const double* __restrict__ in, double lo,
                                                   double hi, double* __restrict__ out) {
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x)
    out[i] = fmin(fmax(in[i], lo), hi);
}
__global__ void __launch_bounds__(256) DivideKernel(int n, const double* __restrict__ in,
                                                    double divisor, double* __restrict__ out) {
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x)
    out[i] = in[i] / divisor;
}
// delta = -y * scale;  S[0] = |delta|^2
__global__ void __launch_bounds__(256) StepKernel(int n, const double* __restrict__ y,
                                                  const double* __restrict__ scale,
                                                  double* __restrict__ delta, double* S,
                                                  const ScalarReduce red) {
  double acc = 0.0;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
    const double d = -y[i] * (scale ? scale[i] : 1.0);
    delta[i] = d;
    acc += d * d;
  }
  const double v[1] = {BlockSum(acc)};
  const int slot[1] = {0};
  FinishScalars<1>(red, v, S, slot);
}
__global__ void __launch_bounds__(256) SquaredNormKernel(int n, const double* __restrict__ x,
                                                         double* S, const ScalarReduce red) {
  double acc = 0.0;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x)
    acc += x[i] * x[i];
  const double v[1] = {BlockSum(acc)};
  const int slot[1] = {0};
  FinishScalars<1>(red, v, S, slot);
}
// max |g|: non-negative doubles order like their bit patterns
__global__ void __launch_bounds__(256) MaxAbsKernel(int n, const double* __restrict__ g,
                                                    unsigned long long* out) {
  double m = 0.0;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x)
    m = fmax(m, fabs(g[i]));
  for (int o = 16; o > 0; o >>= 1) m = fmax(m, __shfl_down_sync(0xffffffffu, m, o));
  if ((threadIdx.x & 31) == 0) atomicMax(out, static_cast<unsigned long long>(__double_as_longlong(m)));
}

// Program::Plus (internal/ceres/program.cc:121-150): one thread per parameter block applies
// x (+) delta for the manifolds the device knows (ceres/manifold.h of this repository:
// SubsetManifold, (Eigen)QuaternionManifold and their products with Euclidean factors,
// internal/ceres/manifold.cc:28-58,184-197).
__device__ __forceinline__ void QuaternionPlusDevice(const double* x, const double* d, double* out,
                                                     int kW, int kX, int kY, int kZ) {
  const double norm = sqrt(d[0] * d[0] + d[1] * d[1] + d[2] * d[2]);
  if (norm == 0.0) {
    for (int i = 0; i < 4; ++i) out[i] = x[i];
    return;
  }
  const double k = sin(norm) / norm;
  const double qw = cos(norm), qx = k * d[0], qy = k * d[1], qz = k * d[2];
  const double xw = x[kW], xx = x[kX], xy = x[kY], xz = x[kZ];
  out[kW] = qw * xw - qx * xx - qy * xy - qz * xz;
  out[kX] = qw * xx + qx * xw + qy * xz - qz * xy;
  out[kY] = qw * xy - qx * xz + qy * xw + qz * xx;
  out[kZ] = qw * xz + qx * xy - qy * xx + qz * xw;
}
__global__ void __launch_bounds__(256) PlusKernel(int num_blocks, const int32_t* __restrict__ table,
                                                  const double* __restrict__ state,
                                                  const double* __restrict__ delta,
                                                  double* __restrict__ out, int32_t* status) {
  for (int b = blockIdx.x * blockDim.x + threadIdx.x; b < num_blocks;
       b += gridDim.x * blockDim.x) {
    const int4 r0 = __ldg(reinterpret_cast<const int4*>(table) + 2 * b);
    const int4 r1 = __ldg(reinterpret_cast<const int4*>(table) + 2 * b + 1);
    const int soff = r0.x, doff = r0.y, kind = r0.w, mparam = r1.x, size = r1.z;
    const double* x = state + soff;
    const double* d = delta + doff;
    double* o = out + soff;
    if (doff < 0) {  // constant block inside the program: unchanged
      for (int i = 0; i < size; ++i) o[i] = x[i];
    } else if (kind == CB200_MANIFOLD_NONE) {
      for (int i = 0; i < size; ++i) o[i] = x[i] + d[i];
    } else if (kind == CB200_MANIFOLD_SUBSET) {
      int j = 0;
      for (int i = 0; i < size; ++i) o[i] = ((mparam >> i) & 1) ? x[i] : x[i] + d[j++];
    } else if (kind == CB200_MANIFOLD_QUATERNION_TAIL) {
      QuaternionPlusDevice(x, d, o, 0, 1, 2, 3);
      for (int i = 4; i < size; ++i) o[i] = x[i] + d[i - 1];
    } else if (kind == CB200_MANIFOLD_EIGEN_QUATERNION_TAIL) {
      QuaternionPlusDevice(x, d, o, 3, 0, 1, 2);
      for (int i = 4; i < size; ++i) o[i] = x[i] + d[i - 1];
    } else {
      *status = 1;
    }
  }
}

}  // namespace

struct cb200_engine {
  int device = 0;
  cudaStream_t stream = nullptr;
  cudaEvent_t ev[5] = {};
  std::string error;
  bool finalized = false;
  bool planning = false;  // CB200_PLANNING_ONLY: no device, structure only

  // parameter blocks
  int32_t num_active = 0, num_constant = 0, num_parameters = 0, num_effective = 0;
  int32_t num_constant_parameters = 0, plus_pool = 0;
  std::vector<cb200_parameter_block> blocks;
  std::vector<double> constant_state;

  // layout
  int32_t jacobian_format = 0, num_rb = 0, num_residuals = 0;
  std::vector<int32_t> residual_layout, jprl, jpro;
  int64_t num_jacobian_values = 0;

  // shard
  int32_t rank = 0, world = 1;
  int32_t rb_begin = 0, rb_end = 0, res_begin = 0, res_end = 0;
  std::vector<Segment> segments;
  int64_t local_jacobian_values = 0;
  // Gradient exchange plan (empty = one all-reduce over [gradient | cost | failed]).
  std::vector<GradientInterval> exchange;
  // Peer exchange (cb200_engine_comm_init sets it up when the plan allows): chunks of this
  // rank's residual blocks with their exclusive gradient ranges, the shared intervals, and a
  // peer-mapped region [2 x gradient | 2 x world slots | flags] on every rank.
  std::vector<int32_t> chunk_table;        // 4 ints per chunk, see cb200_launch_args::chunks
  DeviceBuffer<int32_t> d_chunks;
  int64_t exclusive_begin = 0, exclusive_length = 0;  // this rank's exclusive gradient range
  bool peer_plan = false;                  // the structure allows the peer exchange
  bool peer_ready = false;                 // ... and the region is mapped on every rank
  char* peer_region = nullptr;             // this rank's allocation
  void* peer_base[kMaxRanks] = {};         // every rank's region (own at [rank])
  size_t peer_gradient_stride = 0, peer_slots_offset = 0, peer_flags_offset = 0;  // bytes
  int32_t shared_count = 0;
  unsigned long long epoch = 0;
  DeviceBuffer<unsigned> d_arrivals;
  double* gradcost = nullptr;              // [gradient | cost | failed] of the current evaluation

  std::vector<ResidualType*> types;

  DeviceBuffer<double> d_state, d_plus, d_residuals, d_jacobian, d_gradcost, d_cost_partials;
  DeviceBuffer<int32_t> d_pb_table, d_status;
  int32_t total_cost_partials = 0;
  int32_t chunk_cost_capacity = 0;  // per-chunk cost slots, after the total_cost_partials ones

  // pinned scalars: [cost, status]
  double* h_scalars = nullptr;

  // device-resident Jacobian linear algebra: which outputs of the last evaluation are
  // on the device, and the conjugate-gradient work vectors (allocated on first use)
  bool jacobian_resident = false, residuals_resident = false;
  DeviceBuffer<double> la_col[8];   // x-like: num_effective + 1 each
  DeviceBuffer<double> la_row;      // residual-like: this rank's residuals
  DeviceBuffer<double> la_scalars;  // 3 x kSCount
  DeviceBuffer<double> la_partials; // per-thread-block partial sums of the scalar reductions
  DeviceBuffer<unsigned> la_arrivals;
  double* h_la_scalars = nullptr;   // pinned, 3 x kSCount
  // trust-region state resident in HBM: accepted state and candidate, Jacobi scale, LM
  // diagonal, step
  DeviceBuffer<double> tr_state[2], tr_scale, tr_diagonal, tr_delta;
  bool tr_state_valid = false, tr_scale_valid = false, tr_diagonal_valid = false;
  // la_col[7] holds the squared column norms of the Jacobian as it stands (after the Jacobi
  // scaling): computed once per evaluation - by the scaling pass itself where the per-type
  // kernel runs - and shared by the LM diagonal and the conjugate-gradient preconditioner.
  bool colnorm_valid = false;
  bool plus_on_device = true;       // every manifold of the program is one PlusKernel knows

  void* comm = nullptr;
  double timing[4] = {0, 0, 0, 0};

  int Fail(int code, const char* fmt, ...) {
    char buf[512];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof(buf), fmt, ap);
    va_end(ap);
    error = buf;
    return code;
  }
};

#define CB200_CUDA(e, call)                                                            \
  do {                                                                                 \
    cudaError_t err__ = (call);                                                        \
    if (err__ != cudaSuccess)                                                          \
      return (e)->Fail(CB200_ERROR_CUDA, "%s: %s", #call, cudaGetErrorString(err__));  \
  } while (0)

namespace {
// NVTX range over one C-ABI call (Nsight Systems / Compute timelines: SURVEY.md section 5).
struct NvtxRange {
  explicit NvtxRange(const char* name) { nvtxRangePushA(name); }
  ~NvtxRange() { nvtxRangePop(); }
};
}  // namespace

extern "C" {

const char* cb200_version(void) { return "ceres_b200 0.1 (sm_100a)"; }

int cb200_engine_create(int device, cb200_engine** out) {
  if (!out) return CB200_ERROR_INVALID_ARGUMENT;
  *out = nullptr;
  if (device == CB200_PLANNING_ONLY) {
    // Structure planning without a device: finalize computes this rank's residual
    // block range and Jacobian segments (cb200_engine_shard_info); evaluate fails.
    auto* planner = new cb200_engine;
    planner->device = device;
    planner->planning = true;
    *out = planner;
    return CB200_OK;
  }
  int count = 0;
  if (cudaGetDeviceCount(&count) != cudaSuccess || device < 0 || device >= count) {
    return CB200_ERROR_CUDA;  // fail loudly: there is no CPU fallback
  }
  auto* e = new cb200_engine;
  e->device = device;
  if (cudaSetDevice(device) != cudaSuccess ||
      cudaStreamCreateWithFlags(&e->stream, cudaStreamNonBlocking) != cudaSuccess) {
    delete e;
    return CB200_ERROR_CUDA;
  }
  for (auto& ev : e->ev) cudaEventCreate(&ev);
  cudaHostAlloc(reinterpret_cast<void**>(&e->h_scalars), 4 * sizeof(double), cudaHostAllocDefault);
  *out = e;
  return CB200_OK;
}

void cb200_engine_destroy(cb200_engine* e) {
  if (!e) return;
  if (e->planning) {
    for (auto* t : e->types) delete t;
    delete e;
    return;
  }
  cudaSetDevice(e->device);
  if (e->stream) cudaStreamSynchronize(e->stream);
  if (e->comm) {
    if (NcclApi* n = GetNccl()) n->CommDestroy(e->comm);
  }
  for (auto* t : e->types) {
    t->d_functors.Free(); t->d_loss_table.Free(); t->d_loss_index.Free(); t->d_pb.Free();
    t->d_jpos.Free(); t->d_jstride.Free(); t->d_respos.Free(); t->d_soff.Free(); t->d_doff.Free();
    delete t;
  }
  for (auto& b : e->la_col) b.Free();
  e->la_row.Free(); e->la_scalars.Free(); e->la_partials.Free(); e->la_arrivals.Free();
  for (auto& b : e->tr_state) b.Free();
  e->tr_scale.Free(); e->tr_diagonal.Free(); e->tr_delta.Free();
  if (e->h_la_scalars) cudaFreeHost(e->h_la_scalars);
  e->d_chunks.Free(); e->d_arrivals.Free();
  for (int r = 0; r < kMaxRanks; ++r)
    if (e->peer_base[r] && r != e->rank) cudaIpcCloseMemHandle(e->peer_base[r]);
  if (e->peer_region) cudaFree(e->peer_region);
  e->d_state.Free(); e->d_plus.Free(); e->d_residuals.Free(); e->d_jacobian.Free();
  e->d_gradcost.Free(); e->d_cost_partials.Free(); e->d_pb_table.Free(); e->d_status.Free();
  if (e->h_scalars) cudaFreeHost(e->h_scalars);
  for (auto& ev : e->ev) if (ev) cudaEventDestroy(ev);
  if (e->stream) cudaStreamDestroy(e->stream);
  delete e;
}

const char* cb200_engine_last_error(const cb200_engine* e) { return e ? e->error.c_str() : ""; }

int cb200_engine_set_parameter_blocks(cb200_engine* e, int32_t num_active, int32_t num_constant,
                                      const cb200_parameter_block* blocks, int32_t num_parameters,
                                      int32_t num_effective_parameters,
                                      const double* constant_state,
                                      int32_t num_constant_parameters,
                                      int32_t plus_jacobian_pool_size) {
  if (!e || e->finalized || num_active < 0 || num_constant < 0 ||
      (!blocks && num_active + num_constant > 0))
    return e ? e->Fail(CB200_ERROR_INVALID_ARGUMENT, "set_parameter_blocks: bad arguments")
             : CB200_ERROR_INVALID_ARGUMENT;
  e->num_active = num_active;
  e->num_constant = num_constant;
  e->num_parameters = num_parameters;
  e->num_effective = num_effective_parameters;
  e->num_constant_parameters = num_constant_parameters;
  e->plus_pool = plus_jacobian_pool_size;
  e->blocks.assign(blocks, blocks + num_active + num_constant);
  e->constant_state.assign(constant_state, constant_state + num_constant_parameters);
  return CB200_OK;
}

int cb200_engine_add_residual_blocks(cb200_engine* e, const cb200_residual_type* type, int32_t n,
                                     const int32_t* program_position,
                                     const int32_t* parameter_block_ids, const void* functors,
                                     const void* loss_table, int32_t num_losses,
                                     const int32_t* loss_index) {
  if (!e || e->finalized || !type || !type->launch || n < 0 || num_losses < 1 ||
      type->num_parameter_blocks < 1 || type->num_parameter_blocks > CB200_MAX_PARAMETER_BLOCKS)
    return e ? e->Fail(CB200_ERROR_INVALID_ARGUMENT, "add_residual_blocks: bad arguments")
             : CB200_ERROR_INVALID_ARGUMENT;
  if (num_losses > 1 && !loss_index)
    return e->Fail(CB200_ERROR_INVALID_ARGUMENT, "add_residual_blocks: loss_index required");
  auto* t = new ResidualType;
  t->desc = *type;
  const int nb = type->num_parameter_blocks;
  t->position.assign(program_position, program_position + n);
  t->pb_ids.assign(parameter_block_ids, parameter_block_ids + static_cast<size_t>(n) * nb);
  const char* f = static_cast<const char*>(functors);
  t->functors.assign(f, f + static_cast<size_t>(n) * type->functor_size);
  const char* l = static_cast<const char*>(loss_table);
  t->loss_table.assign(l, l + static_cast<size_t>(num_losses) * type->loss_size);
  t->num_losses = num_losses;
  if (num_losses > 1) t->loss_index.assign(loss_index, loss_index + n);
  e->types.push_back(t);
  return CB200_OK;
}

int cb200_engine_set_layout(cb200_engine* e, int32_t jacobian_format, int32_t num_residual_blocks,
                            int32_t num_residuals, const int32_t* residual_layout,
                            const int32_t* jacobian_per_residual_layout,
                            const int32_t* jacobian_per_residual_offsets, int64_t num_offsets,
                            int64_t num_jacobian_values) {
  if (!e || e->finalized || num_residual_blocks < 0 ||
      (jacobian_format != CB200_JACOBIAN_BLOCK_SPARSE &&
       jacobian_format != CB200_JACOBIAN_COMPRESSED_ROW))
    return e ? e->Fail(CB200_ERROR_INVALID_ARGUMENT, "set_layout: bad arguments")
             : CB200_ERROR_INVALID_ARGUMENT;
  e->jacobian_format = jacobian_format;
  e->num_rb = num_residual_blocks;
  e->num_residuals = num_residuals;
  e->residual_layout.assign(residual_layout, residual_layout + num_residual_blocks);
  e->jprl.assign(jacobian_per_residual_layout, jacobian_per_residual_layout + num_residual_blocks);
  e->jpro.assign(jacobian_per_residual_offsets, jacobian_per_residual_offsets + num_offsets);
  e->num_jacobian_values = num_jacobian_values;
  return CB200_OK;
}

int cb200_engine_set_shard(cb200_engine* e, int32_t rank, int32_t world_size) {
  if (!e || e->finalized || world_size < 1 || rank < 0 || rank >= world_size)
    return e ? e->Fail(CB200_ERROR_INVALID_ARGUMENT, "set_shard: bad arguments")
             : CB200_ERROR_INVALID_ARGUMENT;
  e->rank = rank;
  e->world = world_size;
  return CB200_OK;
}

// Chunk walk instead of the grid stride for large types (measured on B200, BAL L: 1.774 ms with
// chunks of 992 blocks against 1.813 ms; chunks must stay >= ~16 per warp of the persistent
// grid - 148 SMs x 12 warps - or the tail costs more than the walk gains).
constexpr int32_t kUniformChunkBlocks = 992;
constexpr int32_t kUniformChunkMinBlocks = 16 * 148 * 12 * 512;

int cb200_engine_finalize(cb200_engine* e) {
  NvtxRange nvtx_range("cb200_engine_finalize");
  if (!e || e->finalized) return CB200_ERROR_INVALID_ARGUMENT;
  if (!e->planning) CB200_CUDA(e, cudaSetDevice(e->device));
  const int64_t nrb = e->num_rb;
  e->rb_begin = static_cast<int32_t>(nrb * e->rank / e->world);
  e->rb_end = static_cast<int32_t>(nrb * (e->rank + 1) / e->world);
  e->res_begin = e->rb_begin < nrb ? e->residual_layout[e->rb_begin] : e->num_residuals;
  e->res_end = e->rb_end < nrb ? e->residual_layout[e->rb_end] : e->num_residuals;

  // Device parameter-block table (8 ints per block, read as two int4).
  const int npb = e->num_active + e->num_constant;
  std::vector<int32_t> table(static_cast<size_t>(npb) * 8, 0);
  for (int i = 0; i < npb; ++i) {
    const cb200_parameter_block& b = e->blocks[i];
    const bool constant = i >= e->num_active;
    table[8 * i + 0] = constant ? e->num_parameters + b.state_offset : b.state_offset;
    table[8 * i + 1] = constant ? -1 : b.delta_offset;
    table[8 * i + 2] = b.tangent_size;
    table[8 * i + 3] = constant ? CB200_MANIFOLD_NONE : b.manifold_kind;
    table[8 * i + 4] = b.manifold_param;
    table[8 * i + 5] = constant ? -1 : b.plus_jacobian_offset;
    table[8 * i + 6] = b.size;
    if (!constant && b.manifold_kind == CB200_MANIFOLD_GENERIC) e->plus_on_device = false;
  }

  // Gradient exchange plan.  After a Schur ordering the residual blocks of one point
  // are consecutive, so all but a handful of gradient entries are touched by a single
  // rank: those need no reduction, only distribution.  Every rank sees the whole
  // problem here, so all ranks derive the same plan without communicating.
  e->exchange.clear();
  e->chunk_table.clear();
  e->peer_plan = false;
  if (e->world > 1 && e->num_active > 0) {
    std::vector<int32_t> bound(e->world + 1);
    for (int r = 0; r <= e->world; ++r) bound[r] = static_cast<int32_t>(nrb * r / e->world);
    std::vector<int16_t> lo(e->num_active, INT16_MAX), hi(e->num_active, -1);
    // first / last program position of the residual blocks that touch each parameter block
    std::vector<int32_t> first(e->num_active, INT32_MAX), last(e->num_active, -1);
    bool in_program_order = e->types.size() == 1;
    for (ResidualType* t : e->types) {
      const int nb = t->desc.num_parameter_blocks;
      for (size_t k = 0; k < t->position.size(); ++k) {
        const int32_t p = t->position[k];
        if (p < 0 || p >= nrb) continue;  // reported below
        if (p != static_cast<int32_t>(k)) in_program_order = false;
        int r = static_cast<int>(static_cast<int64_t>(p) * e->world / std::max<int64_t>(nrb, 1));
        while (r > 0 && p < bound[r]) --r;
        while (r + 1 < e->world && p >= bound[r + 1]) ++r;
        for (int j = 0; j < nb; ++j) {
          const int32_t id = t->pb_ids[k * nb + j];
          if (id < 0 || id >= e->num_active) continue;
          lo[id] = std::min<int16_t>(lo[id], static_cast<int16_t>(r));
          hi[id] = std::max<int16_t>(hi[id], static_cast<int16_t>(r));
          first[id] = std::min(first[id], p);
          last[id] = std::max(last[id], p);
        }
      }
    }
    // Active blocks are in delta_offset order: merge neighbours of the same class.
    std::vector<GradientInterval> plan;
    for (int i = 0; i < e->num_active; ++i) {
      const cb200_parameter_block& b = e->blocks[i];
      if (b.tangent_size == 0) continue;
      int32_t owner = hi[i] < 0 ? 0 : (lo[i] == hi[i] ? lo[i] : -1);  // untouched: zeros from rank 0
      if (!plan.empty() && plan.back().owner == owner &&
          plan.back().begin + plan.back().length == b.delta_offset) {
        plan.back().length += b.tangent_size;
      } else if (!plan.empty() && hi[i] < 0 &&
                 plan.back().begin + plan.back().length == b.delta_offset) {
        plan.back().length += b.tangent_size;  // untouched entries ride with their neighbour
      } else {
        plan.push_back(GradientInterval{b.delta_offset, b.tangent_size, owner});
      }
    }
    int64_t covered = 0;
    for (const auto& g : plan) covered += g.length;
    if (plan.size() <= 96 && covered == e->num_effective) e->exchange.swap(plan);

    // Peer exchange: possible when the residual blocks are one type in program order, every
    // rank owns at most one exclusive range and the shared part is small.  All of these are
    // properties of the whole problem, so every rank takes the same decision.
    std::vector<int> owned(e->world, 0);
    int64_t shared = 0;
    int shared_intervals = 0;
    for (const GradientInterval& iv : e->exchange) {
      if (iv.owner >= 0) ++owned[iv.owner];
      else { shared += iv.length; ++shared_intervals; }
    }
    bool one_each = !e->exchange.empty();
    for (int c : owned) one_each = one_each && c <= 1;
    const char* mode = getenv("CB200_GRADIENT_EXCHANGE");
    e->peer_plan = one_each && in_program_order && e->world <= kMaxRanks &&
                   shared_intervals <= kMaxSharedIntervals && 4 * shared <= e->num_effective &&
                   !(mode && std::strcmp(mode, "nccl") == 0);
    e->shared_count = static_cast<int32_t>(shared) + 2;
    e->exclusive_begin = e->exclusive_length = 0;
    if (e->peer_plan) {
      // Chunks of this rank's residual blocks whose exclusive gradient entries form a
      // contiguous range touched by no other chunk.  A cut between consecutive parameter
      // blocks i, i + 1 of the exclusive range is valid at residual block position
      // min(first[i + 1 ...]) iff every block up to i was last touched before it.
      // A chunk is a warp's unit of work (tiles of 32 blocks, one fence and one copy at its
      // end), drawn from a counter by the warps of the persistent grid (148 SMs x 12 warps).
      // About 12 chunks per warp bounds the idle tail when the warps run out of chunks; chunk
      // lengths that are multiples of 32 leave no partial tile (at 8 GPUs half a tile in
      // seven was idle lanes).  A cut is taken at the first valid position that makes the
      // length a multiple of 32 once half the target is reached (with ~6.5 blocks per point
      // such a position comes every ~200 blocks); without one by three times the target, at
      // the last valid position within the target.
      const int64_t local_blocks = nrb * (e->rank + 1) / e->world - nrb * e->rank / e->world;
      const int kChunkBlocks = static_cast<int>(std::min<int64_t>(
          4096, std::max<int64_t>(128, 2 * (local_blocks / (148 * 12 * 12) - 104) / 32 * 32)));
      int i0 = -1, i1 = -1;  // active blocks [i0, i1) of this rank's exclusive interval
      for (const GradientInterval& iv : e->exchange) {
        if (iv.owner != e->rank) continue;
        e->exclusive_begin = iv.begin;
        e->exclusive_length = iv.length;
      }
      if (e->exclusive_length > 0) {
        for (int i = 0; i < e->num_active; ++i) {
          const cb200_parameter_block& b = e->blocks[i];
          if (b.tangent_size == 0) continue;
          if (b.delta_offset >= e->exclusive_begin &&
              b.delta_offset < e->exclusive_begin + e->exclusive_length) {
            if (i0 < 0) i0 = i;
            i1 = i + 1;
          }
        }
      }
      const int32_t rb0 = static_cast<int32_t>(nrb * e->rank / e->world);
      const int32_t rb1 = static_cast<int32_t>(nrb * (e->rank + 1) / e->world);
      int32_t start_rb = rb0;
      int64_t start_delta = e->exclusive_begin;
      auto close_chunk = [&](int32_t end_rb, int64_t end_delta) {
        if (end_rb > start_rb) {
          e->chunk_table.push_back(start_rb - rb0);
          e->chunk_table.push_back(end_rb - rb0);
          e->chunk_table.push_back(static_cast<int32_t>(start_delta));
          e->chunk_table.push_back(static_cast<int32_t>(end_delta));
          start_rb = end_rb;
          start_delta = end_delta;
        }
      };
      if (i0 >= 0) {
        std::vector<int32_t> sufmin(static_cast<size_t>(i1 - i0) + 1, INT32_MAX);
        for (int i = i1 - 1; i >= i0; --i) sufmin[i - i0] = std::min(sufmin[i - i0 + 1], first[i]);
        int32_t prefmax = -1, best_rb = -1;
        int64_t best_delta = 0;
        for (int i = i0; i + 1 < i1; ++i) {
          prefmax = std::max(prefmax, last[i]);
          const int32_t cut = sufmin[i + 1 - i0];
          if (cut == INT32_MAX || !(prefmax < cut) || e->blocks[i + 1].tangent_size == 0) continue;
          const int64_t cut_delta = e->blocks[i + 1].delta_offset;
          if (cut <= start_rb) continue;
          // past three times the target without a tile-aligned cut: the best plain one
          while (cut - start_rb > 3 * kChunkBlocks && best_rb > start_rb) {
            close_chunk(best_rb, best_delta);
            best_rb = -1;
          }
          const int32_t length = cut - start_rb;
          if (length > 3 * kChunkBlocks) {  // no cut inside the window: a long chunk
            close_chunk(cut, cut_delta);
            best_rb = -1;
          } else if (length % 32 == 0 && 2 * length >= kChunkBlocks) {
            close_chunk(cut, cut_delta);    // whole tiles only
            best_rb = -1;
          } else if (length <= kChunkBlocks || best_rb <= start_rb) {
            best_rb = cut;
            best_delta = cut_delta;
          }
        }
        if (best_rb > start_rb && rb1 - start_rb > kChunkBlocks) close_chunk(best_rb, best_delta);
      }
      close_chunk(rb1, e->exclusive_begin + e->exclusive_length);
      if (e->chunk_table.size() >= 4)  // the last chunk ends the exclusive range
        e->chunk_table.back() = static_cast<int32_t>(e->exclusive_begin + e->exclusive_length);
    }
  }

  // Pass 1: per type, pick this rank's blocks and find what part of the values
  // array each (type, argument) stream covers.
  struct Stream { int64_t lo, hi, covered; };
  std::vector<Stream> streams;
  std::vector<std::vector<int32_t>> local_index(e->types.size());
  for (size_t ti = 0; ti < e->types.size(); ++ti) {
    ResidualType* t = e->types[ti];
    const int nb = t->desc.num_parameter_blocks, kres = t->desc.num_residuals;
    auto& idx = local_index[ti];
    for (int32_t k = 0; k < static_cast<int32_t>(t->position.size()); ++k) {
      const int32_t p = t->position[k];
      if (p < 0 || p >= nrb)
        return e->Fail(CB200_ERROR_INVALID_ARGUMENT, "residual block position %d out of range", p);
      if (p >= e->rb_begin && p < e->rb_end) idx.push_back(k);
    }
    std::vector<Stream> s(nb, Stream{INT64_MAX, -1, 0});
    for (int32_t k : idx) {
      const int32_t L = e->jprl[t->position[k]];
      int a = 0;
      for (int j = 0; j < nb; ++j) {
        const int32_t id = t->pb_ids[static_cast<size_t>(k) * nb + j];
        if (id < 0 || id >= npb)
          return e->Fail(CB200_ERROR_INVALID_ARGUMENT, "parameter block id %d out of range", id);
        if (id >= e->num_active) continue;  // constant: no Jacobian block
        const int tangent = e->blocks[id].tangent_size;
        for (int r = 0; r < kres; ++r) {
          const int64_t pos = e->jpro[static_cast<size_t>(L) + a * kres + r];
          s[j].lo = std::min(s[j].lo, pos);
          s[j].hi = std::max(s[j].hi, pos + tangent);
          s[j].covered += tangent;
        }
        ++a;
      }
    }
    for (auto& st : s) if (st.hi >= 0) streams.push_back(st);
  }
  // Streams that are dense on their own become segments; otherwise fall back to
  // the union span.  Overlapping / adjacent segments are merged.
  e->segments.clear();
  {
    bool all_dense = true;
    int64_t lo = INT64_MAX, hi = -1, covered = 0;
    for (auto& st : streams) {
      lo = std::min(lo, st.lo); hi = std::max(hi, st.hi); covered += st.covered;
      if (st.covered != st.hi - st.lo) all_dense = false;
    }
    std::vector<std::pair<int64_t, int64_t>> spans;
    if (!streams.empty()) {
      if (all_dense) for (auto& st : streams) spans.emplace_back(st.lo, st.hi);
      else spans.emplace_back(lo, hi);  // interleaved (compressed-row): one span
      (void)covered;
    }
    std::sort(spans.begin(), spans.end());
    int64_t local = 0;
    for (auto& sp : spans) {
      if (!e->segments.empty() &&
          sp.first <= e->segments.back().global_begin + e->segments.back().length) {
        Segment& b = e->segments.back();
        const int64_t new_end = std::max(b.global_begin + b.length, sp.second);
        local += new_end - (b.global_begin + b.length);
        b.length = new_end - b.global_begin;
      } else {
        e->segments.push_back(Segment{sp.first, sp.second - sp.first, local});
        local += sp.second - sp.first;
      }
    }
    e->local_jacobian_values = local;
  }
  auto to_local = [&](int64_t pos) -> int32_t {
    for (const Segment& s : e->segments)
      if (pos >= s.global_begin && pos < s.global_begin + s.length)
        return static_cast<int32_t>(pos - s.global_begin + s.local_begin);
    return -1;
  };

  // Pass 2: build and upload the per-type tables (argument-major SoA).
  e->total_cost_partials = 0;
  for (size_t ti = 0; ti < e->types.size(); ++ti) {
    ResidualType* t = e->types[ti];
    const int nb = t->desc.num_parameter_blocks, kres = t->desc.num_residuals;
    const auto& idx = local_index[ti];
    const int32_t n = static_cast<int32_t>(idx.size());
    t->n_local = n;
    const int tpb = t->desc.threads_per_block > 0 ? t->desc.threads_per_block : 128;
    // Cost partials reserved for the launch: the thunk's (persistent) grid is clamped to
    // this, so the fixed-order reduction reads at most 2048 values per type.
    t->grid = std::min((n + tpb - 1) / tpb, 2048);
    t->cost_partial_offset = e->total_cost_partials;
    e->total_cost_partials += t->grid;
    if (n == 0) continue;
    std::vector<int32_t> pb(static_cast<size_t>(nb) * n), jpos(static_cast<size_t>(nb) * n, -1);
    std::vector<int32_t> soff(static_cast<size_t>(nb) * n), doff(static_cast<size_t>(nb) * n);
    t->plain = true;
    std::vector<int32_t> jstride(n, 0), respos(n), lidx;
    std::vector<char> fun(static_cast<size_t>(n) * t->desc.functor_size);
    if (t->num_losses > 1) lidx.resize(n);
    for (int32_t i = 0; i < n; ++i) {
      const int32_t k = idx[i];
      const int32_t p = t->position[k];
      respos[i] = e->residual_layout[p] - e->res_begin;
      std::memcpy(fun.data() + static_cast<size_t>(i) * t->desc.functor_size,
                  t->functors.data() + static_cast<size_t>(k) * t->desc.functor_size,
                  t->desc.functor_size);
      if (t->num_losses > 1) lidx[i] = t->loss_index[k];
      const int32_t L = e->jprl[p];
      int a = 0;
      for (int j = 0; j < nb; ++j) {
        const int32_t id = t->pb_ids[static_cast<size_t>(k) * nb + j];
        pb[static_cast<size_t>(j) * n + i] = id;
        soff[static_cast<size_t>(j) * n + i] = table[8 * id + 0];
        doff[static_cast<size_t>(j) * n + i] = table[8 * id + 1];
        if (table[8 * id + 1] < 0 || table[8 * id + 3] != CB200_MANIFOLD_NONE ||
            e->blocks[id].tangent_size != e->blocks[id].size)
          t->plain = false;
        if (id >= e->num_active) continue;
        const int64_t pos0 = e->jpro[static_cast<size_t>(L) + a * kres];
        jpos[static_cast<size_t>(j) * n + i] = to_local(pos0);
        if (kres > 1 && jstride[i] == 0)
          jstride[i] = e->jpro[static_cast<size_t>(L) + a * kres + 1] -
                       e->jpro[static_cast<size_t>(L) + a * kres];
        ++a;
      }
    }
    // Arithmetic progressions: a type laid out in program order (bundle adjustment after
    // the Schur ordering, a pose graph's residuals) needs no position tables at all.
    {
      bool res_affine = true, jac_affine = true, delta_is_state = true;
      for (int32_t i = 0; i < n && res_affine; ++i)
        res_affine = respos[i] == respos[0] + static_cast<int64_t>(i) * kres;
      for (int j = 0; j < nb; ++j) {
        const int32_t* jp = jpos.data() + static_cast<size_t>(j) * n;
        const int64_t step = n > 1 ? static_cast<int64_t>(jp[1]) - jp[0] : 0;
        t->jacobian_base[j] = jp[0];
        t->jacobian_step[j] = static_cast<int32_t>(step);
        for (int32_t i = 0; i < n && jac_affine; ++i)
          jac_affine = jp[i] >= 0 && jp[i] == jp[0] + step * i;
        const int32_t* so = soff.data() + static_cast<size_t>(j) * n;
        const int32_t* dof = doff.data() + static_cast<size_t>(j) * n;
        for (int32_t i = 0; i < n && delta_is_state; ++i) delta_is_state = so[i] == dof[i];
      }
      for (int32_t i = 0; i < n && jac_affine; ++i) jac_affine = jstride[i] == jstride[0];
      t->residual_base = respos[0];
      t->row_stride = jstride[0];
      t->affine = (res_affine ? CB200_AFFINE_RESIDUAL : 0u) |
                  (jac_affine ? CB200_AFFINE_JACOBIAN : 0u) |
                  (delta_is_state ? CB200_AFFINE_DELTA_IS_STATE : 0u);
      if (getenv("CB200_NO_AFFINE")) t->affine = 0;  // A/B switch: always read the tables
    }
    if (e->planning) continue;
    CB200_CUDA(e, t->d_pb.Upload(pb, e->stream));
    CB200_CUDA(e, t->d_soff.Upload(soff, e->stream));
    CB200_CUDA(e, t->d_doff.Upload(doff, e->stream));
    CB200_CUDA(e, t->d_jpos.Upload(jpos, e->stream));
    CB200_CUDA(e, t->d_jstride.Upload(jstride, e->stream));
    CB200_CUDA(e, t->d_respos.Upload(respos, e->stream));
    CB200_CUDA(e, t->d_functors.Upload(fun, e->stream));
    CB200_CUDA(e, t->d_loss_table.Upload(t->loss_table, e->stream));
    if (t->num_losses > 1) CB200_CUDA(e, t->d_loss_index.Upload(lidx, e->stream));
    CB200_CUDA(e, cudaStreamSynchronize(e->stream));  // the vectors die at scope end
    // The full-problem host copies are no longer needed.
    std::vector<int32_t>().swap(t->pb_ids);
    std::vector<char>().swap(t->functors);
    std::vector<int32_t>().swap(t->loss_index);
  }

  if (e->planning) {
    e->finalized = true;
    return CB200_OK;
  }
  CB200_CUDA(e, e->d_pb_table.Upload(table, e->stream));
  // (+4: the kernels gather parameter blocks in aligned 16-byte pieces and may read up to
  // two doubles past the last block)
  CB200_CUDA(e, e->d_state.Resize(static_cast<size_t>(e->num_parameters) +
                                  e->num_constant_parameters + 4));
  if (e->num_constant_parameters > 0)
    CB200_CUDA(e, cudaMemcpyAsync(e->d_state.ptr + e->num_parameters, e->constant_state.data(),
                                  e->constant_state.size() * sizeof(double),
                                  cudaMemcpyHostToDevice, e->stream));
  CB200_CUDA(e, e->d_plus.Resize(static_cast<size_t>(e->plus_pool) + 1));
  CB200_CUDA(e, e->d_residuals.Resize(static_cast<size_t>(e->res_end - e->res_begin) + 1));
  CB200_CUDA(e, e->d_jacobian.Resize(static_cast<size_t>(e->local_jacobian_values) + 2));
  CB200_CUDA(e, e->d_gradcost.Resize(static_cast<size_t>(e->num_effective) + 2));
  e->gradcost = e->d_gradcost.ptr;
  if (e->peer_plan && !e->chunk_table.empty())
    CB200_CUDA(e, e->d_chunks.Upload(e->chunk_table, e->stream));
  // the largest chunk count one launch can have: the exchange plan's chunks or uniform ones
  e->chunk_cost_capacity = static_cast<int32_t>(e->chunk_table.size() / 4);
  for (ResidualType* t : e->types)
    e->chunk_cost_capacity = std::max(e->chunk_cost_capacity,
                                      (t->n_local + kUniformChunkBlocks - 1) / kUniformChunkBlocks);
  CB200_CUDA(e, e->d_cost_partials.Resize(static_cast<size_t>(e->total_cost_partials) +
                                          e->chunk_cost_capacity + 1));
  CB200_CUDA(e, e->d_status.Resize(2));  // [failure flag, chunk counter of the chunked kernel]
  CB200_CUDA(e, cudaStreamSynchronize(e->stream));
  // Layout arrays were consumed.
  std::vector<int32_t>().swap(e->jpro);
  e->finalized = true;
  return CB200_OK;
}

// Maps one region per rank into every rank (CUDA IPC over NVLink peer access):
//   [gradient buffer 0 | gradient buffer 1 | slots parity 0 | slots parity 1 | flags]
// Two gradient buffers / slot sets alternate between evaluations so that a fast rank's copies
// for evaluation k + 1 never land in memory a slow rank still reads for evaluation k.  All
// ranks agree (one NCCL sum) on whether the mapping worked; if not, every rank keeps the
// NCCL all-reduce.
static size_t Align256(size_t bytes) { return (bytes + 255) / 256 * 256; }
static int SetupPeerExchange(cb200_engine* e) {
  e->peer_ready = false;
  if (!e->finalized || !e->peer_plan || !e->comm || e->world <= 1) return CB200_OK;
  NcclApi* n = GetNccl();
  if (!n->AllGather) return CB200_OK;
  cudaStream_t s = e->stream;
  e->peer_gradient_stride = Align256((static_cast<size_t>(e->num_effective) + 2) * sizeof(double));
  const size_t slot_bytes = Align256(static_cast<size_t>(e->world) * e->shared_count * sizeof(double));
  e->peer_slots_offset = 2 * e->peer_gradient_stride;
  e->peer_flags_offset = e->peer_slots_offset + 2 * slot_bytes;
  const size_t total = e->peer_flags_offset + 256;
  int failed = 0;
  cudaIpcMemHandle_t mine{};
  if (cudaMalloc(reinterpret_cast<void**>(&e->peer_region), total) != cudaSuccess ||
      cudaMemsetAsync(e->peer_region, 0, total, s) != cudaSuccess ||
      cudaIpcGetMemHandle(&mine, e->peer_region) != cudaSuccess) {
    cudaGetLastError();
    failed = 1;
  }
  // exchange the handles (and, below, the verdicts) through NCCL
  DeviceBuffer<char> wire;
  CB200_CUDA(e, wire.Resize(static_cast<size_t>(e->world) * sizeof(mine) + 2 * sizeof(double)));
  CB200_CUDA(e, cudaMemcpyAsync(wire.ptr + e->rank * sizeof(mine), &mine, sizeof(mine),
                                cudaMemcpyHostToDevice, s));
  if (n->AllGather(wire.ptr + e->rank * sizeof(mine), wire.ptr, sizeof(mine), /*ncclChar*/ 0,
                   e->comm, s) != 0)
    return e->Fail(CB200_ERROR_NCCL, "ncclAllGather of the IPC handles failed");
  std::vector<cudaIpcMemHandle_t> handles(e->world);
  CB200_CUDA(e, cudaMemcpyAsync(handles.data(), wire.ptr, e->world * sizeof(mine),
                                cudaMemcpyDeviceToHost, s));
  CB200_CUDA(e, cudaStreamSynchronize(s));
  for (int r = 0; r < e->world && !failed; ++r) {
    if (r == e->rank) {
      e->peer_base[r] = e->peer_region;
    } else if (cudaIpcOpenMemHandle(&e->peer_base[r], handles[r],
                                    cudaIpcMemLazyEnablePeerAccess) != cudaSuccess) {
      cudaGetLastError();
      e->peer_base[r] = nullptr;
      failed = 1;
    }
  }
  double* verdict = reinterpret_cast<double*>(wire.ptr + e->world * sizeof(mine));
  const double flag = failed;
  CB200_CUDA(e, cudaMemcpyAsync(verdict, &flag, sizeof(double), cudaMemcpyHostToDevice, s));
  if (n->AllReduce(verdict, verdict, 1, kNcclFloat64, kNcclSum, e->comm, s) != 0)
    return e->Fail(CB200_ERROR_NCCL, "NCCL all-reduce failed");
  double total_failed = 1.0;
  CB200_CUDA(e, cudaMemcpyAsync(&total_failed, verdict, sizeof(double), cudaMemcpyDeviceToHost, s));
  CB200_CUDA(e, cudaStreamSynchronize(s));
  wire.Free();
  if (total_failed != 0.0) {
    if (getenv("CB200_VERBOSE"))
      std::fprintf(stderr, "ceres_b200: rank %d: peer mapping unavailable, using the NCCL all-reduce\n",
                   e->rank);
    return CB200_OK;
  }
  CB200_CUDA(e, e->d_arrivals.Resize(1));
  CB200_CUDA(e, cudaMemsetAsync(e->d_arrivals.ptr, 0, sizeof(unsigned), s));
  CB200_CUDA(e, cudaStreamSynchronize(s));
  e->peer_ready = true;
  return CB200_OK;
}

int cb200_nccl_unique_id(void* out) {
  NcclApi* n = GetNccl();
  if (!n || !out) return CB200_ERROR_NCCL;
  return n->GetUniqueId(out) == 0 ? CB200_OK : CB200_ERROR_NCCL;
}

int cb200_engine_comm_init(cb200_engine* e, const void* unique_id, int32_t rank,
                           int32_t world_size) {
  NvtxRange nvtx_range("cb200_engine_comm_init");
  if (!e || !unique_id) return CB200_ERROR_INVALID_ARGUMENT;
  if (e->planning) return e->Fail(CB200_ERROR_CUDA, "planning-only engine");
  NcclApi* n = GetNccl();
  if (!n) return e->Fail(CB200_ERROR_NCCL, "libnccl.so.2 not found");
  CB200_CUDA(e, cudaSetDevice(e->device));
  Uid id;
  std::memcpy(id.internal, unique_id, sizeof(id.internal));
  const int r = n->CommInitRank(&e->comm, world_size, id, rank);
  if (r != 0)
    return e->Fail(CB200_ERROR_NCCL, "ncclCommInitRank: %s",
                   n->GetErrorString ? n->GetErrorString(r) : "?");
  return SetupPeerExchange(e);
}

// Shared by the host-pointer and device-pointer entry points.
static int EvaluateOnDevice(cb200_engine* e, uint32_t flags, bool want_r, bool want_g,
                            bool want_j) {
  cudaStream_t s = e->stream;
  if (want_j) e->jacobian_resident = true;   // values of an older evaluation are overwritten
  if (want_j) e->colnorm_valid = false;
  if (want_r) e->residuals_resident = true;
  CB200_CUDA(e, cudaMemsetAsync(e->d_status.ptr, 0, 2 * sizeof(int32_t), s));
  const size_t ne = static_cast<size_t>(e->num_effective);
  // Several ranks with the peer exchange: this evaluation's [gradient | cost | failed] is
  // one of the two peer-mapped buffers.  Only what this rank's blocks add to is zeroed: the
  // rest of the buffer is written by the other ranks, possibly before this point.
  const bool peer = want_g && e->peer_ready;
  char* region = nullptr;
  if (peer) {
    ++e->epoch;
    region = e->peer_region;
    e->gradcost = reinterpret_cast<double*>(region + (e->epoch & 1) * e->peer_gradient_stride);
    if (e->exclusive_length > 0)
      CB200_CUDA(e, cudaMemsetAsync(e->gradcost + e->exclusive_begin, 0,
                                    e->exclusive_length * sizeof(double), s));
    for (const GradientInterval& iv : e->exchange)
      if (iv.owner < 0)
        CB200_CUDA(e, cudaMemsetAsync(e->gradcost + iv.begin, 0, iv.length * sizeof(double), s));
    CB200_CUDA(e, cudaMemsetAsync(e->gradcost + ne, 0, 2 * sizeof(double), s));
  } else {
    e->gradcost = e->d_gradcost.ptr;
    // Only the gradient accumulates; residuals and Jacobian cells are each written
    // exactly once.  Cost slot and padding are zeroed with it.
    CB200_CUDA(e, cudaMemsetAsync(e->gradcost, 0, (ne + 2) * sizeof(double), s));
  }
  double* peer_gradient[CB200_MAX_PEERS] = {};
  int num_peers = 0;
  if (peer)
    for (int r = 0; r < e->world; ++r)
      if (r != e->rank)
        peer_gradient[num_peers++] = reinterpret_cast<double*>(
            static_cast<char*>(e->peer_base[r]) + (e->epoch & 1) * e->peer_gradient_stride);
  CB200_CUDA(e, cudaEventRecord(e->ev[1], s));
  int launches = 0;
  bool pushed_by_kernel = false;
  int32_t chunk_costs = 0;  // chunks of this evaluation's chunked launch
  for (ResidualType* t : e->types) {
    if (t->n_local == 0) continue;
    cb200_launch_args a{};
    a.n = t->n_local;
    a.output_residuals = want_r;
    a.output_jacobian = want_j;
    a.output_gradient = want_g;
    a.apply_loss_function = (flags & CB200_APPLY_LOSS_FUNCTION) ? 1u : 0u;
    a.crs = e->jacobian_format == CB200_JACOBIAN_COMPRESSED_ROW;
    a.plain = t->plain ? 1u : 0u;
    a.cost_partial_count = t->grid;
    a.state_offset = t->d_soff.ptr;
    a.delta_offset = t->d_doff.ptr;
    a.functors = t->d_functors.ptr;
    a.loss_table = t->d_loss_table.ptr;
    a.loss_index = t->num_losses > 1 ? t->d_loss_index.ptr : nullptr;
    if (t->num_losses == 1 && t->loss_table.size() <= CB200_INLINE_LOSS_BYTES &&
        t->loss_table.size() % 8 == 0 && !t->loss_table.empty()) {
      a.loss_inline_size = static_cast<uint32_t>(t->loss_table.size());
      std::memcpy(a.loss_inline, t->loss_table.data(), t->loss_table.size());
    }
    a.parameter_block = t->d_pb.ptr;
    a.jacobian_pos = t->d_jpos.ptr;
    a.jacobian_row_stride = t->d_jstride.ptr;
    a.residual_pos = t->d_respos.ptr;
    a.parameter_block_table = e->d_pb_table.ptr;
    a.state = e->d_state.ptr;
    a.plus_jacobians = e->d_plus.ptr;
    a.residuals = e->d_residuals.ptr;
    a.jacobian_values = e->d_jacobian.ptr;
    a.gradient = e->gradcost;
    a.cost_partials = e->d_cost_partials.ptr + t->cost_partial_offset;
    a.status = e->d_status.ptr;
    a.affine = t->affine;
    a.residual_base = t->residual_base;
    a.row_stride = t->row_stride;
    std::memcpy(a.jacobian_base, t->jacobian_base, sizeof(a.jacobian_base));
    std::memcpy(a.jacobian_step, t->jacobian_step, sizeof(a.jacobian_step));
    // The chunked variant exists for the plain all-outputs kernel over affine tables (the
    // same test as in the launch thunk); otherwise PushExclusiveKernel below does the copies.
    // One chunked launch per evaluation at most: the chunk counter (status[1]) and the chunk
    // cost slots serve one launch.
    constexpr uint32_t kAffinePlain =
        CB200_AFFINE_RESIDUAL | CB200_AFFINE_JACOBIAN | CB200_AFFINE_DELTA_IS_STATE;
    if (chunk_costs == 0 && peer && t->desc.supports_chunks && e->d_chunks.ptr && t->plain &&
        !a.crs && want_r && want_j && a.apply_loss_function &&
        (t->affine & kAffinePlain) == kAffinePlain &&
        // (measured on B200: with two ranks the copies issued from inside the kernel slow it
        // by more than the separate push costs - 1.15 against 1.05 ms of device time on BAL
        // L - while from four ranks on the fused form wins: 0.37 against 0.55 ms on eight)
        (e->world >= 4 || getenv("CB200_CHUNKED_KERNEL")) && !getenv("CB200_NO_CHUNKED_KERNEL")) {
      a.chunks = e->d_chunks.ptr;
      a.num_chunks = static_cast<int32_t>(e->chunk_table.size() / 4);
      a.num_peers = num_peers;
      std::memcpy(a.peer_gradient, peer_gradient, sizeof(a.peer_gradient));
      pushed_by_kernel = true;
    }
    // Large single-type problems without in-kernel copies: uniform chunks (see chunk_blocks).
    if (chunk_costs == 0 && !a.chunks && t->desc.supports_chunks && t->plain && !a.crs && want_r &&
        want_j && want_g && a.apply_loss_function && (t->affine & kAffinePlain) == kAffinePlain &&
        t->n_local >= kUniformChunkMinBlocks && !getenv("CB200_NO_CHUNKED_KERNEL")) {
      a.chunk_blocks = kUniformChunkBlocks;
      a.num_chunks = (t->n_local + kUniformChunkBlocks - 1) / kUniformChunkBlocks;
      a.num_peers = 0;
    }
    if (a.num_chunks > 0) {
      a.chunk_cost_offset = e->total_cost_partials - t->cost_partial_offset;
      chunk_costs = a.num_chunks;
    }
    const int err = t->desc.launch(&a, s);
    if (err != 0)
      return e->Fail(CB200_ERROR_CUDA, "kernel launch: %s",
                     cudaGetErrorString(static_cast<cudaError_t>(err)));
    ++launches;
  }
  CB200_CUDA(e, cudaEventRecord(e->ev[2], s));
  // [gradient | cost | failed]: the last two slots are written here
  ReduceCostKernel<<<1, kReduceCostThreads, 0, s>>>(
      e->d_cost_partials.ptr, e->total_cost_partials,
      e->d_cost_partials.ptr + e->total_cost_partials, chunk_costs, e->gradcost + ne,
      e->d_status.ptr);
  ++launches;
  if (peer) {
    if (!pushed_by_kernel && e->exclusive_length > 0) {
      PeerPush push{};
      push.num_peers = num_peers;
      push.begin = e->exclusive_begin;
      push.length = e->exclusive_length;
      push.gradient = e->gradcost;
      std::memcpy(push.peer, peer_gradient, sizeof(push.peer));
      const int grid = static_cast<int>(std::min<int64_t>((push.length + 255) / 256, 148 * 4));
      PushExclusiveKernel<<<grid, 256, 0, s>>>(push);
      ++launches;
    }
    SharedExchange x{};
    x.world = e->world;
    x.rank = e->rank;
    int32_t at = 0;
    for (const GradientInterval& iv : e->exchange) {
      if (iv.owner >= 0) continue;
      x.begin[x.num_intervals] = static_cast<int32_t>(iv.begin);
      x.start[x.num_intervals] = at;
      at += static_cast<int32_t>(iv.length);
      ++x.num_intervals;
    }
    x.count = e->shared_count;
    x.gradient = e->gradcost;
    x.cost_offset = e->num_effective;
    const size_t slot_bytes = (e->peer_flags_offset - e->peer_slots_offset) / 2;
    for (int r = 0; r < e->world; ++r) {
      char* base = static_cast<char*>(e->peer_base[r]);
      x.slots[r] = reinterpret_cast<double*>(base + e->peer_slots_offset + (e->epoch & 1) * slot_bytes);
      x.flags[r] = reinterpret_cast<unsigned long long*>(base + e->peer_flags_offset);
    }
    x.epoch = e->epoch;
    x.arrivals = e->d_arrivals.ptr;
    const int grid = std::max(1, std::min((x.count + 255) / 256, 64));
    ExchangeSharedKernel<<<grid, 256, 0, s>>>(x);
    ++launches;
    CB200_CUDA(e, cudaGetLastError());
  } else if (e->comm && e->world > 1) {
    NcclApi* n = GetNccl();
    double* g = e->gradcost;
    // cost-only evaluation: [cost | failed]; otherwise one all-reduce over
    // [gradient | cost | failed] (the path for structures the peer exchange does not cover).
    const int r = want_g ? n->AllReduce(g, g, ne + 2, kNcclFloat64, kNcclSum, e->comm, s)
                         : n->AllReduce(g + ne, g + ne, 2, kNcclFloat64, kNcclSum, e->comm, s);
    if (r != 0) return e->Fail(CB200_ERROR_NCCL, "NCCL collective failed (%d)", r);
  }
  CB200_CUDA(e, cudaEventRecord(e->ev[3], s));
  e->timing[3] = launches;
  return CB200_OK;
}

static int FinishTiming(cb200_engine* e) {
  float ms = 0;
  cudaEventElapsedTime(&ms, e->ev[1], e->ev[2]); e->timing[0] = ms;
  cudaEventElapsedTime(&ms, e->ev[1], e->ev[3]); e->timing[1] = ms;
  cudaEventElapsedTime(&ms, e->ev[0], e->ev[4]); e->timing[2] = ms;
  return CB200_OK;
}

int cb200_engine_evaluate(cb200_engine* e, const double* state, const double* plus_jacobians,
                          uint32_t flags, double* cost, double* residuals, double* gradient,
                          double* jacobian_values) {
  NvtxRange nvtx_range("cb200_engine_evaluate");
  if (!e) return CB200_ERROR_INVALID_ARGUMENT;
  if (!e->finalized) return e->Fail(CB200_ERROR_NOT_FINALIZED, "evaluate before finalize");
  if (e->planning) return e->Fail(CB200_ERROR_CUDA, "planning-only engine: no device, no CPU fallback");
  if (!state || !cost) return e->Fail(CB200_ERROR_INVALID_ARGUMENT, "state and cost are required");
  if (e->plus_pool > 0 && !plus_jacobians)
    return e->Fail(CB200_ERROR_INVALID_ARGUMENT, "plus_jacobians required");
  CB200_CUDA(e, cudaSetDevice(e->device));
  cudaStream_t s = e->stream;
  CB200_CUDA(e, cudaEventRecord(e->ev[0], s));
  CB200_CUDA(e, cudaMemcpyAsync(e->d_state.ptr, state, sizeof(double) * e->num_parameters,
                                cudaMemcpyHostToDevice, s));
  if (e->plus_pool > 0)
    CB200_CUDA(e, cudaMemcpyAsync(e->d_plus.ptr, plus_jacobians, sizeof(double) * e->plus_pool,
                                  cudaMemcpyHostToDevice, s));
  const bool keep_r = (flags & CB200_KEEP_RESIDUALS_ON_DEVICE) != 0;
  const bool keep_j = (flags & CB200_KEEP_JACOBIAN_ON_DEVICE) != 0;
  const int rc = EvaluateOnDevice(e, flags, residuals != nullptr || keep_r, gradient != nullptr,
                                  jacobian_values != nullptr || keep_j);
  if (rc != CB200_OK) return rc;
  CB200_CUDA(e, cudaMemcpyAsync(e->h_scalars, e->gradcost + e->num_effective,
                                2 * sizeof(double), cudaMemcpyDeviceToHost, s));
  if (!(flags & CB200_SKIP_HOST_COPY)) {
    if (residuals && !keep_r && e->res_end > e->res_begin)
      CB200_CUDA(e, cudaMemcpyAsync(residuals + e->res_begin, e->d_residuals.ptr,
                                    sizeof(double) * (e->res_end - e->res_begin),
                                    cudaMemcpyDeviceToHost, s));
    if (gradient && e->num_effective > 0)
      CB200_CUDA(e, cudaMemcpyAsync(gradient, e->gradcost,
                                    sizeof(double) * e->num_effective, cudaMemcpyDeviceToHost, s));
    if (jacobian_values && !keep_j)
      for (const Segment& seg : e->segments)
        CB200_CUDA(e, cudaMemcpyAsync(jacobian_values + seg.global_begin,
                                      e->d_jacobian.ptr + seg.local_begin,
                                      sizeof(double) * seg.length, cudaMemcpyDeviceToHost, s));
  }
  CB200_CUDA(e, cudaEventRecord(e->ev[4], s));
  CB200_CUDA(e, cudaStreamSynchronize(s));  // the only host synchronisation
  FinishTiming(e);
  *cost = e->h_scalars[0];
  return e->h_scalars[1] != 0.0 ? CB200_EVALUATION_FAILED : CB200_OK;
}

int cb200_engine_evaluate_device(cb200_engine* e, const double* state_device,
                                 const double* plus_jacobians_device, uint32_t flags,
                                 int want_residuals, int want_gradient, int want_jacobian,
                                 double* cost) {
  NvtxRange nvtx_range("cb200_engine_evaluate_device");
  if (!e) return CB200_ERROR_INVALID_ARGUMENT;
  if (!e->finalized) return e->Fail(CB200_ERROR_NOT_FINALIZED, "evaluate before finalize");
  if (e->planning) return e->Fail(CB200_ERROR_CUDA, "planning-only engine: no device, no CPU fallback");
  if (!cost) return e->Fail(CB200_ERROR_INVALID_ARGUMENT, "cost is required");
  CB200_CUDA(e, cudaSetDevice(e->device));
  cudaStream_t s = e->stream;
  CB200_CUDA(e, cudaEventRecord(e->ev[0], s));
  if (state_device && state_device != e->d_state.ptr)
    CB200_CUDA(e, cudaMemcpyAsync(e->d_state.ptr, state_device,
                                  sizeof(double) * e->num_parameters, cudaMemcpyDeviceToDevice, s));
  if (plus_jacobians_device && e->plus_pool > 0 && plus_jacobians_device != e->d_plus.ptr)
    CB200_CUDA(e, cudaMemcpyAsync(e->d_plus.ptr, plus_jacobians_device,
                                  sizeof(double) * e->plus_pool, cudaMemcpyDeviceToDevice, s));
  const int rc = EvaluateOnDevice(e, flags, want_residuals != 0, want_gradient != 0,
                                  want_jacobian != 0);
  if (rc != CB200_OK) return rc;
  CB200_CUDA(e, cudaMemcpyAsync(e->h_scalars, e->gradcost + e->num_effective,
                                2 * sizeof(double), cudaMemcpyDeviceToHost, s));
  CB200_CUDA(e, cudaEventRecord(e->ev[4], s));
  CB200_CUDA(e, cudaStreamSynchronize(s));
  FinishTiming(e);
  *cost = e->h_scalars[0];
  return e->h_scalars[1] != 0.0 ? CB200_EVALUATION_FAILED : CB200_OK;
}

void* cb200_engine_device_ptr(cb200_engine* e, int which) {
  if (!e || !e->finalized || e->planning) return nullptr;
  switch (which) {
    case 0: return e->d_residuals.ptr;
    case 1: return e->gradcost;
    case 2: return e->d_jacobian.ptr;
    case 3: return e->d_state.ptr;
    case 4: return e->d_plus.ptr;
    default: return nullptr;
  }
}

// ---- device-resident Jacobian linear algebra --------------------------------------------

static int RunJacobianWalk(cb200_engine* e, int op, const double* x, double* y) {
  cudaStream_t s = e->stream;
  for (ResidualType* t : e->types) {
    if (t->n_local == 0) continue;
    JacobianWalk w{};
    w.n = t->n_local;
    w.nb = t->desc.num_parameter_blocks;
    w.kres = t->desc.num_residuals;
    w.crs = e->jacobian_format == CB200_JACOBIAN_COMPRESSED_ROW;
    w.plain = t->plain;
    for (int j = 0; j < w.nb; ++j) w.sizes[j] = t->desc.parameter_block_sizes[j];
    w.doff = t->d_doff.ptr;
    w.jpos = t->d_jpos.ptr;
    w.pb = t->d_pb.ptr;
    w.jstride = t->d_jstride.ptr;
    w.respos = t->d_respos.ptr;
    w.pb_table = e->d_pb_table.ptr;
    w.values = e->d_jacobian.ptr;
    const int grid = std::min((t->n_local + 255) / 256, 148 * 16);
    // The per-type kernel (compile-time sizes, coalesced cell runs: ceres/internal/
    // normal_kernel.cuh) where the structure allows it; the table-walk kernels otherwise.
    {
      constexpr uint32_t kAffinePlain =
          CB200_AFFINE_RESIDUAL | CB200_AFFINE_JACOBIAN | CB200_AFFINE_DELTA_IS_STATE;
      bool contiguous = t->desc.normal_product != nullptr && t->plain && !w.crs &&
                        (t->affine & kAffinePlain) == kAffinePlain &&
                        !getenv("CB200_GENERIC_NORMAL_PRODUCT");
      for (int j = 0; j < w.nb && contiguous; ++j)
        contiguous = t->jacobian_step[j] == w.kres * w.sizes[j];
      if (!contiguous && getenv("CB200_VERBOSE")) {
        static bool told = false;
        if (!told)
          std::fprintf(stderr,
                       "cb200: table-walk linear algebra (thunk %d plain %d crs %d affine %u steps",
                       t->desc.normal_product != nullptr, int(t->plain), int(w.crs), t->affine);
        for (int j = 0; j < w.nb && !told; ++j) std::fprintf(stderr, " %d", t->jacobian_step[j]);
        if (!told) std::fprintf(stderr, ")\n");
        told = true;
      }
      if (contiguous) {
        cb200_normal_args na{};
        na.n = t->n_local;
        na.offset = t->d_soff.ptr;
        na.values = e->d_jacobian.ptr;
        na.residual_base = t->residual_base;
        std::memcpy(na.base, t->jacobian_base, sizeof(na.base));
        switch (op) {
          case kOpNormal: na.op = CB200_NORMAL_OP_NORMAL; na.x = x; na.y = y; break;
          case kOpLeft: na.op = CB200_NORMAL_OP_LEFT; na.w = const_cast<double*>(x); na.y = y; break;
          case kOpRight: na.op = CB200_NORMAL_OP_RIGHT; na.x = x; na.w = y; break;
          case kOpColumnNorm: na.op = CB200_NORMAL_OP_COLUMN_NORM; na.y = y; break;
          case kOpScaleNorm: na.op = CB200_NORMAL_OP_SCALE_NORM; na.x = x; na.y = y; break;
          default: na.op = -1; break;
        }
        if (na.op >= 0) {
          const int rc = t->desc.normal_product(&na, s);
          if (rc == 0) continue;
          if (rc > 0)
            return e->Fail(CB200_ERROR_CUDA, "per-type linear algebra launch: %s",
                           cudaGetErrorString(static_cast<cudaError_t>(rc)));
          if (getenv("CB200_VERBOSE"))
            std::fprintf(stderr, "cb200: per-type linear algebra kernel declined (%d)\n", rc);
        }
      }
    }
    switch (op) {
      case kOpRight: JacobianWalkKernel<kOpRight><<<grid, 256, 0, s>>>(w, x, y); break;
      case kOpLeft: JacobianWalkKernel<kOpLeft><<<grid, 256, 0, s>>>(w, x, y); break;
      case kOpColumnNorm: JacobianWalkKernel<kOpColumnNorm><<<grid, 256, 0, s>>>(w, x, y); break;
      case kOpScaleNorm:
        JacobianWalkKernel<kOpScale><<<grid, 256, 0, s>>>(w, x, nullptr);
        JacobianWalkKernel<kOpColumnNorm><<<grid, 256, 0, s>>>(w, nullptr, y);
        break;
      case kOpNormal: {
        int cell_doubles = 0;
        for (int j = 0; j < w.nb; ++j) cell_doubles += w.kres * w.sizes[j];
        const size_t smem =
            static_cast<size_t>(kNormalThreads / 32) * 32 * cell_doubles * sizeof(double);
        if (!w.crs && smem <= 96 * 1024) {
          if (smem > 48 * 1024)
            CB200_CUDA(e, cudaFuncSetAttribute(JacobianNormalStagedKernel,
                                               cudaFuncAttributeMaxDynamicSharedMemorySize,
                                               static_cast<int>(smem)));
          const int sgrid = std::min((t->n_local + kNormalThreads - 1) / kNormalThreads, 148 * 16);
          JacobianNormalStagedKernel<<<sgrid, kNormalThreads, smem, s>>>(w, x, y, cell_doubles);
        } else {
          JacobianNormalKernel<<<grid, 256, 0, s>>>(w, x, y);
        }
        break;
      }
      default: JacobianWalkKernel<kOpScale><<<grid, 256, 0, s>>>(w, x, y); break;
    }
  }
  CB200_CUDA(e, cudaGetLastError());
  return CB200_OK;
}

// Sums a column-space vector over the ranks (each holds the contribution of its blocks).
static int SumOverRanks(cb200_engine* e, double* v, size_t count) {
  if (!e->comm || e->world <= 1) return CB200_OK;
  NcclApi* n = GetNccl();
  if (n->AllReduce(v, v, count, kNcclFloat64, kNcclSum, e->comm, e->stream) != 0)
    return e->Fail(CB200_ERROR_NCCL, "NCCL all-reduce failed");
  return CB200_OK;
}

constexpr int kMaxVectorGrid = 148 * 8;
static int PrepareLinearAlgebra(cb200_engine* e, bool need_residuals) {
  if (!e) return CB200_ERROR_INVALID_ARGUMENT;
  if (!e->finalized) return e->Fail(CB200_ERROR_NOT_FINALIZED, "not finalized");
  if (e->planning) return e->Fail(CB200_ERROR_CUDA, "planning-only engine: no device, no CPU fallback");
  if (!e->jacobian_resident)
    return e->Fail(CB200_ERROR_INVALID_ARGUMENT,
                   "no Jacobian on the device: evaluate with a Jacobian first");
  if (need_residuals && !e->residuals_resident)
    return e->Fail(CB200_ERROR_INVALID_ARGUMENT,
                   "no residuals on the device: evaluate with residuals first");
  CB200_CUDA(e, cudaSetDevice(e->device));
  for (auto& b : e->la_col) CB200_CUDA(e, b.Resize(static_cast<size_t>(e->num_effective) + 4));
  CB200_CUDA(e, e->la_row.Resize(static_cast<size_t>(e->res_end - e->res_begin) + 1));
  CB200_CUDA(e, e->la_scalars.Resize(3 * kSCount));
  CB200_CUDA(e, e->la_partials.Resize(3 * kMaxVectorGrid));
  if (!e->la_arrivals.ptr) {
    CB200_CUDA(e, e->la_arrivals.Resize(1));
    CB200_CUDA(e, cudaMemsetAsync(e->la_arrivals.ptr, 0, sizeof(unsigned), e->stream));
  }
  if (!e->h_la_scalars)
    CB200_CUDA(e, cudaHostAlloc(reinterpret_cast<void**>(&e->h_la_scalars),
                                3 * kSCount * sizeof(double), cudaHostAllocDefault));
  return CB200_OK;
}

int cb200_engine_jacobian_multiply(cb200_engine* e, int transpose, const double* x, double* y) {
  NvtxRange nvtx_range("cb200_engine_jacobian_multiply");
  int rc = PrepareLinearAlgebra(e, false);
  if (rc != CB200_OK) return rc;
  if (!x || !y) return e->Fail(CB200_ERROR_INVALID_ARGUMENT, "x and y are required");
  cudaStream_t s = e->stream;
  const size_t ne = e->num_effective, m = e->res_end - e->res_begin;
  double* col = e->la_col[0].ptr;
  double* row = e->la_row.ptr;
  if (!transpose) {
    CB200_CUDA(e, cudaMemcpyAsync(col, x, ne * sizeof(double), cudaMemcpyHostToDevice, s));
    if ((rc = RunJacobianWalk(e, kOpRight, col, row)) != CB200_OK) return rc;
    if (m) CB200_CUDA(e, cudaMemcpyAsync(y + e->res_begin, row, m * sizeof(double),
                                         cudaMemcpyDeviceToHost, s));
  } else {
    if (m) CB200_CUDA(e, cudaMemcpyAsync(row, x + e->res_begin, m * sizeof(double),
                                         cudaMemcpyHostToDevice, s));
    CB200_CUDA(e, cudaMemsetAsync(col, 0, ne * sizeof(double), s));
    if ((rc = RunJacobianWalk(e, kOpLeft, row, col)) != CB200_OK) return rc;
    if ((rc = SumOverRanks(e, col, ne)) != CB200_OK) return rc;
    CB200_CUDA(e, cudaMemcpyAsync(y, col, ne * sizeof(double), cudaMemcpyDeviceToHost, s));
  }
  CB200_CUDA(e, cudaStreamSynchronize(s));
  return CB200_OK;
}

int cb200_engine_jacobian_squared_column_norm(cb200_engine* e, double* out) {
  NvtxRange nvtx_range("cb200_engine_jacobian_squared_column_norm");
  int rc = PrepareLinearAlgebra(e, false);
  if (rc != CB200_OK) return rc;
  if (!out) return e->Fail(CB200_ERROR_INVALID_ARGUMENT, "out is required");
  cudaStream_t s = e->stream;
  const size_t ne = e->num_effective;
  double* col = e->la_col[0].ptr;
  CB200_CUDA(e, cudaMemsetAsync(col, 0, ne * sizeof(double), s));
  if ((rc = RunJacobianWalk(e, kOpColumnNorm, nullptr, col)) != CB200_OK) return rc;
  if ((rc = SumOverRanks(e, col, ne)) != CB200_OK) return rc;
  CB200_CUDA(e, cudaMemcpyAsync(out, col, ne * sizeof(double), cudaMemcpyDeviceToHost, s));
  CB200_CUDA(e, cudaStreamSynchronize(s));
  return CB200_OK;
}

int cb200_engine_jacobian_scale_columns(cb200_engine* e, const double* scale) {
  if (e) e->colnorm_valid = false;
  NvtxRange nvtx_range("cb200_engine_jacobian_scale_columns");
  int rc = PrepareLinearAlgebra(e, false);
  if (rc != CB200_OK) return rc;
  if (!scale) return e->Fail(CB200_ERROR_INVALID_ARGUMENT, "scale is required");
  cudaStream_t s = e->stream;
  double* col = e->la_col[0].ptr;
  CB200_CUDA(e, cudaMemcpyAsync(col, scale, static_cast<size_t>(e->num_effective) * sizeof(double),
                                cudaMemcpyHostToDevice, s));
  if ((rc = RunJacobianWalk(e, kOpScale, col, nullptr)) != CB200_OK) return rc;
  CB200_CUDA(e, cudaStreamSynchronize(s));
  return CB200_OK;
}

// The solve itself.  d_squared: host pointer (copied in), or with d_squared_on_device the
// LM diagonal already in la_col[6]; the solution stays in la_col[0] and is copied to
// `solution` when that is not NULL.
static int CgnrSolve(cb200_engine* e, const double* d_squared, bool d_squared_on_device,
                     const cb200_cgnr_options* options, double* solution,
                     cb200_cgnr_summary* summary) {
  int rc = PrepareLinearAlgebra(e, true);
  if (rc != CB200_OK) return rc;
  if (!options || !summary)
    return e->Fail(CB200_ERROR_INVALID_ARGUMENT, "options and summary are required");
  cudaStream_t s = e->stream;
  const int ne = e->num_effective, m = e->res_end - e->res_begin;
  const size_t col_bytes = static_cast<size_t>(ne) * sizeof(double);
  double *x = e->la_col[0].ptr, *r = e->la_col[1].ptr, *p = e->la_col[2].ptr,
         *q = e->la_col[3].ptr, *b = e->la_col[4].ptr, *minv = e->la_col[5].ptr,
         *d2 = (d_squared || d_squared_on_device) ? e->la_col[6].ptr : nullptr,
         *colnorm = e->la_col[7].ptr;
  double* w = e->la_row.ptr;
  const double* residuals = e->d_residuals.ptr;
  double* S = e->la_scalars.ptr;  // three rotating sets of scalars
  const int vgrid = std::max(1, std::min((ne + 255) / 256, kMaxVectorGrid));
  const int rgrid = std::max(1, std::min((m + 255) / 256, kMaxVectorGrid));
  const ScalarReduce red{e->la_partials.ptr, e->la_arrivals.ptr};
  std::memset(summary, 0, sizeof(*summary));
  bool one_pass = true;
  for (const ResidualType* t : e->types)
    if (t->n_local > 0 && t->desc.num_residuals > kNormalRows) one_pass = false;

  CB200_CUDA(e, cudaEventRecord(e->ev[0], s));
  if (d2 && !d_squared_on_device)
    CB200_CUDA(e, cudaMemcpyAsync(d2, d_squared, col_bytes, cudaMemcpyHostToDevice, s));
  // b = J' residuals, preconditioner from the column norms
  CB200_CUDA(e, cudaMemsetAsync(b, 0, col_bytes, s));
  if ((rc = RunJacobianWalk(e, kOpLeft, residuals, b)) != CB200_OK) return rc;
  if ((rc = SumOverRanks(e, b, ne)) != CB200_OK) return rc;
  if (!e->colnorm_valid) {
    CB200_CUDA(e, cudaMemsetAsync(colnorm, 0, col_bytes, s));
    if ((rc = RunJacobianWalk(e, kOpColumnNorm, nullptr, colnorm)) != CB200_OK) return rc;
    if ((rc = SumOverRanks(e, colnorm, ne)) != CB200_OK) return rc;
    e->colnorm_valid = true;
  }
  CB200_CUDA(e, cudaMemsetAsync(S, 0, 3 * kSCount * sizeof(double), s));
  CgInitKernel<<<vgrid, 256, 0, s>>>(ne, colnorm, d2, b, minv, r, p, x, S, red);
  CB200_CUDA(e, cudaMemcpyAsync(e->h_la_scalars, S, kSCount * sizeof(double),
                                cudaMemcpyDeviceToHost, s));
  CB200_CUDA(e, cudaStreamSynchronize(s));
  const double norm_b = std::sqrt(e->h_la_scalars[kSRnorm2]);
  summary->initial_gradient_norm = norm_b;
  summary->final_residual_norm = norm_b;
  summary->termination = 1;
  double q0 = 0.0;  // Q(x) = -x.(b + r) / 2 at x = 0
  int cur = 0;
  if (!(norm_b > 0.0) || !std::isfinite(norm_b)) {
    summary->termination = std::isfinite(norm_b) ? 0 : 2;
  } else {
    for (int it = 1; it <= options->max_num_iterations; ++it) {
      double* Sc = S + cur * kSCount;
      const int nxt = (cur + 1) % 3;
      double* Sn = S + nxt * kSCount;
      // q = J'(J p): one pass over the values when every type's rows fit in registers
      CB200_CUDA(e, cudaMemsetAsync(q, 0, col_bytes, s));
      if (one_pass) {
        if ((rc = RunJacobianWalk(e, kOpNormal, p, q)) != CB200_OK) return rc;
      } else {
        if ((rc = RunJacobianWalk(e, kOpRight, p, w)) != CB200_OK) return rc;
        if ((rc = RunJacobianWalk(e, kOpLeft, w, q)) != CB200_OK) return rc;
      }
      if ((rc = SumOverRanks(e, q, ne)) != CB200_OK) return rc;
      CgDotKernel<<<vgrid, 256, 0, s>>>(ne, p, q, d2, Sc, red);
      CB200_CUDA(e, cudaMemsetAsync(Sn, 0, kSCount * sizeof(double), s));
      CgUpdateKernel<<<vgrid, 256, 0, s>>>(ne, p, q, d2, minv, b, x, r, Sc, Sn, red);
      CgDirectionKernel<<<vgrid, 256, 0, s>>>(ne, r, minv, p, Sc, Sn);
      CB200_CUDA(e, cudaMemcpyAsync(e->h_la_scalars, S, 3 * kSCount * sizeof(double),
                                    cudaMemcpyDeviceToHost, s));
      CB200_CUDA(e, cudaStreamSynchronize(s));
      const double* hc = e->h_la_scalars + cur * kSCount;
      const double* hn = e->h_la_scalars + nxt * kSCount;
      summary->num_iterations = it;
      const double pq = hc[kSPq], rho = hc[kSRho];
      if (!(pq > 0.0) || !std::isfinite(pq) || !std::isfinite(rho) || !std::isfinite(hn[kSRho])) {
        summary->termination = 2;  // the update used a bad alpha: the caller rejects the step
        break;
      }
      summary->final_residual_norm = std::sqrt(hn[kSRnorm2]);
      const double q1 = -0.5 * hn[kSXbr];
      const double zeta = it * (q1 - q0) / q1;
      q0 = q1;
      cur = nxt;
      if (it >= options->min_num_iterations &&
          (summary->final_residual_norm <= options->r_tolerance * norm_b ||
           zeta < options->q_tolerance)) {
        summary->termination = 0;
        break;
      }
    }
  }
  // model terms for the trust-region step: (J y).b and |J y|^2 over the residuals
  double* Sm = S + ((cur + 2) % 3) * kSCount;
  CB200_CUDA(e, cudaMemsetAsync(Sm, 0, kSCount * sizeof(double), s));
  if ((rc = RunJacobianWalk(e, kOpRight, x, w)) != CB200_OK) return rc;
  CgModelKernel<<<rgrid, 256, 0, s>>>(m, w, residuals, Sm, red);
  if (e->comm && e->world > 1) {
    NcclApi* n = GetNccl();
    if (n->AllReduce(Sm + kSJyB, Sm + kSJyB, 2, kNcclFloat64, kNcclSum, e->comm, s) != 0)
      return e->Fail(CB200_ERROR_NCCL, "NCCL all-reduce failed");
  }
  CB200_CUDA(e, cudaMemcpyAsync(e->h_la_scalars, Sm, kSCount * sizeof(double),
                                cudaMemcpyDeviceToHost, s));
  if (solution)
    CB200_CUDA(e, cudaMemcpyAsync(solution, x, col_bytes, cudaMemcpyDeviceToHost, s));
  CB200_CUDA(e, cudaEventRecord(e->ev[4], s));
  CB200_CUDA(e, cudaStreamSynchronize(s));
  summary->jy_dot_b = e->h_la_scalars[kSJyB];
  summary->jy_squared_norm = e->h_la_scalars[kSJy2];
  float ms = 0;
  cudaEventElapsedTime(&ms, e->ev[0], e->ev[4]);
  summary->solve_ms = ms;
  return CB200_OK;
}

int cb200_engine_cgnr_solve(cb200_engine* e, const double* d_squared,
                            const cb200_cgnr_options* options, double* solution,
                            cb200_cgnr_summary* summary) {
  NvtxRange nvtx_range("cb200_engine_cgnr_solve");
  if (e && !solution) return e->Fail(CB200_ERROR_INVALID_ARGUMENT, "solution is required");
  return CgnrSolve(e, d_squared, false, options, solution, summary);
}

// ---- the trust-region iteration without the host (SURVEY.md section 8(f) 2-3): the state, the
// step and the LM / Jacobi diagonals live in HBM between iterations.
static int PrepareTrustRegion(cb200_engine* e) {
  if (!e) return CB200_ERROR_INVALID_ARGUMENT;
  if (!e->finalized) return e->Fail(CB200_ERROR_NOT_FINALIZED, "not finalized");
  if (e->planning) return e->Fail(CB200_ERROR_CUDA, "planning-only engine: no device, no CPU fallback");
  CB200_CUDA(e, cudaSetDevice(e->device));
  for (auto& b : e->tr_state) CB200_CUDA(e, b.Resize(static_cast<size_t>(e->num_parameters) + 4));
  CB200_CUDA(e, e->tr_scale.Resize(static_cast<size_t>(e->num_effective) + 1));
  CB200_CUDA(e, e->tr_diagonal.Resize(static_cast<size_t>(e->num_effective) + 1));
  CB200_CUDA(e, e->tr_delta.Resize(static_cast<size_t>(e->num_effective) + 1));
  return CB200_OK;
}

int cb200_engine_state_upload(cb200_engine* e, const double* state) {
  NvtxRange nvtx_range("cb200_engine_state_upload");
  int rc = PrepareTrustRegion(e);
  if (rc != CB200_OK) return rc;
  if (!state) return e->Fail(CB200_ERROR_INVALID_ARGUMENT, "state is required");
  CB200_CUDA(e, cudaMemcpyAsync(e->tr_state[0].ptr, state, sizeof(double) * e->num_parameters,
                                cudaMemcpyHostToDevice, e->stream));
  CB200_CUDA(e, cudaStreamSynchronize(e->stream));
  e->tr_state_valid = true;
  return CB200_OK;
}

int cb200_engine_state_download(cb200_engine* e, int which, double* state) {
  NvtxRange nvtx_range("cb200_engine_state_download");
  int rc = PrepareTrustRegion(e);
  if (rc != CB200_OK) return rc;
  if (!state || which < 0 || which > 1 || !e->tr_state_valid)
    return e->Fail(CB200_ERROR_INVALID_ARGUMENT, "state_download: no such state");
  CB200_CUDA(e, cudaMemcpyAsync(state, e->tr_state[which].ptr, sizeof(double) * e->num_parameters,
                                cudaMemcpyDeviceToHost, e->stream));
  CB200_CUDA(e, cudaStreamSynchronize(e->stream));
  return CB200_OK;
}

int cb200_engine_evaluate_state(cb200_engine* e, int which, uint32_t flags, int want_residuals,
                                int want_gradient, int want_jacobian, double* cost) {
  NvtxRange nvtx_range("cb200_engine_evaluate_state");
  int rc = PrepareTrustRegion(e);
  if (rc != CB200_OK) return rc;
  if (which < 0 || which > 1 || !e->tr_state_valid)
    return e->Fail(CB200_ERROR_INVALID_ARGUMENT, "evaluate_state: upload a state first");
  if (e->plus_pool > 0)
    return e->Fail(CB200_ERROR_INVALID_ARGUMENT,
                   "evaluate_state: a manifold needs host plus-Jacobians (use cb200_engine_evaluate)");
  return cb200_engine_evaluate_device(e, e->tr_state[which].ptr, nullptr, flags, want_residuals,
                                      want_gradient, want_jacobian, cost);
}

int cb200_engine_accept_candidate(cb200_engine* e) {
  if (!e || !e->tr_state_valid) return CB200_ERROR_INVALID_ARGUMENT;
  std::swap(e->tr_state[0], e->tr_state[1]);
  return CB200_OK;
}

int cb200_engine_jacobi_scale(cb200_engine* e, int compute) {
  int rc = PrepareLinearAlgebra(e, false);
  if (rc == CB200_OK) rc = PrepareTrustRegion(e);
  if (rc != CB200_OK) return rc;
  cudaStream_t s = e->stream;
  const int ne = e->num_effective;
  const int grid = std::max(1, std::min((ne + 255) / 256, kMaxVectorGrid));
  if (compute) {
    double* col = e->la_col[7].ptr;
    CB200_CUDA(e, cudaMemsetAsync(col, 0, static_cast<size_t>(ne) * sizeof(double), s));
    if ((rc = RunJacobianWalk(e, kOpColumnNorm, nullptr, col)) != CB200_OK) return rc;
    if ((rc = SumOverRanks(e, col, ne)) != CB200_OK) return rc;
    JacobiScaleKernel<<<grid, 256, 0, s>>>(ne, col, e->tr_scale.ptr);
    e->tr_scale_valid = true;
  }
  if (!e->tr_scale_valid)
    return e->Fail(CB200_ERROR_INVALID_ARGUMENT, "jacobi_scale: no scale computed yet");
  {
    // J <- J diag(scale), and the squared column norms of the result in the same pass: the
    // LM diagonal and the preconditioner of this iteration need them (la_col[7])
    double* col = e->la_col[7].ptr;
    CB200_CUDA(e, cudaMemsetAsync(col, 0, static_cast<size_t>(ne) * sizeof(double), s));
    if ((rc = RunJacobianWalk(e, kOpScaleNorm, e->tr_scale.ptr, col)) != CB200_OK) return rc;
    if ((rc = SumOverRanks(e, col, ne)) != CB200_OK) return rc;
    e->colnorm_valid = true;
  }
  CB200_CUDA(e, cudaStreamSynchronize(s));
  return CB200_OK;
}

int cb200_engine_trust_region_step(cb200_engine* e, const cb200_step_options* options,
                                   cb200_step_summary* summary) {
  NvtxRange nvtx_range("cb200_engine_trust_region_step");
  int rc = PrepareLinearAlgebra(e, true);
  if (rc == CB200_OK) rc = PrepareTrustRegion(e);
  if (rc != CB200_OK) return rc;
  if (!options || !summary || !e->tr_state_valid)
    return e->Fail(CB200_ERROR_INVALID_ARGUMENT, "trust_region_step: options, summary and an "
                                                 "uploaded state are required");
  if (!e->plus_on_device)
    return e->Fail(CB200_ERROR_INVALID_ARGUMENT,
                   "trust_region_step: a parameter block has a manifold the device cannot apply");
  cudaStream_t s = e->stream;
  const int ne = e->num_effective;
  const int grid = std::max(1, std::min((ne + 255) / 256, kMaxVectorGrid));
  std::memset(summary, 0, sizeof(*summary));
  // LM diagonal (levenberg_marquardt_strategy.cc:83-96): clamp(diag(J'J)) / radius
  if (!options->reuse_diagonal || !e->tr_diagonal_valid) {
    double* col = e->la_col[7].ptr;
    if (!e->colnorm_valid) {
      CB200_CUDA(e, cudaMemsetAsync(col, 0, static_cast<size_t>(ne) * sizeof(double), s));
      if ((rc = RunJacobianWalk(e, kOpColumnNorm, nullptr, col)) != CB200_OK) return rc;
      if ((rc = SumOverRanks(e, col, ne)) != CB200_OK) return rc;
      e->colnorm_valid = true;
    }
    ClampKernel<<<grid, 256, 0, s>>>(ne, col, options->min_lm_diagonal, options->max_lm_diagonal,
                                     e->tr_diagonal.ptr);
    e->tr_diagonal_valid = true;
  }
  DivideKernel<<<grid, 256, 0, s>>>(ne, e->tr_diagonal.ptr, options->radius, e->la_col[6].ptr);
  if ((rc = CgnrSolve(e, nullptr, true, &options->cg, nullptr, &summary->cg)) != CB200_OK) return rc;
  // step = -y (times the Jacobi scale); |step|, |x|; candidate = x (+) step
  const ScalarReduce red{e->la_partials.ptr, e->la_arrivals.ptr};
  double* S = e->la_scalars.ptr;
  StepKernel<<<grid, 256, 0, s>>>(ne, e->la_col[0].ptr,
                                  e->tr_scale_valid ? e->tr_scale.ptr : nullptr, e->tr_delta.ptr, S,
                                  red);
  const int np = e->num_parameters;
  const int pgrid = std::max(1, std::min((np + 255) / 256, kMaxVectorGrid));
  SquaredNormKernel<<<pgrid, 256, 0, s>>>(np, e->tr_state[0].ptr, S + 1, red);
  const int bgrid = std::max(1, std::min((e->num_active + 255) / 256, 148 * 16));
  CB200_CUDA(e, cudaMemsetAsync(e->d_status.ptr, 0, sizeof(int32_t), s));
  PlusKernel<<<bgrid, 256, 0, s>>>(e->num_active, e->d_pb_table.ptr, e->tr_state[0].ptr,
                                   e->tr_delta.ptr, e->tr_state[1].ptr, e->d_status.ptr);
  CB200_CUDA(e, cudaMemcpyAsync(e->h_la_scalars, S, 2 * sizeof(double), cudaMemcpyDeviceToHost, s));
  CB200_CUDA(e, cudaMemcpyAsync(e->h_la_scalars + 2, e->d_status.ptr, sizeof(int32_t),
                                cudaMemcpyDeviceToHost, s));
  CB200_CUDA(e, cudaStreamSynchronize(s));
  int32_t bad = 0;
  std::memcpy(&bad, e->h_la_scalars + 2, sizeof(bad));
  summary->step_norm = std::sqrt(e->h_la_scalars[0]);
  summary->state_norm = std::sqrt(e->h_la_scalars[1]);
  summary->plus_ok = bad == 0;
  // step = -y: model cost change = (J y).r - |J y|^2 / 2
  summary->model_cost_change = summary->cg.jy_dot_b - 0.5 * summary->cg.jy_squared_norm;
  return CB200_OK;
}

int cb200_engine_gradient_max_norm(cb200_engine* e, double* out) {
  if (!e || !out) return CB200_ERROR_INVALID_ARGUMENT;
  if (!e->finalized || e->planning) return e->Fail(CB200_ERROR_NOT_FINALIZED, "no device state");
  int rc = PrepareLinearAlgebra(e, false);
  if (rc != CB200_OK) return rc;
  cudaStream_t s = e->stream;
  const int ne = e->num_effective;
  const int grid = std::max(1, std::min((ne + 255) / 256, kMaxVectorGrid));
  unsigned long long* slot = reinterpret_cast<unsigned long long*>(e->la_scalars.ptr + 2);
  CB200_CUDA(e, cudaMemsetAsync(slot, 0, sizeof(*slot), s));
  MaxAbsKernel<<<grid, 256, 0, s>>>(ne, e->gradcost, slot);
  CB200_CUDA(e, cudaMemcpyAsync(e->h_la_scalars, slot, sizeof(double), cudaMemcpyDeviceToHost, s));
  CB200_CUDA(e, cudaStreamSynchronize(s));
  *out = e->h_la_scalars[0];
  return CB200_OK;
}

int cb200_engine_shard_info(cb200_engine* e, int32_t* rb_begin, int32_t* rb_end,
                            int32_t* residual_begin, int32_t* residual_end, int64_t* segments,
                            int32_t max_segments) {
  if (!e || !e->finalized) return -1;
  if (rb_begin) *rb_begin = e->rb_begin;
  if (rb_end) *rb_end = e->rb_end;
  if (residual_begin) *residual_begin = e->res_begin;
  if (residual_end) *residual_end = e->res_end;
  const int n = static_cast<int>(e->segments.size());
  for (int i = 0; i < n && i < max_segments; ++i) {
    segments[3 * i + 0] = e->segments[i].global_begin;
    segments[3 * i + 1] = e->segments[i].length;
    segments[3 * i + 2] = e->segments[i].local_begin;
  }
  return n;
}

int cb200_engine_exchange_plan(cb200_engine* e, int32_t* chunks, int32_t max_chunks,
                               int64_t* exclusive, int32_t* shared_count) {
  if (!e || !e->finalized || !e->peer_plan) return -1;
  const int n = static_cast<int>(e->chunk_table.size() / 4);
  if (chunks)
    for (int i = 0; i < n && i < max_chunks; ++i)
      std::memcpy(chunks + 4 * i, e->chunk_table.data() + 4 * i, 4 * sizeof(int32_t));
  if (exclusive) {
    exclusive[0] = e->exclusive_begin;
    exclusive[1] = e->exclusive_length;
  }
  if (shared_count) *shared_count = e->shared_count;
  return n;
}

int cb200_engine_exchange_mode(cb200_engine* e) {
  if (!e || e->world <= 1) return 0;
  return e->peer_ready ? 2 : 1;
}

int cb200_engine_last_timing(cb200_engine* e, double* out4) {
  if (!e || !out4) return CB200_ERROR_INVALID_ARGUMENT;
  for (int i = 0; i < 4; ++i) out4[i] = e->timing[i];
  return CB200_OK;
}

// ---- host memory: lazy anonymous mappings + page-locking of sub-ranges.
namespace {
constexpr uint64_t kPage = 4096;
constexpr uint64_t kAllocMagic = 0x6362323030686d31ULL;
struct AllocHeader {
  uint64_t magic, total_bytes;
};
std::mutex g_pin_mutex;
std::vector<std::pair<uintptr_t, uintptr_t>> g_pinned;  // disjoint [begin, end), sorted

int PinRange(uintptr_t lo, uintptr_t hi) {
  std::lock_guard<std::mutex> lock(g_pin_mutex);
  int count = 0;
  if (cudaGetDeviceCount(&count) != cudaSuccess || count == 0) {
    cudaGetLastError();
    return CB200_OK;  // nothing to DMA to on this machine
  }
  // Register only the pages not covered by an earlier pin.
  std::vector<std::pair<uintptr_t, uintptr_t>> todo;
  uintptr_t cursor = lo;
  for (const auto& r : g_pinned) {
    if (r.second <= cursor) continue;
    if (r.first >= hi) break;
    if (r.first > cursor) todo.emplace_back(cursor, r.first);
    cursor = std::max(cursor, r.second);
    if (cursor >= hi) break;
  }
  if (cursor < hi) todo.emplace_back(cursor, hi);
  for (const auto& t : todo) {
    cudaError_t err = cudaHostRegister(reinterpret_cast<void*>(t.first), t.second - t.first,
                                       cudaHostRegisterPortable);
    if (err != cudaSuccess) {
      cudaGetLastError();
      return CB200_ERROR_CUDA;
    }
    g_pinned.push_back(t);
  }
  std::sort(g_pinned.begin(), g_pinned.end());
  return CB200_OK;
}

void UnpinWithin(uintptr_t lo, uintptr_t hi) {
  std::lock_guard<std::mutex> lock(g_pin_mutex);
  std::vector<std::pair<uintptr_t, uintptr_t>> keep;
  for (const auto& r : g_pinned) {
    if (r.first >= lo && r.second <= hi) {
      cudaHostUnregister(reinterpret_cast<void*>(r.first));
      cudaGetLastError();
    } else {
      keep.push_back(r);
    }
  }
  g_pinned.swap(keep);
}
}  // namespace

void* cb200_host_alloc(uint64_t bytes) {
  const uint64_t total = ((bytes + kPage - 1) / kPage + 1) * kPage;
  void* p = mmap(nullptr, total, PROT_READ | PROT_WRITE, MAP_PRIVATE | MAP_ANONYMOUS, -1, 0);
  if (p == MAP_FAILED) return nullptr;
#ifdef MADV_HUGEPAGE
  // Large arrays (Jacobian values, residuals) are DMA targets: transparent huge pages cut
  // the number of pages the driver has to lock and map (a hint; ignored when unavailable).
  if (total >= (8u << 20)) madvise(p, total, MADV_HUGEPAGE);
#endif
  auto* h = static_cast<AllocHeader*>(p);
  h->magic = kAllocMagic;
  h->total_bytes = total;
  return static_cast<char*>(p) + kPage;
}

int cb200_host_pin(void* ptr, uint64_t bytes) {
  if (!ptr || bytes == 0) return CB200_OK;
  const uintptr_t lo = reinterpret_cast<uintptr_t>(ptr) / kPage * kPage;
  const uintptr_t hi = (reinterpret_cast<uintptr_t>(ptr) + bytes + kPage - 1) / kPage * kPage;
  return PinRange(lo, hi);
}

void cb200_host_free(void* q) {
  if (!q) return;
  char* p = static_cast<char*>(q) - kPage;
  auto* h = reinterpret_cast<AllocHeader*>(p);
  if (h->magic != kAllocMagic) return;
  const uint64_t total = h->total_bytes;
  UnpinWithin(reinterpret_cast<uintptr_t>(p), reinterpret_cast<uintptr_t>(p) + total);
  munmap(p, total);
}

}  // extern "C"
