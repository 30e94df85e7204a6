// The evaluation kernels (sm_100a) and their launch thunk.
//
// One instantiation per <CostFunctor, LossFunctionCUDA, kNumResiduals, Ns...>,
// emitted in the user's translation unit by ProblemCUDA::AddResidualBlock; the
// precompiled engine (csrc/engine.cu) calls it through the C-ABI function pointer
// cb200_launch_fn.  Replaces the reference's EvaluateKernel
// (include/ceres/internal/cuda_evaluator_kernel.h:301-422) and the pieces it
// calls: AutoDifferentiate (include/ceres/internal/autodiff.h:318-381),
// MatrixMultiply J * PlusJacobian (:163-173,355-371), Corrector
// (include/ceres/internal/corrector.h:82-213), ComputeGradient (:193-217) and
// WriteJacobians (:264-294).
//
// Per residual block the order of operations is the CPU evaluator's
// (internal/ceres/residual_block.cc:68-204): autodiff -> finite check ->
// J * PlusJacobian -> s = ||r||^2 (uncorrected) -> rho -> cost = rho[0] / 2 ->
// CorrectJacobian (uses uncorrected r) -> CorrectResiduals -> gradient J^T r
// (both corrected) -> scatter.
//
// Design (DESIGN.md section 3 has the numbers and the measurements behind each choice):
//  * one thread per residual block, Jets with compile-time sparsity masks
//    (ceres/jet.h): ~500 FP64 instructions and 160 registers for the BAL functor, no
//    local-memory spills, no per-thread Jacobian scratch in HBM;
//  * persistent CTAs with a three-stage software pipeline: state offsets two blocks
//    ahead in registers, parameters / functor / per-block integer tables one block ahead
//    through cp.async into shared memory (the parameter gather is warp-cooperative, so a
//    copy instruction touches a few sectors instead of 32), compute from shared memory;
//  * structure-of-arrays inputs, argument-major: every per-block table is read with
//    unit-stride copies;
//  * each Jacobian cell is written exactly once, straight to its final position in the
//    BlockSparseMatrix / CompressedRowSparseMatrix values array (no memset, no second
//    copy): a warp stages its 32 cells in shared memory in global layout and one TMA bulk
//    store moves the run;
//  * gradient: per-lane sums staged in shared memory and added with consecutive lanes on
//    consecutive addresses (red.global.add.f64); long runs of one parameter block are
//    pre-reduced with a segmented warp shuffle;
//  * cost: warp shuffle + one partial per thread block, summed in a fixed order;
//  * variants: Jet-free cost / residual kernel, plain, generic (manifolds, constant
//    blocks), and all-outputs instantiations of the last two with the output flags as
//    compile-time constants.
#ifndef CERES_B200_INTERNAL_EVALUATE_KERNEL_CUH_
#define CERES_B200_INTERNAL_EVALUATE_KERNEL_CUH_

#include <cuda_runtime.h>

#include <cstdint>
#include <type_traits>
#include <utility>

#include "ceres/jet.h"
#include "ceres_b200.h"

namespace ceres {
namespace internal {

constexpr int kEvaluateThreads = 128;  // threads per CTA (measured: see ResidentCtas)
// internal/ceres/array_utils.h: the value autodiff leaves in outputs a functor
// did not write; evaluations containing it are invalid.
constexpr double kImpossibleValue = 1e302;

template <int... Ns>
struct BlockDims {
  static constexpr int kNumBlocks = sizeof...(Ns);
  static constexpr int kNumParameters = (Ns + ... + 0);
  __host__ __device__ static constexpr int Size(int j) {
    constexpr int s[kNumBlocks > 0 ? kNumBlocks : 1] = {Ns...};
    return s[j];
  }
  __host__ __device__ static constexpr int Offset(int j) {
    int o = 0;
    for (int i = 0; i < j; ++i) o += Size(i);
    return o;
  }
  __host__ __device__ static constexpr int MaxSize() {
    int m = 0;
    for (int i = 0; i < kNumBlocks; ++i) m = Size(i) > m ? Size(i) : m;
    return m;
  }
  // 16-byte chunks of the aligned window that contains block j whether its first double
  // sits at an even or an odd offset of the state vector.
  __host__ __device__ static constexpr int WindowChunks(int j) { return Size(j) / 2 + 1; }
  // Cooperative gather: a lane's window of block j occupies WindowPitch(j) chunks, odd, so
  // that the owner's reads (lane stride = pitch * 16 bytes) spread over the banks: an even
  // pitch of 2 or 4 chunks puts 32 lanes on 2 or 4 bank groups (measured on the pose graph
  // <6,7,7>: 217 shared-memory wavefronts per tile for 58 ideal).
  __host__ __device__ static constexpr int WindowPitch(int j) { return WindowChunks(j) | 1; }
  __host__ __device__ static constexpr int PitchChunksBefore(int j) {
    int o = 0;
    for (int i = 0; i < j; ++i) o += WindowPitch(i);
    return o;
  }
};

template <typename Dims, typename Functor, typename T, std::size_t... Is>
__device__ __forceinline__ bool CallFunctor(const Functor& f, const T* x, T* out,
                                            std::index_sequence<Is...>) {
  return f((x + Dims::Offset(Is))..., out);
}

template <typename F, std::size_t... Js>
__device__ __forceinline__ void ForEachBlock(F&& f, std::index_sequence<Js...>) {
  (f(std::integral_constant<int, static_cast<int>(Js)>{}), ...);
}

// sqrt(rho') of the Corrector.  rho' is 1 for most blocks and a positive finite number
// otherwise: reciprocal square root + one correction step (within 1 ulp) instead of the
// library's sequence with its slow-path call; other arguments take the library function.
__device__ __forceinline__ double DeviceSqrt(double x) {
  if (x > 0.0 && x < 1.7976931348623157e308) {
    const double r = rsqrt(x);
    const double y = x * r;
    const double root = fma(fma(-y, y, x), 0.5 * r, y);
    return x == 1.0 ? 1.0 : root;  // (exactly 1 in the quadratic region of a robust loss)
  }
  return ::sqrt(x);
}

__device__ __forceinline__ bool IsValidValue(double x) {
  return ::fabs(x) <= 1.7976931348623157e308 && x != 1e302;
}

// Sums `v` over runs of consecutive lanes; `run_end` is one past the last lane of
// the calling lane's run.  Afterwards the first lane of every run holds its total.
template <int kCount>
__device__ __forceinline__ void WarpSegmentedSum(int run_end, double (&v)[kCount], int lane) {
#pragma unroll
  for (int d = 1; d < 32; d <<= 1) {
    const bool take = lane + d < run_end;
#pragma unroll
    for (int c = 0; c < kCount; ++c) {
      const double o = __shfl_down_sync(0xffffffffu, v[c], d);
      if (take) v[c] += o;
    }
  }
}

__device__ __forceinline__ int VolatileLaneId() {
  int lane;
  asm volatile("mov.u32 %0, %%laneid;" : "=r"(lane));
  return lane;
}

// (row, column) of element 32 * round + lane in a row-major [32][kSize] array.
template <int kSize>
struct RoundIndex {
  int row, c;
  __device__ __forceinline__ explicit RoundIndex(int lane) : row(lane / kSize), c(lane % kSize) {}
  __device__ __forceinline__ void Next() {
    row += 32 / kSize;
    c += 32 % kSize;
    if (c >= kSize) {
      c -= kSize;
      ++row;
    }
  }
};

__device__ __forceinline__ void RedAdd(double* address, double value) {
  // No return value wanted: red.global.add.f64 instead of an atom round trip.
  asm volatile("red.global.add.f64 [%0], %1;" ::"l"(address), "d"(value) : "memory");
}

// Predicated form: the compiler branches around an atomic inside an `if`; one predicated
// instruction avoids the BSSY / BRA / BSYNC per reduction round.
__device__ __forceinline__ void RedAddIf(bool condition, double* address, double value) {
  asm volatile(
      "{\n"
      "  .reg .pred p;\n"
      "  setp.ne.u32 p, %2, 0;\n"
      "  @p red.global.add.f64 [%0], %1;\n"
      "}" ::"l"(address), "d"(value), "r"(static_cast<unsigned>(condition))
      : "memory");
}

// Jacobian block helpers.  B is the kRes x kSize ambient block.
template <int kRes, int kSize>
struct BlockEpilogue {
  // B <- B * P, P row-major kSize x tangent (cuda_evaluator_kernel.h:355-371); used for
  // manifolds the device does not know (CB200_MANIFOLD_GENERIC).
  static __device__ __forceinline__ void MultiplyPlusJacobian(double (&B)[kRes][kSize],
                                                              const double* __restrict__ P,
                                                              int tangent) {
    double out[kRes][kSize];
#pragma unroll
    for (int c = 0; c < kSize; ++c) {
      if (c < tangent) {
        double p[kSize];
#pragma unroll
        for (int k = 0; k < kSize; ++k) p[k] = P[k * tangent + c];
#pragma unroll
        for (int r = 0; r < kRes; ++r) {
          double acc = 0.0;
#pragma unroll
          for (int k = 0; k < kSize; ++k) acc += B[r][k] * p[k];
          out[r][c] = acc;
        }
      } else {
#pragma unroll
        for (int r = 0; r < kRes; ++r) out[r][c] = 0.0;
      }
    }
#pragma unroll
    for (int r = 0; r < kRes; ++r)
#pragma unroll
      for (int c = 0; c < kSize; ++c) B[r][c] = out[r][c];
  }

  // corrector.h:174-213 CorrectJacobian, column by column.
  static __device__ __forceinline__ void Correct(double (&B)[kRes][kSize],
                                                 const double (&res)[kRes], double sqrt_rho1,
                                                 double alpha_sq_norm) {
    if (alpha_sq_norm == 0.0) {
#pragma unroll
      for (int r = 0; r < kRes; ++r)
#pragma unroll
        for (int c = 0; c < kSize; ++c) B[r][c] *= sqrt_rho1;
      return;
    }
#pragma unroll
    for (int c = 0; c < kSize; ++c) {
      double r_transpose_j = 0.0;
#pragma unroll
      for (int r = 0; r < kRes; ++r) r_transpose_j += B[r][c] * res[r];
#pragma unroll
      for (int r = 0; r < kRes; ++r)
        B[r][c] = sqrt_rho1 * (B[r][c] - alpha_sq_norm * res[r] * r_transpose_j);
    }
  }
};

// ---- asynchronous global -> shared copies (LDGSTS), used to prefetch the next
// residual block's parameters and functor while the current one is computed.
__device__ __forceinline__ void CpAsync8(void* smem, const void* gmem) {
  asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"(
                   static_cast<unsigned>(__cvta_generic_to_shared(smem))),
               "l"(gmem)
               : "memory");
}
__device__ __forceinline__ void CpAsync4(void* smem, const void* gmem) {
  asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"(
                   static_cast<unsigned>(__cvta_generic_to_shared(smem))),
               "l"(gmem)
               : "memory");
}
__device__ __forceinline__ void CpAsync16(void* smem, const void* gmem) {
  asm volatile("cp.async.ca.shared.global [%0], [%1], 16;" ::"r"(
                   static_cast<unsigned>(__cvta_generic_to_shared(smem))),
               "l"(gmem)
               : "memory");
}
__device__ __forceinline__ void CpAsyncCommit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int kPending>
__device__ __forceinline__ void CpAsyncWait() {
  asm volatile("cp.async.wait_group %0;" ::"n"(kPending) : "memory");
}

// ---- TMA bulk store shared -> global (cp.async.bulk): one instruction moves a
// warp's whole run of Jacobian cells; no LDS / STG / address arithmetic per element.
__device__ __forceinline__ void FenceProxyAsyncShared() {
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}
__device__ __forceinline__ void BulkStore(void* gmem, const void* smem, unsigned bytes) {
  asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(gmem),
               "r"(static_cast<unsigned>(__cvta_generic_to_shared(smem))), "r"(bytes)
               : "memory");
}
__device__ __forceinline__ void BulkCommit() {
  asm volatile("cp.async.bulk.commit_group;" ::: "memory");
}
// Waits until the bulk copies issued by this thread have finished READING shared memory.
__device__ __forceinline__ void BulkWaitRead() {
  asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
}
__device__ __forceinline__ void BulkWaitAll() {
  asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");
}

__host__ __device__ constexpr int MaxInt(int a, int b) { return a > b ? a : b; }

// Accumulates evidence of a non-finite value; Bad() is true iff one was seen.
struct FiniteCheck {
  // Every accumulator stays 0 iff its values are finite (0 * Inf = NaN).  One chain measured
  // fastest on B200 (BAL L: 2.28 ms against 2.32 ms with four - the extra accumulators cost
  // registers).  The chain array and its counter stay although kChains is 1: where a
  // caller's loop is not fully unrolled, a plain scalar accumulator changes the kernel's
  // registers and stack frame (the pose-graph cost kernels, test functors), unmeasured.
  static constexpr int kChains = 1;
  double acc[kChains] = {};
  int next = 0;  // folds to a constant once the callers' loops are unrolled
  __device__ __forceinline__ void Add(double x) {
    acc[next] = ::fma(x, 0.0, acc[next]);
    next = next + 1 == kChains ? 0 : next + 1;
  }
  __device__ __forceinline__ bool Bad() const {
    double sum = acc[0];
#pragma unroll
    for (int k = 1; k < kChains; ++k) sum += acc[k];
    return !(sum == 0.0);
  }
};

// Loss classes may declare `static constexpr bool kNonPositiveCurvature = true` (rho'' <= 0
// for every s, e.g. Huber, Cauchy): the Corrector's alpha branch is then dead code.
template <typename Loss, typename = void>
struct LossCurvature {
  static constexpr bool kNonPositive = false;
};
template <typename Loss>
struct LossCurvature<Loss, std::enable_if_t<Loss::kNonPositiveCurvature || true>> {
  static constexpr bool kNonPositive = Loss::kNonPositiveCurvature;
};

// Kernel variants.
constexpr int kVariantCost = 0;     // cost / residuals only: plain doubles, no Jets
constexpr int kVariantPlain = 1;    // Jets; no manifold and no constant block in this type
constexpr int kVariantGeneric = 2;  // Jets; per-block manifold projection / constant blocks
// kVariantPlain specialised for the call the minimizer makes after every accepted step: all
// outputs, loss applied, block-sparse values.  The output flags become compile-time
// constants, which removes their (uniform) branches and lets the compiler schedule across.
constexpr int kVariantPlainAll = 3;
constexpr int kVariantGenericAll = 4;  // kVariantGeneric with all outputs (either value layout)
// The two all-outputs variants are instantiated twice: reading the per-block integer tables
// (any program), and `kAffine`, for types whose tables are arithmetic progressions
// (cb200_launch_args::affine: one residual-block type laid out in program order, e.g. bundle
// adjustment): positions are computed from the block index, nothing is fetched, the
// contiguity of a warp's Jacobian cells is known without a vote, and 16-20 bytes per block
// of index traffic disappear.

// ---- derivative passes.  Wide problems (pose graphs: 14 derivative lanes x 6 residuals
// = 90 live doubles of output alone) are differentiated in several passes, each seeding
// only some parameter blocks (Jet width = their total size, all other blocks constants):
// the scalar part is recomputed per pass but registers per thread drop by the pass count,
// which removes the local-memory spills that otherwise dominate.  Small problems use one pass.
template <int kRes, int... Ns>
struct PassPlan {
  using Dims = BlockDims<Ns...>;
  static constexpr int kNB = Dims::kNumBlocks;
  // Live output doubles (residuals x parameters) up to which one pass is used.  BAL (2 x 12)
  // in two passes, i.e. a limit of 20, measured 2.09 ms against 1.84 ms on B200 (DESIGN.md 3.1).
  static constexpr int kSinglePassLimit = 40;
  static constexpr bool kSinglePass = kRes * Dims::kNumParameters <= kSinglePassLimit;
  static constexpr int kMaxWidth = Dims::MaxSize() > 8 ? Dims::MaxSize() : 8;
  // pass index of block j: greedy grouping of consecutive blocks up to kMaxWidth lanes
  __host__ __device__ static constexpr int PassOf(int j) {
    if (kSinglePass) return 0;
    int pass = 0, width = 0;
    for (int i = 0; i <= j; ++i) {
      if (width + Dims::Size(i) > kMaxWidth && width > 0) { ++pass; width = 0; }
      width += Dims::Size(i);
    }
    return pass;
  }
  static constexpr int kNumPasses = PassOf(kNB - 1) + 1;
  __host__ __device__ static constexpr int FirstBlock(int pass) {
    for (int j = 0; j < kNB; ++j) if (PassOf(j) == pass) return j;
    return kNB;
  }
  __host__ __device__ static constexpr int EndBlock(int pass) {
    int e = 0;
    for (int j = 0; j < kNB; ++j) if (PassOf(j) == pass) e = j + 1;
    return e;
  }
  __host__ __device__ static constexpr int Width(int pass) {
    int w = 0;
    for (int j = 0; j < kNB; ++j) if (PassOf(j) == pass) w += Dims::Size(j);
    return w;
  }
  __host__ __device__ static constexpr int MaxWidth() {
    int w = 0;
    for (int p = 0; p < kNumPasses; ++p) w = Width(p) > w ? Width(p) : w;
    return w;
  }
  // derivative lane of parameter i of block j inside its pass
  __host__ __device__ static constexpr int Lane(int j, int i) {
    return Dims::Offset(j) - Dims::Offset(FirstBlock(PassOf(j))) + i;
  }
};

__host__ __device__ constexpr int StagePitch(int n) { return n | 1; }
// Cells of at least this many doubles that do not form one run are written cooperatively
// (stage, then cell after cell with coalesced 16-byte stores) instead of by their thread.
constexpr int kCooperativeCellDoubles = 32;
// Where argument j's 32 cells start in a warp's Jacobian staging region, for a pass that
// begins at block `first`; j == `end` gives the size of the region.  Arguments whose cells
// can take the cooperative path get four doubles of slack per lane for its padded pitch.
template <int kRes, typename Dims>
__host__ __device__ constexpr int StageOffset(int first, int j) {
  int doubles = 0;
  for (int i = first; i < j; ++i)
    doubles += kRes * Dims::Size(i) + (kRes * Dims::Size(i) >= kCooperativeCellDoubles ? 4 : 0);
  return 32 * doubles;
}
template <int kRes, int... Ns>
__host__ __device__ constexpr int MaxStageDoubles() {
  using Plan = PassPlan<kRes, Ns...>;
  int m = 0;
  for (int p = 0; p < Plan::kNumPasses; ++p) {
    const int d = StageOffset<kRes, BlockDims<Ns...>>(Plan::FirstBlock(p), Plan::EndBlock(p));
    m = d > m ? d : m;
  }
  return m;
}

// CTAs per SM the Jet kernels are compiled for.  Measured on B200 for the BAL functor
// (scripts/kbench.cu, profiles/r2_kbench_variants.txt): 3 CTAs x 128 threads (162 registers)
// 1.98 ms; 4 x 128 (128 registers, no spills) 2.08; 2 x 128 (242 registers) 2.36; 5 x 96 2.16;
// 3 x 160 2.19; 7 x 64 2.19 - more warps cost the compiler the registers it uses to overlap
// independent Jet lanes, fewer warps cost latency hiding.  Wide problems get 2 CTAs.
constexpr int kResidentCtasSmall = 3;
constexpr int kResidentCtasCost = 6;    // CTAs per SM wanted for the Jet-free variant
constexpr int kResidentCtasTables = 3;  // variants that stage the int tables: more shared memory
__host__ __device__ constexpr int ResidentCtas(int num_residuals, int num_parameters,
                                               bool int_tables = false) {
  return (num_parameters <= 13 && num_residuals <= 3)
             ? (int_tables ? kResidentCtasTables : kResidentCtasSmall)
             : 2;
}
// Dynamic shared memory a CTA may use so that `ctas` of them fit on an SM (228 KB per SM,
// 1 KB reserved per CTA, at most 227 KB for one CTA).
__host__ __device__ constexpr int SmemBudget(int ctas) {
  const int share = 228 * 1024 / ctas - 1024;
  return share < 227 * 1024 ? share : 227 * 1024;
}

// Shared memory plan of a kernel instantiation.  Per CTA:
//   [parameters, two stages: per warp, the 16-byte windows of its 32 blocks]
//   [functor slot per thread, two stages]
//   [per-block integer tables, two stages — absent when kInts is false]
//   [per warp: Jacobian staging | gradient staging]
// Parameters, functor and tables are double-buffered: the copies for residual block k+1 are
// issued at the top of iteration k, into the stage block k-1 used, and land while block k is
// computed.
template <typename Functor, bool kInts, int kRes, int... Ns>
struct SmemPlan {
  using Dims = BlockDims<Ns...>;
  static constexpr int kNB = Dims::kNumBlocks;
  // bytes per thread of one parameter stage
  static constexpr int kParamBytes = Dims::PitchChunksBefore(kNB) * 16;
  static constexpr bool kFunctorInSmem =
      (sizeof(Functor) % 4 == 0) && (alignof(Functor) <= 16) && (sizeof(Functor) <= 128);
  static constexpr int kFunctorBytes = kFunctorInSmem ? static_cast<int>(sizeof(Functor)) : 0;
  // Functor slots are padded to 16 bytes so every slot is 16-byte aligned.
  static constexpr int kFunctorSlot = (kFunctorBytes + 15) / 16 * 16;
  // Per-block int tables that travel with the parameters: [delta offset or block id]
  // and [Jacobian position] per argument, residual position, CRS row stride, loss index.
  static constexpr int kIntSlots = 2 * kNB + 3;
  static constexpr int kSlotDelta = 0, kSlotJpos = kNB, kSlotResidual = 2 * kNB,
                       kSlotRowStride = 2 * kNB + 1, kSlotLoss = 2 * kNB + 2;
  static constexpr int kIntStageBytes = kInts ? kIntSlots * 4 * kEvaluateThreads : 0;

  static constexpr int kParamOffset = 0;
  static constexpr int kParamStageBytes = kParamBytes * kEvaluateThreads;
  static constexpr int kFunctorOffset = 2 * kParamStageBytes;
  static constexpr int kFunctorStageBytes = kFunctorSlot * kEvaluateThreads;
  static constexpr int kIntOffset = kFunctorOffset + 2 * kFunctorStageBytes;
  static constexpr int kPrefetchRaw = kIntOffset + 2 * kIntStageBytes;
  static constexpr bool kFits = kPrefetchRaw <= 96 * 1024;
  static constexpr int kPrefetchBytes = kFits ? kPrefetchRaw : 0;

  static constexpr int kCtas = ResidentCtas(kRes, Dims::kNumParameters, kInts);
  // per warp: the cells of the arguments of one derivative pass side by side (Jacobian
  // staging; with several passes the region is reused pass after pass) ...
  static constexpr int kJacobianDoubles = MaxStageDoubles<kRes, Ns...>();
  // ... and one padded row per lane for the staged gradient reductions plus, per staged
  // element, its destination in the gradient (an int; -1 = nothing to add).  Within a
  // derivative pass every gradient is out before the first cell is staged, so the gradient
  // staging reuses the Jacobian staging buffer.
  static constexpr int kGradientStage = 48 * StagePitch(Dims::MaxSize());
  // (several passes: each pass waits for the previous pass's stores to leave the staging
  // region before its own gradient uses it, so the alias holds pass by pass)
  static constexpr bool kGradientAliasesJacobian = kGradientStage <= kJacobianDoubles;
  static constexpr int kGradientDoubles = kGradientAliasesJacobian ? 0 : kGradientStage;
  static constexpr int kWarps = kEvaluateThreads / 32;
  static constexpr bool kStageJacobian =
      kPrefetchBytes + kWarps * (kJacobianDoubles + kGradientDoubles) * 8 <= SmemBudget(kCtas);
  static constexpr int kGradientOffset =
      (kStageJacobian && !kGradientAliasesJacobian) ? kJacobianDoubles : 0;
  static constexpr int kWarpDoubles =
      kStageJacobian ? kJacobianDoubles + kGradientDoubles : kGradientStage;
  static constexpr int kJetBytes = kPrefetchBytes + kWarps * kWarpDoubles * 8;
  static constexpr int kCostBytes = kPrefetchBytes > 0 ? kPrefetchBytes : 64;
};

// The Jet-free cost / residual kernel needs ~80 registers and only the prefetch buffers, so
// more of its CTAs fit on an SM; it is latency bound (argument reduction of sincos,
// divisions), and the extra warps hide that.
__host__ __device__ constexpr int VariantCtas(int variant, int resident, int cost_bytes) {
  if (variant != kVariantCost) return resident;
  const int by_smem = (227 * 1024) / (cost_bytes + 1024);
  const int wanted = kResidentCtasCost;
  return by_smem < resident ? resident : (by_smem < wanted ? by_smem : wanted);
}

// One thread evaluates one residual block at a time and walks the type's blocks with a
// grid stride (persistent CTAs).  Software pipeline per thread:
//   iteration k:  [cp.async parameters + functor (+ int tables) of block k+1 -> other stage]
//                 [state offsets of block k+2 -> registers]
//                 [wait for block k's copies] functor of block k from shared memory
//                 epilogue of block k (loss, gradient, scatter)
// so the two dependent global loads (offset, then the gathered parameters) of a block are
// in flight while the blocks before it are computed instead of stalling
// the warp (v1 of this kernel: long-scoreboard stalls 7.5 of 15 cycles per issue, FP64 pipe
// 22% busy; profiles/r1_v1_ncu_summary.txt).  a.state must be 16-byte aligned and followed
// by at least two doubles of slack (the engine's state buffer is).
//
// kChunked (several ranks, cb200_launch_args::chunks): a warp evaluates whole CHUNKS of
// consecutive residual blocks instead of a grid stride.  The gradient entries of a chunk's
// exclusive range (the points of a bundle adjustment problem) are touched by that chunk
// only, so when its last tile is done the thread block copies them straight into the
// gradient buffers of the other ranks over NVLink (peer-mapped memory): the exchange of one
// chunk overlaps the evaluation of the next ones, tile by tile, inside the same kernel.
template <int kVariant, bool kAffine, bool kChunked, typename Functor, typename Loss, int kRes,
          int... Ns>
__global__ void __launch_bounds__(
    kEvaluateThreads,
    VariantCtas(kVariant,
                ResidentCtas(kRes, (Ns + ... + 0),
                             kVariant != kVariantCost &&
                                 (!kAffine || kVariant == kVariantGenericAll)),
                SmemPlan<Functor, false, kRes, Ns...>::kCostBytes))
    EvaluateKernel(const cb200_launch_args a) {
  using Dims = BlockDims<Ns...>;
  using Plan = PassPlan<kRes, Ns...>;
  constexpr int kNB = Dims::kNumBlocks;
  constexpr int kNP = Dims::kNumParameters;
  constexpr bool kJets = kVariant != kVariantCost;
  constexpr bool kGeneric = kVariant == kVariantGeneric || kVariant == kVariantGenericAll;
  constexpr bool kAll = kVariant == kVariantPlainAll || kVariant == kVariantGenericAll;
  static_assert(!kAffine || kAll, "affine tables are for the all-outputs variants");
  static_assert(!kChunked || (kAffine && !kGeneric), "chunks: plain all-outputs affine variant");
  // The int tables ride the cp.async pipeline except where positions are computed (affine)
  // and in the Jet-free variant (it needs one or two of them: read directly).
  // Generic variants keep the parameter-block ids there even when positions are computed:
  // the id heads a chain of two dependent loads that must not start inside the iteration.
  constexpr bool kInts = kJets && (!kAffine || kGeneric);
  using Smem = SmemPlan<Functor, kInts, kRes, Ns...>;
  const bool out_residuals = kAll || a.output_residuals;
  const bool out_jacobian = kAll || a.output_jacobian;
  const bool out_gradient = kAll || a.output_gradient;
  const bool apply_loss = kAll || a.apply_loss_function;
  const bool crs = kVariant != kVariantPlainAll && a.crs;
  constexpr bool kPrefetch = Smem::kFits;
  constexpr bool kStage = kJets && Smem::kStageJacobian;

  extern __shared__ __align__(16) unsigned char smem[];
  double* const wbuf = reinterpret_cast<double*>(smem + Smem::kPrefetchBytes) +
                       (threadIdx.x >> 5) * Smem::kWarpDoubles;
  double* const jbuf = wbuf;                                              // Jacobian staging
  double* const gbuf = wbuf + Smem::kGradientOffset;                      // gradient staging
  int* const obuf = reinterpret_cast<int*>(gbuf + 32 * StagePitch(Dims::MaxSize()));

  const int tid = threadIdx.x;
  const int lane = tid & 31;
  const int n = a.n;
  const int stride = gridDim.x * kEvaluateThreads;
  const int first = blockIdx.x * kEvaluateThreads + tid;
  // Every thread of a CTA runs the same number of iterations (warp collectives).
  const int cta_first = blockIdx.x * kEvaluateThreads;
  const int iterations = cta_first < n ? (n - cta_first + stride - 1) / stride : 0;

  auto clamp = [&](int rb) { return rb < n ? rb : n - 1; };
  // this warp's region of parameter stage `stage`
  auto stage_params = [&](int stage) {
    double* base =
        reinterpret_cast<double*>(smem + Smem::kParamOffset + stage * Smem::kParamStageBytes);
    return base + (tid >> 5) * 32 * (Smem::kParamBytes / 8);
  };
  auto stage_functor = [&](int stage) {
    return smem + Smem::kFunctorOffset + stage * Smem::kFunctorStageBytes +
           tid * Smem::kFunctorSlot;
  };
  auto stage_ints = [&](int stage) {
    return reinterpret_cast<int*>(smem + Smem::kIntOffset + stage * Smem::kIntStageBytes) + tid;
  };
  auto load_offsets = [&](int rb, int (&soff)[kNB]) {
    const int r = clamp(rb);
#pragma unroll
    for (int j = 0; j < kNB; ++j) soff[j] = __ldg(a.state_offset + static_cast<size_t>(j) * n + r);
  };
  // bit j: block j starts at an odd double of the state vector
  auto parity_of = [&](const int (&soff)[kNB]) {
    unsigned p = 0;
#pragma unroll
    for (int j = 0; j < kNB; ++j) p |= static_cast<unsigned>(soff[j] & 1) << j;
    return p;
  };
  // Issues the copies of residual block rb: its parameter blocks (into its warp's region of
  // parameter stage `stage`), its functor, and — table variants — its integers.
  auto prefetch = [&](int stage, int rb, const int (&soff)[kNB]) {
    if constexpr (kPrefetch) {
      double* dst = stage_params(stage);
      // The aligned window [start & ~1, ...) of W = Size/2 + 1 16-byte pieces holds a block
      // for either parity of its start; the owner reads from (start & 1) on.  The warp copies
      // the 32 windows of argument j as one stream of 32 * W pieces: consecutive lanes fetch
      // consecutive pieces of a window, so a copy instruction touches a handful of cache lines
      // instead of 32; shared layout [argument][lane][odd pitch of W | 1 pieces].
#pragma unroll
      for (int j = 0; j < kNB; ++j) {
        const int kW = Dims::WindowChunks(j);  // constant after unrolling
#pragma unroll
        for (int it = 0; it < kW; ++it) {
          const int e = it * 32 + lane;
          const int owner = e / kW;
          const int c = e - owner * kW;
          const int so = __shfl_sync(0xffffffffu, soff[j], owner);
          CpAsync16(dst + 2 * (32 * Dims::PitchChunksBefore(j) + owner * Dims::WindowPitch(j) + c),
                    a.state + ((so & ~1) + 2 * c));
        }
      }
      // The int tables of the block (consumed in the epilogue, from shared memory, so
      // no register is held across the functor).
      if constexpr (kInts) {
        const int r = clamp(rb);
        int* idst = stage_ints(stage);
#pragma unroll
        for (int j = 0; j < kNB; ++j) {
          const int32_t* tab = kGeneric ? a.parameter_block : a.delta_offset;
          CpAsync4(idst + (Smem::kSlotDelta + j) * kEvaluateThreads,
                   tab + static_cast<size_t>(j) * n + r);
          if (out_jacobian && !kAffine)
            CpAsync4(idst + (Smem::kSlotJpos + j) * kEvaluateThreads,
                     a.jacobian_pos + static_cast<size_t>(j) * n + r);
        }
        if (crs && out_jacobian && !kAffine)
          CpAsync4(idst + Smem::kSlotRowStride * kEvaluateThreads, a.jacobian_row_stride + r);
        if (out_residuals && !kAffine)
          CpAsync4(idst + Smem::kSlotResidual * kEvaluateThreads, a.residual_pos + r);
        if (a.loss_index)
          CpAsync4(idst + Smem::kSlotLoss * kEvaluateThreads, a.loss_index + r);
      }
      if constexpr (Smem::kFunctorInSmem) {
        const unsigned char* src = static_cast<const unsigned char*>(a.functors) +
                                   static_cast<size_t>(clamp(rb)) * sizeof(Functor);
        unsigned char* my_functor = stage_functor(stage);
        if constexpr (sizeof(Functor) % 16 == 0) {
#pragma unroll
          for (int b = 0; b < static_cast<int>(sizeof(Functor)); b += 16) CpAsync16(my_functor + b, src + b);
        } else if constexpr (sizeof(Functor) % 8 == 0) {
#pragma unroll
          for (int b = 0; b < static_cast<int>(sizeof(Functor)); b += 8) CpAsync8(my_functor + b, src + b);
        } else {
#pragma unroll
          for (int b = 0; b < static_cast<int>(sizeof(Functor)); b += 4) CpAsync4(my_functor + b, src + b);
        }
      }
      CpAsyncCommit();
    }
  };

  double cost_sum = 0.0;
  bool all_ok = true;
  bool bulk_pending = false;  // warp-uniform: a bulk store may still read the staging buffer

  // ---- the sequence of residual blocks of this thread.  Grid stride: first + k * stride.
  // Chunked: the tiles (kEvaluateThreads blocks) of chunks blockIdx.x, + gridDim.x, ...;
  // `walk` runs two tiles ahead of the one being computed (offsets are fetched two ahead,
  // copies issued one ahead).
  struct Walk { int c, t, lo, hi; };
  const int4* const chunk_table = reinterpret_cast<const int4*>(a.chunks);
  auto load_chunk = [&](Walk& w) {
    if (w.c < a.num_chunks) {
      if (chunk_table) {
        const int4 rec = __ldg(chunk_table + w.c);
        w.lo = rec.x;
        w.hi = rec.y;
      } else {  // uniform chunks, nothing to copy (cb200_launch_args::chunk_blocks)
        w.lo = w.c * a.chunk_blocks;
        w.hi = min(n, w.lo + a.chunk_blocks);
      }
    } else {
      w.lo = w.hi = n;
    }
  };
  // (chunks belong to WARPS: a warp that finishes a chunk fences and copies on its own while
  // the other warps of the thread block keep evaluating)
  // Chunks are drawn from a counter (a.status[1], zero at launch), one ahead: a static
  // round-robin leaves the warps with 8 or 9 chunks each (10 % of the kernel at 8 GPUs).
  auto draw_chunk = [&]() {
    int c = 0;
    if (lane == 0) c = atomicAdd(a.status + 1, 1);
    return __shfl_sync(0xffffffffu, c, 0);
  };
  int chunk_ahead = 0;
  auto walk_rb = [&](const Walk& w) { return w.lo + w.t * 32 + lane; };
  auto walk_advance = [&](Walk& w) {
    ++w.t;
    if (w.lo + w.t * 32 >= w.hi) {
      w.c = chunk_ahead;
      chunk_ahead = draw_chunk();
      w.t = 0;
      load_chunk(w);
    }
  };
  Walk walk{0, 0, 0, 0};
  int rb0 = first, hi0 = n, c0 = 0, rb1 = first + stride, hi1 = n, c1 = 0;
  if constexpr (kChunked) {
    walk.c = draw_chunk();
    chunk_ahead = draw_chunk();
    load_chunk(walk);
    rb0 = walk_rb(walk); hi0 = walk.hi; c0 = walk.c;
    walk_advance(walk);
    rb1 = walk_rb(walk); hi1 = walk.hi; c1 = walk.c;
    walk_advance(walk);
  }

  int soff_next[kNB];   // state offsets of the block whose prefetch is issued next
  int soff_cur[kNB];    // state offsets of the block being computed (fallback path)
  load_offsets(rb0, soff_cur);
  prefetch(0, rb0, soff_cur);
  unsigned parity_cur = parity_of(soff_cur);
  load_offsets(rb1, soff_next);

#pragma unroll 1
  for (int k = 0; kChunked ? c0 < a.num_chunks : k < iterations; ++k) {
    const int rb = kChunked ? rb0 : first + k * stride;
    const int limit = kChunked ? hi0 : n;  // blocks [.., limit) belong to this tile's chunk
    const bool valid = rb < limit;
    const int tt = valid ? rb : limit - 1;
    const int stage = k & 1;
    // first residual block of this warp: affine positions of a whole warp derive from it
    const int warp_rb = rb - lane;
    const bool warp_valid = warp_rb + 31 < limit;
    const int rb_next = kChunked ? rb1 : rb + stride;

    // The offsets of the next block arrived during the previous iteration: its copies go to
    // the other stage now and land while this block is computed.
    int soff_issue[kNB];
#pragma unroll
    for (int j = 0; j < kNB; ++j) soff_issue[j] = soff_next[j];
    const unsigned parity_issue = parity_of(soff_issue);
    // (a lambda called once: inlined as a unit, it keeps the instruction schedule the kernel
    // was measured with; the same statements written inline make the compiler order the loop
    // differently, e.g. 32 more instructions and 2 more registers in the affine BAL kernel)
    auto issue_next = [&]() {
      prefetch(stage ^ 1, rb_next, soff_issue);
      // The offsets of block k+2 are fetched right after the copies of block k+1 are issued:
      // the load then writes the registers the copies just released and is not needed for a
      // whole iteration.  Fetched before, ptxas keeps the loaded value in a temporary and
      // moves it into the loop-carried register at once, i.e. it waits for a load it issued
      // ~40 instructions earlier (one fifth of the kernel's stall samples,
      // profiles/r2_v10_offset_load_stall.txt).
      load_offsets(kChunked ? walk_rb(walk) : rb + 2 * stride, soff_next);
    };
    issue_next();

    if constexpr (kPrefetch) {
      // this thread's copies for block k have landed (block k+1's may be in flight) ...
      CpAsyncWait<1>();
      __syncwarp();  // ... and its warp's
    }

    // Per-block int tables: from the prefetched stage, computed (affine), or straight
    // from global memory (Jet-free variant; parameters too large for shared memory).
    const int* sints = stage_ints(stage);
    auto table = [&](int slot, const int32_t* global_table, size_t index) -> int {
      if constexpr (kPrefetch && kInts) {
        return sints[slot * kEvaluateThreads];
      } else {
        return __ldg(global_table + index);
      }
    };
    // Per argument: where the gradient goes, where the Jacobian block goes, how the
    // ambient columns map to tangent columns.
    int delta_off[kNB], jpos[kNB], tangent[kNB], kind[kNB], mparam[kNB], plus_off[kNB], key[kNB];
    if constexpr (kJets) {
#pragma unroll
      for (int j = 0; j < kNB; ++j) {
        const size_t at = static_cast<size_t>(j) * n + tt;
        if constexpr (kGeneric) {
          const int id = table(Smem::kSlotDelta + j, a.parameter_block, at);
          const int4* rec = reinterpret_cast<const int4*>(a.parameter_block_table) + 2 * id;
          const int4 r0 = __ldg(rec), r1 = __ldg(rec + 1);
          delta_off[j] = r0.y;
          tangent[j] = r0.z;
          kind[j] = r0.w;
          mparam[j] = r1.x;
          plus_off[j] = r1.y;
          key[j] = id;
        } else {
          // affine plain types have delta offset == state offset (cb200_launch_args::affine)
          delta_off[j] = kAffine ? 0 : table(Smem::kSlotDelta + j, a.delta_offset, at);
          tangent[j] = Dims::Size(j);
          kind[j] = CB200_MANIFOLD_NONE;
          mparam[j] = 0;
          plus_off[j] = -1;
          key[j] = delta_off[j];
        }
        if constexpr (kAffine) {
          jpos[j] = a.jacobian_base[j] + tt * a.jacobian_step[j];
        } else {
          jpos[j] = out_jacobian ? table(Smem::kSlotJpos + j, a.jacobian_pos, at) : 0;
        }
      }
    }
    int respos = 0;
    if (out_residuals) {
      // (the Jet-free variant has no affine instantiation and reads its tables straight from
      // global memory: take the computed position when the engine found the table affine)
      const bool computed = kAffine || (!kJets && (a.affine & CB200_AFFINE_RESIDUAL));
      respos = computed ? a.residual_base + tt * kRes : table(Smem::kSlotResidual, a.residual_pos, tt);
    }
    int row_stride_crs = 0;
    if constexpr (kJets) {
      if (crs && out_jacobian)
        row_stride_crs =
            kAffine ? a.row_stride : table(Smem::kSlotRowStride, a.jacobian_row_stride, tt);
    }
    const Loss* __restrict__ losses = static_cast<const Loss*>(a.loss_table);
    int loss_at = 0;
    if (a.loss_index)
      loss_at = table(Smem::kSlotLoss, a.loss_index, tt);  // (direct load when not staged)
    // One loss object for the whole type (the usual case): its bytes ride in the kernel
    // arguments, i.e. the constant bank, and become instruction operands; otherwise they
    // are loaded from the table (a global load per block whose latency is exposed: 4-8 % of
    // the Jet-free kernel's stall samples, profiles/r2_costonly_ncu_summary.txt).
    // (the loss table already holds byte copies of the host objects - with their unused
    // host vtable pointer - so a byte copy is all a loss needs to support)
    constexpr bool kInlineLoss = sizeof(Loss) % 8 == 0 && sizeof(Loss) <= CB200_INLINE_LOSS_BYTES;
    constexpr int kLossWords = kInlineLoss ? static_cast<int>(sizeof(Loss) / 8) : 1;
    struct alignas(8) LossBytes { unsigned long long w[kLossWords]; } loss_bytes;
    if constexpr (kInlineLoss) {
      if (a.loss_inline_size == sizeof(Loss)) {
#pragma unroll
        for (int w = 0; w < kLossWords; ++w) loss_bytes.w[w] = a.loss_inline[w];
      } else {
        const unsigned long long* src = reinterpret_cast<const unsigned long long*>(losses + loss_at);
#pragma unroll
        for (int w = 0; w < kLossWords; ++w) loss_bytes.w[w] = __ldg(src + w);
      }
    }
    const Loss& loss = kInlineLoss ? *reinterpret_cast<const Loss*>(&loss_bytes) : losses[loss_at];

    const double* sp = stage_params(stage);
    const Functor* functor_ptr;
    if constexpr (kPrefetch && Smem::kFunctorInSmem) {
      functor_ptr = reinterpret_cast<const Functor*>(stage_functor(stage));
    } else {
      functor_ptr = static_cast<const Functor*>(a.functors) + tt;
    }
    const Functor& functor = *functor_ptr;

    double xval[kNP];
    if constexpr (kPrefetch) {
      // The owner reads its windows in 16-byte pieces (lane pitch odd in pieces: conflict
      // free, 4 wavefronts per instruction) and picks the doubles by the block's parity; the
      // 8-byte reads at an even lane pitch are two-way bank conflicted (72 wavefronts per tile
      // for 48 ideal, against 28 this way) and the shared-memory pipe is the busiest unit.
#pragma unroll
      for (int j = 0; j < kNB; ++j) {
        constexpr int kMaxW = Dims::MaxSize() / 2 + 1;
        double2 w[kMaxW];
        const double2* src = reinterpret_cast<const double2*>(sp) +
                             (32 * Dims::PitchChunksBefore(j) + lane * Dims::WindowPitch(j));
#pragma unroll
        for (int c = 0; c < kMaxW; ++c)
          if (c < Dims::WindowChunks(j)) w[c] = src[c];
        const bool odd = (parity_cur >> j) & 1u;
#pragma unroll
        for (int i = 0; i < Dims::Size(j); ++i) {
          // element i of the block is double (parity + i) of the window
          const double even_pick = (i & 1) ? w[i / 2].y : w[i / 2].x;
          const double odd_pick = ((i + 1) & 1) ? w[(i + 1) / 2].y : w[(i + 1) / 2].x;
          xval[Dims::Offset(j) + i] = odd ? odd_pick : even_pick;
        }
      }
    } else {
#pragma unroll
      for (int j = 0; j < kNB; ++j)
#pragma unroll
        for (int i = 0; i < Dims::Size(j); ++i)
          xval[Dims::Offset(j) + i] = __ldg(a.state + soff_cur[j] + i);
    }

    double res[kRes];
    bool ok = true;
    double cost = 0.0;
    const double kNaN = __longlong_as_double(0x7ff8000000000000LL);

    if constexpr (!kJets) {
      // AutoDiffCostFunction::Evaluate with jacobians == nullptr.
#pragma unroll
      for (int r = 0; r < kRes; ++r) res[r] = kNaN;  // unwritten outputs stay invalid
      ok = CallFunctor<Dims>(functor, xval, res, std::make_index_sequence<kNB>{});
      FiniteCheck check;
#pragma unroll
      for (int r = 0; r < kRes; ++r) check.Add(res[r]);
      ok = ok && !check.Bad();

      double s = 0.0;
#pragma unroll
      for (int r = 0; r < kRes; ++r) s += res[r] * res[r];
      if (apply_loss) {
        double rho[3];
        loss.Evaluate(s, rho);
        cost = 0.5 * rho[0];
        if (out_residuals) {
          // corrector.h:82-147 then :159-166
          const double sqrt_rho1 = DeviceSqrt(rho[1]);
          double scaling = sqrt_rho1;
          if (!(s == 0.0 || rho[2] <= 0.0)) {
            const double D = 1.0 + 2.0 * s * rho[2] / rho[1];
            const double alpha = 1.0 - ::sqrt(D);
            scaling = sqrt_rho1 / (1 - alpha);
          }
#pragma unroll
          for (int r = 0; r < kRes; ++r) res[r] *= scaling;
        }
      } else {
        cost = 0.5 * s;
      }
    } else {
      // ---- where the Jacobian leaves through shared memory + TMA (warp-uniform plan)
      // BlockSparse: argument j's 32 cells are one run of the values array (always true
      // inside the E or F region); CompressedRow: the warp's 32 row groups are one run.
      bool bulk_arg[kNB];
      bool coop_arg[kNB];  // cells staged and written cooperatively, cell after cell
      bool bulk_all = false;
      int bulk_base[kNB];
      int bulk_all_base = 0;
#pragma unroll
      for (int j = 0; j < kNB; ++j) { bulk_arg[j] = false; coop_arg[j] = false; bulk_base[j] = 0; }
      // (made after the first functor call: the generic variants read tangent sizes and
      // gradient offsets from the parameter-block table, a dependent global load issued at
      // the top of the iteration; consumed here, before the functor, it stalled the warp for
      // the whole L2 round trip - 12 % of the pose-graph kernel's stall samples)
      auto make_store_plan = [&]() {
      if constexpr (kStage) {
        if (out_jacobian) {
          if (!crs) {
#pragma unroll
            for (int j = 0; j < kNB; ++j) {
              if constexpr (kAffine && !kGeneric) {
                // positions are an arithmetic progression: contiguity is a property of
                // the type, only the evenness of the warp's first cell varies
                const int base = a.jacobian_base[j] + warp_rb * a.jacobian_step[j];
                bulk_arg[j] = warp_valid && a.jacobian_step[j] == kRes * Dims::Size(j) &&
                              ((base & 1) == 0);
                bulk_base[j] = base;
              } else {
                const int t0 = __shfl_sync(0xffffffffu, tangent[j], 0);
                const int base = __shfl_sync(0xffffffffu, jpos[j], 0);
                const bool mine = valid && delta_off[j] >= 0 && tangent[j] == t0 &&
                                  jpos[j] == base + lane * kRes * t0;
                bulk_arg[j] = __all_sync(0xffffffffu, mine) && ((base & 1) == 0);
                bulk_base[j] = base;
                if (!bulk_arg[j]) {
                  const bool separate = valid && delta_off[j] >= 0 && tangent[j] == t0 &&
                                        ((jpos[j] & 1) == 0) && ((kRes * t0) % 2 == 0);
                  coop_arg[j] = kRes * Dims::Size(j) >= kCooperativeCellDoubles &&
                                __all_sync(0xffffffffu, separate);
                }
              }
            }
          } else {
            int lo = 0x7fffffff;
#pragma unroll
            for (int j = 0; j < kNB; ++j)
              if (delta_off[j] >= 0) lo = min(lo, jpos[j]);
            const int s0 = __shfl_sync(0xffffffffu, row_stride_crs, 0);
            const int base = __shfl_sync(0xffffffffu, lo, 0);
            const bool mine = valid && row_stride_crs == s0 && lo == base + lane * kRes * s0;
            bulk_all = Plan::kNumPasses == 1 && __all_sync(0xffffffffu, mine) &&
                       ((base & 1) == 0) && s0 > 0;
            bulk_all_base = base;
          }
        }
      }
      };
      double sqrt_rho1 = 1.0, residual_scaling = 1.0, alpha_sq_norm = 0.0;
      bool correct = false;
      double res_corrected[kRes];

      // ---- derivative passes
      auto pass = [&](auto pc) {
        constexpr int p = decltype(pc)::value;
        constexpr int kW = Plan::Width(p);
        constexpr int kFirst = Plan::FirstBlock(p), kEnd = Plan::EndBlock(p);
        using JetT = Jet<double, kW>;
        JetT x[kNP];
#pragma unroll
        for (int j = 0; j < kNB; ++j)
#pragma unroll
          for (int i = 0; i < Dims::Size(j); ++i)
            x[Dims::Offset(j) + i] = (j >= kFirst && j < kEnd)
                                         ? JetT(xval[Dims::Offset(j) + i], Plan::Lane(j, i))
                                         : JetT(xval[Dims::Offset(j) + i]);
        JetT out[kRes];
        // autodiff.h:358-363 invalidates the outputs with kImpossibleValue and the CPU
        // evaluator rejects evaluations that still contain it
        // (residual_block_utils.cc:70-95).  Here unwritten outputs are NaN, so the
        // finite check below covers both conditions.
#pragma unroll
        for (int r = 0; r < kRes; ++r) out[r] = JetT::Filled(kNaN, kNaN);
        ok = CallFunctor<Dims>(functor, x, out, std::make_index_sequence<kNB>{}) && ok;
        if constexpr (p == 0) make_store_plan();

        FiniteCheck check;
#pragma unroll
        for (int r = 0; r < kRes; ++r) {
          if (p == 0) check.Add(out[r].a);
#pragma unroll
          for (int i = 0; i < kW; ++i)
            if (out[r].lane(i)) check.Add(out[r].v[i]);
        }
        ok = ok && !check.Bad();

        if constexpr (p == 0) {
          double s = 0.0;
#pragma unroll
          for (int r = 0; r < kRes; ++r) {
            res[r] = out[r].a;
            s += res[r] * res[r];
          }
          if (apply_loss) {
            double rho[3];
            loss.Evaluate(s, rho);
            cost = 0.5 * rho[0];
            sqrt_rho1 = DeviceSqrt(rho[1]);
            residual_scaling = sqrt_rho1;
            if (!LossCurvature<Loss>::kNonPositive && !(s == 0.0 || rho[2] <= 0.0)) {
              const double D = 1.0 + 2.0 * s * rho[2] / rho[1];
              const double alpha = 1.0 - ::sqrt(D);
              residual_scaling = sqrt_rho1 / (1 - alpha);
              alpha_sq_norm = alpha / s;
            }
            // Multiplying by exactly 1 changes nothing: skip the correction for blocks
            // in the quadratic region of the loss (rho' = 1, rho'' = 0).
            correct = !(sqrt_rho1 == 1.0 && alpha_sq_norm == 0.0);
          } else {
            cost = 0.5 * s;
          }
#pragma unroll
          for (int r = 0; r < kRes; ++r) res_corrected[r] = res[r] * residual_scaling;
        }

        // The staging buffer may still be read by last iteration's bulk stores: wait
        // here, after the functor, so the copy has the whole evaluation to complete.
        if (kStage && bulk_pending) {
          if (lane == 0) BulkWaitRead();
          __syncwarp();
          bulk_pending = false;
        }

        // Per parameter block of this pass, in three sweeps so that the gradient staging
        // can reuse the Jacobian staging buffer: (1) project onto the tangent space and
        // apply the loss correction in place, (2) gradient, (3) scatter.
        unsigned live[kNB];  // ambient columns that are tangent columns, per argument
#pragma unroll
        for (int j = 0; j < kNB; ++j) live[j] = 0u;

        auto prepare = [&](auto jc) {
          constexpr int j = decltype(jc)::value;
          if constexpr (j >= kFirst && j < kEnd) {
            constexpr int kSize = Dims::Size(j);
            constexpr int kLane0 = Plan::Lane(j, 0);
            constexpr unsigned kAllLive = kSize >= 32 ? 0xffffffffu : ((1u << kSize) - 1u);
            const bool active = kGeneric ? delta_off[j] >= 0 : true;
            double B[kRes][kSize];
#pragma unroll
            for (int r = 0; r < kRes; ++r)
#pragma unroll
              for (int c = 0; c < kSize; ++c) B[r][c] = out[r].v[kLane0 + c];
            unsigned lv = kAllLive;
            if constexpr (kGeneric) {
              if (kind[j] == CB200_MANIFOLD_SUBSET) {
                lv = kAllLive & ~static_cast<unsigned>(mparam[j]);  // column selection
              } else if (kind[j] == CB200_MANIFOLD_QUATERNION_TAIL ||
                         kind[j] == CB200_MANIFOLD_EIGEN_QUATERNION_TAIL) {
                if constexpr (kSize >= 4) {
                  // d(q (+) delta)/d delta at delta = 0, 4 x 3, from the state itself
                  // (manifold.cc:62-79); Euclidean tail columns shift left by one.
                  const bool eigen_order = kind[j] == CB200_MANIFOLD_EIGEN_QUATERNION_TAIL;
                  const double* q = xval + Dims::Offset(j);
                  const double qw = eigen_order ? q[3] : q[0];
                  const double qx = eigen_order ? q[0] : q[1];
                  const double qy = eigen_order ? q[1] : q[2];
                  const double qz = eigen_order ? q[2] : q[3];
#pragma unroll
                  for (int r = 0; r < kRes; ++r) {
                    const double bw = eigen_order ? B[r][3] : B[r][0];
                    const double bx = eigen_order ? B[r][0] : B[r][1];
                    const double by = eigen_order ? B[r][1] : B[r][2];
                    const double bz = eigen_order ? B[r][2] : B[r][3];
                    B[r][0] = -bw * qx + bx * qw - by * qz + bz * qy;
                    B[r][1] = -bw * qy + bx * qz + by * qw - bz * qx;
                    B[r][2] = -bw * qz - bx * qy + by * qx + bz * qw;
#pragma unroll
                    for (int c = 3; c + 1 < kSize; ++c) B[r][c] = B[r][c + 1];
                  }
                  lv = kAllLive >> 1;
                }
              } else if (kind[j] == CB200_MANIFOLD_GENERIC && active) {
                BlockEpilogue<kRes, kSize>::MultiplyPlusJacobian(
                    B, a.plus_jacobians + plus_off[j], tangent[j]);
                lv = tangent[j] >= 32 ? 0xffffffffu : ((1u << tangent[j]) - 1u);
              }
            }
            live[j] = lv;
            if (correct)
              BlockEpilogue<kRes, kSize>::Correct(B, res, sqrt_rho1, alpha_sq_norm);
#pragma unroll
            for (int r = 0; r < kRes; ++r)
#pragma unroll
              for (int c = 0; c < kSize; ++c) out[r].v[kLane0 + c] = B[r][c];
          }
        };

        auto gradient = [&](auto jc) {
          constexpr int j = decltype(jc)::value;
          if constexpr (j >= kFirst && j < kEnd) {
            constexpr int kSize = Dims::Size(j);
            constexpr int kLane0 = Plan::Lane(j, 0);
            constexpr unsigned kAllLive = kSize >= 32 ? 0xffffffffu : ((1u << kSize) - 1u);
            const bool active = kGeneric ? delta_off[j] >= 0 : true;
            const unsigned lv = kGeneric ? live[j] : kAllLive;
            // affine plain types: the gradient offset is the state offset, still in the
            // registers that fetched this block's parameters
            const int doff = (kAffine && !kGeneric) ? soff_cur[j] : delta_off[j];
            const int run_key = (kAffine && !kGeneric) ? doff : key[j];
            double g[kSize];
#pragma unroll
            for (int c = 0; c < kSize; ++c) {
              double acc = 0.0;
#pragma unroll
              for (int r = 0; r < kRes; ++r) acc += out[r].v[kLane0 + c] * res_corrected[r];
              g[c] = acc;
            }
            // Long runs of consecutive blocks sharing this parameter block (few distinct
            // blocks in the warp) are summed in the warp first, so one lane per run adds
            // to memory.  Short runs (the 3-10 observations of a BAL point) go out
            // directly: lanes of one red instruction that hit the same sector share one
            // L2 request, which is cheaper than 5 shuffle steps per value.
            const int k_ = (valid && active) ? run_key : -1 - lane;
            const int prev_key = __shfl_up_sync(0xffffffffu, k_, 1);
            bool head = (lane == 0) || (prev_key != k_);
            const unsigned heads = __ballot_sync(0xffffffffu, head);
            if (__popc(heads) <= 4) {
#pragma unroll
              for (int c = 0; c < kSize; ++c) g[c] = (valid && ok && active) ? g[c] : 0.0;
              const unsigned above = lane == 31 ? 0u : (heads & ~((2u << lane) - 1u));
              const int run_end = above ? __ffs(above) - 1 : 32;
              WarpSegmentedSum<kSize>(run_end, g, lane);
            } else {
              head = true;  // every lane adds its own contribution
            }
            const bool emit = head && valid && ok && active;
            const unsigned emit_mask = __ballot_sync(0xffffffffu, emit);
            if (__popc(emit_mask) >= 12) {
              // Most lanes own a distinct block (the cameras of a BAL warp): stage the
              // per-lane sums and let consecutive lanes add to consecutive addresses, so
              // one red instruction touches a few sectors instead of 32.  Each lane also
              // stages the destination of every element it stages, so a reduction round is
              // two shared loads, one 64-bit multiply-add for the address and the red (4
              // instructions); recomputing the (row, column) of the element in every round
              // took 9 (measured: 111 of the BAL kernel's 1184 instructions per tile were
              // address arithmetic of the rounds).
              constexpr int kPitch = StagePitch(kSize);
              int next = doff;  // destination of the next live column
#pragma unroll
              for (int c = 0; c < kSize; ++c) {
                gbuf[lane * kPitch + c] = g[c];
                const bool live_c = !kGeneric || ((lv >> c) & 1u);
                obuf[lane * kPitch + c] = (emit && live_c) ? next : -1;
                next += kGeneric ? static_cast<int>(live_c) : 1;
              }
              if constexpr (kPitch > kSize) obuf[lane * kPitch + kSize] = -1;  // the pad slot
              __syncwarp();
              // rounds walk the staged rows as they lie (pad slots included: no division)
              if (!kGeneric && kPitch == kSize && emit_mask == 0xffffffffu) {
#pragma unroll
                for (int it = 0; it < kPitch; ++it)
                  RedAdd(a.gradient + obuf[it * 32 + lane], gbuf[it * 32 + lane]);
              } else {
#pragma unroll
                for (int it = 0; it < kPitch; ++it) {
                  const int d = obuf[it * 32 + lane];
                  RedAddIf(d >= 0, a.gradient + d, gbuf[it * 32 + lane]);
                }
              }
              __syncwarp();
            } else if (emit) {
              double* __restrict__ dst = a.gradient + doff;
#pragma unroll
              for (int c = 0; c < kSize; ++c)
                if (!kGeneric || ((lv >> c) & 1u))
                  RedAdd(dst + (kGeneric ? __popc(lv & ((1u << c) - 1u)) : c), g[c]);
            }
          }
        };

        auto scatter = [&](auto jc) {
          constexpr int j = decltype(jc)::value;
          if constexpr (j >= kFirst && j < kEnd) {
            constexpr int kSize = Dims::Size(j);
            constexpr int kLane0 = Plan::Lane(j, 0);
            constexpr unsigned kAllLive = kSize >= 32 ? 0xffffffffu : ((1u << kSize) - 1u);
            const bool active = kGeneric ? delta_off[j] >= 0 : true;
            const unsigned lv = kGeneric ? live[j] : kAllLive;
            // tangent column of every ambient column: a running count of the live columns
            // before it (once per argument; a population count per element and row measured
            // 145 instructions per tile in the generic bundle-adjustment kernel)
            int tangent_column[kSize];
            {
              int col = 0;
#pragma unroll
              for (int c = 0; c < kSize; ++c) {
                tangent_column[c] = kGeneric ? col : c;
                if constexpr (kGeneric) col += static_cast<int>((lv >> c) & 1u);
              }
            }
            auto dcol = [&](int c) -> int { return tangent_column[c]; };
            auto is_live = [&](int c) -> bool { return kGeneric ? ((lv >> c) & 1u) : true; };
            const int tan = kGeneric ? tangent[j] : kSize;
            const int row_stride = crs ? row_stride_crs : tan;
            if (kStage && (bulk_arg[j] || bulk_all)) {
              // Stage the cell exactly as it lies in global memory.
              double* cell = bulk_all ? jbuf + (jpos[j] - bulk_all_base)
                                      : jbuf + StageOffset<kRes, Dims>(kFirst, j) +
                                            lane * kRes * tan;
              if (!kGeneric && !crs && (kRes * kSize) % 2 == 0) {
                double2* mine = reinterpret_cast<double2*>(cell);  // conflict-free 128-bit
#pragma unroll
                for (int e = 0; e < kRes * kSize; e += 2)
                  mine[e / 2] = make_double2(out[e / kSize].v[kLane0 + e % kSize],
                                             out[(e + 1) / kSize].v[kLane0 + (e + 1) % kSize]);
              } else {
#pragma unroll
                for (int r = 0; r < kRes; ++r)
#pragma unroll
                  for (int c = 0; c < kSize; ++c)
                    if (is_live(c)) cell[r * row_stride + dcol(c)] = out[r].v[kLane0 + c];
              }
            } else if (kStage && !crs && coop_arg[j]) {
              // The warp's cells of this argument are not one run (two cells per row block,
              // a pose graph) but each cell is contiguous: stage them side by side, then
              // write cell after cell with consecutive lanes on consecutive 16-byte pieces,
              // so a store instruction fills whole sectors (a thread writing its own cell
              // with 8-byte stores at a 288-byte stride costs four requests per sector:
              // 2340 L2 write requests per tile measured on the pose graph for 576 ideal).
              // (cells padded to a pitch whose 16-byte multiple is odd mod 8: a 288-byte
              // pitch puts every fourth lane on the same banks, 604 wavefronts for 172)
              const int cell_doubles = kRes * tan;
              constexpr int kPitch = (kRes * kSize + 2) | 2;  // even, and pitch / 2 is odd
              static_assert(kPitch <= kRes * kSize + 4, "stage pitch within the argument's slack");
              double* stage = jbuf + StageOffset<kRes, Dims>(kFirst, j);
              double* cell = stage + lane * kPitch;
#pragma unroll
              for (int r = 0; r < kRes; ++r)
#pragma unroll
                for (int c = 0; c < kSize; ++c)
                  if (is_live(c)) cell[r * tan + dcol(c)] = out[r].v[kLane0 + c];
              __syncwarp();
              const int pairs = cell_doubles / 2;
              constexpr int kMaxPairs = kRes * kSize / 2;
#pragma unroll 8
              for (int owner = 0; owner < 32; ++owner) {
                const int base = __shfl_sync(0xffffffffu, jpos[j], owner);
                double2* __restrict__ dst = reinterpret_cast<double2*>(a.jacobian_values + base);
                const double2* src = reinterpret_cast<const double2*>(stage + owner * kPitch);
#pragma unroll
                for (int w0 = 0; w0 < kMaxPairs; w0 += 32)
                  if (w0 + lane < pairs) dst[w0 + lane] = src[w0 + lane];
              }
              __syncwarp();
            } else if (valid && active) {
              double* __restrict__ dst = a.jacobian_values + jpos[j];
              if (!kGeneric && row_stride == kSize && ((jpos[j] & 1) == 0) &&
                  ((kRes * kSize) % 2 == 0)) {
                double2* __restrict__ d2 = reinterpret_cast<double2*>(dst);
#pragma unroll
                for (int e = 0; e < kRes * kSize; e += 2)
                  d2[e / 2] = make_double2(out[e / kSize].v[kLane0 + e % kSize],
                                           out[(e + 1) / kSize].v[kLane0 + (e + 1) % kSize]);
              } else {
#pragma unroll
                for (int r = 0; r < kRes; ++r)
#pragma unroll
                  for (int c = 0; c < kSize; ++c)
                    if (is_live(c)) dst[r * row_stride + dcol(c)] = out[r].v[kLane0 + c];
              }
            }
          }
        };

        if (out_jacobian || out_gradient) {
          ForEachBlock(prepare, std::make_index_sequence<kNB>{});
          if (out_gradient) ForEachBlock(gradient, std::make_index_sequence<kNB>{});
          if (out_jacobian) {
            ForEachBlock(scatter, std::make_index_sequence<kNB>{});
            if constexpr (kStage) {
              // One proxy fence for all the cells staged in this pass, then one bulk store
              // per argument (the fence costs ~2 % of the kernel each time it runs).
              bool any = false;
#pragma unroll
              for (int j = kFirst; j < kEnd; ++j) any = any || bulk_arg[j];
              if (any) {
                FenceProxyAsyncShared();
                __syncwarp();
                if (lane == 0) {
#pragma unroll
                  for (int j = kFirst; j < kEnd; ++j)
                    if (bulk_arg[j])
                      BulkStore(a.jacobian_values + bulk_base[j],
                                jbuf + StageOffset<kRes, Dims>(kFirst, j),
                                32 * kRes * (kGeneric ? tangent[j] : Dims::Size(j)) * 8);
                  BulkCommit();
                }
                bulk_pending = true;  // the next pass (or block) waits before it restages
              }
            }
          }
        }
      };
      ForEachBlock(pass, std::make_index_sequence<Plan::kNumPasses>{});

      if constexpr (kStage) {
        if (bulk_all) {
          FenceProxyAsyncShared();
          __syncwarp();
          const int s0 = __shfl_sync(0xffffffffu, row_stride_crs, 0);
          if (lane == 0) {
            BulkStore(a.jacobian_values + bulk_all_base, jbuf, 32 * kRes * s0 * 8);
            BulkCommit();
          }
          bulk_pending = true;
        }
      }
#pragma unroll
      for (int r = 0; r < kRes; ++r) res[r] = res_corrected[r];
    }

    if (valid) {
      all_ok = all_ok && ok;
      if (ok) cost_sum += cost;
      if (out_residuals) {
        double* __restrict__ dst = a.residuals + respos;
        if ((kRes % 2 == 0) && ((respos & 1) == 0)) {
#pragma unroll
          for (int r = 0; r < kRes; r += 2)
            reinterpret_cast<double2*>(dst)[r / 2] = make_double2(res[r], res[r + 1 < kRes ? r + 1 : r]);
        } else {
#pragma unroll
          for (int r = 0; r < kRes; ++r) dst[r] = res[r];
        }
      }
    }
#pragma unroll
    for (int j = 0; j < kNB; ++j) soff_cur[j] = soff_issue[j];
    parity_cur = parity_issue;

    if constexpr (kChunked) {
      // Last tile of a chunk: the chunk's cost goes to a slot of its own (summed in chunk
      // order by the engine, whichever warp drew the chunk).
      if (warp_rb + 32 >= limit) {
        double chunk_cost = cost_sum;
#pragma unroll
        for (int d = 16; d > 0; d >>= 1) chunk_cost += __shfl_down_sync(0xffffffffu, chunk_cost, d);
        if (lane == 0) a.cost_partials[a.chunk_cost_offset + c0] = chunk_cost;
        cost_sum = 0.0;
      }
      // Last tile of a chunk: its exclusive gradient range is final (no other chunk, on
      // any rank, adds to it).  Make this warp's reductions visible, then copy the range
      // into every other rank's gradient buffer; meanwhile the other warps of this SM keep
      // evaluating.
      if (warp_rb + 32 >= limit && a.num_peers > 0) {
        // The range was added to by this warp's lanes only: ordering among them is all the
        // reads below need (a device-wide fence here waited for every red of the chunk to be
        // acknowledged, once per chunk and warp).  The peers read the copies after the
        // system-scope flag exchange of ExchangeSharedKernel.
        __threadfence_block();
        __syncwarp();
        const int4 rec = __ldg(chunk_table + c0);
        // The range goes to the peers through the copy engine (one bulk store per peer and
        // piece, shared -> peer memory over NVLink): stores issued by the lanes themselves sit
        // in the SM's load/store queue until NVLink takes them and hold up every other warp's
        // memory instructions behind them.  Staged in this tile's parameter stage, which is
        // free until the next iteration's prefetch; 16-byte granularity, odd ends by lane 0/1.
        if constexpr (kPrefetch) {
          const int d0 = rec.z, d1 = rec.w;
          const int a0 = (d0 + 1) & ~1, a1 = d1 & ~1;
          if (lane == 0 && d0 < a0 && d0 < d1) {
            const double v = __ldcg(a.gradient + d0);
            for (int q = 0; q < a.num_peers; ++q) __stcg(a.peer_gradient[q] + d0, v);
          }
          if (lane == 1 && a1 < d1 && a1 >= a0 && a1 >= d0) {
            const double v = __ldcg(a.gradient + a1);
            for (int q = 0; q < a.num_peers; ++q) __stcg(a.peer_gradient[q] + a1, v);
          }
          double* const piece = const_cast<double*>(stage_params(stage));
          constexpr int kCapacity = (32 * (Smem::kParamBytes / 8)) & ~1;
          for (int base = a0; base < a1; base += kCapacity) {
            const int count = min(kCapacity, a1 - base);
            for (int i0 = lane; i0 < count; i0 += 128) {
              double v[4];
#pragma unroll
              for (int u = 0; u < 4; ++u)
                v[u] = i0 + 32 * u < count ? __ldcg(a.gradient + base + i0 + 32 * u) : 0.0;
#pragma unroll
              for (int u = 0; u < 4; ++u)
                if (i0 + 32 * u < count) piece[i0 + 32 * u] = v[u];
            }
            FenceProxyAsyncShared();
            __syncwarp();
            if (lane == 0) {
              for (int q = 0; q < a.num_peers; ++q)
                BulkStore(a.peer_gradient[q] + base, piece, static_cast<unsigned>(count) * 8u);
              BulkCommit();
              BulkWaitRead();  // (also covers this tile's Jacobian stores: their stage is free)
            }
            __syncwarp();
            bulk_pending = false;
          }
        } else {
          // (no parameter stage to stage in: the lanes store the range themselves)
          // four independent loads in flight per lane: the loop is latency bound otherwise
          for (int i0 = rec.z + lane; i0 < rec.w; i0 += 128) {
            double v[4];
#pragma unroll
            for (int u = 0; u < 4; ++u)
              v[u] = i0 + 32 * u < rec.w ? __ldcg(a.gradient + i0 + 32 * u) : 0.0;
#pragma unroll 1
            for (int q = 0; q < a.num_peers; ++q) {
              double* __restrict__ dst = a.peer_gradient[q];
#pragma unroll
              for (int u = 0; u < 4; ++u)
                if (i0 + 32 * u < rec.w) __stcg(dst + i0 + 32 * u, v[u]);
            }
          }
        }
      }
      rb0 = rb1; hi0 = hi1; c0 = c1;
      rb1 = walk_rb(walk); hi1 = walk.hi; c1 = walk.c;
      walk_advance(walk);
    }
  }
  if constexpr (kPrefetch) CpAsyncWait<0>();
  // (the chunked variant may have peer copies in flight whose staging was already released)
  if ((bulk_pending || kChunked) && lane == 0) BulkWaitAll();

  if (!all_ok) *a.status = 1;

  // Cost: warp shuffle, then one partial per CTA (summed in a fixed order by the
  // engine, so the cost is reproducible run to run for a given grid).  Chunked: zero, every
  // chunk's cost is in its own slot already.
  double c = cost_sum;
#pragma unroll
  for (int d = 16; d > 0; d >>= 1) c += __shfl_down_sync(0xffffffffu, c, d);
  __syncthreads();  // every warp is done with the prefetch buffers: reuse their first bytes
  double* const warp_cost = reinterpret_cast<double*>(smem);
  if (lane == 0) warp_cost[tid >> 5] = c;
  __syncthreads();
  if (tid == 0) {
    double total = 0.0;
#pragma unroll
    for (int w = 0; w < kEvaluateThreads / 32; ++w) total += warp_cost[w];
    a.cost_partials[blockIdx.x] = total;
    for (int p = blockIdx.x + gridDim.x; p < a.cost_partial_count; p += gridDim.x)
      a.cost_partials[p] = 0.0;
  }
}

// The launch thunk whose address goes through the C ABI.  Nothing is cached per process:
// the opt-in to large dynamic shared memory is a per-device function attribute and an
// application may run engines on several devices (Solver::Options::cuda_device), so it is
// set for the kernel being launched on the current device every time (~1 us).
template <typename Kernel>
int LaunchVariant(Kernel kernel, int wanted_ctas_per_sm, int smem_bytes,
                  const cb200_launch_args* args, cudaStream_t s, int work_items = -1) {
  int device = 0, sms = 0;
  cudaError_t e = cudaGetDevice(&device);
  if (e == cudaSuccess) e = cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, device);
  if (e == cudaSuccess)
    e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_bytes);
  if (e != cudaSuccess) return static_cast<int>(e);
  const int wanted = (sms > 0 ? sms : 148) * wanted_ctas_per_sm;
  // one thread block per tile of kEvaluateThreads residual blocks, or per chunk
  const int needed =
      work_items >= 0 ? work_items : (args->n + kEvaluateThreads - 1) / kEvaluateThreads;
  int grid = needed < wanted ? needed : wanted;
  if (grid > args->cost_partial_count) grid = args->cost_partial_count;
  kernel<<<grid, kEvaluateThreads, smem_bytes, s>>>(*args);
  return static_cast<int>(cudaGetLastError());
}

template <typename Functor, typename Loss, int kRes, int... Ns>
int LaunchEvaluate(const cb200_launch_args* args, void* stream) {
  if (args->n <= 0) return 0;
  using Tables = SmemPlan<Functor, true, kRes, Ns...>;    // int tables in shared memory
  using Computed = SmemPlan<Functor, false, kRes, Ns...>; // affine / Jet-free: none
  constexpr int kJetCtas = ResidentCtas(kRes, (Ns + ... + 0), true);      // table variants
  constexpr int kAffineCtas = ResidentCtas(kRes, (Ns + ... + 0), false);  // affine variants
  constexpr int kCostCtas = VariantCtas(kVariantCost, kAffineCtas, Computed::kCostBytes);
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  const bool all = args->output_residuals && args->output_jacobian && args->output_gradient &&
                   args->apply_loss_function;
  constexpr unsigned kAffinePlain =
      CB200_AFFINE_RESIDUAL | CB200_AFFINE_JACOBIAN | CB200_AFFINE_DELTA_IS_STATE;
  constexpr unsigned kAffineGeneric = CB200_AFFINE_RESIDUAL | CB200_AFFINE_JACOBIAN;
  if (!(args->output_jacobian || args->output_gradient)) {
    return LaunchVariant(EvaluateKernel<kVariantCost, false, false, Functor, Loss, kRes, Ns...>, kCostCtas,
                         Computed::kCostBytes, args, s);
  }
  if (all && args->plain && !args->crs) {
    if ((args->chunks || args->num_chunks > 0) && (args->affine & kAffinePlain) == kAffinePlain)
      return LaunchVariant(
          EvaluateKernel<kVariantPlainAll, true, true, Functor, Loss, kRes, Ns...>, kAffineCtas,
          Computed::kJetBytes, args, s,
          (args->num_chunks + kEvaluateThreads / 32 - 1) / (kEvaluateThreads / 32));
    if ((args->affine & kAffinePlain) == kAffinePlain)
      return LaunchVariant(EvaluateKernel<kVariantPlainAll, true, false, Functor, Loss, kRes, Ns...>,
                           kAffineCtas, Computed::kJetBytes, args, s);
    return LaunchVariant(EvaluateKernel<kVariantPlainAll, false, false, Functor, Loss, kRes, Ns...>,
                         kJetCtas, Tables::kJetBytes, args, s);
  }
  if (all && !args->plain) {
    if ((args->affine & kAffineGeneric) == kAffineGeneric)
      return LaunchVariant(EvaluateKernel<kVariantGenericAll, true, false, Functor, Loss, kRes, Ns...>,
                           kJetCtas, Tables::kJetBytes, args, s);  // (block ids stay staged)
    return LaunchVariant(EvaluateKernel<kVariantGenericAll, false, false, Functor, Loss, kRes, Ns...>,
                         kJetCtas, Tables::kJetBytes, args, s);
  }
  if (args->plain)
    return LaunchVariant(EvaluateKernel<kVariantPlain, false, false, Functor, Loss, kRes, Ns...>, kJetCtas,
                         Tables::kJetBytes, args, s);
  return LaunchVariant(EvaluateKernel<kVariantGeneric, false, false, Functor, Loss, kRes, Ns...>, kJetCtas,
                       Tables::kJetBytes, args, s);
}

// ceres/internal/normal_kernel.cuh (included at the end of this file)
template <int kRes, int... Ns>
int LaunchNormalProduct(const cb200_normal_args* args, void* stream);

template <typename Functor, typename Loss, int kRes, int... Ns>
cb200_residual_type MakeResidualType() {
  static_assert(sizeof...(Ns) >= 1 && sizeof...(Ns) <= CB200_MAX_PARAMETER_BLOCKS,
                "between 1 and 10 parameter blocks per residual block");
  cb200_residual_type t{};
  t.num_residuals = kRes;
  t.num_parameter_blocks = sizeof...(Ns);
  const int sizes[] = {Ns...};
  for (int i = 0; i < static_cast<int>(sizeof...(Ns)); ++i) t.parameter_block_sizes[i] = sizes[i];
  t.functor_size = static_cast<int32_t>(sizeof(Functor));
  t.loss_size = static_cast<int32_t>(sizeof(Loss));
  t.threads_per_block = kEvaluateThreads;
  t.supports_chunks = 1;
  t.launch = &LaunchEvaluate<Functor, Loss, kRes, Ns...>;
  t.normal_product = &LaunchNormalProduct<kRes, Ns...>;
  return t;
}

}  // namespace internal
}  // namespace ceres

#include "ceres/internal/normal_kernel.cuh"

#endif  // CERES_B200_INTERNAL_EVALUATE_KERNEL_CUH_
