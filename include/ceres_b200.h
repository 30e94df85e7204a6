/* ceres_b200.h — C ABI of the B200-native residual/Jacobian evaluation engine.
 *
 * This is the drop-in boundary for the one hot path of jwmak/ceres-solver-cuda:
 * ProgramEvaluatorCUDA::Evaluate -> RegisteredCUDAEvaluators::{Init,Evaluate}
 * -> per-type AutoDiffResidualBlockCUDAEvaluator::{Init,Evaluate} -> EvaluateKernel.
 * Plain pointers and sizes only; every function returns an int status, no C++
 * exceptions cross the boundary.  Each entry point cites the reference interface
 * it replaces (paths relative to the reference tree).
 *
 * The only templated, user-TU-compiled piece is the launch thunk
 * (cb200_launch_fn): user functors are templates on the scalar type, so the
 * kernel that calls them has to be instantiated by nvcc in the user's translation
 * unit (include/ceres/internal/evaluate_kernel.cuh emits it); everything else
 * — device buffers, layouts, reductions, transfers, NCCL — is in libceres_b200.so.
 */
#ifndef CERES_B200_H_
#define CERES_B200_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define CB200_MAX_PARAMETER_BLOCKS 10 /* include/ceres/internal/parameter_dims.h users: <= 10 */
#define CB200_MAX_PEERS 15             /* other ranks of one NVLink domain */

/* status codes */
#define CB200_OK 0
#define CB200_EVALUATION_FAILED 1 /* a functor returned false or produced a non-finite value:
                                     Evaluator::Evaluate returns false (internal/ceres/evaluator.h:119-124) */
#define CB200_ERROR_CUDA (-1)
#define CB200_ERROR_INVALID_ARGUMENT (-2)
#define CB200_ERROR_NOT_FINALIZED (-3)
#define CB200_ERROR_NCCL (-4)

/* cb200_engine_evaluate flags */
#define CB200_APPLY_LOSS_FUNCTION 1u /* Evaluator::EvaluateOptions::apply_loss_function */
#define CB200_SKIP_HOST_COPY 2u      /* leave outputs on the device (see cb200_engine_device_ptr) */
#define CB200_KEEP_RESIDUALS_ON_DEVICE 4u /* compute the residuals, do not copy them to the host
                                             (the residuals argument may then be NULL) */
#define CB200_KEEP_JACOBIAN_ON_DEVICE 8u  /* compute the Jacobian and leave it on the device for the
                                             cb200_engine_jacobian_* / cb200_engine_cgnr_solve calls
                                             (the jacobian_values argument may then be NULL) */

#define CB200_JACOBIAN_BLOCK_SPARSE 0   /* BlockJacobianWriter  (internal/ceres/block_jacobian_writer.cc) */
#define CB200_JACOBIAN_COMPRESSED_ROW 1 /* CompressedRowJacobianWriter (compressed_row_jacobian_writer.cc) */

typedef struct cb200_engine cb200_engine;

/* One parameter block of the (reduced) program; replaces the device AoS record
 * ParameterBlockCUDA (include/ceres/internal/parameter_block_cuda.h:44-117).
 * Blocks [0, num_active) are Program::parameter_blocks() in order, blocks
 * [num_active, num_active + num_constant) are Program::constant_parameter_blocks(). */
typedef struct cb200_parameter_block {
  int32_t size;                 /* ambient size */
  int32_t tangent_size;         /* == size without a manifold */
  int32_t state_offset;         /* active: into the state vector; constant: into constant_state */
  int32_t delta_offset;         /* active: into the gradient / Jacobian columns; constant: -1 */
  int32_t plus_jacobian_offset; /* CB200_MANIFOLD_GENERIC: offset (doubles) of the row-major
                                   size x tangent_size plus-Jacobian in the pool passed to
                                   cb200_engine_evaluate; -1 otherwise */
  int32_t manifold_kind;        /* CB200_MANIFOLD_*: manifolds the kernel applies by itself need
                                   no plus-Jacobian from the host (Manifold::PlusJacobian,
                                   internal/ceres/manifold.cc:62-79,199-214) */
  int32_t manifold_param;       /* SUBSET: bit i set = coordinate i held constant (size <= 32) */
} cb200_parameter_block;

#define CB200_MANIFOLD_NONE 0
#define CB200_MANIFOLD_SUBSET 1                /* SubsetManifold */
#define CB200_MANIFOLD_QUATERNION_TAIL 2       /* (w,x,y,z) at [0,4) then Euclidean coordinates:
                                                  QuaternionManifold, ProductManifold<Quaternion, Euclidean<k>> */
#define CB200_MANIFOLD_EIGEN_QUATERNION_TAIL 3 /* (x,y,z,w) at [0,4) then Euclidean coordinates */
#define CB200_MANIFOLD_GENERIC 4               /* any other manifold: plus-Jacobian from the pool */

/* Arguments of one kernel launch for one residual-block type.  All pointers are
 * device pointers owned by the engine.  Structure-of-arrays, argument-major:
 * entry (arg j, residual block t) of a per-argument table is at [j * n + t]. */
#define CB200_INLINE_LOSS_BYTES 64

typedef struct cb200_launch_args {
  int32_t n;                      /* residual blocks of this type on this rank */
  uint32_t output_residuals;
  uint32_t output_jacobian;
  uint32_t output_gradient;
  uint32_t apply_loss_function;
  uint32_t crs;                   /* 1: Jacobian rows use the per-block row stride below */
  uint32_t plain;                 /* 1: no block of this type has a manifold or is constant */
  int32_t cost_partial_count;     /* entries of cost_partials reserved for this launch; the
                                     kernel writes all of them (unused ones with zero) */
  const void* functors;           /* n cost functors, sizeof(CostFunctor) each */
  const void* loss_table;         /* distinct loss objects of this type */
  const int32_t* loss_index;      /* per block index into loss_table, or NULL when there is one entry */
  const int32_t* parameter_block; /* [num_blocks][n] index into parameter_block_table */
  const int32_t* state_offset;    /* [num_blocks][n] offset of the block's parameters in state */
  const int32_t* delta_offset;    /* [num_blocks][n] offset in the gradient, -1 for a constant block */
  const int32_t* jacobian_pos;    /* [num_blocks][n] offset of element (0,0) of the block in
                                     jacobian_values (rank-local), -1 for a constant block */
  const int32_t* jacobian_row_stride; /* [n] compressed-row: values between consecutive rows */
  const int32_t* residual_pos;    /* [n] offset of the block's residuals (rank-local) */
  const int32_t* parameter_block_table; /* 8 ints per block: state_offset, delta_offset,
                                      tangent_size, manifold_kind, manifold_param,
                                      plus_jacobian_offset, 0, 0; constant blocks have
                                      delta_offset -1 and state_offset already shifted past the
                                      active state */
  const double* state;            /* [num_parameters | constant state]; 16-byte aligned and
                                     followed by >= 2 doubles of slack (the kernel gathers
                                     parameter blocks in aligned 16-byte pieces) */
  const double* plus_jacobians;
  double* residuals;
  double* jacobian_values;
  double* gradient;
  double* cost_partials;          /* one per thread block of this launch */
  int32_t* status;                /* set non-zero when a functor fails / yields a non-finite value;
                                     status[1] (zero at launch) is the work counter the
                                     chunked variant draws its chunks from */
  /* Tables that are arithmetic progressions need not be read (found by cb200_engine_finalize;
   * typical of a single residual-block type laid out in program order, e.g. bundle adjustment):
   *   CB200_AFFINE_RESIDUAL        residual_pos[t] == residual_base + t * num_residuals
   *   CB200_AFFINE_JACOBIAN        jacobian_pos[j][t] == jacobian_base[j] + t * jacobian_step[j] for
   *                                every argument (none constant), and jacobian_row_stride[t] ==
   *                                row_stride for the compressed-row layout
   *   CB200_AFFINE_DELTA_IS_STATE  delta_offset[j][t] == state_offset[j][t] */
  uint32_t affine;
  int32_t residual_base;
  int32_t row_stride;
  int32_t jacobian_base[CB200_MAX_PARAMETER_BLOCKS];
  int32_t jacobian_step[CB200_MAX_PARAMETER_BLOCKS];
  /* Several ranks, gradient exchange fused into the evaluation kernel (NULL otherwise): a
   * warp evaluates whole chunks; chunk c is residual blocks [chunks[4c], chunks[4c+1])
   * of this launch and gradient entries [chunks[4c+2], chunks[4c+3]) are touched by it alone,
   * so the kernel copies them into peer_gradient[0 .. num_peers) — the gradient buffers of
   * the other ranks, peer-mapped — as soon as the chunk is done. */
  const int32_t* chunks;
  int32_t num_chunks;
  int32_t num_peers;
  /* chunks == NULL and num_chunks > 0: the same warp-private walk over uniform chunks of
   * chunk_blocks residual blocks (a multiple of 32), nothing copied - on large problems the
   * walk itself is ~2 % faster than the grid stride (profiles/r2_kbench_variants.txt). */
  int32_t chunk_blocks;
  /* Both chunked forms: the cost of chunk c goes to cost_partials[chunk_cost_offset + c] and
   * the per-thread-block entries hold zero, so the sum of the entries in order does not depend
   * on which warp drew which chunk. */
  int32_t chunk_cost_offset;
  double* peer_gradient[CB200_MAX_PEERS];
  /* A copy of the loss object when the type has exactly one (loss_index == NULL) and it fits:
   * kernel arguments live in the constant bank, so the kernel reads the loss parameters as
   * instruction operands instead of loading them from loss_table for every residual block.
   * loss_inline_size == 0: not provided, read loss_table. */
  uint32_t loss_inline_size;
  uint32_t reserved0;
  uint64_t loss_inline[CB200_INLINE_LOSS_BYTES / 8];
} cb200_launch_args;

#define CB200_AFFINE_RESIDUAL 1u
#define CB200_AFFINE_JACOBIAN 2u
#define CB200_AFFINE_DELTA_IS_STATE 4u

/* Launch thunk: the single symbol compiled in the user's translation unit per
 * <CostFunctor, LossFunctionCUDA, kNumResiduals, Ns...>.  Replaces
 * AutoDiffResidualBlockCUDAEvaluator::Evaluate's kernel launch
 * (include/ceres/internal/autodiff_residual_block_cuda_evaluator.h:248-250).
 * `stream` is a cudaStream_t.  Returns a cudaError_t value. */
typedef int (*cb200_launch_fn)(const cb200_launch_args* args, void* stream);

/* y += J'(J x) and the other one-pass operations (CB200_NORMAL_OP_*) for one residual-block
 * type on the Jacobian values left in HBM (conjugate
 * gradients on the normal equations; reference: CgnrSolver's two SpMVs per iteration,
 * internal/ceres/cgnr_solver.cc:190-330).  Compiled per <kNumResiduals, Ns...> next to the
 * launch thunk (ceres/internal/normal_kernel.cuh).  Only for block-sparse values of a type
 * without manifolds or constant blocks whose cells are an arithmetic progression with step
 * num_residuals * size[j]; the engine's generic kernels serve everything else. */
#define CB200_NORMAL_OP_NORMAL 0       /* y += J'(J x) */
#define CB200_NORMAL_OP_LEFT 1         /* y += J' w                (LeftMultiplyAndAccumulate) */
#define CB200_NORMAL_OP_RIGHT 2        /* w  = J x                 (RightMultiplyAndAccumulate into zero) */
#define CB200_NORMAL_OP_COLUMN_NORM 3  /* y += squared column norms (SquaredColumnNorm) */
#define CB200_NORMAL_OP_SCALE_NORM 4   /* J <- J diag(x) in place (ScaleColumns), then y += its
                                          squared column norms: one pass instead of two */

typedef struct cb200_normal_args {
  int32_t n;               /* residual blocks of this type on this rank */
  const int32_t* offset;   /* [num_blocks][n] gradient (== state) offset of every argument */
  const double* x;         /* 16-byte aligned, followed by >= 2 doubles of slack */
  double* y;
  double* values;          /* this rank's Jacobian values (written by CB200_NORMAL_OP_SCALE_NORM) */
  int32_t base[CB200_MAX_PARAMETER_BLOCKS]; /* cell (t, j) starts at base[j] + t * kRes * size[j] */
  int32_t op;              /* CB200_NORMAL_OP_* */
  int32_t residual_base;   /* rows of block t are w[residual_base + t * kRes ...] (affine) */
  double* w;               /* residual-space vector of LEFT (read) and RIGHT (written) */
} cb200_normal_args;
typedef int (*cb200_normal_fn)(const cb200_normal_args* args, void* stream);

/* Static description of a residual-block type; replaces the template arguments of
 * AutoDiffResidualBlockCUDAEvaluator<CostFunctor, LossFunctionCUDA, kNumResiduals, Ns...>
 * (include/ceres/internal/autodiff_residual_block_cuda_evaluator.h:60-94). */
typedef struct cb200_residual_type {
  int32_t num_residuals;
  int32_t num_parameter_blocks;
  int32_t parameter_block_sizes[CB200_MAX_PARAMETER_BLOCKS];
  int32_t functor_size;      /* bytes */
  int32_t loss_size;         /* bytes */
  int32_t threads_per_block; /* of the launch thunk; fixes the number of cost partials */
  int32_t supports_chunks;   /* the thunk honours cb200_launch_args::chunks (fused exchange) */
  cb200_launch_fn launch;
  cb200_normal_fn normal_product; /* may be NULL; returns -1 when the sizes do not fit */
} cb200_residual_type;

/* ---- lifetime.  Replaces ContextImpl::InitCuda + RegisteredCUDAEvaluators ctor
 * (internal/ceres/context_impl.cc:112-174, include/ceres/internal/registered_cuda_evaluators.h:64-70). */
#define CB200_PLANNING_ONLY (-1) /* device argument: plan the sharding on a host without a GPU */
int cb200_engine_create(int device, cb200_engine** engine);
void cb200_engine_destroy(cb200_engine* engine);
const char* cb200_engine_last_error(const cb200_engine* engine);

/* ---- structure upload.  Together these replace RegisteredCUDAEvaluators::Init
 * (internal/ceres/registered_cuda_evaluators.cc:226-280). */

/* SetupParameterBlocks (registered_cuda_evaluators.cc:123-198). */
int cb200_engine_set_parameter_blocks(cb200_engine* engine, int32_t num_active,
                                      int32_t num_constant,
                                      const cb200_parameter_block* blocks,
                                      int32_t num_parameters,
                                      int32_t num_effective_parameters,
                                      const double* constant_state,
                                      int32_t num_constant_parameters,
                                      int32_t plus_jacobian_pool_size);

/* SetupResidualBlocks + per-type Init/SetupResidualBlocksOnDevice
 * (registered_cuda_evaluators.cc:200-224,
 *  autodiff_residual_block_cuda_evaluator.h:96-133,153-180).
 * program_position[t] is the block's POSITION in program->residual_blocks()
 * (the loop index the CPU evaluator uses, program_evaluator.h:186-236), not
 * ResidualBlock::index().  parameter_block_ids is [n][num_parameter_blocks].
 * loss_index may be NULL when num_losses == 1. */
int cb200_engine_add_residual_blocks(cb200_engine* engine, const cb200_residual_type* type,
                                     int32_t n, const int32_t* program_position,
                                     const int32_t* parameter_block_ids, const void* functors,
                                     const void* loss_table, int32_t num_losses,
                                     const int32_t* loss_index);

/* The layouts ProgramEvaluatorCUDA's constructor builds
 * (internal/ceres/program_evaluator_cuda.h:69-91,159-170) exactly as the reference's
 * writers emit them: residual_layout[num_residual_blocks],
 * jacobian_per_residual_layout[num_residual_blocks] and
 * jacobian_per_residual_offsets[sum over blocks of active_args * num_residuals]
 * (BlockJacobianWriter / CompressedRowJacobianWriter::CreateJacobianPerResidualLayout,
 *  block_jacobian_writer.cc:154-160, compressed_row_jacobian_writer.cc:240-300). */
int cb200_engine_set_layout(cb200_engine* engine, int32_t jacobian_format,
                            int32_t num_residual_blocks, int32_t num_residuals,
                            const int32_t* residual_layout,
                            const int32_t* jacobian_per_residual_layout,
                            const int32_t* jacobian_per_residual_offsets,
                            int64_t num_offsets, int64_t num_jacobian_values);

/* Multi-GPU: this rank evaluates the contiguous range of residual blocks
 * [floor(rank * n / world), floor((rank + 1) * n / world)) in program order
 * (no reference equivalent; the reference is single-GPU).  Call before finalize. */
int cb200_engine_set_shard(cb200_engine* engine, int32_t rank, int32_t world_size);

/* Builds the device tables.  After this the structure is immutable. */
int cb200_engine_finalize(cb200_engine* engine);

/* NCCL communicator for the cost/gradient all-reduce.  unique_id is the 128-byte
 * ncclUniqueId created by cb200_nccl_unique_id on rank 0 and broadcast by the caller. */
int cb200_nccl_unique_id(void* unique_id_128_bytes);
int cb200_engine_comm_init(cb200_engine* engine, const void* unique_id_128_bytes,
                           int32_t rank, int32_t world_size);

/* ---- the hot call.  Replaces RegisteredCUDAEvaluators::Evaluate
 * (internal/ceres/registered_cuda_evaluators.cc:46-103).  All pointers are HOST
 * pointers.  state has num_parameters doubles; plus_jacobians is the pool described
 * by cb200_parameter_block::plus_jacobian_offset (may be NULL when the pool is
 * empty).  cost must not be NULL; residuals / gradient / jacobian_values may each be
 * NULL, exactly as in Evaluator::Evaluate (internal/ceres/evaluator.h:119-124).
 * jacobian_values is the values array of the matrix returned by CreateJacobian();
 * with sharding only this rank's slices are written.
 * Returns CB200_OK, CB200_EVALUATION_FAILED, or an error. */
int cb200_engine_evaluate(cb200_engine* engine, const double* state,
                          const double* plus_jacobians, uint32_t flags, double* cost,
                          double* residuals, double* gradient, double* jacobian_values);

/* Device-resident variant: same work, inputs already on the device (state_device
 * has num_parameters doubles, plus_jacobians_device may be NULL), outputs stay on
 * the device; want_* select what is computed.  *cost is read back (8 bytes). */
int cb200_engine_evaluate_device(cb200_engine* engine, const double* state_device,
                                 const double* plus_jacobians_device, uint32_t flags,
                                 int want_residuals, int want_gradient, int want_jacobian,
                                 double* cost);

/* Device buffers of the last evaluation, for a device-side consumer (a GPU linear
 * solver).  which: 0 residuals, 1 gradient, 2 jacobian_values, 3 state. */
void* cb200_engine_device_ptr(cb200_engine* engine, int which);

/* This rank's slices: residual range and up to max_segments Jacobian value ranges
 * as (global_offset, length, local_offset) triples.  Returns the segment count. */
int cb200_engine_shard_info(cb200_engine* engine, int32_t* rb_begin, int32_t* rb_end,
                            int32_t* residual_begin, int32_t* residual_end,
                            int64_t* segments, int32_t max_segments);

/* Multi-GPU gradient exchange plan of this rank (derived by cb200_engine_finalize from the
 * whole problem; works on planning-only engines).  Returns the number of chunks, or -1 when
 * the structure does not allow the peer exchange (several residual-block types, no
 * exclusive ranges, ...: the ranks then use one NCCL all-reduce).  chunks receives up to
 * max_chunks records of 4 ints (cb200_launch_args::chunks); exclusive = {begin, length} of
 * the gradient range only this rank's residual blocks touch; *shared_count = entries several
 * ranks add to, plus cost and status. */
int cb200_engine_exchange_plan(cb200_engine* engine, int32_t* chunks, int32_t max_chunks,
                               int64_t* exclusive, int32_t* shared_count);

/* ---- linear algebra on the device-resident Jacobian of the last evaluation
 * (SURVEY.md section 8(f) items 1-2).  The 5.6 GB of Jacobian values of a large bundle
 * adjustment problem then never cross PCIe.  They replace, for a Jacobian that stays in HBM,
 * BlockSparseMatrix / CompressedRowSparseMatrix::{RightMultiplyAndAccumulate,
 * LeftMultiplyAndAccumulate, SquaredColumnNorm, ScaleColumns}
 * (internal/ceres/block_sparse_matrix.cc:150-280, compressed_row_sparse_matrix.cc:300-470),
 * their CUDA counterparts (internal/ceres/cuda_sparse_matrix.cc) and the CUDA CGNR solver
 * (internal/ceres/cgnr_solver.cc:190-330).  Vectors are HOST pointers: x-like vectors have
 * num_effective_parameters entries, residual-like vectors num_residuals (with sharding a
 * rank reads / writes only its residual slice; column-space results are summed over ranks). */

/* transpose == 0: y = J x;  transpose != 0: y = J' x. */
int cb200_engine_jacobian_multiply(cb200_engine* engine, int transpose, const double* x,
                                   double* y);
/* out[c] = sum over rows of J(r, c)^2 */
int cb200_engine_jacobian_squared_column_norm(cb200_engine* engine, double* out);
/* J <- J diag(scale) */
int cb200_engine_jacobian_scale_columns(cb200_engine* engine, const double* scale);

typedef struct cb200_cgnr_options {
  int32_t min_num_iterations;
  int32_t max_num_iterations;
  double r_tolerance; /* stop when |residual| <= r_tolerance * |J'b|  (conjugate_gradients_solver.h) */
  double q_tolerance; /* stop when the relative decrease of the quadratic model falls below this */
} cb200_cgnr_options;

typedef struct cb200_cgnr_summary {
  int32_t num_iterations;
  int32_t termination;        /* 0 converged, 1 iteration limit, 2 breakdown (non-positive curvature / non-finite) */
  double initial_gradient_norm; /* |J'b| */
  double final_residual_norm;
  double jy_dot_b;            /* (J y).b and |J y|^2 for the trust-region model: with the step */
  double jy_squared_norm;     /* -y, model_cost_change = (J y).b - |J y|^2 / 2 */
  double solve_ms;            /* device time of the call */
} cb200_cgnr_summary;

/* Solves (J'J + diag(d_squared)) y = J'b by preconditioned conjugate gradients on the
 * normal equations without forming them, b = the residuals of the last evaluation (on the
 * device) and J its Jacobian (CB200_KEEP_*_ON_DEVICE), preconditioner
 * diag(J'J + d_squared)^-1.  d_squared may be NULL (zero).  solution: num_effective doubles. */
int cb200_engine_cgnr_solve(cb200_engine* engine, const double* d_squared,
                            const cb200_cgnr_options* options, double* solution,
                            cb200_cgnr_summary* summary);

/* ---- the trust-region iteration with the state in HBM (SURVEY.md section 8(f) 2-3).
 * Replaces, for CGNR + CUDA_SPARSE, what TrustRegionMinimizer does on the host around the
 * evaluator (internal/ceres/trust_region_minimizer.cc:246-275,518,780): Jacobi scaling
 * (SquaredColumnNorm / ScaleColumns), the LM diagonal (levenberg_marquardt_strategy.cc:83-96),
 * the linear solve, Program::Plus (program.cc:121-150, manifolds of manifold.cc:28-58,184-197)
 * and the step / state / gradient norms.  Per iteration only a few scalars cross PCIe.
 * State slot 0 is the accepted state, slot 1 the candidate x (+) step. */
typedef struct cb200_step_options {
  double radius;            /* LM diagonal = clamp(diag(J'J), min, max) / radius */
  double min_lm_diagonal;
  double max_lm_diagonal;
  int32_t reuse_diagonal;   /* keep diag(J'J) of the last accepted point (step was rejected) */
  cb200_cgnr_options cg;
} cb200_step_options;

typedef struct cb200_step_summary {
  cb200_cgnr_summary cg;
  double model_cost_change; /* (J y).r - |J y|^2 / 2 for the step -y */
  double step_norm;         /* |delta| in the parameters' scale */
  double state_norm;        /* |x| */
  int32_t plus_ok;          /* 0: a block has a manifold only the host can apply */
} cb200_step_summary;

int cb200_engine_state_upload(cb200_engine* engine, const double* state);
int cb200_engine_state_download(cb200_engine* engine, int which, double* state);
/* cb200_engine_evaluate_device at state slot `which` (no host plus-Jacobians: every manifold
 * must be one the kernel applies by itself). */
int cb200_engine_evaluate_state(cb200_engine* engine, int which, uint32_t flags,
                                int want_residuals, int want_gradient, int want_jacobian,
                                double* cost);
/* compute != 0: scale = 1 / (1 + sqrt(diag(J'J))) of the resident Jacobian, kept in HBM; then
 * (always) J <- J diag(scale). */
int cb200_engine_jacobi_scale(cb200_engine* engine, int compute);
/* LM diagonal, conjugate gradients, step = -y * scale, candidate = state (+) step. */
int cb200_engine_trust_region_step(cb200_engine* engine, const cb200_step_options* options,
                                   cb200_step_summary* summary);
int cb200_engine_accept_candidate(cb200_engine* engine); /* candidate becomes the state */
int cb200_engine_gradient_max_norm(cb200_engine* engine, double* max_norm);
/* 0: one rank; 1: NCCL all-reduce of [gradient | cost | failed]; 2: peer exchange fused into
 * the evaluation kernel (cb200_engine_exchange_plan). */
int cb200_engine_exchange_mode(cb200_engine* engine);

/* Timing of the last evaluation in milliseconds (CUDA events on the engine's
 * stream): out[0] kernels only, out[1] kernels + reductions + all-reduce,
 * out[2] whole call including host<->device copies.  out[3] = kernel launches. */
int cb200_engine_last_timing(cb200_engine* engine, double* out4);

/* Host memory for the caller's arrays (the values of CreateJacobian(), the state,
 * residual and gradient vectors).  cb200_host_alloc returns zero-filled, page-aligned,
 * lazily committed memory (untouched pages cost nothing, so a rank of a sharded run
 * can hold a full-size values array and only ever touch its slices); cb200_host_pin
 * page-locks a sub-range for full-rate DMA (cudaHostRegister; a no-op without a
 * device).  Ranges may overlap earlier pins.  Replaces the pageable
 * std::unique_ptr<double[]> of internal/ceres/block_sparse_matrix.h:163-167 that makes
 * the reference's device->host copy its bottleneck (README.md:198-200). */
void* cb200_host_alloc(uint64_t bytes);
int cb200_host_pin(void* ptr, uint64_t bytes);
void cb200_host_free(void* ptr);

const char* cb200_version(void);

#ifdef __cplusplus
}
#endif

#endif /* CERES_B200_H_ */
