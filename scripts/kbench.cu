// Stand-alone micro-benchmark of the BAL evaluation kernel: builds a synthetic
// BAL-shaped table set directly in C++ (no engine, no Python) and times
// LaunchEvaluate<SnavelyReprojectionError, HuberLossCUDA, 2, 9, 3>.  To A/B a kernel
// variant on the GPU, edit evaluate_kernel.cuh in a scratch copy of the tree and build
// both copies with scripts/kbench_build.sh.
//   nvcc -gencode arch=compute_100a,code=sm_100a -O3 -std=c++17 -Iinclude \
//        -Iceres-solver-cuda_b200/include -Iceres-solver-cuda_b200/examples scripts/kbench.cu
#include <algorithm>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <random>
#include <vector>

#include "ceres/internal/evaluate_kernel.cuh"
#include "ceres/loss_function_cuda.h"
#include "snavely_reprojection_error.h"

using Functor = ceres::examples::SnavelyReprojectionError;
using Loss = ceres::HuberLossCUDA;

#define CK(x) do { cudaError_t e_ = (x); if (e_ != cudaSuccess) { std::printf("%s: %s\n", #x, cudaGetErrorString(e_)); std::exit(1);} } while (0)

template <typename T> T* Upload(const std::vector<T>& v) {
  T* d; CK(cudaMalloc(&d, v.size() * sizeof(T) + 16));
  CK(cudaMemcpy(d, v.data(), v.size() * sizeof(T), cudaMemcpyHostToDevice)); return d;
}

int main(int argc, char** argv) {
  const int nc = argc > 1 ? std::atoi(argv[1]) : 13682;
  const int np = argc > 2 ? std::atoi(argv[2]) : 4456117;
  const int n = argc > 3 ? std::atoi(argv[3]) : 28987644;
  const int want_g = argc > 4 ? std::atoi(argv[4]) : 1;
  const int want_j = argc > 5 ? std::atoi(argv[5]) : 1;
  std::mt19937_64 rng(3);
  std::normal_distribution<double> N01(0, 1);
  std::uniform_real_distribution<double> U(0, 1);
  std::vector<double> state(3 * (size_t)np + 9 * (size_t)nc);
  for (int i = 0; i < 3 * np; ++i) state[i] = N01(rng);
  for (int c = 0; c < nc; ++c) {
    double* cam = &state[3 * (size_t)np + 9 * (size_t)c];
    for (int k = 0; k < 3; ++k) cam[k] = 0.1 * N01(rng);
    cam[3] = 0.5 * N01(rng); cam[4] = 0.5 * N01(rng); cam[5] = -8 + 0.5 * N01(rng);
    cam[6] = 400 + 800 * U(rng); cam[7] = 1e-7 * N01(rng); cam[8] = 1e-13 * N01(rng);
  }
  std::vector<int> soff(2 * (size_t)n), doff(2 * (size_t)n), jpos(2 * (size_t)n), respos(n);
  std::vector<Functor> functors; functors.reserve(n);
  // observations grouped by point, ~n/np per point, cameras distinct ascending per point
  size_t k = 0;
  for (int p = 0; p < np && k < (size_t)n; ++p) {
    int deg = (int)((size_t)n * (p + 1) / np - (size_t)n * p / np);
    if (deg < 1) deg = 1;
    int cam = (int)(nc * U(rng) * U(rng));
    for (int d = 0; d < deg && k < (size_t)n; ++d, ++k) {
      cam = (cam + 1 + (int)(U(rng) * (nc / (deg + 1)))) % nc;
      soff[k] = 3 * np + 9 * cam; soff[n + k] = 3 * p;
      doff[k] = 3 * np + 9 * cam; doff[n + k] = 3 * p;
      jpos[k] = 6 * n + 18 * (int)k; jpos[n + k] = 6 * (int)k;  // F then E region (int32 like the layouts)
      respos[k] = 2 * (int)k;
      // exact projection + noise so residuals are pixel-sized
      const double* c9 = &state[soff[k]]; const double* X = &state[3 * (size_t)p];
      double th = std::sqrt(c9[0]*c9[0]+c9[1]*c9[1]+c9[2]*c9[2]), P[3];
      double w[3] = {c9[0]/th, c9[1]/th, c9[2]/th}, ct = std::cos(th), st = std::sin(th);
      double wx[3] = {w[1]*X[2]-w[2]*X[1], w[2]*X[0]-w[0]*X[2], w[0]*X[1]-w[1]*X[0]};
      double wd = (w[0]*X[0]+w[1]*X[1]+w[2]*X[2])*(1-ct);
      for (int i = 0; i < 3; ++i) P[i] = X[i]*ct + wx[i]*st + w[i]*wd + c9[3+i];
      double xp = -P[0]/P[2], yp = -P[1]/P[2], r2 = xp*xp+yp*yp, dd = 1 + r2*(c9[7]+c9[8]*r2);
      double noise = U(rng) < 0.02 ? 20.0 : 0.5;
      functors.emplace_back(c9[6]*dd*xp + noise*N01(rng), c9[6]*dd*yp + noise*N01(rng));
    }
  }
  std::printf("blocks %zu (jacobian %.2f GB)\n", k, 192.0 * k / 1e9);
  Loss loss(1.0);
  cb200_launch_args a{};
  a.n = n; a.output_residuals = 1; a.output_jacobian = want_j; a.output_gradient = want_g;
  a.apply_loss_function = 1; a.crs = 0; a.plain = 1;
  const int affine = argc > 7 ? std::atoi(argv[7]) : 1;
  if (affine) {
    a.affine = CB200_AFFINE_RESIDUAL | CB200_AFFINE_JACOBIAN | CB200_AFFINE_DELTA_IS_STATE;
    a.residual_base = 0; a.row_stride = 9;
    a.jacobian_base[0] = 6 * n; a.jacobian_step[0] = 18;
    a.jacobian_base[1] = 0; a.jacobian_step[1] = 6;
  }
  // KBENCH_GENERIC=1: BASELINE config 4 - every camera has SubsetManifold(9, {0}) (8 tangent
  // columns), compressed-row values (per block 2 rows of 3 point + 8 camera entries), the
  // generic all-outputs variant with the parameter-block table.
  const bool generic = std::getenv("KBENCH_GENERIC") != nullptr;
  std::vector<int> pbid, pbtab;
  if (generic) {
    a.plain = 0; a.crs = 1;
    a.affine = CB200_AFFINE_RESIDUAL | CB200_AFFINE_JACOBIAN;
    a.residual_base = 0; a.row_stride = 11;
    a.jacobian_base[0] = 3; a.jacobian_step[0] = 22;   // camera cell: after the point's 3 columns
    a.jacobian_base[1] = 0; a.jacobian_step[1] = 22;
    pbid.resize(2 * (size_t)n);
    pbtab.assign(8 * ((size_t)np + nc), 0);
    for (int p = 0; p < np; ++p) {
      int* r = &pbtab[8 * (size_t)p];
      r[0] = 3 * p; r[1] = 3 * p; r[2] = 3; r[3] = CB200_MANIFOLD_NONE; r[4] = 0; r[5] = -1;
    }
    for (int c = 0; c < nc; ++c) {
      int* r = &pbtab[8 * ((size_t)np + c)];
      r[0] = 3 * np + 9 * c; r[1] = 3 * np + 8 * c; r[2] = 8; r[3] = CB200_MANIFOLD_SUBSET; r[4] = 1; r[5] = -1;
    }
    for (size_t i = 0; i < (size_t)n; ++i) {
      pbid[i] = np + (soff[i] - 3 * np) / 9;
      pbid[n + i] = soff[n + i] / 3;
      jpos[i] = 22 * (int)i + 3; jpos[n + i] = 22 * (int)i;
    }
  }
  constexpr int kThreads = ceres::internal::kEvaluateThreads;
  const int grid_max = std::min((n + kThreads - 1) / kThreads, 4096);
  a.cost_partial_count = grid_max;
  a.functors = Upload(functors);
  std::vector<char> lb((char*)&loss, (char*)&loss + sizeof(loss));
  a.loss_table = Upload(lb); a.loss_index = nullptr;
#ifdef CB200_INLINE_LOSS_BYTES
  if (!std::getenv("KBENCH_NO_INLINE_LOSS")) { a.loss_inline_size = sizeof(loss); std::memcpy(a.loss_inline, &loss, sizeof(loss)); }
#endif
  a.state_offset = Upload(soff); a.delta_offset = Upload(doff); a.jacobian_pos = Upload(jpos);
  a.residual_pos = Upload(respos); a.parameter_block = nullptr; a.parameter_block_table = nullptr;
  a.jacobian_row_stride = nullptr;
  if (generic) {
    a.parameter_block = Upload(pbid); a.parameter_block_table = Upload(pbtab);
    std::vector<int> rs(n, 11); a.jacobian_row_stride = Upload(rs);
  } a.state = Upload(state); a.plus_jacobians = nullptr;
  // KBENCH_CHUNK=<blocks>: the chunked (multi-GPU) variant on one GPU, no peers: what the chunk
  // walk itself costs against the grid-stride walk
  if (const char* cb = std::getenv("KBENCH_CHUNK")) {
    const int chunk = std::atoi(cb);
    std::vector<int> table;
    for (int lo = 0; lo < n; lo += chunk) {
      const int hi = std::min(n, lo + chunk);
      table.push_back(lo); table.push_back(hi);
      // KBENCH_PEERS=k: the chunk's point gradient range is copied to k local stand-in buffers
      const bool copy = std::getenv("KBENCH_PEERS") != nullptr;
      table.push_back(copy ? soff[(size_t)n + lo] : 0);
      table.push_back(copy ? (hi < n ? soff[(size_t)n + hi] : 3 * np) : 0);
    }
    a.chunks = Upload(table); a.num_chunks = (int)(table.size() / 4); a.num_peers = 0;
    if (std::getenv("KBENCH_UNIFORM")) { a.chunks = nullptr; a.chunk_blocks = chunk; }  // table-free form
    if (const char* pe = std::getenv("KBENCH_PEERS")) {
      a.num_peers = std::atoi(pe);
      for (int q = 0; q < a.num_peers; ++q) CK(cudaMalloc(&a.peer_gradient[q], 8 * state.size()));
    }
  }
  // chunked: one cost slot per chunk after the per-thread-block ones
  const int cost_slots = grid_max + a.num_chunks;
  a.chunk_cost_offset = grid_max;
  double *res, *jac, *grad, *cp; int* status;
  CK(cudaMalloc(&res, 16 * (size_t)n)); CK(cudaMalloc(&jac, 192 * (size_t)n));
  CK(cudaMalloc(&grad, 8 * state.size())); CK(cudaMalloc(&cp, 8 * (size_t)cost_slots)); CK(cudaMalloc(&status, 8));
  CK(cudaMemset(status, 0, 8));
  a.residuals = res; a.jacobian_values = jac; a.gradient = grad; a.cost_partials = cp; a.status = status;
  cudaStream_t s; CK(cudaStreamCreate(&s));
  cudaEvent_t e0, e1; cudaEventCreate(&e0); cudaEventCreate(&e1);
  float best = 1e9f, sum = 0; const int reps = 10;
  for (int it = 0; it < reps + 3; ++it) {
    CK(cudaMemsetAsync(grad, 0, 8 * state.size(), s));
    CK(cudaMemsetAsync(status, 0, 8, s));
    cudaEventRecord(e0, s);
    int rc = ceres::internal::LaunchEvaluate<Functor, Loss, 2, 9, 3>(&a, s);
    cudaEventRecord(e1, s);
    CK(cudaStreamSynchronize(s));
    if (rc) { std::printf("launch failed %d\n", rc); return 1; }
    float ms; cudaEventElapsedTime(&ms, e0, e1);
    if (it >= 3) { best = ms < best ? ms : best; sum += ms; }
  }
  if (std::getenv("KBENCH_NORMAL")) {
    // y += J'(J x) on the Jacobian just written (the conjugate-gradient product)
    cb200_normal_args na{};
    na.n = n; na.offset = a.state_offset; na.x = a.state; na.values = jac; na.op = std::getenv("KBENCH_NORMAL_OP") ? std::atoi(std::getenv("KBENCH_NORMAL_OP")) : 0; na.w = res; na.residual_base = 0;
    na.base[0] = 6 * n; na.base[1] = 0;
    double* y; CK(cudaMalloc(&y, 8 * state.size() + 16));
    na.y = y;
    float nbest = 1e9f, nsum = 0;
    for (int it = 0; it < reps + 3; ++it) {
      CK(cudaMemsetAsync(y, 0, 8 * state.size(), s));
      cudaEventRecord(e0, s);
      int rc = ceres::internal::LaunchNormalProduct<2, 9, 3>(&na, s);
      cudaEventRecord(e1, s);
      CK(cudaStreamSynchronize(s));
      if (rc) { std::printf("normal product launch failed %d\n", rc); return 1; }
      float ms; cudaEventElapsedTime(&ms, e0, e1);
      if (it >= 3) { nbest = ms < nbest ? ms : nbest; nsum += ms; }
    }
    std::vector<double> yh(state.size());
    CK(cudaMemcpy(yh.data(), y, 8 * yh.size(), cudaMemcpyDeviceToHost));
    double ys = 0, ya = 0; for (double v : yh) { ys += v; ya += std::fabs(v); }
    std::printf("KNORMAL %s : mean %.3f ms best %.3f ms (%.0f GB/s of Jacobian values)  y sum %.12e abs %.12e\n",
                argc > 6 ? argv[6] : "", nsum / reps, nbest, 192.0 * n / (nsum / reps) / 1e6, ys, ya);
  }
  int st; CK(cudaMemcpy(&st, status, 4, cudaMemcpyDeviceToHost));
  std::vector<double> part(cost_slots); CK(cudaMemcpy(part.data(), cp, 8 * (size_t)cost_slots, cudaMemcpyDeviceToHost));
  double cost = 0; for (double v : part) cost += v;
  {
    std::vector<double> gh(state.size()), jh(1 << 16);
    CK(cudaMemcpy(gh.data(), grad, 8 * gh.size(), cudaMemcpyDeviceToHost));
    CK(cudaMemcpy(jh.data(), jac + 6 * (size_t)n, 8 * jh.size(), cudaMemcpyDeviceToHost));
    double gs = 0, ga = 0, js = 0;
    for (double v : gh) { gs += v; ga += std::fabs(v); }
    for (double v : jh) js += std::fabs(v);
    std::printf("checksums: gradient sum %.12e abs %.12e  jacobian abs %.12e\n", gs, ga, js);
  }
  {
    using Plan = ceres::internal::SmemPlan<Functor, false, 2, 9, 3>;
    std::printf("smem plan: %d bytes per CTA, %d CTAs per SM, Jacobian staged %d, passes %d\n",
                Plan::kJetBytes, Plan::kCtas, (int)Plan::kStageJacobian,
                ceres::internal::PassPlan<2, 9, 3>::kNumPasses);
  }
  std::printf("KBENCH %s affine=%d g=%d j=%d : mean %.3f ms best %.3f ms  (%.2f G blocks/s)  status=%d cost=%.6e\n",
              argc > 6 ? argv[6] : "", affine, want_g, want_j, sum / reps, best, n / (sum / reps) / 1e6, st, cost);
  return 0;
}
