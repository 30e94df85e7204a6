// Bundle adjustment with the CUDA evaluator, written against the same API as the
// reference's examples/bundle_adjuster.cu.cc (BuildProblem :302-366, SetOrdering :225-268,
// SolveProblem :368-392): one AddResidualBlock<SnavelyReprojectionError, 2, 9, 3> per
// observation, HuberLossCUDA(1) when --robustify, points eliminated before cameras.
//
//   bundle_adjuster --input=problem.txt [--robustify] [--num_iterations=20]
//                   [--loss=huber|cauchy|soft_l1|arctan|tolerant|tukey]   (scale 1)
//                   [--linear_solver=iterative_schur|cgnr|cgnr_cuda] [--constant_first_camera]
//                   [--preconditioner=identity|jacobi|scalar_jacobi]   (cgnr_cuda only)
//   bundle_adjuster --synthetic=16,2000,8000 ...
//   bundle_adjuster --input=problem.txt --check_input     (parse only, no GPU needed)
//
// The input is a BAL text file (https://grail.cs.washington.edu/projects/bal/):
// "num_cameras num_points num_observations", then "camera point x y" per observation,
// then 9 doubles per camera and 3 per point, one per line.
#include <cstdio>
#include <cstdlib>
#include <algorithm>
#include <cstring>
#include <memory>
#include <random>
#include <string>
#include <thread>
#include <vector>

#include "ceres/problem_cuda.h"
#include "snavely_reprojection_error.h"

struct BalProblem {
  int num_cameras = 0, num_points = 0, num_observations = 0;
  std::vector<int> camera_index, point_index;
  std::vector<double> observations, cameras, points;

  bool Load(const char* path) {
    FILE* f = std::fopen(path, "r");
    if (!f) return false;
    bool ok = std::fscanf(f, "%d %d %d", &num_cameras, &num_points, &num_observations) == 3;
    camera_index.resize(num_observations);
    point_index.resize(num_observations);
    observations.resize(2 * static_cast<size_t>(num_observations));
    for (int i = 0; ok && i < num_observations; ++i)
      ok = std::fscanf(f, "%d %d %lf %lf", &camera_index[i], &point_index[i],
                       &observations[2 * i], &observations[2 * i + 1]) == 4;
    cameras.resize(9 * static_cast<size_t>(num_cameras));
    points.resize(3 * static_cast<size_t>(num_points));
    for (size_t i = 0; ok && i < cameras.size(); ++i) ok = std::fscanf(f, "%lf", &cameras[i]) == 1;
    for (size_t i = 0; ok && i < points.size(); ++i) ok = std::fscanf(f, "%lf", &points[i]) == 1;
    std::fclose(f);
    return ok;
  }

  // A small random scene observed with noise, perturbed away from the truth.
  void Synthesize(int nc, int np, int nobs, unsigned seed) {
    std::mt19937_64 rng(seed);
    std::normal_distribution<double> N(0, 1);
    std::uniform_real_distribution<double> U(0, 1);
    num_cameras = nc; num_points = np; num_observations = nobs;
    cameras.resize(9 * static_cast<size_t>(nc));
    points.resize(3 * static_cast<size_t>(np));
    for (int c = 0; c < nc; ++c) {
      double* cam = &cameras[9 * c];
      for (int k = 0; k < 3; ++k) cam[k] = 0.1 * N(rng);
      cam[3] = 0.5 * N(rng); cam[4] = 0.5 * N(rng); cam[5] = -8 + 0.5 * N(rng);
      cam[6] = 400 + 800 * U(rng); cam[7] = 1e-7 * N(rng); cam[8] = 1e-13 * N(rng);
    }
    for (double& v : points) v = N(rng);
    camera_index.resize(nobs); point_index.resize(nobs); observations.resize(2 * static_cast<size_t>(nobs));
    for (int i = 0; i < nobs; ++i) {
      point_index[i] = static_cast<int>(static_cast<long long>(i) * np / nobs);
      camera_index[i] = (i * 7 + point_index[i]) % nc;
      double r[2];
      ceres::examples::SnavelyReprojectionError zero(0, 0);
      zero(&cameras[9 * camera_index[i]], &points[3 * point_index[i]], r);
      observations[2 * i] = r[0] + 0.5 * N(rng);
      observations[2 * i + 1] = r[1] + 0.5 * N(rng);
    }
    for (double& v : points) v += 0.02 * N(rng);
    for (int c = 0; c < nc; ++c)
      for (int k = 0; k < 6; ++k) cameras[9 * c + k] += 0.005 * N(rng);
  }
};

static const char* Flag(int argc, char** argv, const char* name) {
  const size_t n = std::strlen(name);
  for (int i = 1; i < argc; ++i)
    if (!std::strncmp(argv[i], name, n)) return argv[i][n] == '=' ? argv[i] + n + 1 : "";
  return nullptr;
}

// One residual block per observation, each with a copy of *loss (null: no loss).  bulk: all
// observations in one call sharing one loss object, no heap object per residual block (the
// reference's per-block objects make its preprocessor take 47 s on the 29 M-block problem,
// README.md:186).
template <typename Loss>
void AddObservations(ceres::ProblemCUDA* problem, BalProblem& bal, bool bulk, const Loss* loss) {
  if (bulk) {
    ceres::Problem::Options problem_options;
    problem_options.loss_function_ownership = ceres::DO_NOT_TAKE_OWNERSHIP;
    *problem = ceres::ProblemCUDA(problem_options);
    static std::unique_ptr<Loss> shared_loss;
    if (loss) shared_loss.reset(new Loss(*loss));
    std::vector<ceres::examples::SnavelyReprojectionError> functors;
    std::vector<double*> blocks;
    functors.reserve(bal.num_observations);
    blocks.reserve(2 * static_cast<size_t>(bal.num_observations));
    for (int i = 0; i < bal.num_observations; ++i) {
      functors.emplace_back(bal.observations[2 * i], bal.observations[2 * i + 1]);
      blocks.push_back(&bal.cameras[9 * static_cast<size_t>(bal.camera_index[i])]);
      blocks.push_back(&bal.points[3 * static_cast<size_t>(bal.point_index[i])]);
    }
    problem->AddResidualBlocks<ceres::examples::SnavelyReprojectionError, 2, 9, 3>(
        bal.num_observations, functors.data(), shared_loss.get(), blocks.data());
    return;
  }
  for (int i = 0; i < bal.num_observations; ++i) {
    ceres::CostFunction* cost_function = ceres::examples::SnavelyReprojectionError::Create(
        bal.observations[2 * i], bal.observations[2 * i + 1]);
    double* camera = &bal.cameras[9 * static_cast<size_t>(bal.camera_index[i])];
    double* point = &bal.points[3 * static_cast<size_t>(bal.point_index[i])];
    problem->AddResidualBlock<ceres::examples::SnavelyReprojectionError, 2, 9, 3>(
        cost_function, loss ? new Loss(*loss) : nullptr, camera, point);
  }
}

// --loss=<name>: the loss of every residual block, all with scale 1 (Tolerant: a = b = 1).
// Returns false for an unknown name.
static bool AddObservations(ceres::ProblemCUDA* problem, BalProblem& bal, bool bulk,
                            const char* loss) {
  if (!loss) {
    AddObservations(problem, bal, bulk, static_cast<const ceres::TrivialLossCUDA*>(nullptr));
  } else if (!std::strcmp(loss, "huber")) {
    const ceres::HuberLossCUDA l(1.0);
    AddObservations(problem, bal, bulk, &l);
  } else if (!std::strcmp(loss, "cauchy")) {
    const ceres::CauchyLossCUDA l(1.0);
    AddObservations(problem, bal, bulk, &l);
  } else if (!std::strcmp(loss, "soft_l1")) {
    const ceres::SoftLOneLossCUDA l(1.0);
    AddObservations(problem, bal, bulk, &l);
  } else if (!std::strcmp(loss, "arctan")) {
    const ceres::ArctanLossCUDA l(1.0);
    AddObservations(problem, bal, bulk, &l);
  } else if (!std::strcmp(loss, "tolerant")) {
    const ceres::TolerantLossCUDA l(1.0, 1.0);
    AddObservations(problem, bal, bulk, &l);
  } else if (!std::strcmp(loss, "tukey")) {
    const ceres::TukeyLossCUDA l(1.0);
    AddObservations(problem, bal, bulk, &l);
  } else {
    return false;
  }
  return true;
}

int main(int argc, char** argv) {
  BalProblem bal;
  if (const char* in = Flag(argc, argv, "--input")) {
    if (!bal.Load(in)) { std::fprintf(stderr, "cannot read %s\n", in); return 1; }
  } else if (const char* syn = Flag(argc, argv, "--synthetic")) {
    int nc = 16, np = 2000, nobs = 8000;
    std::sscanf(syn, "%d,%d,%d", &nc, &np, &nobs);
    bal.Synthesize(nc, np, nobs, 1);
  } else {
    std::fprintf(stderr, "usage: %s --input=<bal file> | --synthetic=nc,np,nobs [--robustify] "
                 "[--loss=huber|cauchy|soft_l1|arctan|tolerant|tukey] "
                 "[--num_iterations=N] [--linear_solver=iterative_schur|cgnr|cgnr_cuda] [--bulk] "
                 "[--preconditioner=identity|jacobi|scalar_jacobi]\n", argv[0]);
    return 1;
  }
  if (Flag(argc, argv, "--check_input")) {
    // what the reader understood, without touching a GPU (tests/test_bal_reader.py)
    double sum = 0.0;
    for (double v : bal.observations) sum += v;
    for (double v : bal.cameras) sum += v;
    for (double v : bal.points) sum += v;
    long long index_sum = 0;
    for (int i = 0; i < bal.num_observations; ++i)
      index_sum += bal.camera_index[i] + 3LL * bal.point_index[i];
    std::printf("cameras %d points %d observations %d index_sum %lld value_sum %.17g\n",
                bal.num_cameras, bal.num_points, bal.num_observations, index_sum, sum);
    return 0;
  }
  const bool robustify = Flag(argc, argv, "--robustify") != nullptr;
  const char* ls = Flag(argc, argv, "--linear_solver");
  const char* iters = Flag(argc, argv, "--num_iterations");

  const char* loss = Flag(argc, argv, "--loss");
  if (!loss && robustify) loss = "huber";

  ceres::ProblemCUDA problem;
  if (!AddObservations(&problem, bal, Flag(argc, argv, "--bulk") != nullptr, loss)) {
    std::fprintf(stderr, "unknown --loss=%s\n", loss);
    return 1;
  }
  if (Flag(argc, argv, "--constant_first_camera")) problem.SetParameterBlockConstant(&bal.cameras[0]);

  ceres::Solver::Options options;
  options.max_num_iterations = iters ? std::atoi(iters) : 20;
  options.minimizer_progress_to_stdout = true;
  const char* threads = Flag(argc, argv, "--num_threads");
  options.num_threads = threads ? std::atoi(threads)
                                : static_cast<int>(std::max(1u, std::thread::hardware_concurrency()));
  options.linear_solver_type = ceres::ITERATIVE_SCHUR;
  if (ls && !std::strcmp(ls, "cgnr")) options.linear_solver_type = ceres::CGNR;
  if (ls && !std::strcmp(ls, "cgnr_cuda")) {
    // the Jacobian never leaves the device: evaluation and conjugate gradients both run there
    options.linear_solver_type = ceres::CGNR;
    options.sparse_linear_algebra_library_type = ceres::CUDA_SPARSE;
  }
  if (const char* pc = Flag(argc, argv, "--preconditioner")) {
    if (!std::strcmp(pc, "identity")) {
      options.preconditioner_type = ceres::IDENTITY;
    } else if (!std::strcmp(pc, "jacobi")) {
      options.preconditioner_type = ceres::JACOBI;
    } else if (!std::strcmp(pc, "scalar_jacobi")) {
      options.preconditioner_type = ceres::SCALAR_JACOBI;
    } else {
      std::fprintf(stderr, "unknown --preconditioner=%s\n", pc);
      return 1;
    }
  }
  // The points come before the cameras.
  auto* ordering = new ceres::ParameterBlockOrdering;
  for (int i = 0; i < bal.num_points; ++i) ordering->AddElementToGroup(&bal.points[3 * i], 0);
  for (int i = 0; i < bal.num_cameras; ++i) ordering->AddElementToGroup(&bal.cameras[9 * i], 1);
  options.linear_solver_ordering.reset(ordering);

  ceres::Solver::Summary summary;
  ceres::Solve(options, &problem, &summary);
  std::printf("%s\n", summary.FullReport().c_str());
  return summary.IsSolutionUsable() ? 0 : 2;
}
