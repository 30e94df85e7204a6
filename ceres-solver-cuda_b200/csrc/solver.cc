// Minimal TRUST_REGION driver around the CUDA evaluator; see ceres/solver.h for scope.
#include "ceres/solver.h"

#include "ceres/internal/parallel_for.h"

#include <algorithm>
#include <chrono>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <nvtx3/nvToolsExt.h>

namespace ceres {
namespace {

double Seconds() {
  return std::chrono::duration<double>(std::chrono::steady_clock::now().time_since_epoch())
      .count();
}

// The vectors that cross PCIe every iteration (state, gradient, step, LM diagonal) live in
// page-locked memory: pageable copies of 108 MB run at a fraction of the link rate.
class PinnedVector {
 public:
  explicit PinnedVector(size_t n = 0, double value = 0.0) { assign(n, value); }
  ~PinnedVector() { Release(); }
  PinnedVector(const PinnedVector&) = delete;
  PinnedVector& operator=(const PinnedVector&) = delete;
  void assign(size_t n, double value) {
    if (n != size_) {
      Release();
      size_ = n;
      if (n > 0) {
        data_ = static_cast<double*>(cb200_host_alloc(n * sizeof(double)));
        cb200_host_pin(data_, n * sizeof(double));
      }
    }
    std::fill(begin(), end(), value);
  }
  double* data() { return data_; }
  double& operator[](size_t i) { return data_[i]; }
  double* begin() { return data_; }
  double* end() { return data_ + size_; }

 private:
  void Release() {
    if (data_) cb200_host_free(data_);
    data_ = nullptr;
    size_ = 0;
  }
  double* data_ = nullptr;
  size_t size_ = 0;
};

// Element-wise pass over [0, n) on num_threads threads; f(i) must only touch index i.
template <typename F>
void ForEach(int num_threads, int64_t n, F&& f) {
  internal::ParallelFor(num_threads, n, [&](int64_t begin, int64_t end, int) {
    for (int64_t i = begin; i < end; ++i) f(i);
  });
}
// Sum (or maximum) of f(i) over [0, n) with one partial per thread.
template <typename F>
double Reduce(int num_threads, int64_t n, bool maximum, F&& f) {
  std::vector<double> partial(std::max(1, num_threads), 0.0);
  internal::ParallelFor(num_threads, n, [&](int64_t begin, int64_t end, int t) {
    double acc = 0.0;
    for (int64_t i = begin; i < end; ++i) acc = maximum ? std::max(acc, f(i)) : acc + f(i);
    partial[t] = acc;
  });
  double total = 0.0;
  for (double p : partial) total = maximum ? std::max(total, p) : total + p;
  return total;
}

// Solves (J'J + D^2) y = J'r with Jacobi-preconditioned conjugate gradients (CGNR);
// stand-in for the reference's linear solvers.  Returns the iteration count.
int SolveNormalEquations(const internal::SparseMatrix& J, const double* D2, const double* r,
                         int max_iterations, double tolerance, PinnedVector* y) {
  const int n = J.num_cols(), m = J.num_rows();
  std::vector<double> b(n, 0.0), res(n), z(n), p(n), Ap(n), tmp(m), precond(n);
  J.LeftMultiplyAndAccumulate(r, b.data());
  J.SquaredColumnNorm(precond.data());
  for (int i = 0; i < n; ++i) precond[i] = 1.0 / (precond[i] + D2[i]);
  y->assign(n, 0.0);
  res = b;
  double norm_b = 0.0;
  for (int i = 0; i < n; ++i) norm_b += b[i] * b[i];
  norm_b = std::sqrt(norm_b);
  if (norm_b == 0.0) return 0;
  double rho = 0.0;
  int it = 0;
  for (; it < max_iterations; ++it) {
    for (int i = 0; i < n; ++i) z[i] = precond[i] * res[i];
    double rho_new = 0.0;
    for (int i = 0; i < n; ++i) rho_new += res[i] * z[i];
    if (it == 0) {
      p = z;
    } else {
      const double beta = rho_new / rho;
      for (int i = 0; i < n; ++i) p[i] = z[i] + beta * p[i];
    }
    rho = rho_new;
    std::fill(tmp.begin(), tmp.end(), 0.0);
    J.RightMultiplyAndAccumulate(p.data(), tmp.data());
    for (int i = 0; i < n; ++i) Ap[i] = D2[i] * p[i];
    J.LeftMultiplyAndAccumulate(tmp.data(), Ap.data());
    double pAp = 0.0;
    for (int i = 0; i < n; ++i) pAp += p[i] * Ap[i];
    if (!(pAp > 0.0)) break;
    const double alpha = rho / pAp;
    double norm_res = 0.0;
    for (int i = 0; i < n; ++i) {
      (*y)[i] += alpha * p[i];
      res[i] -= alpha * Ap[i];
      norm_res += res[i] * res[i];
    }
    if (std::sqrt(norm_res) <= tolerance * norm_b) { ++it; break; }
  }
  return it;
}

}  // namespace

bool Solver::Options::IsValid(std::string* error) const {
  // solver.cc:702-708: the CUDA evaluator supports TRUST_REGION only.
  if (use_cuda_for_evaluator && minimizer_type != TRUST_REGION) {
    *error = "Using CUDA for cost function evaluation is currently only supported for "
             "TRUST_REGION minimizers.";
    return false;
  }
  if (minimizer_type != TRUST_REGION) {
    *error = "Only TRUST_REGION minimization is provided by this library.";
    return false;
  }
  if (use_cuda_for_evaluator && registered_cuda_evaluators == nullptr) {
    *error = "use_cuda_for_evaluator requires registered_cuda_evaluators (use "
             "ceres::Solve(options, ProblemCUDA*, summary)).";
    return false;
  }
  if (max_num_iterations < 0) { *error = "max_num_iterations < 0"; return false; }
  // only the conjugate gradients on the device-resident Jacobian read the preconditioner
  if (preconditioner_type != SCALAR_JACOBI &&
      (linear_solver_type != CGNR || sparse_linear_algebra_library_type != CUDA_SPARSE)) {
    *error = "preconditioner_type IDENTITY and JACOBI require linear_solver_type = CGNR and "
             "sparse_linear_algebra_library_type = CUDA_SPARSE.";
    return false;
  }
  return true;
}

std::string Solver::Summary::BriefReport() const {
  char buf[256];
  std::snprintf(buf, sizeof(buf), "Ceres Solver Report: Iterations: %d, Initial cost: %e, "
                "Final cost: %e, Termination: %s",
                num_successful_steps + num_unsuccessful_steps, initial_cost, final_cost,
                termination_type == CONVERGENCE ? "CONVERGENCE"
                : termination_type == NO_CONVERGENCE ? "NO_CONVERGENCE" : "FAILURE");
  return buf;
}

std::string Solver::Summary::FullReport() const {
  char buf[2048];
  std::snprintf(
      buf, sizeof(buf),
      "\nSolver Summary (B200 evaluation engine)\n\n"
      "                                     Original                  Reduced\n"
      "Parameter blocks                 %12d             %12d\n"
      "Parameters                       %12d             %12d\n"
      "Effective parameters             %12d             %12d\n"
      "Residual blocks                  %12d             %12d\n"
      "Residuals                        %12d             %12d\n\n"
      "Cost:\nInitial                          %e\nFinal                            %e\n"
      "Change                           %e\n\n"
      "Minimizer iterations             %12d\nSuccessful steps                 %12d\n"
      "Unsuccessful steps               %12d\n\n"
      "Time (in seconds):\nPreprocessor                     %12.6f\n\n"
      "  Residual only evaluation       %12.6f (%d)\n"
      "  Jacobian & residual evaluation %12.6f (%d)\n"
      "  Linear solver                  %12.6f\n"
      "Minimizer                        %12.6f\n\nTotal                            %12.6f\n\n"
      "Termination:                     %s (%s)\n",
      num_parameter_blocks, num_parameter_blocks_reduced, num_parameters, num_parameters_reduced,
      num_effective_parameters, num_effective_parameters_reduced, num_residual_blocks,
      num_residual_blocks_reduced, num_residuals, num_residuals_reduced, initial_cost, final_cost,
      initial_cost - final_cost, num_successful_steps + num_unsuccessful_steps,
      num_successful_steps, num_unsuccessful_steps, preprocessor_time_in_seconds,
      residual_evaluation_time_in_seconds, num_residual_evaluations,
      jacobian_evaluation_time_in_seconds, num_jacobian_evaluations,
      linear_solver_time_in_seconds, minimizer_time_in_seconds, total_time_in_seconds,
      termination_type == CONVERGENCE ? "CONVERGENCE"
      : termination_type == NO_CONVERGENCE ? "NO_CONVERGENCE" : "FAILURE",
      message.c_str());
  return buf;
}

namespace {
// The Levenberg-Marquardt loop (trust_region_minimizer.cc step acceptance,
// levenberg_marquardt_strategy.cc radius update) is written once, in Minimize.  What an
// iteration asks of the place where the state, gradient and Jacobian live is behind
// TrustRegionState: DeviceState keeps them in HBM, HostState in host memory.
// kRejected: an evaluation or the step failed numerically; kError: an engine call failed,
// and error() holds the call's name and the engine's message.
enum Result { kDone, kRejected, kError };

// levenberg_marquardt_strategy.cc:97-118: inexact step, stopped by the relative decrease of
// the quadratic model (eta) and not by the residual (r_tolerance = -1)
cb200_cgnr_options ConjugateGradientOptions(const Solver::Options& options) {
  const int32_t preconditioner = options.preconditioner_type == JACOBI
                                     ? CB200_PRECONDITIONER_BLOCK_JACOBI
                                 : options.preconditioner_type == IDENTITY
                                     ? CB200_PRECONDITIONER_IDENTITY
                                     : CB200_PRECONDITIONER_SCALAR_JACOBI;
  return {options.min_linear_solver_iterations, options.max_linear_solver_iterations, -1.0,
          options.eta, preconditioner};
}

class TrustRegionState {
 public:
  virtual ~TrustRegionState() = default;
  // Cost, gradient and Jacobian at the accepted state (the first call: the initial state).
  virtual Result EvaluateJacobian(double* cost) = 0;
  // J <- J diag(scale); compute: scale = 1 / (1 + sqrt(diag(J'J))) of this Jacobian first.
  virtual Result ScaleJacobian(bool compute) = 0;
  // LM diagonal, linear solve, delta = -y * scale, the norms and the candidate x (+) delta,
  // reported as the engine's trust-region step reports them.
  virtual Result ComputeStep(double radius, bool reuse_diagonal, cb200_step_summary* step) = 0;
  virtual Result EvaluateCandidate(double* cost) = 0;  // cost only
  virtual void AcceptCandidate() = 0;
  virtual double GradientMaxNorm() = 0;
  // The accepted state into the caller's x; evaluation counts, evaluation and linear solver
  // times into the summary.
  virtual void Finish(Solver::Summary* summary) = 0;
  const std::string& error() const { return error_; }

 protected:
  Result Fail(cb200_engine* engine, const char* call) {
    error_ = std::string(call) + ": " + cb200_engine_last_error(engine);
    return kError;
  }
  std::string error_;
};

// State, step, gradient and diagonals in HBM (cb200_engine_trust_region_step and friends,
// include/ceres_b200.h): per iteration the host reads a handful of scalars.  The state
// crosses PCIe twice, up and down at the end, and HostState's work vectors are never
// allocated: page-locking those costs 0.5 s on BAL L.
class DeviceState final : public TrustRegionState {
 public:
  DeviceState(const Solver::Options& options, cb200_engine* engine, double* x)
      : options_(options), engine_(engine), x_(x) {}
  Result EvaluateJacobian(double* cost) override {
    if (!uploaded_ && cb200_engine_state_upload(engine_, x_) != CB200_OK)
      return Fail("cb200_engine_state_upload");
    uploaded_ = true;
    return Evaluate(0, true, cost);
  }
  Result ScaleJacobian(bool compute) override {
    if (cb200_engine_jacobi_scale(engine_, compute) != CB200_OK) return Fail("cb200_engine_jacobi_scale");
    return kDone;
  }
  Result ComputeStep(double radius, bool reuse_diagonal, cb200_step_summary* step) override {
    cb200_step_options so{};
    so.radius = radius;
    so.min_lm_diagonal = options_.min_lm_diagonal;
    so.max_lm_diagonal = options_.max_lm_diagonal;
    so.reuse_diagonal = reuse_diagonal;
    so.cg = ConjugateGradientOptions(options_);
    const double ls_start = Seconds();
    if (cb200_engine_trust_region_step(engine_, &so, step) != CB200_OK)
      return Fail("cb200_engine_trust_region_step");
    linear_solver_seconds_ += Seconds() - ls_start;
    return kDone;
  }
  Result EvaluateCandidate(double* cost) override { return Evaluate(1, false, cost); }
  void AcceptCandidate() override { cb200_engine_accept_candidate(engine_); }
  double GradientMaxNorm() override {
    double gmax = 0.0;
    cb200_engine_gradient_max_norm(engine_, &gmax);
    return gmax;
  }
  void Finish(Solver::Summary* summary) override {
    cb200_engine_state_download(engine_, 0, x_);
    summary->linear_solver_time_in_seconds = linear_solver_seconds_;
    summary->residual_evaluation_time_in_seconds = evaluation_seconds_[0];
    summary->num_residual_evaluations = evaluation_calls_[0];
    summary->jacobian_evaluation_time_in_seconds = evaluation_seconds_[1];
    summary->num_jacobian_evaluations = evaluation_calls_[1];
  }

 private:
  Result Fail(const char* call) { return TrustRegionState::Fail(engine_, call); }
  // at state slot `which`: 0 the accepted state, 1 the candidate
  Result Evaluate(int which, bool jacobian, double* cost) {
    const double t0 = Seconds();
    const int rc = cb200_engine_evaluate_state(
        engine_, which,
        CB200_APPLY_LOSS_FUNCTION | CB200_KEEP_JACOBIAN_ON_DEVICE | CB200_KEEP_RESIDUALS_ON_DEVICE,
        jacobian, jacobian, jacobian, cost);
    evaluation_seconds_[jacobian] += Seconds() - t0;
    ++evaluation_calls_[jacobian];
    if (rc < 0) return Fail("cb200_engine_evaluate_state");
    return rc == CB200_OK ? kDone : kRejected;
  }

  const Solver::Options& options_;
  cb200_engine* const engine_;
  double* const x_;
  bool uploaded_ = false;
  double linear_solver_seconds_ = 0.0, evaluation_seconds_[2] = {0.0, 0.0};
  int evaluation_calls_[2] = {0, 0};
};

// State, gradient, step and diagonals in host memory around the evaluator.  The linear solve
// runs where the evaluator keeps the Jacobian: conjugate gradients in HBM for a
// device-resident one (cb200_engine_cgnr_solve), SolveNormalEquations for a host one.
class HostState final : public TrustRegionState {
 public:
  HostState(const Solver::Options& options, const internal::Program& program,
            internal::Evaluator* evaluator, internal::SparseMatrix* jacobian, PinnedVector* x)
      : options_(options), evaluator_(evaluator), jacobian_(jacobian),
        resident_(dynamic_cast<internal::DeviceResidentJacobian*>(jacobian)),
        n_(program.NumParameters()), ne_(program.NumEffectiveParameters()),
        nt_(std::max(1, options.num_threads)), x_(*x), x_plus_(n_), gradient_(ne_),
        scale_(ne_, 1.0), diagonal_(ne_), D2_(ne_), y_(ne_), delta_(ne_) {
    // only the host linear solver reads the residuals and the model on the host; with a
    // device-resident Jacobian the residuals stay on the device as well
    if (!resident_) {
      residuals_.resize(program.NumResiduals());
      model_.resize(program.NumResiduals());
    }
  }
  Result EvaluateJacobian(double* cost) override {
    double* const residuals = resident_ ? nullptr : residuals_.data();
    const bool ok = evaluator_->Evaluate(x_.data(), cost, residuals, gradient_.data(), jacobian_);
    return ok ? kDone : kRejected;
  }
  Result ScaleJacobian(bool compute) override {
    if (compute) {
      jacobian_->SquaredColumnNorm(scale_.data());
      ForEach(nt_, ne_, [&](int64_t i) { scale_[i] = 1.0 / (1.0 + std::sqrt(scale_[i])); });
    }
    jacobian_->ScaleColumns(scale_.data());
    return kDone;
  }
  Result ComputeStep(double radius, bool reuse_diagonal, cb200_step_summary* step) override {
    if (!reuse_diagonal) {
      jacobian_->SquaredColumnNorm(diagonal_.data());
      ForEach(nt_, ne_, [&](int64_t i) {
        diagonal_[i] =
            std::min(std::max(diagonal_[i], options_.min_lm_diagonal), options_.max_lm_diagonal);
      });
    }
    ForEach(nt_, ne_, [&](int64_t i) { D2_[i] = diagonal_[i] / radius; });
    const double ls_start = Seconds();
    if (resident_) {
      const cb200_cgnr_options cg_options = ConjugateGradientOptions(options_);
      y_.assign(ne_, 0.0);
      if (cb200_engine_cgnr_solve(resident_->engine(), D2_.data(), &cg_options, y_.data(),
                                  &step->cg) != CB200_OK)
        return Fail(resident_->engine(), "cb200_engine_cgnr_solve");
      // step = -y: model cost change = (J y).r - |J y|^2 / 2
      step->model_cost_change = step->cg.jy_dot_b - 0.5 * step->cg.jy_squared_norm;
      ForEach(nt_, ne_, [&](int64_t i) { y_[i] = -y_[i]; });
    } else {
      step->cg.num_iterations =
          SolveNormalEquations(*jacobian_, D2_.data(), residuals_.data(),
                               options_.max_linear_solver_iterations, 1e-2 * options_.eta, &y_);
      // step = -y (scaled space); model cost change = -m'(r + m/2), m = J step
      std::fill(model_.begin(), model_.end(), 0.0);
      for (int i = 0; i < ne_; ++i) y_[i] = -y_[i];
      jacobian_->RightMultiplyAndAccumulate(y_.data(), model_.data());
      double model_cost_change = 0.0;
      for (size_t i = 0; i < model_.size(); ++i)
        model_cost_change -= model_[i] * (residuals_[i] + 0.5 * model_[i]);
      step->model_cost_change = model_cost_change;
    }
    linear_solver_seconds_ += Seconds() - ls_start;
    ForEach(nt_, ne_, [&](int64_t i) { delta_[i] = y_[i] * scale_[i]; });
    step->step_norm = std::sqrt(Reduce(nt_, ne_, false, [&](int64_t i) { return delta_[i] * delta_[i]; }));
    step->state_norm = std::sqrt(Reduce(nt_, n_, false, [&](int64_t i) { return x_[i] * x_[i]; }));
    step->plus_ok = step->cg.termination != 2 && step->model_cost_change > 0.0 &&
                    evaluator_->Plus(x_.data(), delta_.data(), x_plus_.data());
    return kDone;
  }
  Result EvaluateCandidate(double* cost) override {
    return evaluator_->Evaluate(x_plus_.data(), cost, nullptr, nullptr, nullptr) ? kDone : kRejected;
  }
  void AcceptCandidate() override { ForEach(nt_, n_, [&](int64_t i) { x_[i] = x_plus_[i]; }); }
  double GradientMaxNorm() override {
    return Reduce(nt_, ne_, true, [&](int64_t i) { return std::fabs(gradient_[i]); });
  }
  void Finish(Solver::Summary* summary) override {
    summary->linear_solver_time_in_seconds = linear_solver_seconds_;
    for (const auto& kv : evaluator_->Statistics()) {
      if (kv.first == "Evaluator::Residual") {
        summary->residual_evaluation_time_in_seconds = kv.second.time;
        summary->num_residual_evaluations = kv.second.calls;
      } else if (kv.first == "Evaluator::Jacobian") {
        summary->jacobian_evaluation_time_in_seconds = kv.second.time;
        summary->num_jacobian_evaluations = kv.second.calls;
      }
    }
  }

 private:
  const Solver::Options& options_;
  internal::Evaluator* const evaluator_;
  internal::SparseMatrix* const jacobian_;
  internal::DeviceResidentJacobian* const resident_;
  const int n_, ne_, nt_;
  double linear_solver_seconds_ = 0.0;
  PinnedVector& x_;
  PinnedVector x_plus_, gradient_, scale_, diagonal_, D2_, y_;
  std::vector<double> delta_, residuals_, model_;
};

// The state stays in HBM unless the program needs the host: bounds, a manifold only the host
// knows, an EvaluationCallback that must see the parameter blocks.
bool DeviceLoopPossible(const internal::Program& program, const internal::ProblemImpl& problem) {
  if (std::getenv("CB200_HOST_TRUST_REGION")) return false;
  if (problem.options().evaluation_callback != nullptr) return false;
  for (const internal::ParameterBlock* pb : program.parameter_blocks()) {
    if (pb->lower_bounds || pb->upper_bounds) return false;
    int kind = 0, param = 0;
    if (pb->manifold && !pb->manifold->DeviceDescription(&kind, &param)) return false;
  }
  return true;
}

// Returns without Finish when the initial evaluation or Jacobi scaling fails.
void Minimize(const Solver::Options& options, TrustRegionState* state, double fixed_cost,
              double start, Solver::Summary* summary) {
  auto fail = [&](const std::string& message) {
    summary->termination_type = FAILURE;
    summary->message = message;
  };
  double cost = 0.0;
  Result result = state->EvaluateJacobian(&cost);
  if (result != kDone) {
    summary->message = "Initial residual and Jacobian evaluation failed.";
    if (result == kError) fail(state->error());
    return;
  }
  summary->initial_cost = cost + fixed_cost;
  if (options.jacobi_scaling && state->ScaleJacobian(true) != kDone) return fail(state->error());
  double radius = options.initial_trust_region_radius, decrease_factor = 2.0;
  bool reuse_diagonal = false;
  summary->termination_type = NO_CONVERGENCE;
  summary->message = "Maximum number of iterations reached.";
  if (options.minimizer_progress_to_stdout)
    std::printf("iter      cost      cost_change  |gradient|   |step|    tr_ratio  tr_radius  ls_iter\n"
                "%4d  %.6e    %.2e   %.2e   %.2e  %.2e  %.2e   %5d\n",
                0, cost + fixed_cost, 0.0, 0.0, 0.0, 0.0, radius, 0);
  const bool timing = std::getenv("CB200_SOLVER_TIMING") != nullptr;
  for (int it = 1; it <= options.max_num_iterations; ++it) {
    if (Seconds() - start > options.max_solver_time_in_seconds) {
      summary->message = "Maximum solver time reached.";
      break;
    }
    cb200_step_summary step{};
    const double step_start = Seconds();
    if (state->ComputeStep(radius, reuse_diagonal, &step) != kDone) { fail(state->error()); break; }
    if (timing)
      std::fprintf(stderr, "iteration %d: trust-region step %.1f ms wall, %d linear solver iterations, "
                   "%.1f ms of them on the device\n", it, (Seconds() - step_start) * 1e3,
                   step.cg.num_iterations, step.cg.solve_ms);
    Solver::IterationSummary is;
    is.iteration = it;
    is.linear_solver_iterations = step.cg.num_iterations;
    is.step_norm = step.step_norm;
    double new_cost = 0.0;
    bool ok = step.cg.termination != 2 && step.model_cost_change > 0.0 && step.plus_ok;
    if (ok) {
      result = state->EvaluateCandidate(&new_cost);
      if (result == kError) { fail(state->error()); break; }
      ok = result == kDone;
    }
    const double relative_decrease = ok ? (cost - new_cost) / step.model_cost_change : -1.0;
    is.relative_decrease = relative_decrease;
    if (ok && relative_decrease > options.min_relative_decrease) {
      is.step_is_successful = true;
      is.cost_change = cost - new_cost;
      state->AcceptCandidate();
      if (state->EvaluateJacobian(&cost) != kDone) { fail("Residual and Jacobian evaluation failed."); break; }
      if (options.jacobi_scaling && state->ScaleJacobian(false) != kDone) { fail(state->error()); break; }
      radius = std::min(options.max_trust_region_radius,
                        radius / std::max(1.0 / 3.0, 1.0 - std::pow(2.0 * relative_decrease - 1.0, 3)));
      decrease_factor = 2.0;
      reuse_diagonal = false;
      ++summary->num_successful_steps;
    } else {
      radius /= decrease_factor;
      decrease_factor *= 2.0;
      reuse_diagonal = true;
      ++summary->num_unsuccessful_steps;
    }
    const double gmax = state->GradientMaxNorm();
    is.cost = cost + fixed_cost;
    is.gradient_max_norm = gmax;
    is.trust_region_radius = radius;
    summary->iterations.push_back(is);
    if (options.minimizer_progress_to_stdout)
      std::printf("%4d  %.6e    %.2e   %.2e   %.2e  %.2e  %.2e   %5d\n", it, is.cost, is.cost_change,
                  gmax, step.step_norm, relative_decrease, radius, step.cg.num_iterations);
    const char* converged = nullptr;
    if (!is.step_is_successful)
      converged = radius < options.min_trust_region_radius ? "Minimum trust region radius reached." : nullptr;
    else if (std::fabs(is.cost_change) <= options.function_tolerance * cost)
      converged = "Function tolerance reached.";
    else if (gmax <= options.gradient_tolerance)
      converged = "Gradient tolerance reached.";
    else if (step.step_norm <= options.parameter_tolerance * (step.state_norm + options.parameter_tolerance))
      converged = "Parameter tolerance reached.";
    if (converged) {
      summary->termination_type = CONVERGENCE;
      summary->message = converged;
      break;
    }
  }
  state->Finish(summary);
  summary->final_cost = cost + fixed_cost;
}
}  // namespace

namespace internal {
// The parameter blocks that only ever appear as argument j of their residual blocks form an
// independent set: every residual block holds exactly one of them (the points of a bundle
// adjustment problem for j = 1).  Puts them in group 0 and everything else in group 1 for the
// argument slot with the most such blocks; false when no slot covers half of the variable
// blocks (a small first group is not worth its own region of the Jacobian).
bool ArgumentSlotOrdering(const ProblemImpl& problem, ParameterBlockOrdering* ordering) {
  const auto& pbs = problem.parameter_blocks();
  std::vector<uint32_t> slots(pbs.size(), 0u);
  int common_slots = CB200_MAX_PARAMETER_BLOCKS;
  for (const ResidualTypeStore& t : problem.types()) {
    const int nb = t.desc.num_parameter_blocks;
    if (t.size() == 0) continue;
    common_slots = std::min(common_slots, nb);
    for (size_t k = 0; k < t.parameter_blocks.size(); ++k)
      slots[t.parameter_blocks[k]] |= 1u << (k % nb);
  }
  int best_slot = -1;
  size_t best_count = 0, variable = 0;
  for (size_t i = 0; i < pbs.size(); ++i) variable += !pbs[i]->IsConstant();
  for (int j = 0; j < common_slots; ++j) {
    size_t count = 0;
    for (size_t i = 0; i < pbs.size(); ++i) count += slots[i] == (1u << j) && !pbs[i]->IsConstant();
    if (count > best_count) { best_count = count; best_slot = j; }
  }
  if (best_slot < 0 || 2 * best_count < variable) return false;
  for (size_t i = 0; i < pbs.size(); ++i)
    ordering->AddElementToGroup(pbs[i]->user_state, slots[i] == (1u << best_slot) ? 0 : 1);
  return true;
}
}  // namespace internal

void Solver::Solve(const Options& options, Problem* problem, Summary* summary) {
  const double start = Seconds();
  *summary = Summary();
  if (!options.IsValid(&summary->message)) {
    summary->termination_type = FAILURE;
    return;
  }
  if (!options.use_cuda_for_evaluator) {
    summary->message = "This library only provides the CUDA evaluator: solve a ProblemCUDA "
                       "with ceres::Solve(options, ProblemCUDA*, summary).";
    return;
  }
  internal::ProblemImpl* impl = problem->mutable_impl();
  summary->num_parameter_blocks = impl->NumParameterBlocks();
  summary->num_parameters = impl->NumParameters();
  summary->num_residual_blocks = impl->NumResidualBlocks();
  summary->num_residuals = impl->NumResiduals();
  for (const auto& pb : impl->parameter_blocks())
    summary->num_effective_parameters += pb->TangentSize();

  // ---- preprocessing (trust_region_preprocessor.cc:373-407)
  internal::Program full(impl);
  std::vector<double*> removed;
  double fixed_cost = 0.0;
  std::unique_ptr<internal::Program> program =
      full.CreateReducedProgram(&removed, &fixed_cost, &summary->message);
  if (!program) return;
  summary->fixed_cost = fixed_cost;
  if (program->NumParameterBlocks() == 0) {
    summary->termination_type = CONVERGENCE;
    summary->message = "Function tolerance reached. No non-constant parameter blocks found.";
    summary->initial_cost = summary->final_cost = fixed_cost;
    return;
  }
  const bool schur = options.linear_solver_type == DENSE_SCHUR ||
                     options.linear_solver_type == SPARSE_SCHUR ||
                     options.linear_solver_type == ITERATIVE_SCHUR;
  // CGNR with CUDA_SPARSE keeps the Jacobian in HBM (below): its layout is private to the
  // device, so a two-group ordering is applied there too.  With the first group's cells in one
  // region and the rest in another, the 32 cells a warp writes per argument are one contiguous
  // run, which is what the bulk stores of the evaluation kernel and the per-type J'(J p) kernel
  // need; in the row-by-row layout of num_eliminate_blocks = 0 both fall back to their
  // per-thread paths (measured on BAL L: evaluation 2.63 instead of 1.83 ms, 11.7 instead of
  // 1.43 ms per conjugate-gradient product; profiles/r2_solve_L_launches_rowwise_layout.csv).
  const bool resident_cgnr = options.linear_solver_type == CGNR &&
                             options.sparse_linear_algebra_library_type == CUDA_SPARSE;
  const ParameterBlockOrdering* ordering = options.linear_solver_ordering.get();
  // No ordering given for the resident layout: the argument-slot independent set (above)
  // becomes the first group.
  ParameterBlockOrdering slot_ordering;
  if (resident_cgnr && !ordering && internal::ArgumentSlotOrdering(*impl, &slot_ordering))
    ordering = &slot_ordering;
  int num_eliminate_blocks = 0;
  if ((schur || resident_cgnr) && ordering) {
    // ApplyOrdering + size of the first elimination group (reorder_program.cc:469-560).
    program->ReorderParameterBlocksByGroup(ordering->element_to_group());
    const int first = ordering->MinGroup();
    for (const internal::ParameterBlock* pb : program->parameter_blocks())
      num_eliminate_blocks += ordering->GroupId(pb->user_state) == first;
    if (num_eliminate_blocks > 0 && num_eliminate_blocks < program->NumParameterBlocks())
      program->LexicographicallyOrderResidualBlocks(num_eliminate_blocks);
    else
      num_eliminate_blocks = 0;
  }
  internal::Evaluator::Options eo;
  eo.num_threads = options.num_threads;
  eo.num_eliminate_blocks = num_eliminate_blocks;
  eo.linear_solver_type = options.linear_solver_type;
  eo.sparse_linear_algebra_library_type = options.sparse_linear_algebra_library_type;
  eo.use_cuda = true;
  eo.registered_cuda_evaluators = options.registered_cuda_evaluators;
  eo.evaluation_callback = impl->options().evaluation_callback;
  eo.device = options.cuda_device;
  // CGNR with CUDA_SPARSE is the reference's device-resident combination
  // (cgnr_solver.cc CudaCgnrSolver): the Jacobian stays in HBM and conjugate gradients on
  // the normal equations run there (cb200_engine_cgnr_solve).
  eo.jacobian_on_device = options.linear_solver_type == CGNR &&
                          options.sparse_linear_algebra_library_type == CUDA_SPARSE;
  std::unique_ptr<internal::Evaluator> evaluator =
      internal::Evaluator::Create(eo, program.get(), &summary->message);
  if (!evaluator) return;
  std::unique_ptr<internal::SparseMatrix> jacobian = evaluator->CreateJacobian();
  summary->num_parameter_blocks_reduced = program->NumParameterBlocks();
  summary->num_parameters_reduced = program->NumParameters();
  summary->num_effective_parameters_reduced = program->NumEffectiveParameters();
  summary->num_residual_blocks_reduced = program->NumResidualBlocks();
  summary->num_residuals_reduced = program->NumResiduals();
  summary->preprocessor_time_in_seconds = Seconds() - start;

  // ---- trust-region loop
  const double minimizer_start = Seconds();
  PinnedVector x(program->NumParameters());
  program->ParameterBlocksToStateVector(x.data());
  auto* resident = dynamic_cast<internal::DeviceResidentJacobian*>(jacobian.get());
  std::unique_ptr<TrustRegionState> state;
  if (resident && DeviceLoopPossible(*program, *impl))
    state.reset(new DeviceState(options, resident->engine(), x.data()));
  else
    state.reset(new HostState(options, *program, evaluator.get(), jacobian.get(), &x));
  Minimize(options, state.get(), fixed_cost, start, summary);
  program->StateVectorToParameterBlocks(x.data());  // results back into the user's arrays
  summary->minimizer_time_in_seconds = Seconds() - minimizer_start;
  summary->total_time_in_seconds = Seconds() - start;
}

void Solve(const Solver::Options& options, Problem* problem, Solver::Summary* summary) {
  nvtxRangePushA("ceres::Solve");
  Solver solver;
  solver.Solve(options, problem, summary);
  nvtxRangePop();
}

}  // namespace ceres
