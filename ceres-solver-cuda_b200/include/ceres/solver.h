// ceres::Solver — the option/summary plumbing of the evaluation path and a minimal
// TRUST_REGION (Levenberg-Marquardt) loop that drives it.
//
// Scope.  The reference routes `Solver::Options::use_cuda_for_evaluator` /
// `registered_cuda_evaluators` (include/ceres/solver.h:831-841) through
// solver.cc:675-758 and trust_region_preprocessor.cc:260-289 into Evaluator::Create,
// and rejects non-TRUST_REGION minimizers for the CUDA evaluator (solver.cc:702-708).
// This header keeps that surface so code written for the reference
// (examples/bundle_adjuster.cu.cc) compiles and runs:
//     ceres::Solver::Options options;  options.linear_solver_type = ceres::ITERATIVE_SCHUR;
//     ceres::Solve(options, &problem_cuda, &summary);  std::cout << summary.FullReport();
// The minimizer and the linear solvers themselves are OUT OF SCOPE for this repository
// (they stay on the reference's implementation, DESIGN.md section 7): what is here is the
// preprocessing the evaluator depends on (reduced program, ordering, Schur residual
// order; trust_region_preprocessor.cc:373-407), the LM bookkeeping
// (levenberg_marquardt_strategy.cc:68-165, trust_region_minimizer.cc step acceptance) and
// a Jacobi-preconditioned CGNR on the host as the stand-in linear solver for every
// linear_solver_type.
#ifndef CERES_B200_SOLVER_H_
#define CERES_B200_SOLVER_H_

#include <map>
#include <memory>
#include <string>
#include <unordered_map>
#include <vector>

#include "ceres/internal/evaluator.h"
#include "ceres/problem.h"
#include "ceres/types.h"

namespace ceres {

// include/ceres/ordered_groups.h: group id per parameter block, lower groups are
// eliminated first.
class ParameterBlockOrdering {
 public:
  bool AddElementToGroup(const double* element, int group) {
    groups_[element] = group;
    return true;
  }
  int GroupId(const double* element) const {
    auto it = groups_.find(element);
    return it == groups_.end() ? -1 : it->second;
  }
  int NumElements() const { return static_cast<int>(groups_.size()); }
  int GroupSize(int group) const {
    int n = 0;
    for (const auto& kv : groups_) n += kv.second == group;
    return n;
  }
  int MinGroup() const {
    int m = 0x7fffffff;
    for (const auto& kv : groups_) m = kv.second < m ? kv.second : m;
    return m;
  }
  const std::unordered_map<const double*, int>& element_to_group() const { return groups_; }

 private:
  std::unordered_map<const double*, int> groups_;
};

namespace internal {
class ProblemImpl;
// Two-group ordering from the argument slots of the residual blocks (csrc/solver.cc): used for
// the device-resident Jacobian layout when the caller gives no linear_solver_ordering.
bool ArgumentSlotOrdering(const ProblemImpl& problem, ParameterBlockOrdering* ordering);
}  // namespace internal

enum TerminationType { CONVERGENCE, NO_CONVERGENCE, FAILURE, USER_SUCCESS, USER_FAILURE };

class Solver {
 public:
  struct Options {
    MinimizerType minimizer_type = TRUST_REGION;
    int max_num_iterations = 50;
    double max_solver_time_in_seconds = 1e9;
    int num_threads = 1;
    double initial_trust_region_radius = 1e4;
    double max_trust_region_radius = 1e16;
    double min_trust_region_radius = 1e-32;
    double min_relative_decrease = 1e-3;
    double min_lm_diagonal = 1e-6;
    double max_lm_diagonal = 1e32;
    double function_tolerance = 1e-6;
    double gradient_tolerance = 1e-10;
    double parameter_tolerance = 1e-8;
    LinearSolverType linear_solver_type = SPARSE_NORMAL_CHOLESKY;
    SparseLinearAlgebraLibraryType sparse_linear_algebra_library_type = NO_SPARSE;
    // IDENTITY and JACOBI need CGNR with CUDA_SPARSE.  The default is SCALAR_JACOBI rather
    // than Ceres' JACOBI so that existing callers keep the steps they had before this option
    // existed.
    PreconditionerType preconditioner_type = SCALAR_JACOBI;
    std::shared_ptr<ParameterBlockOrdering> linear_solver_ordering;
    int min_linear_solver_iterations = 0;
    int max_linear_solver_iterations = 500;
    double eta = 1e-1;
    bool jacobi_scaling = true;
    bool minimizer_progress_to_stdout = false;
    bool use_nonmonotonic_steps = false;
    bool use_inner_iterations = false;
    // The evaluation path (include/ceres/solver.h:831-841 of the reference).
    bool use_cuda_for_evaluator = false;
    internal::RegisteredCUDAEvaluators* registered_cuda_evaluators = nullptr;
    // Extension: CUDA device ordinal.
    int cuda_device = 0;

    bool IsValid(std::string* error) const;
  };

  struct IterationSummary {
    int iteration = 0;
    bool step_is_successful = false;
    double cost = 0.0, cost_change = 0.0, gradient_max_norm = 0.0, step_norm = 0.0;
    double relative_decrease = 0.0, trust_region_radius = 0.0;
    int linear_solver_iterations = 0;
  };

  struct Summary {
    TerminationType termination_type = FAILURE;
    std::string message = "ceres::Solve was not called.";
    double initial_cost = -1.0, final_cost = -1.0, fixed_cost = -1.0;
    std::vector<IterationSummary> iterations;
    int num_successful_steps = 0, num_unsuccessful_steps = 0;
    int num_parameter_blocks = 0, num_parameters = 0, num_effective_parameters = 0;
    int num_residual_blocks = 0, num_residuals = 0;
    int num_parameter_blocks_reduced = 0, num_parameters_reduced = 0;
    int num_effective_parameters_reduced = 0, num_residual_blocks_reduced = 0;
    int num_residuals_reduced = 0;
    double preprocessor_time_in_seconds = 0.0, minimizer_time_in_seconds = 0.0;
    double total_time_in_seconds = 0.0, linear_solver_time_in_seconds = 0.0;
    double residual_evaluation_time_in_seconds = 0.0, jacobian_evaluation_time_in_seconds = 0.0;
    int num_residual_evaluations = 0, num_jacobian_evaluations = 0;
    bool IsSolutionUsable() const {
      return termination_type == CONVERGENCE || termination_type == NO_CONVERGENCE ||
             termination_type == USER_SUCCESS;
    }
    std::string BriefReport() const;
    // Same "Time (in seconds)" block as the reference (internal/ceres/solver.cc:1101-1112),
    // the lines its README benchmarks quote.
    std::string FullReport() const;
  };

  void Solve(const Options& options, Problem* problem, Summary* summary);
};

void Solve(const Solver::Options& options, Problem* problem, Solver::Summary* summary);

}  // namespace ceres

#endif  // CERES_B200_SOLVER_H_
