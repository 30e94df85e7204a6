// C interface of the test/bench driver for the conjugate-gradient preconditioners
// (Solver::Options::preconditioner_type, cb200_cgnr_options::preconditioner).  Python binds it
// with ctypes (ceres-solver-cuda_b200/binding.py).
#include <cstdlib>

#include "driver.h"

using driver::DriverProblem;

extern "C" {

// cb200_engine_cgnr_solve on the Jacobian the last evaluation left in HBM.  preconditioner:
// CB200_PRECONDITIONER_*.  out: [iterations, termination, |J'b|, final residual norm, (Jy).b,
// |Jy|^2, ms]
int drv_cgnr_solve_preconditioned(void* h, const double* d_squared, int min_iterations,
                                  int max_iterations, double r_tolerance, double q_tolerance,
                                  int preconditioner, double* solution, double* out) {
  auto* dp = static_cast<DriverProblem*>(h);
  if (!dp->evaluator) return -100;
  cb200_cgnr_options o{min_iterations, max_iterations, r_tolerance, q_tolerance, preconditioner};
  cb200_cgnr_summary s;
  const int rc = cb200_engine_cgnr_solve(dp->evaluator->engine(), d_squared, &o, solution, &s);
  if (rc != CB200_OK) { dp->error = cb200_engine_last_error(dp->evaluator->engine()); return rc; }
  out[0] = s.num_iterations; out[1] = s.termination; out[2] = s.initial_gradient_norm;
  out[3] = s.final_residual_norm; out[4] = s.jy_dot_b; out[5] = s.jy_squared_norm;
  out[6] = s.solve_ms;
  return rc;
}

// ceres::Solve(options, ProblemCUDA*, summary) on the driver's problem with
// options.preconditioner_type = preconditioner (a ceres::PreconditionerType).  ordering: group
// id per parameter block (or NULL).  out: [initial_cost, final_cost, iterations,
// successful_steps, termination_type, num_jacobian_evaluations, num_residual_evaluations,
// linear solver seconds, linear solver iterations over all steps].  The solution is written to
// the driver's parameter values (drv_user_values).
int drv_solve_preconditioned(void* h, int linear_solver_type, int cuda_sparse, int preconditioner,
                             int max_num_iterations, const int* ordering, int device,
                             double* out) {
  auto* dp = static_cast<DriverProblem*>(h);
  ceres::Solver::Options options;
  options.linear_solver_type = static_cast<ceres::LinearSolverType>(linear_solver_type);
  if (cuda_sparse) options.sparse_linear_algebra_library_type = ceres::CUDA_SPARSE;
  options.preconditioner_type = static_cast<ceres::PreconditionerType>(preconditioner);
  options.max_num_iterations = max_num_iterations;
  options.cuda_device = device;
  // (tests that compare two trust-region loops ask for near-exact steps: with the default
  // eta = 0.1 the point where conjugate gradients stop depends on the last bits of the sums)
  if (const char* eta = std::getenv("CB200_DRIVER_ETA")) options.eta = std::atof(eta);
  if (ordering) {
    auto* o = new ceres::ParameterBlockOrdering;
    for (size_t k = 0; k < dp->pb_offset.size(); ++k)
      o->AddElementToGroup(dp->pb(static_cast<int>(k)), ordering[k]);
    options.linear_solver_ordering.reset(o);
  }
  ceres::Solver::Summary summary;
  ceres::Solve(options, &dp->problem, &summary);
  dp->error = summary.message;
  out[0] = summary.initial_cost;
  out[1] = summary.final_cost;
  out[2] = static_cast<double>(summary.iterations.size());
  out[3] = summary.num_successful_steps;
  out[4] = static_cast<double>(summary.termination_type);
  out[5] = summary.num_jacobian_evaluations;
  out[6] = summary.num_residual_evaluations;
  out[7] = summary.linear_solver_time_in_seconds;
  out[8] = 0;
  for (const auto& it : summary.iterations) out[8] += it.linear_solver_iterations;
  return summary.IsSolutionUsable() ? 1 : 0;
}

// Solver::Options::IsValid with the CUDA evaluator requested, for a minimizer type (0
// LINE_SEARCH, 1 TRUST_REGION), a linear solver type and a preconditioner (ceres enum values;
// < 0 keeps the default) and CUDA_SPARSE or not.  Returns 1 when valid; the message is copied to
// msg.
int drv_options_is_valid_for(void* h, int minimizer_type, int linear_solver_type, int cuda_sparse,
                             int preconditioner, char* msg, int msg_size) {
  auto* dp = static_cast<DriverProblem*>(h);
  ceres::Solver::Options options;
  options.minimizer_type = static_cast<ceres::MinimizerType>(minimizer_type);
  if (linear_solver_type >= 0)
    options.linear_solver_type = static_cast<ceres::LinearSolverType>(linear_solver_type);
  if (cuda_sparse) options.sparse_linear_algebra_library_type = ceres::CUDA_SPARSE;
  if (preconditioner >= 0)
    options.preconditioner_type = static_cast<ceres::PreconditionerType>(preconditioner);
  options.use_cuda_for_evaluator = true;
  options.registered_cuda_evaluators = dp->problem.mutable_registered_cuda_evaluators();
  std::string error;
  const bool ok = options.IsValid(&error);
  std::snprintf(msg, msg_size, "%s", error.c_str());
  return ok ? 1 : 0;
}

}  // extern "C"
