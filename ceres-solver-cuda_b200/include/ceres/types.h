// Enums of the public API that the evaluation path reads
// (reference: include/ceres/types.h; only the members the path dispatches on).
#ifndef CERES_B200_TYPES_H_
#define CERES_B200_TYPES_H_

namespace ceres {

// Argument type used in interfaces that can optionally take ownership of a
// passed in argument.
enum Ownership { DO_NOT_TAKE_OWNERSHIP, TAKE_OWNERSHIP };

// Selects the Jacobian container (internal/ceres/evaluator.cc:57-92).
enum LinearSolverType {
  DENSE_NORMAL_CHOLESKY,
  DENSE_QR,
  SPARSE_NORMAL_CHOLESKY,
  DENSE_SCHUR,
  SPARSE_SCHUR,
  ITERATIVE_SCHUR,
  CGNR
};

enum SparseLinearAlgebraLibraryType {
  SUITE_SPARSE,
  EIGEN_SPARSE,
  ACCELERATE_SPARSE,
  CUDA_SPARSE,
  NO_SPARSE
};

// Preconditioner of the iterative linear solvers; this library reads it for CGNR with
// CUDA_SPARSE (the conjugate gradients on the device-resident Jacobian).
//   IDENTITY       no preconditioning.
//   JACOBI         the block diagonal of J'J + D'D, one dense block per parameter block,
//                  inverted (Ceres' CGNR JACOBI).
//   SCALAR_JACOBI  extension of this library, not a Ceres name: the scalar diagonal
//                  diag(J'J + D'D)^-1.
enum PreconditionerType { IDENTITY, JACOBI, SCALAR_JACOBI };

enum MinimizerType { LINE_SEARCH, TRUST_REGION };

constexpr int DYNAMIC = -1;

}  // namespace ceres

#endif  // CERES_B200_TYPES_H_
