// The SoftLOne, Arctan, Tolerant, Tukey, scaled and composed loss kinds of the test driver
// (driver_losses.cu, driver_losses2.cu), numbered after driver.h's LossKind; see problems.py.
#ifndef TESTS_DRIVER_DRIVER_LOSSES_H_
#define TESTS_DRIVER_DRIVER_LOSSES_H_

#include "driver.h"

namespace driver {

// SoftLOne(a), Arctan(a), Tolerant(a, b), Tukey(a), Scaled(SoftLOne(a), b), Scaled(Tukey(a), b),
// Composed(Scaled(SoftLOne(a), b), Cauchy(a))
enum NewLossKind { kSoftLOne = 8, kArctan, kTolerant, kTukey, kScaledSoftLOne, kScaledTukey,
                   kComposed };

// kComposed: more than CB200_INLINE_LOSS_BYTES, so the kernel reads it from the loss table.
using ComposedLoss =
    ceres::ComposedLossCUDA<ceres::ScaledLossCUDA<ceres::SoftLOneLossCUDA>, ceres::CauchyLossCUDA>;
static_assert(sizeof(ComposedLoss) > CB200_INLINE_LOSS_BYTES, "meant for the loss-table path");

// Same contract as driver.h's AddRun* functions, for the kinds above.
bool AddRunLosses(DriverProblem& dp, int type, int loss_kind, double a, double b, int n,
                  const int* pb, const double* fdata, bool bulk, bool* handled);
bool AddRunScaledAndComposedLosses(DriverProblem& dp, int type, int loss_kind, double a, double b,
                                   int n, const int* pb, const double* fdata, bool bulk,
                                   bool* handled);

}  // namespace driver

#endif  // TESTS_DRIVER_DRIVER_LOSSES_H_
