// (a translation unit of its own: see driver_losses.cu)  The scaled and composed loss kinds
// 12-14 on SnavelyReprojectionError<2, 9, 3>.
#include "driver_losses.h"
#include "snavely_reprojection_error.h"

namespace driver {
bool AddRunScaledAndComposedLosses(DriverProblem& dp, int type, int loss_kind, double a, double b,
                                   int n, const int* pb, const double* fdata, bool bulk,
                                   bool* handled) {
  using namespace ceres;
  using examples::SnavelyReprojectionError;
  *handled = true;
  if (type != 0) return false;
  auto snavely = [](const double* d) { return SnavelyReprojectionError(d[0], d[1]); };
  switch (loss_kind) {
    case kScaledSoftLOne:
      AddRun<SnavelyReprojectionError, 2, 9, 3>(
          dp, dp.GetLoss<ScaledLossCUDA<SoftLOneLossCUDA>>(loss_kind, a, b, SoftLOneLossCUDA(a), b),
          n, pb, fdata, 2, bulk, snavely);
      return true;
    case kScaledTukey:
      AddRun<SnavelyReprojectionError, 2, 9, 3>(
          dp, dp.GetLoss<ScaledLossCUDA<TukeyLossCUDA>>(loss_kind, a, b, TukeyLossCUDA(a), b), n,
          pb, fdata, 2, bulk, snavely);
      return true;
    case kComposed:
      AddRun<SnavelyReprojectionError, 2, 9, 3>(
          dp,
          dp.GetLoss<ComposedLoss>(loss_kind, a, b,
                                   ScaledLossCUDA<SoftLOneLossCUDA>(SoftLOneLossCUDA(a), b),
                                   CauchyLossCUDA(a)),
          n, pb, fdata, 2, bulk, snavely);
      return true;
  }
  return false;
}
}  // namespace driver
