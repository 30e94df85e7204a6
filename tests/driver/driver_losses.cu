// The SoftLOne, Arctan, Tolerant and Tukey losses (loss kinds 8-11, see driver_losses.h) on
// SnavelyReprojectionError<2, 9, 3>, and SoftLOne on RelativePoseError<6, 7, 7>; the scaled and
// composed kinds 12-14 are in driver_losses2.cu.  Translation units of their own, so that these
// instantiations compile in parallel with the others and add no variant to driver_bal.cu.
// Also the C entry points that add residual blocks with these losses to a driver problem
// (drv_add_residual_blocks) and evaluate every loss object on the host (drv_loss_evaluate).
#include <string>

#include "driver_losses.h"
#include "relative_pose_error.h"
#include "snavely_reprojection_error.h"

namespace driver {
bool AddRunLosses(DriverProblem& dp, int type, int loss_kind, double a, double b, int n,
                  const int* pb, const double* fdata, bool bulk, bool* handled) {
  using namespace ceres;
  using examples::RelativePoseError;
  using examples::SnavelyReprojectionError;
  *handled = false;
  if (loss_kind < kSoftLOne) return false;
  *handled = true;
  auto snavely = [](const double* d) { return SnavelyReprojectionError(d[0], d[1]); };
  if (type == 0) {
    switch (loss_kind) {
      case kSoftLOne:
        AddRun<SnavelyReprojectionError, 2, 9, 3>(
            dp, dp.GetLoss<SoftLOneLossCUDA>(loss_kind, a, b, a), n, pb, fdata, 2, bulk, snavely);
        return true;
      case kArctan:
        AddRun<SnavelyReprojectionError, 2, 9, 3>(
            dp, dp.GetLoss<ArctanLossCUDA>(loss_kind, a, b, a), n, pb, fdata, 2, bulk, snavely);
        return true;
      case kTolerant:
        AddRun<SnavelyReprojectionError, 2, 9, 3>(
            dp, dp.GetLoss<TolerantLossCUDA>(loss_kind, a, b, a, b), n, pb, fdata, 2, bulk,
            snavely);
        return true;
      case kTukey:
        AddRun<SnavelyReprojectionError, 2, 9, 3>(
            dp, dp.GetLoss<TukeyLossCUDA>(loss_kind, a, b, a), n, pb, fdata, 2, bulk, snavely);
        return true;
    }
  }
  if (type == 4 && loss_kind == kSoftLOne) {
    AddRun<RelativePoseError, 6, 7, 7>(
        dp, dp.GetLoss<SoftLOneLossCUDA>(loss_kind, a, b, a), n, pb, fdata, 7, bulk,
        [](const double* d) { return RelativePoseError(d); });
    return true;
  }
  return AddRunScaledAndComposedLosses(dp, type, loss_kind, a, b, n, pb, fdata, bulk, handled);
}
}  // namespace driver

namespace {
using namespace ceres;
using HuberOfCauchy = ComposedLossCUDA<HuberLossCUDA, CauchyLossCUDA>;
using TolerantOfTukey = ComposedLossCUDA<TolerantLossCUDA, TukeyLossCUDA>;
static_assert(HuberOfCauchy::kNonPositiveCurvature, "both curvatures are <= 0");
static_assert(!TolerantOfTukey::kNonPositiveCurvature, "Tolerant has rho'' > 0");
static_assert(!driver::ComposedLoss::kNonPositiveCurvature, "ScaledLossCUDA declares none");

// Calls fn with the loss object of a kind (driver.h) and parameters a, b.  False for kinds
// without one.
template <typename Fn>
bool WithLoss(int kind, double a, double b, Fn fn) {
  switch (kind) {
    case driver::kTrivial: fn(TrivialLossCUDA()); return true;
    case driver::kHuber: fn(HuberLossCUDA(a)); return true;
    case driver::kCauchy: fn(CauchyLossCUDA(a)); return true;
    case driver::kSoftLOne: fn(SoftLOneLossCUDA(a)); return true;
    case driver::kArctan: fn(ArctanLossCUDA(a)); return true;
    case driver::kTolerant: fn(TolerantLossCUDA(a, b)); return true;
    case driver::kTukey: fn(TukeyLossCUDA(a)); return true;
    case driver::kScaledSoftLOne:
      fn(ScaledLossCUDA<SoftLOneLossCUDA>(SoftLOneLossCUDA(a), b));
      return true;
    case driver::kScaledTukey: fn(ScaledLossCUDA<TukeyLossCUDA>(TukeyLossCUDA(a), b)); return true;
    case driver::kComposed:
      fn(driver::ComposedLoss(ScaledLossCUDA<SoftLOneLossCUDA>(SoftLOneLossCUDA(a), b),
                              CauchyLossCUDA(a)));
      return true;
  }
  return false;
}

// rho(s) through HostLossThunk, as Problem::EvaluateResidualBlock evaluates a loss.
struct EvaluateOnHost {
  double s;
  double* rho;
  template <typename Loss>
  void operator()(const Loss& loss) const {
    ceres::internal::HostLossThunk<Loss>(&loss, s, rho);
  }
};
}  // namespace

extern "C" {

// Adds residual blocks to a problem made by drv_create (which adds the parameter blocks with
// their manifolds and constant flags; call it with num_rb = 0): the same arrays as drv_create's,
// and the number of parameter blocks and functor doubles of every cost type id.  Runs of one
// type and loss go to the new loss kinds' translation units first, then to the others.
// Returns 1 on success; otherwise drv_error tells why.
int drv_add_residual_blocks(void* h, int num_rb, const int* rb_type, const int* rb_pb,
                            const int* rb_loss_kind, const double* rb_loss_a,
                            const double* rb_loss_b, const double* fdata, int bulk,
                            int num_types, const int* type_blocks, const int* type_fdata) {
  auto* dp = static_cast<driver::DriverProblem*>(h);
  if (!dp->error.empty()) return 0;
  int64_t pb_cursor = 0, fd_cursor = 0;
  int i = 0;
  while (i < num_rb) {
    const int type = rb_type[i];
    if (type < 0 || type >= num_types) { dp->error = "unknown cost type"; return 0; }
    int j = i + 1;
    while (j < num_rb && rb_type[j] == type && rb_loss_kind[j] == rb_loss_kind[i] &&
           rb_loss_a[j] == rb_loss_a[i] && rb_loss_b[j] == rb_loss_b[i])
      ++j;
    const int n = j - i;
    const int* pb = rb_pb + pb_cursor;
    const double* fd = fdata + fd_cursor;
    const int kind = rb_loss_kind[i];
    const double a = rb_loss_a[i], b = rb_loss_b[i];
    bool handled = false, ok = false;
    ok = driver::AddRunLosses(*dp, type, kind, a, b, n, pb, fd, bulk != 0, &handled);
    if (!handled) ok = driver::AddRunBal(*dp, type, kind, a, b, n, pb, fd, bulk != 0, &handled);
    if (!handled) ok = driver::AddRunPose(*dp, type, kind, a, b, n, pb, fd, bulk != 0, &handled);
    if (!handled) ok = driver::AddRunTests(*dp, type, kind, a, b, n, pb, fd, bulk != 0, &handled);
    if (!handled || !ok) {
      dp->error = "cost type / loss combination not instantiated in the test driver";
      return 0;
    }
    pb_cursor += static_cast<int64_t>(n) * type_blocks[type];
    fd_cursor += static_cast<int64_t>(n) * type_fdata[type];
    i = j;
  }
  return 1;
}

// rho(s) of the loss object of a kind, evaluated on the host.  Returns 0 for a kind without one.
int drv_loss_evaluate(int kind, double a, double b, double s, double* rho) {
  return WithLoss(kind, a, b, EvaluateOnHost{s, rho}) ? 1 : 0;
}

// Host evaluation of two compositions no loss kind names: which = 0: Huber(a) of Cauchy(b);
// 1: Tolerant(a, b) of Tukey(a).  Returns 0 for another `which`.
int drv_composed_loss_evaluate(int which, double a, double b, double s, double* rho) {
  if (which == 0) {
    const HuberOfCauchy loss{HuberLossCUDA(a), CauchyLossCUDA(b)};
    ceres::internal::HostLossThunk<HuberOfCauchy>(&loss, s, rho);
    return 1;
  }
  if (which == 1) {
    const TolerantOfTukey loss{TolerantLossCUDA(a, b), TukeyLossCUDA(a)};
    ceres::internal::HostLossThunk<TolerantOfTukey>(&loss, s, rho);
    return 1;
  }
  return 0;
}

}  // extern "C"
