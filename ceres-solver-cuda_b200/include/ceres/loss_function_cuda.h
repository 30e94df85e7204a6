// Loss functions evaluated on the device.
//
// Same classes and Evaluate(s, rho[3]) contract as the reference's
// include/ceres/loss_function_cuda.h:52-149 (which mirror the CPU losses of
// internal/ceres/loss_function.cc:44-82): rho[0] = rho(s), rho[1] = rho'(s),
// rho[2] = rho''(s) for s = ||r||^2.  Beyond the reference, the SoftLOne, Arctan, Tolerant,
// Tukey and composed losses of loss_function.cc.  No virtual Evaluate: the kernel is
// instantiated per loss type.  LossFunctionCUDABase exists only so ProblemCUDA can
// own heterogeneous loss objects (problem_cuda.h:455-460).
#ifndef CERES_B200_LOSS_FUNCTION_CUDA_H_
#define CERES_B200_LOSS_FUNCTION_CUDA_H_

#include <cmath>
#include <limits>
#include <type_traits>

#include "ceres/internal/cuda_defs.h"

namespace ceres {

class LossFunctionCUDABase {
 public:
  virtual ~LossFunctionCUDABase() {}
};

namespace loss_internal {
// rho <- (value, first derivative, second derivative)
HOST_DEVICE inline void Set(double rho[3], double value, double d1, double d2) {
  rho[0] = value;
  rho[1] = d1;
  rho[2] = d2;
}
// Square root and its reciprocal of a positive finite x, for device code: one MUFU.RSQ64H with
// its Newton step (rsqrt) and one correction step for the root, instead of the library's
// sqrt followed by a division (each a 20-instruction sequence with a slow-path call).  The
// root is within 1 ulp; anything else (0, negative, Inf, NaN) takes the library functions.
HOST_DEVICE inline void RootAndReciprocal(double x, double* root, double* inv_root) {
#ifdef __CUDA_ARCH__
  if (x > 0.0 && x < 1.7976931348623157e308) {
    const double r = rsqrt(x);
    const double y = x * r;
    *root = fma(fma(-y, y, x), 0.5 * r, y);
    *inv_root = r;
    return;
  }
#endif
  *root = sqrt(x);
  *inv_root = 1.0 / *root;
}
// max(x, numeric_limits<double>::min()): rho' is kept strictly positive
// (loss_function.cc:56,70).
HOST_DEVICE inline double AtLeastTiny(double x) {
  const double tiny = 2.2250738585072014e-308;
  return x > tiny ? x : tiny;
}
// True when L declares kNonPositiveCurvature = true.
template <typename L, typename = void>
struct DeclaresNonPositiveCurvature : std::false_type {};
template <typename L>
struct DeclaresNonPositiveCurvature<L, std::void_t<decltype(L::kNonPositiveCurvature)>>
    : std::integral_constant<bool, L::kNonPositiveCurvature> {};
}  // namespace loss_internal

// rho(s) = s
class TrivialLossCUDA : public LossFunctionCUDABase {
 public:
  // rho'' <= 0 everywhere: the evaluation kernel skips the Corrector's alpha branch
  // (corrector.cc:105-110 takes it only for rho'' > 0) and never needs rho[2].
  static constexpr bool kNonPositiveCurvature = true;
  HOST_DEVICE void Evaluate(double s, double rho[3]) const {
    loss_internal::Set(rho, s, 1.0, 0.0);
  }
};

// rho(s) = s for s <= a^2, 2 a sqrt(s) - a^2 beyond.
class HuberLossCUDA : public LossFunctionCUDABase {
 public:
  // rho'' <= 0 everywhere: the evaluation kernel skips the Corrector's alpha branch
  // (corrector.cc:105-110 takes it only for rho'' > 0) and never needs rho[2].
  static constexpr bool kNonPositiveCurvature = true;
  HOST_DEVICE explicit HuberLossCUDA(double a) : a_(a), b_(a * a) {}
  HOST_DEVICE void Evaluate(double s, double rho[3]) const {
    if (!(s > b_)) {  // inlier region (and NaN, as in the reference): the identity
      loss_internal::Set(rho, s, 1.0, 0.0);
      return;
    }
    double root, inv_root;
    loss_internal::RootAndReciprocal(s, &root, &inv_root);
#ifdef __CUDA_ARCH__
    const double slope = loss_internal::AtLeastTiny(a_ * inv_root);
#else
    // (host evaluation, e.g. Problem::EvaluateResidualBlock: the reference's expression)
    const double slope = loss_internal::AtLeastTiny(a_ / root);
#endif
    loss_internal::Set(rho, 2.0 * a_ * root - b_, slope, -slope / (2.0 * s));
  }

 private:
  double a_;
  double b_;
};

// rho(s) = a^2 log(1 + s / a^2)
class CauchyLossCUDA : public LossFunctionCUDABase {
 public:
  // rho'' <= 0 everywhere: the evaluation kernel skips the Corrector's alpha branch
  // (corrector.cc:105-110 takes it only for rho'' > 0) and never needs rho[2].
  static constexpr bool kNonPositiveCurvature = true;
  HOST_DEVICE explicit CauchyLossCUDA(double a) : b_(a * a), c_(1 / b_) {}
  HOST_DEVICE void Evaluate(double s, double rho[3]) const {
    const double one_plus = 1.0 + s * c_;
    const double reciprocal = 1.0 / one_plus;
    loss_internal::Set(rho, b_ * log(one_plus), loss_internal::AtLeastTiny(reciprocal),
                       -c_ * (reciprocal * reciprocal));
  }

 private:
  double b_;
  double c_;
};

// rho(s) = 2 a^2 (sqrt(1 + s / a^2) - 1), a smooth L1 (loss_function.cc SoftLOneLoss).
class SoftLOneLossCUDA : public LossFunctionCUDABase {
 public:
  // rho'' <= 0 everywhere: no Corrector alpha branch in the evaluation kernel.
  static constexpr bool kNonPositiveCurvature = true;
  HOST_DEVICE explicit SoftLOneLossCUDA(double a) : b_(a * a), c_(1 / b_) {}
  HOST_DEVICE void Evaluate(double s, double rho[3]) const {
    const double sum = 1.0 + s * c_;
    // (host: sqrt and 1 / sqrt as the reference writes them; device: one rsqrt, within 1 ulp)
    double root, inv_root;
    loss_internal::RootAndReciprocal(sum, &root, &inv_root);
    const double d1 = loss_internal::AtLeastTiny(inv_root);
    double d2 = -(c_ * d1) / (2.0 * sum);
#ifdef __CUDA_ARCH__
    // (<= 0 already, except NaN for a NaN s, which fails the block anyway): shown to the
    // compiler, so that the Jet-free kernel, which tests rho'' for the Corrector's alpha branch,
    // drops that branch; with it the kernel spilled at its 80-register bound
    d2 = fmin(d2, 0.0);
#endif
    loss_internal::Set(rho, 2.0 * b_ * (root - 1.0), d1, d2);
  }

 private:
  double b_;
  double c_;
};

// rho(s) = a atan(s / a) (loss_function.cc ArctanLoss).
class ArctanLossCUDA : public LossFunctionCUDABase {
 public:
  // rho'' <= 0 for s >= 0: no Corrector alpha branch in the evaluation kernel.
  static constexpr bool kNonPositiveCurvature = true;
  HOST_DEVICE explicit ArctanLossCUDA(double a) : a_(a), b_(1 / (a * a)) {}
  HOST_DEVICE void Evaluate(double s, double rho[3]) const {
    const double sum = 1 + s * s * b_;
    const double inv = 1 / sum;
    loss_internal::Set(rho, a_ * atan2(s, a_), loss_internal::AtLeastTiny(inv),
                       -2.0 * s * b_ * (inv * inv));
  }

 private:
  double a_;
  double b_;
};

// rho(s) = b log(1 + exp((s - a) / b)) - b log(1 + exp(-a / b)), a >= 0, b > 0
// (loss_function.cc TolerantLoss): close to 0 below a, close to s - a above.
class TolerantLossCUDA : public LossFunctionCUDABase {
 public:
  // rho'' > 0: the evaluation kernel takes the Corrector's alpha branch, so no
  // kNonPositiveCurvature.
  HOST_DEVICE TolerantLossCUDA(double a, double b)
      : a_(a), b_(b), c_(b * log(1.0 + exp(-a / b))) {}
  HOST_DEVICE void Evaluate(double s, double rho[3]) const {
    const double x = (s - a_) / b_;
    // Beyond ln(2^53) 1 + e^x rounds to e^x: the linear tail (and no overflow of exp).
    if (x > 36.7) {
      loss_internal::Set(rho, s - a_ - c_, 1.0, 0.0);
      return;
    }
    const double e = exp(x);
#ifdef __CUDA_ARCH__
    // cosh(x) from the exponential already in hand.  Written as e/2 + 0.5/e rather than
    // (e + 1/e)/2 so that it overflows where cosh does (x < -710.47, not already at
    // 1/e > DBL_MAX, x < -709.78): in between rho'' stays positive, as on the host.
    const double cosh_x = 0.5 * e + 0.5 / e;
#else
    const double cosh_x = cosh(x);
#endif
    loss_internal::Set(rho, b_ * log(1.0 + e) - c_, loss_internal::AtLeastTiny(e / (1.0 + e)),
                       0.5 / (b_ * (1.0 + cosh_x)));
  }

 private:
  double a_;
  double b_;
  double c_;
};

// rho(s) = a^2 / 6 (1 - (1 - s / a^2)^3) for s <= a^2, a^2 / 6 beyond (loss_function.cc
// TukeyLoss).  Redescending: rho' = 0 for the outliers, whose residuals and Jacobian rows the
// Corrector then sets to zero.
class TukeyLossCUDA : public LossFunctionCUDABase {
 public:
  // rho'' <= 0 everywhere: no Corrector alpha branch in the evaluation kernel.
  static constexpr bool kNonPositiveCurvature = true;
  HOST_DEVICE explicit TukeyLossCUDA(double a) : a_squared_(a * a) {}
  HOST_DEVICE void Evaluate(double s, double rho[3]) const {
    if (s <= a_squared_) {
      const double value = 1.0 - s / a_squared_;
      const double value_sq = value * value;
      loss_internal::Set(rho, a_squared_ / 6.0 * (1.0 - value_sq * value), 0.5 * value_sq,
                         -1.0 / a_squared_ * value);
      return;
    }
    loss_internal::Set(rho, a_squared_ / 6.0, 0.0, 0.0);
  }

 private:
  double a_squared_;
};

// a * rho(s)
template <typename LossFunctionCUDA>
class ScaledLossCUDA : public LossFunctionCUDABase {
 public:
  HOST_DEVICE ScaledLossCUDA(const LossFunctionCUDA& rho, double a) : rho_(rho), a_(a) {}
  HOST_DEVICE void Evaluate(double s, double rho[3]) const {
    rho_.Evaluate(s, rho);
    loss_internal::Set(rho, rho[0] * a_, rho[1] * a_, rho[2] * a_);
  }

 private:
  LossFunctionCUDA rho_;
  double a_;
};

template <>
class ScaledLossCUDA<TrivialLossCUDA> : public LossFunctionCUDABase {
 public:
  HOST_DEVICE ScaledLossCUDA(const TrivialLossCUDA&, double a) : a_(a) {}
  HOST_DEVICE void Evaluate(double s, double rho[3]) const {
    loss_internal::Set(rho, a_ * s, a_, 0.0);
  }

 private:
  double a_;
};

// rho(s) = f(g(s)) (loss_function.cc ComposedLoss).  f and g are held by value, so a
// composition is one object the kernel copies like any other loss; past
// CB200_INLINE_LOSS_BYTES it is read from the type's loss table.
template <typename F, typename G>
class ComposedLossCUDA : public LossFunctionCUDABase {
 public:
  // f'' g'^2 + f' g'' <= 0 when both curvatures are (f' >= 0).
  static constexpr bool kNonPositiveCurvature =
      loss_internal::DeclaresNonPositiveCurvature<F>::value &&
      loss_internal::DeclaresNonPositiveCurvature<G>::value;
  HOST_DEVICE ComposedLossCUDA(const F& f, const G& g) : f_(f), g_(g) {}
  HOST_DEVICE void Evaluate(double s, double rho[3]) const {
    double rho_f[3], rho_g[3];
    g_.Evaluate(s, rho_g);
    f_.Evaluate(rho_g[0], rho_f);
    loss_internal::Set(rho, rho_f[0], rho_f[1] * rho_g[1],
                       rho_f[2] * rho_g[1] * rho_g[1] + rho_f[1] * rho_g[2]);
  }

 private:
  F f_;
  G g_;
};

}  // namespace ceres

#endif  // CERES_B200_LOSS_FUNCTION_CUDA_H_
