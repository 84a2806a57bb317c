// Rotation-vector helpers shared by the calibration-noise model and the rig bundle adjustment (fp64).  openmpl_b200/synth.py
// (so3_exp) and tests/rig_calibration_oracle.py restate them in numpy.
#pragma once

namespace mpl {

// Below theta^2 = kSo3TaylorTheta2 the three coefficients sin t / t, (1 - cos t) / t^2 and (t - sin t) / t^3 come from their
// Taylor series through t^8 (truncation < 1e-19 relative at t = 0.1), where the closed forms lose digits to cancellation.
constexpr double kSo3TaylorTheta2 = 1e-2;

__device__ __forceinline__ void so3_coeffs(double t2, double& a, double& b, double& c) {
  if (t2 < kSo3TaylorTheta2) {
    a = 1.0 - t2 / 6.0 * (1.0 - t2 / 20.0 * (1.0 - t2 / 42.0 * (1.0 - t2 / 72.0)));
    b = 0.5 * (1.0 - t2 / 12.0 * (1.0 - t2 / 30.0 * (1.0 - t2 / 56.0 * (1.0 - t2 / 90.0))));
    c = (1.0 - t2 / 20.0 * (1.0 - t2 / 42.0 * (1.0 - t2 / 72.0 * (1.0 - t2 / 110.0)))) / 6.0;
  } else {
    const double t = sqrt(t2), s = sin(t), co = cos(t);
    a = s / t;
    b = (1.0 - co) / t2;
    c = (t - s) / (t2 * t);
  }
}

// M = I + p [w]x + q [w]x^2, row-major; [w]x^2 = w w^T - |w|^2 I.
__device__ __forceinline__ void so3_poly(const double (&w)[3], double t2, double p, double q, double (&M)[9]) {
#pragma unroll
  for (int i = 0; i < 3; ++i)
#pragma unroll
    for (int k = 0; k < 3; ++k) M[3 * i + k] = (i == k ? 1.0 - q * t2 : 0.0) + q * w[i] * w[k];
  M[1] -= p * w[2];
  M[2] += p * w[1];
  M[3] += p * w[2];
  M[5] -= p * w[0];
  M[6] -= p * w[1];
  M[7] += p * w[0];
}

// Exp(w) (Rodrigues) and, when Jl != nullptr, the left Jacobian J_l(w) = I + (1 - cos t) / t^2 [w]x + (t - sin t) / t^3 [w]x^2.
__device__ __forceinline__ void so3_exp(const double (&w)[3], double (&E)[9]) {
  const double t2 = w[0] * w[0] + w[1] * w[1] + w[2] * w[2];
  double a, b, c;
  so3_coeffs(t2, a, b, c);
  so3_poly(w, t2, a, b, E);
}
__device__ __forceinline__ void so3_left_jacobian(const double (&w)[3], double (&Jl)[9]) {
  const double t2 = w[0] * w[0] + w[1] * w[1] + w[2] * w[2];
  double a, b, c;
  so3_coeffs(t2, a, b, c);
  so3_poly(w, t2, b, c, Jl);
}

// out = E R (3 x 3, row-major), sums in index order.
__device__ __forceinline__ void mat3_mul(const double (&E)[9], const double* R, double (&out)[9]) {
#pragma unroll
  for (int i = 0; i < 3; ++i)
#pragma unroll
    for (int k = 0; k < 3; ++k) out[3 * i + k] = E[3 * i] * R[k] + E[3 * i + 1] * R[3 + k] + E[3 * i + 2] * R[6 + k];
}

}  // namespace mpl
