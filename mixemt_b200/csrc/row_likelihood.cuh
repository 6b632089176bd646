// The one rule that sends a row to log space, shared by the EM's log-space step
// (em_kernels.cuh: em_logspace_*) and the log-space redo of the log-likelihood (loglik.cu).
#pragma once

namespace mxb {

// A row whose mixture likelihood t = sum_j L_ij pi_j lies below kRowLikelihoodMin, or is NaN,
// cannot be carried in linear space.  The coefficient w / t overflows to +inf once
// t < w / DBL_MAX, which covers every subnormal t and, with large weights, normal t too; the
// column sums then hold inf * L and inf * 0 and every proportion becomes NaN.  Above 2^-960 the
// coefficient is at most w * 2^960 and a column sum at most W * 2^960 (L <= 1), finite for any
// total weight W < 2^63; subnormal products L_ij pi_j change t by at most H * 2^-1075 =
// H * 2^-115 of t, below an ulp for any H < 2^62.
constexpr double kRowLikelihoodMin = 0x1p-960;
__device__ __forceinline__ bool row_needs_logspace(double t) { return !(t >= kRowLikelihoodMin); }

}  // namespace mxb
