// Binary traits (logistic mixed model, PQL) and the saddlepoint-calibrated score test.  The reference has no
// counterpart.
//
// slmm_glmm_working: the elementwise step between two PQL iterations, fused: the BLUP identity for eta, the clamped
// logistic mean, the weight and the new working vector, written in place into the session's phenotype and into the
// value array of the diagonal component W^-1.
//
// slmm_assoc_spa: the saddlepoint p-value (SAIGE's Get_Saddle_Prob without its sparse split, Lugannani-Rice tail) of
// a block of flagged variants, one CTA per variant.  Every sum over the n individuals is taken by a fixed thread-to-row
// map and a fixed tree, with no atomics, so a variant's p-value has the same bits whatever block it is computed in.
#include "common.h"

#include <math_constants.h>

namespace slmm {

constexpr double GLMM_MU_EPS = 2.220446049250313e-16;   // mu is clamped to [eps, 1 - eps], as R's binomial()
constexpr int SPA_THREADS = 512;
constexpr int SPA_MAXC = 31;          // covariates (c x c inverse staged in shared memory)
constexpr int SPA_MAX_DOUBLINGS = 64; // bracket doublings before a variant falls back to the normal p
constexpr int SPA_MAX_STEPS = 200;    // safeguarded Newton steps per side (bisection alone would need < 110)
constexpr double SPA_TOL = 1e-10;     // relative Newton step at which the root is accepted
constexpr double SPA_MIN_W = 1e-3;    // |w| below this is the 0/0 point of the Lugannani-Rice formula

__global__ void glmm_working_kernel(double* __restrict__ yt, const double* __restrict__ vir, double* __restrict__ d,
                                    const double* __restrict__ y, int64_t n, double* __restrict__ eta_out,
                                    double* __restrict__ mu_out, int* __restrict__ flag) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const double yi = y[i];
  if (!(yi == 0.0 || yi == 1.0)) *flag = 1;
  const double eta = yt[i] - d[i] * vir[i];
  double mu = 1.0 / (1.0 + exp(-eta));
  mu = fmin(fmax(mu, GLMM_MU_EPS), 1.0 - GLMM_MU_EPS);
  const double w = mu * (1.0 - mu);
  yt[i] = eta + (yi - mu) / w;
  d[i] = 1.0 / w;
  eta_out[i] = eta;
  mu_out[i] = mu;
}

// Sum of three per-thread values over the CTA: shuffles within the warp, then warp 0 over the warp partials, in a
// fixed order.  Every thread returns the totals.
__device__ __forceinline__ void spa_sum3(double& a, double& b, double& c, double (*red)[SPA_THREADS / 32]) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    a += __shfl_down_sync(0xffffffffu, a, o);
    b += __shfl_down_sync(0xffffffffu, b, o);
    c += __shfl_down_sync(0xffffffffu, c, o);
  }
  __syncthreads();                     // the previous sum's totals have been read
  if (lane == 0) { red[0][warp] = a; red[1][warp] = b; red[2][warp] = c; }
  __syncthreads();
  if (warp == 0) {
    a = lane < SPA_THREADS / 32 ? red[0][lane] : 0.0;
    b = lane < SPA_THREADS / 32 ? red[1][lane] : 0.0;
    c = lane < SPA_THREADS / 32 ? red[2][lane] : 0.0;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      a += __shfl_down_sync(0xffffffffu, a, o);
      b += __shfl_down_sync(0xffffffffu, b, o);
      c += __shfl_down_sync(0xffffffffu, c, o);
    }
    if (lane == 0) { red[0][0] = a; red[1][0] = b; red[2][0] = c; }
  }
  __syncthreads();
  a = red[0][0];
  b = red[1][0];
  c = red[2][0];
}

// K(t), K'(t), K''(t) of S = sum_i g_i (Y_i - mu_i) with independent Y_i ~ Bernoulli(mu_i).  With a = g t, b = -|a|,
// E = expm1(b) and m = mu (a < 0) or 1 - mu (a >= 0), every term is free of overflow and of cancellation:
//   log(1 - mu + mu e^a) - a mu = log1p(m E) - b m,
//   g (p - mu) = -sign(a) g mu (1 - mu) E / (1 + m E),       p = mu e^a / (1 - mu + mu e^a),
//   g^2 p (1 - p) = g^2 mu (1 - mu) (1 + E) / (1 + m E)^2.
__device__ __noinline__ void spa_cgf(const double* __restrict__ g, const double* __restrict__ mu,
                                        const double* __restrict__ w, int64_t n, double t, double& K, double& K1,
                                        double& K2, double (*red)[SPA_THREADS / 32]) {
  double s0 = 0.0, s1 = 0.0, s2 = 0.0;
  for (int64_t i = threadIdx.x; i < n; i += SPA_THREADS) {
    const double gi = g[i], mi = mu[i], wi = w[i];
    const double a = gi * t;
    const double b = -fabs(a);
    const double E = expm1(b);
    const double m = a < 0.0 ? mi : 1.0 - mi;
    const double mE = m * E;
    const double r = 1.0 / (1.0 + mE);
    s0 += log1p(mE) - b * m;
    const double wr = wi * r;
    s1 = fma(a < 0.0 ? gi : -gi, wr * E, s1);
    s2 = fma(gi * gi, wr * r * (1.0 + E), s2);
  }
  spa_sum3(s0, s1, s2, red);
  K = s0;
  K1 = s1;
  K2 = s2;
}

// One CTA per flagged variant j of the block:
//   h = Minv proj[:, j] with Minv = (C'WC)^-1 and proj = (WC)' x~ (slmm_assoc_genotypes with P = WC);
//   g~ = x~ - C h, written to gt[j * n ...]; Var* = sum g~^2 w = K''(0); q = U sqrt(Var* / Var(U));
//   per side s = +1, -1: the root of K'(zeta) = s |q| by Newton steps safeguarded by a bracket that starts at [0, t1]
//   (t1 the Newton step from 0) and doubles until it holds the root; then the Lugannani-Rice tail of that side.
// status: 1 = p is the saddlepoint p-value, -1 = no root in range, not bracketed, or |w| < 1e-3 on a side (p NaN).
// iters: cumulant-generating-function passes over the n individuals, both sides.
__global__ void __launch_bounds__(SPA_THREADS) assoc_spa_kernel(
    const double* __restrict__ X, int64_t n, int b, const double* __restrict__ proj, int c,
    const double* __restrict__ Minv, const double* __restrict__ C, const double* __restrict__ mu,
    const double* __restrict__ w, const double* __restrict__ score, const double* __restrict__ var,
    double* __restrict__ gt, double* __restrict__ p_out, int* __restrict__ status_out, int* __restrict__ iters_out) {
  __shared__ double h[SPA_MAXC];
  __shared__ double red[3][SPA_THREADS / 32];
  const int j = blockIdx.x;
  if (threadIdx.x < c) {
    double s = 0.0;
    for (int l = 0; l < c; l++) s = fma(Minv[threadIdx.x * c + l], proj[(int64_t)l * b + j], s);
    h[threadIdx.x] = s;
  }
  __syncthreads();
  double* g = gt + (int64_t)j * n;
  double v2 = 0.0, lim_hi = 0.0, lim_lo = 0.0;
  for (int64_t i = threadIdx.x; i < n; i += SPA_THREADS) {
    double gi = X[i * b + j];
    const double* ci = C + i * c;
    for (int k = 0; k < c; k++) gi = fma(-ci[k], h[k], gi);
    g[i] = gi;
    const double mi = mu[i];
    v2 = fma(gi * gi, w[i], v2);
    lim_hi = fma(gi, (gi > 0.0 ? 1.0 : 0.0) - mi, lim_hi);     // K'(+inf)
    lim_lo = fma(gi, (gi < 0.0 ? 1.0 : 0.0) - mi, lim_lo);     // K'(-inf)
  }
  spa_sum3(v2, lim_hi, lim_lo, red);
  __syncthreads();                     // g is read by other threads from here on
  const double q = fabs(score[j] * sqrt(v2 / var[j]));
  bool ok = v2 > 0.0 && isfinite(q);
  int iters = 0;
  double total = 0.0;
  for (int side = 1; side >= -1 && ok; side -= 2) {
    const double target = side * q;
    if (!(lim_lo < target && target < lim_hi)) { ok = false; break; }
    double K, K1, K2;
    double a = 0.0, t = target / v2;     // a: residual K' - target of sign -side
    spa_cgf(g, mu, w, n, t, K, K1, K2, red);
    iters++;
    int dbl = 0;
    while (side * (K1 - target) < 0.0) {
      if (++dbl > SPA_MAX_DOUBLINGS) { ok = false; break; }
      a = t;
      t *= 2.0;
      spa_cgf(g, mu, w, n, t, K, K1, K2, red);
      iters++;
    }
    if (!ok) break;
    double bnd = t;                      // residual of sign side (or 0)
    for (int step = 0;; step++) {
      const double res = K1 - target;
      if (side * res < 0.0) a = t; else bnd = t;
      const double dt = -res / K2;
      if (res == 0.0 || fabs(dt) <= SPA_TOL * fabs(t)) break;
      if (step >= SPA_MAX_STEPS || !isfinite(K1)) { ok = false; break; }
      double tn = t + dt;
      if (!(tn > fmin(a, bnd) && tn < fmax(a, bnd))) tn = 0.5 * (a + bnd);
      t = tn;
      spa_cgf(g, mu, w, n, t, K, K1, K2, red);
      iters++;
    }
    if (!ok) break;
    const double wlr = side * sqrt(fmax(2.0 * (t * target - K), 0.0));
    const double vlr = t * sqrt(K2);
    if (!(fabs(wlr) >= SPA_MIN_W)) { ok = false; break; }
    const double corr = exp(-0.5 * wlr * wlr) * (0.5 * M_2_SQRTPI * M_SQRT1_2) * (1.0 / vlr - 1.0 / wlr);
    total += side > 0 ? 0.5 * erfc(wlr * M_SQRT1_2) + corr : 0.5 * erfc(-wlr * M_SQRT1_2) - corr;
  }
  if (ok && !(isfinite(total) && total >= 0.0)) ok = false;
  if (threadIdx.x == 0) {
    p_out[j] = ok ? fmin(total, 1.0) : CUDART_NAN;
    status_out[j] = ok ? 1 : -1;
    iters_out[j] = iters;
  }
}

namespace {
struct GlmmFlag {
  DevPtr<int> buf;
  int device = -1;
  int* get() {
    int dev = 0;
    CUDA_OK(cudaGetDevice(&dev));
    if (dev != device) {
      buf.reset();
      buf = dev_alloc<int>(1);
      device = dev;
    }
    return buf.get();
  }
};
GlmmFlag g_glmm_flag;
}  // namespace

}  // namespace slmm

using namespace slmm;

extern "C" {

int slmm_glmm_working(double* d_ytilde, const double* d_vir, double* d_dvals, const double* d_y, int64_t n,
                      double* d_eta, double* d_mu) {
  SLMM_TRY
  if (!d_ytilde || !d_vir || !d_dvals || !d_y || !d_eta || !d_mu || n <= 0) throw std::invalid_argument("bad arguments");
  int* flag = g_glmm_flag.get();
  CUDA_OK(cudaMemsetAsync(flag, 0, sizeof(int), 0));
  glmm_working_kernel<<<(unsigned)((n + 255) / 256), 256>>>(d_ytilde, d_vir, d_dvals, d_y, n, d_eta, d_mu, flag);
  g_launch_count += 1;
  CUDA_OK(cudaGetLastError());
  int bad = 0;
  CUDA_OK(cudaMemcpy(&bad, flag, sizeof(int), cudaMemcpyDeviceToHost));
  if (bad) throw std::invalid_argument("slmm_glmm_working: y entries must be 0 or 1");
  return SLMM_OK;
  SLMM_CATCH
}

int slmm_assoc_spa(const double* d_X, int64_t n, int32_t b, const double* d_proj, int32_t c, const double* d_Minv,
                   const double* d_C, const double* d_mu, const double* d_w, const double* d_score,
                   const double* d_var, double* d_work, double* d_p, int32_t* d_status, int32_t* d_iters) {
  SLMM_TRY
  if (!d_X || !d_proj || !d_Minv || !d_C || !d_mu || !d_w || !d_score || !d_var || !d_work || !d_p || !d_status ||
      !d_iters || n <= 0 || b <= 0)
    throw std::invalid_argument("bad arguments");
  if (c < 1 || c > SPA_MAXC) throw std::invalid_argument("slmm_assoc_spa: need 1 <= c <= 31 covariates");
  assoc_spa_kernel<<<b, SPA_THREADS>>>(d_X, n, b, d_proj, c, d_Minv, d_C, d_mu, d_w, d_score, d_var, d_work, d_p,
                                       d_status, d_iters);
  g_launch_count += 1;
  CUDA_OK(cudaGetLastError());
  return SLMM_OK;
  SLMM_CATCH
}

}  // extern "C"
