// Shared device helpers of the vimure_b200 kernels (sm_100a).
#pragma once
#include <cuda_runtime.h>
#include <math.h>
#include <stdint.h>

#include "vimure_b200.h"

#define VM_LOG2E 1.4426950408889634074
// fp64 exp(x) rounds to 0 below this: a row whose every log-weight is below it stays all-zero in the
// reference (model.py:807-811 normalises only where the sum is > 0, quirk Q3)
#define VM_DEAD_LN (-745.13321910194122)
#define VM_DEAD_LOG2 ((float)(VM_DEAD_LN * VM_LOG2E))
#define VM_CLAMP_LOG2 120.0f

#define VM_DENSE_THREADS 256

// per-TU function table (see vm_kernels.cu / vm_api.cu)
struct vm_tu_api {
  int (*materialize_prior)(const vm_ctx*, void*);
  int (*refresh_cache)(const vm_ctx*, void*);
  int (*init_stats)(const vm_ctx*, void*);
  int (*phase_gamma)(const vm_ctx*, void*);
  int (*phase_phi)(const vm_ctx*, void*);
  int (*phase_rho)(const vm_ctx*, int, void*);
  int (*dense_only)(const vm_ctx*, int, void*);
  int (*phase_finish)(const vm_ctx*, int, void*);
  int (*iteration)(const vm_ctx*, int, void*);
  int (*run)(const vm_ctx*, int, int, int, void*);
  int (*infer)(const vm_ctx*, int, double, uint8_t*, void*);
  int (*materialize_rows)(const vm_ctx*, int64_t, int64_t, float*, void*);
};

// Column tile of the dense kernels: TW = 128*NCH columns; NCH is K-dependent so that the per-lane column accumulators
// (NCH*4*(K-1) registers) stay in registers.
#ifndef VM_NCH2
#define VM_NCH2 4
#endif
template <int K>
struct DenseCfg {
  static constexpr int NCH = (K <= 2) ? VM_NCH2 : (K == 3) ? 4 : (K <= 5) ? 2 : 1;
  static constexpr int TW = 128 * NCH;
};
static inline int64_t vm_dense_tile_w_host(int64_t K) {
  if (K < 2 || K > VM_MAX_K) return VM_EINVAL;
  return K <= 2 ? DenseCfg<2>::TW : K == 3 ? DenseCfg<3>::TW : K <= 5 ? DenseCfg<4>::TW : DenseCfg<6>::TW;
}
// fixed-point scale of the integer-atomic per-reporter accumulators: 2^42, i.e. |sum| < 2^21 = 2.1e6 fits an int64 and the
// resolution is 2.3e-13.  A reporter of an ego mask has at most 2N special ties, each contributing less than 1 in
// magnitude, and no slab with N > 4.2e5 fits eight 180 GB GPUs (K = 2, L = 1): the sum cannot overflow at any size the
// path can run.  (Round 1 used 2^44, which a hub with more than 5.2e5 special ties would have overflowed silently.)
#define VM_FIX_SCALE 4398046511104.0
#define VM_FIX_INV (1.0 / 4398046511104.0)

// ------------------------------------------------------------------ special functions (fp64)
// digamma: recurrence up to x >= 10, then the asymptotic series (truncation error < 1e-16 there).
// Replaces scipy.special.psi used at model.py:596, 604-605, 676-677, 684, 911-912, 940-942, 1302.
__device__ __forceinline__ double vm_digamma(double x) {
  double r = 0.0;
  while (x < 10.0) {
    r -= 1.0 / x;
    x += 1.0;
  }
  const double f = 1.0 / (x * x);
  const double t =
      f * (-1.0 / 12.0 +
           f * (1.0 / 120.0 +
                f * (-1.0 / 252.0 +
                     f * (1.0 / 240.0 + f * (-1.0 / 132.0 + f * (691.0 / 32760.0 + f * (-1.0 / 12.0)))))));
  return r + log(x) - 0.5 / x + t;
}

// _gamma_elbo_term, model.py:1300-1303
__device__ __forceinline__ double vm_gamma_elbo_term(double pa, double pb, double qa, double qb) {
  return lgamma(qa) - pa * log(qb) + (pa - qa) * vm_digamma(qa) + qa * (1.0 - pb / qb);
}

// ------------------------------------------------------------------ deterministic reductions
__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_down_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_down_sync(0xffffffffu, v, o);
  return v;
}

__device__ __forceinline__ double warp_max(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmax(v, __shfl_down_sync(0xffffffffu, v, o));
  return v;
}
template <int NT>
__device__ __forceinline__ double block_max(double v, double* sm) {
  v = warp_max(v);
  const int w = threadIdx.x >> 5, lane = threadIdx.x & 31;
  __syncthreads();
  if (lane == 0) sm[w] = v;
  __syncthreads();
  if (w == 0) {
    v = (lane < NT / 32) ? sm[lane] : -1e300;
    v = warp_max(v);
  }
  return v;
}

// Sum over the block in a fixed order; result valid in thread 0. `sm` holds >= NT/32 doubles.
template <int NT>
__device__ __forceinline__ double block_sum(double v, double* sm) {
  v = warp_sum(v);
  const int w = threadIdx.x >> 5, lane = threadIdx.x & 31;
  __syncthreads();
  if (lane == 0) sm[w] = v;
  __syncthreads();
  if (w == 0) {
    v = (lane < NT / 32) ? sm[lane] : 0.0;
    v = warp_sum(v);
  }
  return v;
}

// ------------------------------------------------------------------ fast fp32 primitives
__device__ __forceinline__ float vm_ex2(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
__device__ __forceinline__ float vm_rcp(float x) {
  float y;
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}

// fp64 reciprocal (IEEE round-to-nearest; cheaper than a full division, no numerator scaling).  NOTE: a hand-rolled
// `rcp.approx.ftz.f64` + Newton version was tried and miscompiled (register-pair clobber) with nvcc 12.9 -- keep this.
__device__ __forceinline__ double vm_rcp64(double a) { return __drcp_rn(a); }

// ------------------------------------------------------------------ the per-tie closed form
// Posterior of a tie that carries no X entry (one-hot prior [1,0,..], model.py:536-556):
//   rho_k  proportional to  (pr_k+EPS) * exp(-S * E[lambda_k]),   S = sum of E[theta_m] over the tie's reporters
// (model.py:800-811 with an empty `_sp_uttkrp_rho` contribution).  `a[k]`, k>=1, is the log2-odds against k=0,
// a[0] the log2 weight of k=0 itself (only needed for the dead-row check).  fp32; the same function is used by
// the dense kernel and by the special-tie kernel (which subtracts it again), so the two agree bit for bit.
template <int K>
__device__ __forceinline__ void vm_formula_rho(const float* a, bool may_dead, float* out, float& epsr, bool& dead) {
  float r[K];
  float s = 0.f;
#pragma unroll
  for (int k = 1; k < K; ++k) {
    r[k] = vm_ex2(fminf(a[k], VM_CLAMP_LOG2));
    s = __fadd_rn(s, r[k]);
  }
  epsr = s;
  const float inv = vm_rcp(__fadd_rn(1.f, s));
  out[0] = inv;
#pragma unroll
  for (int k = 1; k < K; ++k) out[k] = __fmul_rn(r[k], inv);
  dead = false;
  if (may_dead) {
    float mx = 0.f;
#pragma unroll
    for (int k = 1; k < K; ++k) mx = fmaxf(mx, a[k]);
    if (__fadd_rn(a[0], mx) < VM_DEAD_LOG2) {
      dead = true;
#pragma unroll
      for (int k = 0; k < K; ++k) out[k] = 0.f;
    }
  }
}

// log1p for fp32: series below 0.05 (exact to ~1e-10 relative), MUFU-based above
__device__ __forceinline__ float vm_log1p_fast(float x) {
  if (fabsf(x) < 4e-4f) return x * (1.f - 0.5f * x);  // (the usual case: x ~ EPS; truncation x^2/3 < 6e-8 relative)
  if (fabsf(x) < 0.05f) {
    const float t = -0.16666667f;
    return x * (1.f + x * (-0.5f + x * (0.33333334f + x * (-0.25f + x * (0.2f + x * t)))));
  }
  return __logf(1.f + x);
}

// categorical ELBO term of such a tie: sum_k rho_k (log(pr_k+EPS) - log(rho_k+EPS)), model.py:1306-1313,
// written so that the ~1e-12 contributions survive fp32 (log(rho_0+EPS) = log1p(EPS*s) - log1p(s-1)).
template <int K>
__device__ __forceinline__ float vm_formula_cat(const float* out, float epsr, bool dead, float lp0, float lpk,
                                                float eps) {
  if (dead) return 0.f;
  const float s = __fadd_rn(1.f, epsr);
  float t = __fmul_rn(out[0], __fsub_rn(lp0, __fsub_rn(vm_log1p_fast(__fmul_rn(eps, s)), vm_log1p_fast(epsr))));
#pragma unroll
  for (int k = 1; k < K; ++k) t = __fadd_rn(t, __fmul_rn(out[k], __fsub_rn(lpk, __logf(__fadd_rn(out[k], eps)))));
  return t;
}

// ------------------------------------------------------------------ Poisson allocation (fp64)
// `_update_cache`, model.py:676-696: dz1_k = x z1_k/(z1_k+z2), dz2_k = x z2/(z1_k+z2), with the
// zero-denominator rule of model.py:692 (Q5); mutuality=False: dz1 = x, dz2 = 0 (model.py:679-681).
template <int K>
__device__ __forceinline__ void vm_alloc(bool mut, double x, double xT, double Gth, const double* Gl, double Gnu,
                                         double* dz1, double* dz2) {
  if (!mut) {
#pragma unroll
    for (int k = 0; k < K; ++k) {
      dz1[k] = x;
      dz2[k] = 0.0;
    }
    return;
  }
  const double z2 = Gnu * xT;
#pragma unroll
  for (int k = 0; k < K; ++k) {
    const double z1 = Gth * Gl[k];
    const double den = z1 + z2;
    const double xi = (den == 0.0) ? 0.0 : x * vm_rcp64(den);  // den == 0 => z1 == z2 == 0 (model.py:692)
    dz1[k] = xi * z1;
    dz2[k] = xi * z2;
  }
}

// layout of the per-layer constants block
#define VM_LC_STRIDE(K) (3 * (K) + 5)
#define VM_LC_C(k) (k)                 // c_k: log2-odds intercept (k>=1), log2 weight of k=0 (k=0)
#define VM_LC_D(K, k) ((K) + (k))      // d_k: slope in S
#define VM_LC_SALL(K) (2 * (K))        // sum_m E[theta_lm]
#define VM_LC_LP0(K) (2 * (K) + 1)     // log(1+EPS)
#define VM_LC_LPK(K) (2 * (K) + 2)     // log(EPS)
#define VM_LC_DEAD(K) (2 * (K) + 3)    // != 0: some closed-form row of this layer may underflow completely
#define VM_LC_SIMPLE(K) (2 * (K) + 4)  // != 0: the fp32 kernels (k_dense_sc / k_all32) evaluate the special ties of this layer
#define VM_LC_G(K, k) (2 * (K) + 5 + (k))  // (E[log lambda_k] - E[log lambda_0]) log2e
// fixed-point scale of fixP (sums of rho_k X over the simple ties of a layer: up to ~1e7)
#define VM_FIXP_SCALE 1073741824.0
