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
  int (*edges)(const vm_ctx*, const vm_edges_args*, int, void*);  // int: 0 = vm_edges_count, 1 = vm_edges_emit
  int (*rho_at)(const vm_ctx*, int64_t, int64_t, const int64_t*, float*, void*);
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

// ------------------------------------------------------------------ posterior sampling (model.py:1062-1096)
// Philox4x32-10 (Salmon et al. 2011), counter = (global tie id, block of 4 draws), key = seed: the stream of a tie does
// not depend on the launch geometry nor on how the ties are sharded over ranks.
__device__ __forceinline__ uint4 vm_philox4x32(uint4 ctr, uint2 key) {
#pragma unroll
  for (int r = 0; r < 10; ++r) {
    const uint32_t hi0 = __umulhi(0xD2511F53u, ctr.x), lo0 = 0xD2511F53u * ctr.x;
    const uint32_t hi1 = __umulhi(0xCD9E8D57u, ctr.z), lo1 = 0xCD9E8D57u * ctr.z;
    ctr = make_uint4(hi1 ^ ctr.y ^ key.x, lo1, hi0 ^ ctr.w ^ key.y, lo0);
    key.x += 0x9E3779B9u;
    key.y += 0xBB67AE85u;
  }
  return ctr;
}

// The label vm_sample gives the tie `gt` (global flat id) of posterior r[0..K): n_trials draws from Categorical(r) -> the
// category drawn most often (first one on a draw), i.e. `multinomial(n, rho).argmax(-1)` of model.py:1086-1088.  A draw
// that exceeds the cumulative sum (rounding, or an all-zero row) falls into the LAST category, as numpy's multinomial
// assigns the remainder.  Shared by the dense (k_sample) and the sparse (k_edges) consumers.
__device__ __forceinline__ int vm_sample_label(const float* r, int K, int64_t n_trials, uint64_t gt, uint2 key) {
  float p[VM_MAX_K];
  int cnt[VM_MAX_K];
  float sum = 0.f;
  for (int k = 0; k < K; ++k) {
    p[k] = r[k];
    sum += p[k];
    cnt[k] = 0;
  }
  // Every draw lands in category 0 when the fp32 sum equals p[0] > 0: the first cumulative sum is p[0] = sum, and the
  // uniform below is v*sum with v = ((x>>9)+0.5)*2^-23 <= 1-2^-24 (exact), so v*sum <= sum - sum*2^-24.  For sum in
  // [2^e, 2^(e+1)) that is at least ulp(sum)/2 below sum, strictly unless sum = 2^e, where sum - 2^(e-24) is itself
  // representable: fl(v*sum) < sum = cum in every case, and the draw stops at k = 0.  (sum = 0, a dead tie, goes to the
  // last category below; a NaN fails the test.)  Most ties of a sparse network: no Philox evaluation needed.
  if (sum == p[0] && sum > 0.f) return 0;
  for (int64_t d0 = 0; d0 < n_trials; d0 += 4) {
    const uint64_t blk = (uint64_t)(d0 >> 2);
    const uint4 x = vm_philox4x32(make_uint4((uint32_t)gt, (uint32_t)(gt >> 32), (uint32_t)blk, (uint32_t)(blk >> 32)), key);
    const uint32_t xs[4] = {x.x, x.y, x.z, x.w};
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      if (d0 + q >= n_trials) break;
      // uniform strictly inside (0, sum): 23 random bits + 1/2 is exact in fp32 (24 bits would round up to 1.0)
      const float u = ((float)(xs[q] >> 9) + 0.5f) * (1.0f / 8388608.0f) * sum;
      float cum = 0.f;
      int k = 0;
      for (; k < K - 1; ++k) {
        cum += p[k];
        if (u < cum) break;
      }
      cnt[k] += 1;
    }
  }
  int best = 0;
  for (int k = 1; k < K; ++k)
    if (cnt[k] > cnt[best]) best = k;
  return best;
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
