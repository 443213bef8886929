// vimure_b200 -- hand-written sm_100a kernels of the CAVI hot path + the extern "C" launcher layer.
//
// What runs where (one CAVI iteration = reference `_update_CAVI`, model.py:623-660):
//   phase gamma : k_gamma_partial (reporter-sorted) | k_gamma_partial_ts (tie-sorted, few reporters) -> k_gamma_reduce  (red1)
//   phase phi   : k_gamma_finish -> k_phi_partial -> k_phi_reduce         (red2)
//   phase rho   : k_phi_finish -> k_tables
//                 -> special ties: k_special<K> (fp64; every special tie on ELBO iterations, the non-shortcut ones otherwise)
//                                  | k_all32<K> (all-reporter mask, fp32, entry-parallel)
//                 -> every tie:    k_dense_tma<K> (TMA bulk stores; the HBM-bound kernel), or k_dense_sc<K> (the same, also
//                                  evaluating the shortcut ties in fp32; ego mask, no ELBO), + k_dense<K> (partial tiles,
//                                  general masks, dead rows) on the aux stream, k_sums_stage1 / k_elbo_b next to them (and
//                                  next to k_dense_sc, the list-mode k_special) -> [k_patch_rest]
//                 -> k_col_reduce -> k_stats_* -> k_sums_reduce   (red3)
//   phase finish: [k_elbo_partial] -> k_finish
// All reductions are two-pass (block partials, then a fixed-order second pass) or integer atomics on fixed-point values:
// results are bit-reproducible run to run.  No floating-point atomics anywhere.
#include <stdio.h>
#include <stdlib.h>

#include "vm_common.cuh"

// This file is compiled once per translation unit (TU), each TU instantiating the kernels for a few values of K
// (vimure_b200/build.py generates `_gen/vm_tu_<id>.cu`, which defines VM_TU_ID and VM_DISPATCH_CASES and includes
// this file).  csrc/vm_api.cu holds the extern "C" entry points and routes to the TU that owns ctx->K.
#ifndef VM_TU_ID
#error "compile through vimure_b200/build.py (VM_TU_ID / VM_DISPATCH_CASES must be defined)"
#endif
#define VM_PASTE2(a, b) a##b
#define VM_PASTE(a, b) VM_PASTE2(a, b)
namespace VM_PASTE(vmtu, VM_TU_ID) {

// VM_DEBUG_SYNC=1 in the environment: synchronise after every launch and report the failing launch site
static bool vm_debug_sync() {
  static int v = -1;
  if (v < 0) {
    const char* e = getenv("VM_DEBUG_SYNC");
    v = (e && e[0] == '1') ? 1 : 0;
  }
  return v == 1;
}
#define VM_CHECK_LAUNCH()                                                                          \
  do {                                                                                             \
    cudaError_t e__ = cudaGetLastError();                                                          \
    if (e__ == cudaSuccess && vm_debug_sync()) e__ = cudaDeviceSynchronize();                      \
    if (e__ != cudaSuccess) {                                                                      \
      if (vm_debug_sync()) fprintf(stderr, "vimure_b200: launch before line %d failed: %s\n", __LINE__, cudaGetErrorString(e__)); \
      return (int)e__;                                                                             \
    }                                                                                              \
  } while (0)

// slots of the special-tie block partials, stored slot-major: part[slot * n_upart + block]
#define UP_NU 0
#define UP_CAT 1
#define UP_T2 2
#define UP_DELTA 3        // + k
#define UP_P0(K) (3 + (K))  // + k: rho_k * u_x0sum (E0 part of the next phi-shape sums)
#define UP_SLOTS(K) (3 + 2 * (K))

// fp32 posterior of one special tie (K consecutive floats, 4K-byte aligned for K = 2, 4)
template <int K>
__device__ __forceinline__ void vm_load_rho32(const float* p, float* r) {
  if (K == 2) {
    const float2 v = *reinterpret_cast<const float2*>(p);
    r[0] = v.x; r[1] = v.y;
  } else if (K == 4) {
    const float4 v = *reinterpret_cast<const float4*>(p);
    r[0] = v.x; r[1] = v.y; r[2] = v.z; r[3] = v.w;
  } else {
#pragma unroll
    for (int k = 0; k < K; ++k) r[k] = p[k];
  }
}

// =====================================================================================================
// phase gamma
// =====================================================================================================
// One warp per reporter chunk (<= 256 entries of one reporter (l,m), reporter-sorted copies => coalesced):
// sum_k rho_k * dz1_k per entry.  Replaces `_sp_uttkrp_theta` (model.py:851-859), whose python loop is 65% of the
// reference's CAVI time.
template <int K>
__global__ void __launch_bounds__(256) k_gamma_partial(const __grid_constant__ vm_ctx c, double* part) {
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int64_t chunk = (int64_t)blockIdx.x * 8 + warp;
  if (chunk >= c.n_gchunk) return;
  const int lm = c.g_chunk_lm[chunk];
  const int l = lm / (int)c.M;
  const bool mut = c.mutuality != 0;
  const double Gth = c.G_theta[lm];
  const double Gnu = c.nu[VM_NU_G];
  double Gl[K];
#pragma unroll
  for (int k = 0; k < K; ++k) Gl[k] = c.G_lambda[l * K + k];
  double acc = 0.0;
  const int64_t p1 = c.g_chunk_ptr[chunk + 1];
  // a chunk holds <= 256 entries = 8 per lane: rounds of NQ independent gathers.  NQ = 1 for K > 8: with 4 entries in
  // flight nvcc 12.9 generated a kernel for K = 12 that faulted ("misaligned address" with every access naturally
  // aligned: a clobbered return address of the fp64 reciprocal's out-of-line slow path) -- see also vm_rcp64.
  constexpr int NQ = (K <= 8) ? 4 : 1;
  for (int64_t pb = c.g_chunk_ptr[chunk] + lane; pb < p1; pb += 32 * NQ) {
    int64_t u[NQ];
    float x[NQ], xT[NQ];
#pragma unroll
    for (int q = 0; q < NQ; ++q) {
      const int64_t p = pb + 32 * q;
      const bool ok = p < p1;
      u[q] = ok ? (int64_t)c.g_u[p] : 0;
      x[q] = ok ? c.g_x[p] : 0.f;
      xT[q] = ok ? c.g_xT[p] : 0.f;
    }
    float r[NQ][K];  // the fp32 posterior of the tie (8 bytes at K=2: half the gather of the fp64 copy)
#pragma unroll
    for (int q = 0; q < NQ; ++q) vm_load_rho32<K>(c.rho_u32 + u[q] * K, r[q]);
#pragma unroll
    for (int q = 0; q < NQ; ++q) {
      double dz1[K], dz2[K];
      vm_alloc<K>(mut, (double)x[q], (double)xT[q], Gth, Gl, Gnu, dz1, dz2);  // x == 0 for padding lanes
#pragma unroll
      for (int k = 0; k < K; ++k) acc += (double)r[q][k] * dz1[k];
    }
  }
  acc = warp_sum(acc);
  if (lane == 0) part[chunk] = acc;
}

__global__ void __launch_bounds__(256) k_gamma_reduce(const __grid_constant__ vm_ctx c, const double* part) {
  // one warp per reporter: a reporter that reports every tie owns thousands of chunks
  const int lane = threadIdx.x & 31;
  const int64_t lm = (int64_t)blockIdx.x * 8 + (threadIdx.x >> 5);
  if (lm >= c.L * c.M) return;
  double s = 0.0;
  for (int64_t q = c.g_lm_cptr[lm] + lane; q < c.g_lm_cptr[lm + 1]; q += 32) s += part[q];
  s = warp_sum(s);
  // + the entries without a reciprocal report: dz1 = x, so their share is sum x (minus the ties that underflowed)
  if (lane == 0) c.red1[lm] = s + c.g0[lm] + (double)c.fixG[lm] * VM_FIX_INV;
}

// Tie-sorted variant of the gamma pass (vm_ctx.gamma_ts: all-reporter mask, M <= 256).  Grid and chunking of k_phi_partial
// (blocks of phi_chunk consecutive E1 entries of a layer, sorted by tie: the posterior gather is sequential); the
// per-reporter sums of a block are accumulated in shared memory, per warp, in FIXED POINT (2^-30; three 20-bit limbs in
// 32-bit words, so that plain 32-bit shared atomics neither overflow -- a warp adds at most phi_chunk/8 = 512 terms -- nor
// depend on the order: bit-reproducible).  One partial per (block, reporter); k_gamma_reduce_ts sums them.
template <int K>
__global__ void __launch_bounds__(256) k_gamma_partial_ts(const __grid_constant__ vm_ctx c, double* part) {
  extern __shared__ __align__(16) unsigned char gts_smem[];
  const int l = blockIdx.y, M = (int)c.M, warp = threadIdx.x >> 5;
  double* s_Gth = reinterpret_cast<double*>(gts_smem);                     // [M]
  unsigned int* s_acc = reinterpret_cast<unsigned int*>(s_Gth + M);        // [8][M][3]
  for (int m = threadIdx.x; m < M; m += 256) s_Gth[m] = c.G_theta[(int64_t)l * M + m];
  for (int t = threadIdx.x; t < 8 * M * 3; t += 256) s_acc[t] = 0u;
  __syncthreads();
  const int64_t s0 = c.lay_eptr[l] + (int64_t)blockIdx.x * c.phi_chunk;
  const int64_t s1 = min(s0 + c.phi_chunk, c.lay_eptr[l + 1]);
  const bool mut = c.mutuality != 0;
  const double Gnu = c.nu[VM_NU_G];
  double Gl[K];
#pragma unroll
  for (int k = 0; k < K; ++k) Gl[k] = c.G_lambda[l * K + k];
  unsigned int* acc = s_acc + (size_t)warp * M * 3;
  constexpr int NQ = 4;
  for (int64_t eb = s0 + threadIdx.x; eb < s1; eb += 256 * NQ) {
    int64_t u[NQ];
    int m[NQ];
    float x[NQ], xT[NQ];
#pragma unroll
    for (int q = 0; q < NQ; ++q) {
      const int64_t e = eb + 256 * q;
      const bool ok = e < s1;
      u[q] = ok ? (int64_t)c.f_u[e] : 0;
      m[q] = ok ? c.f_m[e] : 0;
      x[q] = ok ? c.f_x[e] : 0.f;
      xT[q] = ok ? c.f_xT[e] : 0.f;
    }
    float r[NQ][K];
#pragma unroll
    for (int q = 0; q < NQ; ++q) vm_load_rho32<K>(c.rho_u32 + u[q] * K, r[q]);
#pragma unroll
    for (int q = 0; q < NQ; ++q) {
      double dz1[K], dz2[K];
      vm_alloc<K>(mut, (double)x[q], (double)xT[q], s_Gth[m[q]], Gl, Gnu, dz1, dz2);  // x == 0 for padding
      double sv = 0.0;
#pragma unroll
      for (int k = 0; k < K; ++k) sv += (double)r[q][k] * dz1[k];
      const unsigned long long v = (unsigned long long)__double2ll_rn(sv * 1073741824.0);  // sv >= 0
      if (v != 0ull) {
        unsigned int* a = acc + m[q] * 3;
        atomicAdd(a, (unsigned int)(v & 0xfffffull));
        atomicAdd(a + 1, (unsigned int)((v >> 20) & 0xfffffull));
        const unsigned int hi = (unsigned int)(v >> 40);
        if (hi) atomicAdd(a + 2, hi);
      }
    }
  }
  __syncthreads();
  for (int mm = threadIdx.x; mm < M; mm += 256) {
    unsigned long long tot = 0ull;
    for (int w = 0; w < 8; ++w) {
      const unsigned int* a = s_acc + ((size_t)w * M + mm) * 3;
      tot += (unsigned long long)a[0] + ((unsigned long long)a[1] << 20) + ((unsigned long long)a[2] << 40);
    }
    part[((int64_t)l * c.n_phichunk + blockIdx.x) * M + mm] = (double)tot * (1.0 / 1073741824.0);
  }
}

__global__ void __launch_bounds__(256) k_gamma_reduce_ts(const __grid_constant__ vm_ctx c, const double* part) {
  // one warp per reporter: fixed-order sum of its block partials
  const int lane = threadIdx.x & 31;
  const int64_t lm = (int64_t)blockIdx.x * 8 + (threadIdx.x >> 5);
  if (lm >= c.L * c.M) return;
  const int64_t l = lm / c.M, m = lm - l * c.M;
  double s = 0.0;
  for (int64_t q = lane; q < c.n_phichunk; q += 32) s += part[(l * c.n_phichunk + q) * c.M + m];
  s = warp_sum(s);
  if (lane == 0) c.red1[lm] = s + c.g0[lm] + (double)c.fixG[lm] * VM_FIX_INV;
}

// =====================================================================================================
// phase phi
// =====================================================================================================
__device__ __forceinline__ void vm_store_theta_cache(const vm_ctx& c, int64_t lm, double shp, double rte, double& et,
                                                     double& el) {
  el = vm_digamma(shp) - log(rte);
  et = shp / rte;
  const double g = exp(el);
  c.Elog_theta[lm] = el;
  c.G_theta[lm] = g;
  c.E_theta[lm] = et;
  c.GE_theta[2 * lm] = g;
  c.GE_theta[2 * lm + 1] = el;
}

// per-block partials of k_gamma_finish, consumed by k_phi_finish: sum_m E[theta_m] A[m,k] (k < K), sum_m E[theta_m],
// max E[theta], max -E[log theta], max E[log theta]
#define VM_GF_SLOTS(K) ((K) + 4)
#define VM_GF_THREADS 256

// `_update_gamma` (model.py:698-718) from the (all-reduced) shape sums and A, then the theta part of
// `_update_cache` (model.py:676).  gamma_rte[l,m] = beta + sum_k A[l,m,k] E[lambda_lk].
// Grid (ceil(M/256), L).  The same pass produces the block partials of what `_update_phi` needs from the NEW theta
// (phi_rte[l,k] = beta + sum_m E[theta_lm] A[l,m,k], model.py:742-749) and clears the fixed-point accumulators of the
// coming rho update (fixA: consumed by the last k_stats_ego; fixG: consumed by k_gamma_reduce just before).
template <int K>
__global__ void __launch_bounds__(VM_GF_THREADS) k_gamma_finish(const __grid_constant__ vm_ctx c) {
  __shared__ double sm[VM_GF_THREADS / 32];
  const int l = blockIdx.y;
  const int64_t m = (int64_t)blockIdx.x * VM_GF_THREADS + threadIdx.x;
  double acc[K + 1];
#pragma unroll
  for (int k = 0; k <= K; ++k) acc[k] = 0.0;
  double emax = 0.0, nelmax = -1e300, elmax = -1e300;
  if (m < c.M) {
    const int64_t lm = (int64_t)l * c.M + m;
    const double shp = c.alpha_theta[lm] + c.red1[lm];
    double r = 0.0, a[K];
#pragma unroll
    for (int k = 0; k < K; ++k) {
      a[k] = c.A[lm * K + k];
      r += a[k] * c.E_lambda[l * K + k];
    }
    const double rte = c.beta_theta[lm] + r;
    c.gamma_shp[lm] = shp;
    c.gamma_rte[lm] = rte;
    double et, el;
    vm_store_theta_cache(c, lm, shp, rte, et, el);
#pragma unroll
    for (int k = 0; k < K; ++k) acc[k] = et * a[k];
    acc[K] = et;
    emax = et;
    nelmax = -el;
    elmax = el;
    if (c.r_mode == VM_R_EGO) {
#pragma unroll
      for (int k = 0; k < K; ++k) c.fixA[lm * K + k] = 0;
    }
    c.fixG[lm] = 0;
  }
  double* out = c.gfpart + ((int64_t)l * gridDim.x + blockIdx.x) * VM_GF_SLOTS(K);
#pragma unroll
  for (int k = 0; k <= K; ++k) {
    const double v = block_sum<VM_GF_THREADS>(acc[k], sm);
    if (threadIdx.x == 0) out[k] = v;
  }
  emax = block_max<VM_GF_THREADS>(emax, sm);
  if (threadIdx.x == 0) out[K + 1] = emax;
  nelmax = block_max<VM_GF_THREADS>(nelmax, sm);
  if (threadIdx.x == 0) out[K + 2] = nelmax;
  elmax = block_max<VM_GF_THREADS>(elmax, sm);
  if (threadIdx.x == 0) out[K + 3] = elmax;
}

// `_sp_uttkrp_lambda` (model.py:880-887): per-layer sums of rho_k*dz1_k over the X entries (new theta cache).
template <int K>
__global__ void __launch_bounds__(256) k_phi_partial(const __grid_constant__ vm_ctx c, double* part) {
  __shared__ double sm[8];
  const int l = blockIdx.y;
  const int64_t s0 = c.lay_eptr[l] + (int64_t)blockIdx.x * c.phi_chunk;
  const int64_t s1 = min(s0 + c.phi_chunk, c.lay_eptr[l + 1]);
  const bool mut = c.mutuality != 0;
  const double Gnu = c.nu[VM_NU_G];
  double Gl[K], acc[K];
#pragma unroll
  for (int k = 0; k < K; ++k) {
    Gl[k] = c.G_lambda[l * K + k];
    acc[k] = 0.0;
  }
  constexpr int NQ = (K <= 8) ? 4 : 1;  // (see k_gamma_partial)
  for (int64_t eb = s0 + threadIdx.x; eb < s1; eb += 256 * NQ) {
    int64_t u[NQ];
    int m[NQ];
    float x[NQ], xT[NQ];
#pragma unroll
    for (int q = 0; q < NQ; ++q) {
      const int64_t e = eb + 256 * q;
      const bool ok = e < s1;
      u[q] = ok ? (int64_t)c.f_u[e] : 0;
      m[q] = ok ? c.f_m[e] : 0;
      x[q] = ok ? c.f_x[e] : 0.f;
      xT[q] = ok ? c.f_xT[e] : 0.f;
    }
    float r[NQ][K];
    double Gth[NQ];
#pragma unroll
    for (int q = 0; q < NQ; ++q) {
      Gth[q] = c.G_theta[(int64_t)l * c.M + m[q]];
      vm_load_rho32<K>(c.rho_u32 + u[q] * K, r[q]);
    }
#pragma unroll
    for (int q = 0; q < NQ; ++q) {
      double dz1[K], dz2[K];
      vm_alloc<K>(mut, (double)x[q], (double)xT[q], Gth[q], Gl, Gnu, dz1, dz2);  // x == 0 for padding
#pragma unroll
      for (int k = 0; k < K; ++k) acc[k] += (double)r[q][k] * dz1[k];
    }
  }
#pragma unroll
  for (int k = 0; k < K; ++k) {
    const double v = block_sum<256>(acc[k], sm);
    if (threadIdx.x == 0) part[((int64_t)l * c.n_phichunk + blockIdx.x) * K + k] = v;
  }
}

template <int K>
__global__ void __launch_bounds__(256) k_phi_reduce(const __grid_constant__ vm_ctx c, const double* part) {
  __shared__ double sm[8];
  const int l = blockIdx.x;
#pragma unroll
  for (int k = 0; k < K; ++k) {
    double v = 0.0;
    for (int64_t q = threadIdx.x; q < c.n_phichunk; q += 256) v += part[((int64_t)l * c.n_phichunk + q) * K + k];
    v = block_sum<256>(v, sm);
    if (threadIdx.x == 0) c.red2[l * K + k] = v + c.phi0[l * K + k];  // + the E0 entries (from the last rho update)
  }
}

// =====================================================================================================
// phase rho
// =====================================================================================================
// `_update_phi` (model.py:729-749): phi_rte[l,k] = beta + sum_m E[theta_lm](new) A[l,m,k] from the block partials of
// k_gamma_finish; lambda part of the cache; then the per-layer constants of the closed-form tie posterior.
template <int K>
__global__ void __launch_bounds__(256) k_phi_finish(const __grid_constant__ vm_ctx c) {
  __shared__ double sm[8];
  __shared__ double rte_s[K + 1];
  const int l = blockIdx.x;
  const int64_t nb = (c.M + VM_GF_THREADS - 1) / VM_GF_THREADS;
  const double* gp = c.gfpart + (int64_t)l * nb * VM_GF_SLOTS(K);
  double acc[K + 1];
  double emax = 0.0, nelmax = -1e300, elmax = -1e300;  // max E[theta]; max of -E[log theta]; max E[log theta]
#pragma unroll
  for (int k = 0; k <= K; ++k) acc[k] = 0.0;
  for (int64_t b = threadIdx.x; b < nb; b += 256) {
#pragma unroll
    for (int k = 0; k <= K; ++k) acc[k] += gp[b * VM_GF_SLOTS(K) + k];
    emax = fmax(emax, gp[b * VM_GF_SLOTS(K) + K + 1]);
    nelmax = fmax(nelmax, gp[b * VM_GF_SLOTS(K) + K + 2]);
    elmax = fmax(elmax, gp[b * VM_GF_SLOTS(K) + K + 3]);
  }
#pragma unroll
  for (int k = 0; k <= K; ++k) {
    const double v = block_sum<256>(acc[k], sm);
    if (threadIdx.x == 0) rte_s[k] = v;
  }
  emax = block_max<256>(emax, sm);
  nelmax = block_max<256>(nelmax, sm);
  elmax = block_max<256>(elmax, sm);
  if (c.simple_mode && threadIdx.x < K) c.fixP[l * K + threadIdx.x] = 0;
  if (threadIdx.x == 0) {
    if (l == 0) {
      c.dev_flags[VM_FLAG_DEAD] = 0;
      c.dev_flags[VM_FLAG_FIXNU] = 0;
    }
    double El[K], Ell[K], Gl[K];
#pragma unroll
    for (int k = 0; k < K; ++k) {
      const double shp = c.alpha_lambda[l * K + k] + c.red2[l * K + k];
      const double rte = c.beta_lambda[l * K + k] + rte_s[k];
      c.phi_shp[l * K + k] = shp;
      c.phi_rte[l * K + k] = rte;
      const double el = vm_digamma(shp) - log(rte);
      Ell[k] = el;
      c.Elog_lambda[l * K + k] = el;
      Gl[k] = exp(el);
      c.G_lambda[l * K + k] = Gl[k];
      El[k] = shp / rte;
      c.E_lambda[l * K + k] = El[k];
    }
    double* lc = c.layer_consts + (int64_t)l * VM_LC_STRIDE(K);
    const double lp0 = log1p(c.eps), lpk = log(c.eps);
    lc[VM_LC_C(0)] = lp0 * VM_LOG2E;
    lc[VM_LC_D(K, 0)] = El[0] * VM_LOG2E;
#pragma unroll
    for (int k = 1; k < K; ++k) {
      lc[VM_LC_C(k)] = (lpk - lp0) * VM_LOG2E;
      lc[VM_LC_D(K, k)] = (El[k] - El[0]) * VM_LOG2E;
    }
    lc[VM_LC_SALL(K)] = rte_s[K];
    lc[VM_LC_LP0(K)] = lp0;
    lc[VM_LC_LPK(K)] = lpk;
    // no closed-form row can underflow completely if even the largest possible S keeps k=0 alive
    const double s_max = (c.r_mode == VM_R_EGO) ? 2.0 * emax : rte_s[K];
    lc[VM_LC_DEAD(K)] = (c.r_mode == VM_R_CSR || lp0 - s_max * El[0] < VM_DEAD_LN + 8.0) ? 1.0 : 0.0;
#pragma unroll
    for (int k = 0; k < K; ++k) lc[VM_LC_G(K, k)] = (Ell[k] - Ell[0]) * VM_LOG2E;
    // shortcut ties (see vm_ctx.simple_mode): evaluated by the fp32 kernels only if
    //  (i) none of them can underflow completely: the log-weight of category k is
    //      >= min log(pr_k+EPS) - S_max E[lambda_k] + X_max min(0, min E[log theta] + E[log lambda_k])
    //      (every entry's dz1_k lies in [0, x]), and it is enough that ONE category stays above the threshold, and
    //  (ii) the fp32 Poisson split of the SINGLE ties stays in range: z2 = G_nu x^T and z1 = G_theta G_lambda_k
    //       within [1e-30, 1e30] at their largest / z2 at its smallest (x^T >= 1)
    bool simple_ok = false;
    if (((c.simple_mode && c.r_mode == VM_R_EGO) || (c.all32_mode && c.r_mode == VM_R_ALL)) && c.may_dead == 0 &&
        lc[VM_LC_DEAD(K)] == 0.0) {
      // (a tie is alive if ANY category's log-weight is: the bound of the most favourable category decides; the
      // all-reporter kernel checks every tie itself -- with many reporters per tie this bound is far too pessimistic)
      double lwb = -1e300;
#pragma unroll
      for (int k = 0; k < K; ++k)
        lwb = fmax(lwb, c.simple_consts[3 + k] - s_max * El[k] + c.simple_consts[1] * fmin(0.0, -nelmax + Ell[k]));
      simple_ok = c.r_mode == VM_R_ALL || lwb >= VM_DEAD_LN + 8.0;
      if (c.mutuality) {
        const double gnu = c.nu[VM_NU_G];
        double glmax = 0.0;
#pragma unroll
        for (int k = 0; k < K; ++k) glmax = fmax(glmax, Gl[k]);
        simple_ok = simple_ok && gnu >= 1e-30 && gnu * fmax(1.0, c.simple_consts[2]) <= 1e30 &&
                    exp(fmin(elmax, 80.0)) * glmax <= 1e30;
      }
    }
    lc[VM_LC_SIMPLE(K)] = simple_ok ? 1.0 : 0.0;
  }
}

// theta/lambda/nu caches from the current shapes and rates (`_update_cache`, model.py:676-684); used once after the
// initial state has been injected.
__global__ void k_refresh_cache(const __grid_constant__ vm_ctx c) {
  const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t < c.L * c.M) {
    double et, el;
    vm_store_theta_cache(c, t, c.gamma_shp[t], c.gamma_rte[t], et, el);
  }
  if (t < c.L * c.K) {
    const double el = vm_digamma(c.phi_shp[t]) - log(c.phi_rte[t]);
    c.Elog_lambda[t] = el;
    c.G_lambda[t] = exp(el);
    c.E_lambda[t] = c.phi_shp[t] / c.phi_rte[t];
  }
  if (t == 0) {
    double* nu = c.nu;
    nu[VM_NU_E] = nu[VM_NU_SHP] / nu[VM_NU_RTE];
    nu[VM_NU_G] = c.mutuality ? exp(vm_digamma(nu[VM_NU_SHP]) - log(nu[VM_NU_RTE])) : 0.0;
    nu[VM_NU_G_STALE] = nu[VM_NU_G];
  }
}

__device__ __forceinline__ double vm_Er(const vm_ctx& c, int l, int n) {
  // E[theta] of node n acting as reporter in layer l (0 when it is not an active reporter)
  return (n < (int)c.M && c.rep[(int64_t)l * c.M + n]) ? c.E_theta[(int64_t)l * c.M + n] : 0.0;
}

// per-node table of the shortcut ties (k_dense_sc): q_1..q_{K-1}, G_theta, E[log theta] log2e, active flag
template <int K>
struct NodeTab {
  static constexpr int STRIDE = (K == 2) ? 4 : (K <= 6 ? 8 : K + 2);
};

// Row/column tables of the separable log2-odds: a_k(l,i,j) = tab_p[lrow,k] + tab_q[l,j,k] since for the ego mask
// S = E[theta_i]+E[theta_j], and for the all-reporter mask S is a per-layer constant.
template <int K>
__global__ void k_tables(const __grid_constant__ vm_ctx c) {
  const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int64_t nq = c.L * c.N, np = c.L * c.nloc;
  if (t < nq) {
    const int l = (int)(t / c.N), n = (int)(t - (int64_t)l * c.N);
    const double* lc = c.layer_consts + (int64_t)l * VM_LC_STRIDE(K);
    const double er = (c.r_mode == VM_R_EGO) ? vm_Er(c, l, n) : 0.0;
    c.er_node[t] = er;
#pragma unroll
    for (int k = 0; k < K; ++k) c.tab_q[t * K + k] = (float)(-er * lc[VM_LC_D(K, k)]);
    if (c.simple_mode) {  // per-node table of the shortcut-tie kernel
      float* nt = c.nodetab + t * NodeTab<K>::STRIDE;
#pragma unroll
      for (int k = 1; k < K; ++k) nt[k - 1] = (float)(-er * lc[VM_LC_D(K, k)]);
      double2 ge = make_double2(0.0, 0.0);
      if (n < (int)c.M) ge = *reinterpret_cast<const double2*>(c.GE_theta + 2 * ((int64_t)l * c.M + n));
      nt[K - 1] = (float)ge.x;
      nt[K] = (float)(ge.y * VM_LOG2E);
      nt[K + 1] = er > 0.0 ? 1.f : 0.f;
    }
  }
  if (t < np) {
    const int l = (int)(t / c.nloc), i = (int)(t - (int64_t)l * c.nloc) + (int)c.row0;
    const double* lc = c.layer_consts + (int64_t)l * VM_LC_STRIDE(K);
    const double s = (c.r_mode == VM_R_EGO) ? vm_Er(c, l, i) : lc[VM_LC_SALL(K)];
#pragma unroll
    for (int k = 0; k < K; ++k) c.tab_p[t * K + k] = (float)(lc[VM_LC_C(k)] - s * lc[VM_LC_D(K, k)]);
  }
}

template <int K>
__device__ __forceinline__ bool vm_may_dead(const vm_ctx& c, int l) {
  return c.may_dead != 0 || c.layer_consts[(int64_t)l * VM_LC_STRIDE(K) + VM_LC_DEAD(K)] != 0.0;
}

// fp32 S of a tie under the general (CSR) mask, in CSR order -- shared by k_dense<CSR> and k_special.
__device__ __forceinline__ float vm_csr_S32(const vm_ctx& c, int l, int64_t tie) {
  float s = 0.f;
  for (int64_t e = c.r_ptr[tie]; e < c.r_ptr[tie + 1]; ++e)
    s = __fmaf_rn((float)c.E_theta[(int64_t)l * c.M + c.r_m[e]], c.r_val[e], s);
  return s;
}

template <int K>
__device__ __forceinline__ void vm_tie_logodds(const vm_ctx& c, int l, int64_t lrow, int j, float* a) {
  if (c.r_mode == VM_R_CSR) {
    const double* lc = c.layer_consts + (int64_t)l * VM_LC_STRIDE(K);
    const float s = vm_csr_S32(c, l, lrow * c.N + j);
#pragma unroll
    for (int k = 0; k < K; ++k) a[k] = __fmaf_rn(-s, (float)lc[VM_LC_D(K, k)], (float)lc[VM_LC_C(k)]);
  } else {
#pragma unroll
    for (int k = 0; k < K; ++k)
      a[k] = __fadd_rn(c.tab_p[lrow * K + k], c.tab_q[((int64_t)l * c.N + j) * K + k]);
  }
}

#define VM_LONG_TIE 8  // ties with more X entries than this are swept cooperatively by the warp

// contribution of one X entry to the log-weights of its tie and to the nu statistic:
// lw_k += dz1_k (E[log theta_m] + E[log lambda_k]),  Dz_k += dz2_k   (model.py:693-696, 916-921)
template <int K>
__device__ __forceinline__ void vm_entry_accumulate(bool mut, double x, double xT, double2 ge, double Gnu,
                                                    const double* s_Gl, const double* s_Ell, double* lw, double* Dz) {
  if (mut && xT != 0.0) {
    const double z2 = Gnu * xT;
#pragma unroll
    for (int k = 0; k < K; ++k) {
      const double z1 = ge.x * s_Gl[k];
      const double den = z1 + z2;
      const double xi = (den == 0.0) ? 0.0 : x * vm_rcp64(den);  // model.py:692 (Q5)
      lw[k] += (xi * z1) * (ge.y + s_Ell[k]);
      Dz[k] += xi * z2;
    }
  } else {
    // no reciprocal report (or no mutuality): z2 = 0, so dz1_k = x and dz2_k = 0 -- no division needed; with mutuality
    // an underflowed z1_k = 0 makes the denominator 0 and the reference's rule (model.py:692) gives dz1_k = 0
#pragma unroll
    for (int k = 0; k < K; ++k) {
      const bool zero = mut && (ge.x * s_Gl[k] == 0.0);
      if (!zero) lw[k] += x * (ge.y + s_Ell[k]);
    }
  }
}

// Per-reporter accumulation of d[k] = (posterior of a special tie) - (closed form the dense kernel counts for it),
// ego mask: the tie (i,j) is reported by i and by j (the diagonal tie once, and only if the mask contains it).
// Fixed point + integer atomics: the sum is exact in any order, so the result is bit-reproducible.
// d[0] is not accumulated: sum_k d[k] = (special tie alive) - (closed form alive), which is 0 unless a row
// underflowed completely; only that residual goes to slot 0 and k_stats_ego rebuilds d[0] = resid - sum_{k>=1} d[k].
template <int K>
__device__ __forceinline__ void vm_fix_accumulate(unsigned long long* fix_l, bool ego_diag, bool valid, int lrow, int i,
                                                  int j, double ti, double tj, const double* d, int resid) {
  // WARP-COLLECTIVE: every lane of the warp must call it (valid = false for lanes without a tie).
  // Consecutive lanes hold consecutive special ties, i.e. mostly the SAME row: the row-reporter contributions are
  // combined with a segmented warp scan first (one atomic per row segment instead of 32 on one address); the
  // column-reporter contributions go to distinct addresses and are issued directly.  `fix_l` = fixA of the layer.
  const unsigned full = 0xffffffffu;
  const int lane = threadIdx.x & 31;
  const bool diag = (i == j);
  const bool use = valid && !(diag && !ego_diag);
  const bool act_i = use && ti > 0.0, act_j = use && !diag && tj > 0.0;  // E[theta] > 0 <=> active reporter
  const int key = valid ? lrow : (-1 - lane);
  bool same[5];
#pragma unroll
  for (int s = 0; s < 5; ++s) {
    const int kn = __shfl_up_sync(full, key, 1 << s);
    same[s] = (lane >= (1 << s)) && (kn == key);
  }
  const int knext = __shfl_down_sync(full, key, 1);
  const bool tail = valid && ((lane == 31) || (knext != key));
#pragma unroll
  for (int k = 1; k < K; ++k) {
    const long long q = valid ? __double2ll_rn(d[k] * VM_FIX_SCALE) : 0ll;
    long long qr = act_i ? q : 0ll;
#pragma unroll
    for (int s = 0; s < 5; ++s) {
      const long long qn = __shfl_up_sync(full, qr, 1 << s);
      if (same[s]) qr += qn;
    }
    if (tail && qr != 0) atomicAdd(fix_l + i * K + k, (unsigned long long)qr);
    if (act_j && q != 0) atomicAdd(fix_l + j * K + k, (unsigned long long)q);
  }
  if (resid != 0) {  // rare: a row underflowed completely
    const unsigned long long q = (unsigned long long)((long long)resid * (long long)VM_FIX_SCALE);
    if (act_i) atomicAdd(fix_l + i * K, q);
    if (act_j) atomicAdd(fix_l + j * K, q);
  }
}

// ---- special ties (ties that carry X entries, and the diagonal): the full `_update_rho` in fp64 -------------
// log rho_k = log(pr_k+EPS) + sum_{entries} dz1_k (E[log theta_m] + E[log lambda_k]) - S E[lambda_k]   (model.py:800-804,
// 911-921), softmax over k (model.py:807-811), nu statistic (model.py:822-825), ELBO pieces (model.py:967-995, 1306-1313).
// One thread per tie, VM_SPECIAL_TIES_PER_BLOCK ties per block (4 per thread, strided for coalescing).
// All per-layer base pointers are hoisted and the per-tie indices are 32-bit: the kernel is issue-bound, and 64-bit
// index arithmetic was ~1/4 of its instructions.
#ifndef VM_SPECIAL_MINBLK
#define VM_SPECIAL_MINBLK 3
#endif
// LIST (ego mask, no ELBO), for the iterations on which k_dense_sc evaluates the shortcut ties of the layers flagged
// VM_LC_SIMPLE.  LIST = 1 handles those layers: it walks the special ties that take NO shortcut through their compacted
// copies of the per-tie arrays (`cx_*`: coalesced; walking the original arrays at low density multiplied the DRAM bytes
// read per tie, profiles/ncu_r1_simple_dense_fast_special.txt); its grid covers that list only (n_cxblk blocks per
// layer).  LIST = 2 handles the other layers exactly like LIST = 0.  Each block of a (layer, block) grid does its work
// in exactly one of the two launches and returns in the other.
template <int K, bool ELBO, int RMODE, int LIST = 0>
__global__ void __launch_bounds__(256, (K <= 2 ? (ELBO ? 3 : VM_SPECIAL_MINBLK) : 2)) k_special(const __grid_constant__ vm_ctx c, double* part) {
  __shared__ double s_Gl[K], s_Ell[K], s_El[K];
  const int l = blockIdx.y;
  const int nloc = (int)c.nloc, nct = (int)c.nct, N = (int)c.N, M = (int)c.M, row0 = (int)c.row0;
  const int u0 = c.utile_ptr[(int64_t)l * nloc * nct], u1 = c.utile_ptr[(int64_t)(l + 1) * nloc * nct];
  int blk = blockIdx.x;  // block index within the layer
  constexpr bool elbo = ELBO;
  constexpr bool COOP = (RMODE != VM_R_EGO);
  const bool mut = c.mutuality != 0;
  const bool may_dead = vm_may_dead<K>(c, l);
  const bool ego_diag = c.ego_diag != 0;
  const double eps = c.eps;
  const double* lc = c.layer_consts + (int64_t)l * VM_LC_STRIDE(K);
  const double Gnu = c.nu[VM_NU_G];
  // per-layer bases
  const double* er_l = c.er_node + (int64_t)l * N;
  const double* ge_l = c.GE_theta + 2 * (int64_t)l * M;
  const double* et_l = c.E_theta + (int64_t)l * M;
  const float* tabq_l = c.tab_q + (int64_t)l * N * K;
  const float* tabp = c.tab_p;
  unsigned long long* fix_l = reinterpret_cast<unsigned long long*>(c.fixA) + (int64_t)l * M * K;
  const float cat_lp0 = (float)lc[VM_LC_LP0(K)], cat_lpk = (float)lc[VM_LC_LPK(K)], epsf = (float)eps;
  if (LIST != 0 && (lc[VM_LC_SIMPLE(K)] != 0.0) != (LIST == 1)) return;  // the other launch owns this layer
  if (threadIdx.x < K) {
    s_Gl[threadIdx.x] = c.G_lambda[l * K + threadIdx.x];
    s_Ell[threadIdx.x] = c.Elog_lambda[l * K + threadIdx.x];
    s_El[threadIdx.x] = c.E_lambda[l * K + threadIdx.x];
  }
  __syncthreads();
  // LIST = 2 is launched with a small grid whose blocks stride over the layer's block indices (on most fits no layer is
  // its to do: thousands of blocks that only return cost 15 us per iteration at config 3)
  do {
  double nu_acc = 0.0, cat_acc = 0.0, t2_acc = 0.0;
  double dsum[K], p0[K];
#pragma unroll
  for (int k = 0; k < K; ++k) dsum[k] = p0[k] = 0.0;

  constexpr int TPT = VM_SPECIAL_TIES_PER_BLOCK / 256;
  // positions [base, end): tie indices themselves, or (LIST) positions in cx_idx
  int base = u0, end = u1;  // positions: tie indices, or (LIST = 1) positions in the compacted arrays
  if (LIST == 1) {
    base = (int)c.cx_ptr[l];
    end = (int)c.cx_ptr[l + 1];
  }
  const int ub = base + blk * VM_SPECIAL_TIES_PER_BLOCK + threadIdx.x;
  // per-tie data of the first tie (incl. its first X entry, stored inline); the next tie's is fetched while the
  // current one is processed, so only ONE dependent gather level (tables indexed by node / reporter) is exposed
  int n_lrow = 0, n_col = 0, n_m0 = 0, n_cnt = 0;
  float n_x0 = 0.f, n_xT0 = 0.f, n_x0s = 0.f;
  double n_logpr[K];
#pragma unroll
  for (int k = 0; k < K; ++k) n_logpr[k] = 0.0;
  // per-tie arrays: the originals indexed by tie, or (LIST = 1) their compacted copies indexed by position
  const int32_t* a_lrow = (LIST == 1) ? c.cx_lrow : c.u_lrow;
  const int32_t* a_col = (LIST == 1) ? c.cx_col : c.u_col;
  const int32_t* a_cnt = (LIST == 1) ? c.cx_cnt : c.u_cnt;
  const int32_t* a_m0 = (LIST == 1) ? c.cx_m0 : c.u_m0;
  const float* a_x0 = (LIST == 1) ? c.cx_x0 : c.u_x0;
  const float* a_xT0 = (LIST == 1) ? c.cx_xT0 : c.u_xT0;
  const float* a_x0s = (LIST == 1) ? c.cx_x0sum : c.u_x0sum;
  const double* a_logpr = (LIST == 1) ? c.cx_logpr : c.u_logpr;
  int n_u = ub;  // (LIST = 1) tie index of the tie whose data sits in n_*
  if (ub < end) {
    if (LIST == 1) n_u = c.cx_idx[ub];
    n_lrow = a_lrow[ub];
    n_col = a_col[ub];
    n_cnt = a_cnt[ub];
    n_m0 = a_m0[ub];
    n_x0 = a_x0[ub];
    n_xT0 = a_xT0[ub];
    n_x0s = a_x0s[ub];
#pragma unroll
    for (int k = 0; k < K; ++k) n_logpr[k] = a_logpr[(size_t)ub * K + k];
  }
#pragma unroll 1
  for (int it = 0; it < TPT; ++it) {
    const int pos = ub + it * 256;
    const bool valid = pos < end;
    const int u = (LIST == 1) ? n_u : pos;
    // ---- stage A (per thread): tie data, S, prior; entries of SHORT ties
    int lrow = 0, i = 0, j = 0, cnt = 0;
    int64_t e0 = 0;
    double ti = 0.0, tj = 0.0, x0s = 0.0;
    double lw[K], Dz[K], logpr[K];
    float a[K];
#pragma unroll
    for (int k = 0; k < K; ++k) {
      lw[k] = Dz[k] = logpr[k] = 0.0;
      a[k] = 0.f;
    }
    if (valid) {
      lrow = n_lrow;
      j = n_col;
      cnt = n_cnt;
      const int m0 = n_m0;
      const float x0 = n_x0, xT0 = n_xT0;
      x0s = (double)n_x0s;
#pragma unroll
      for (int k = 0; k < K; ++k) logpr[k] = n_logpr[k];
      const int posn = pos + 256;
      if (it + 1 < TPT && posn < end) {
        const int un = posn;
        if (LIST == 1) n_u = c.cx_idx[un];
        n_lrow = a_lrow[un];
        n_col = a_col[un];
        n_cnt = a_cnt[un];
        n_m0 = a_m0[un];
        n_x0 = a_x0[un];
        n_xT0 = a_xT0[un];
        n_x0s = a_x0s[un];
#pragma unroll
        for (int k = 0; k < K; ++k) n_logpr[k] = a_logpr[(size_t)un * K + k];
      }
      i = lrow - l * nloc + row0;
      // the one dependent gather level: reporter cache of the first entry, prior, closed-form tables, S
      double2 ge0 = make_double2(0.0, 0.0);
      if (cnt > 0 && (!COOP || cnt <= VM_LONG_TIE)) ge0 = *reinterpret_cast<const double2*>(ge_l + 2 * m0);
      if (RMODE == VM_R_CSR) {
        vm_tie_logodds<K>(c, l, lrow, j, a);
      } else {
        const float* tp = tabp + lrow * K;
        const float* tq = tabq_l + j * K;
#pragma unroll
        for (int k = 0; k < K; ++k) a[k] = __fadd_rn(tp[k], tq[k]);
      }
      // S = sum over the tie's reporters of E[theta] * R.vals (model.py:766-792)
      double S;
      if (RMODE == VM_R_EGO) {
        ti = er_l[i];
        tj = er_l[j];
        S = (i == j) ? (ego_diag ? ti : 0.0) : ti + tj;
      } else if (RMODE == VM_R_ALL) {
        S = lc[VM_LC_SALL(K)];
      } else {
        S = 0.0;
        const int64_t tie = (int64_t)lrow * N + j;
        for (int64_t e = c.r_ptr[tie]; e < c.r_ptr[tie + 1]; ++e) S += et_l[c.r_m[e]] * (double)c.r_val[e];
      }
#pragma unroll
      for (int k = 0; k < K; ++k) lw[k] = logpr[k] - S * s_El[k];
      if (cnt > 1 || elbo) e0 = c.u_ptr[u];
      if (!COOP || cnt <= VM_LONG_TIE) {
        for (int q = 0; q < cnt; ++q) {
          double2 ge = ge0;  // (G_theta, Elog_theta)
          double x = (double)x0, xT = (double)xT0;
          if (q > 0) {
            const int64_t e = e0 + q;
            ge = *reinterpret_cast<const double2*>(ge_l + 2 * c.e_m[e]);
            x = (double)c.e_x[e];
            xT = (double)c.e_xT[e];
          }
          vm_entry_accumulate<K>(mut, x, xT, ge, Gnu, s_Gl, s_Ell, lw, Dz);
        }
      }
    }
    // ---- stage B (warp-cooperative): ties with many entries (e.g. every reporter reports the tie) are swept by the
    // whole warp, 32 entries at a time, instead of serialising one lane
    if (COOP) {  // an ego mask has at most two reporters per tie: no long ties, stage compiled out
      unsigned longmask = __ballot_sync(0xffffffffu, valid && cnt > VM_LONG_TIE);
      const int lane_b = threadIdx.x & 31;
      while (longmask) {
        const int b = __ffs(longmask) - 1;
        longmask &= longmask - 1;
        const int64_t be0 = __shfl_sync(0xffffffffu, e0, b);
        const int bcnt = __shfl_sync(0xffffffffu, cnt, b);
        double plw[K], pDz[K];
#pragma unroll
        for (int k = 0; k < K; ++k) plw[k] = pDz[k] = 0.0;
        for (int q = lane_b; q < bcnt; q += 32) {
          const int64_t e = be0 + q;
          const double2 ge = *reinterpret_cast<const double2*>(ge_l + 2 * c.e_m[e]);
          vm_entry_accumulate<K>(mut, (double)c.e_x[e], (double)c.e_xT[e], ge, Gnu, s_Gl, s_Ell, plw, pDz);
        }
#pragma unroll
        for (int k = 0; k < K; ++k) {
          plw[k] = warp_sum(plw[k]);  // fixed order; total in lane 0
          pDz[k] = warp_sum(pDz[k]);
          plw[k] = __shfl_sync(0xffffffffu, plw[k], 0);
          pDz[k] = __shfl_sync(0xffffffffu, pDz[k], 0);
          if (lane_b == b) {
            lw[k] += plw[k];
            Dz[k] += pDz[k];
          }
        }
      }
    }
    // ---- stage C (per thread): softmax, statistics, stores
    int o_resid = 0;
    double o_dk[K];
#pragma unroll
    for (int k = 0; k < K; ++k) o_dk[k] = 0.0;
    if (valid) {
      double mx = lw[0];
#pragma unroll
      for (int k = 1; k < K; ++k) mx = fmax(mx, lw[k]);
      double rho[K];
      const bool alive_u = mx >= VM_DEAD_LN;
      if (!alive_u) {
#pragma unroll
        for (int k = 0; k < K; ++k) rho[k] = 0.0;
        c.dev_flags[VM_FLAG_DEAD] = 1;  // benign race: every writer stores the same value
        // its E0 entries no longer contribute x to the gamma-shape sums: take them out of the constant g0
        if (cnt > 0) {
          const int64_t ef = c.u_ptr[u];
          for (int64_t e = ef; e < ef + cnt; ++e)
            if (!mut || c.e_xT[e] == 0.f)
              atomicAdd(reinterpret_cast<unsigned long long*>(c.fixG) + (int64_t)l * M + c.e_m[e],
                        (unsigned long long)(-__double2ll_rn((double)c.e_x[e] * VM_FIX_SCALE)));
        }
      } else if (K == 2) {
        // two categories: the larger weight is exp(0) = 1, only one exponential is needed
        const double e = exp(-fabs(lw[1] - lw[0]));
        const double inv = vm_rcp64(1.0 + e);
        const bool one_max = lw[1] > lw[0];
        rho[0] = one_max ? e * inv : inv;
        rho[1] = one_max ? inv : e * inv;
      } else {
        double sum = 0.0;
#pragma unroll
        for (int k = 0; k < K; ++k) {
          rho[k] = exp(lw[k] - mx);
          sum += rho[k];
        }
        const double inv = vm_rcp64(sum);
#pragma unroll
        for (int k = 0; k < K; ++k) rho[k] *= inv;
      }
      {
#pragma unroll
        for (int k = 0; k < K; ++k) {
          nu_acc += Dz[k] * rho[k];  // sum_e sum_k dz2_k rho_k (model.py:822-825)
          p0[k] += rho[k] * x0s;     // E0 part of the next phi-shape sums (model.py:880-887 with dz1 = x)
        }
      }
      // closed-form value the dense kernel uses for this tie: subtract it again from the statistics
      float f[K], epsr;
      bool dead;
      vm_formula_rho<K>(a, may_dead, f, epsr, dead);
      {
        // closed-form k=0 as the statistics count it: the exact complement of the others (F_0 = n - dead - sum F_k)
        double fk = 0.0;
#pragma unroll
        for (int k = 1; k < K; ++k) fk += (double)f[k];
        double* ru = c.rho_u + (size_t)u * K;
        float* ru32 = c.rho_u32 + (size_t)u * K;
#pragma unroll
        for (int k = 0; k < K; ++k) {
          const double fv = (k == 0) ? (dead ? 0.0 : 1.0 - fk) : (double)f[k];
          o_dk[k] = rho[k] - fv;
          ru[k] = rho[k];
          ru32[k] = (float)rho[k];
          dsum[k] += o_dk[k];
        }
        o_resid = (alive_u ? 1 : 0) - (dead ? 0 : 1);
      }
      if (elbo) {
        // log-Poisson-mean term: uses exp(rho) (Q1) and only the entries that are also in R (model.py:967-995)
        double erho[K];
#pragma unroll
        for (int k = 0; k < K; ++k) erho[k] = exp(rho[k]);
        for (int64_t e = e0; e < e0 + cnt; ++e) {
          const double Gth = ge_l[2 * c.e_m[e]], x = (double)c.e_x[e], z2 = Gnu * (double)c.e_xT[e];
          double val = 0.0;
          if (c.e_flags[e] & 1) {
#pragma unroll
            for (int k = 0; k < K; ++k) val += erho[k] * (Gth * s_Gl[k] + z2);
          }
          t2_acc += x * log(val + eps);
        }
#pragma unroll
        for (int k = 0; k < K; ++k) cat_acc += rho[k] * (logpr[k] - log(rho[k] + eps));
        cat_acc -= (double)vm_formula_cat<K>(f, epsr, dead, cat_lp0, cat_lpk, epsf);
      }
    }  // valid
    if (RMODE == VM_R_EGO) vm_fix_accumulate<K>(fix_l, ego_diag, valid, lrow, i, j, ti, tj, o_dk, o_resid);
  }
  // per-WARP partials (no block barrier: a warp retires as soon as its own ties are done)
  const int64_t nup = c.L * c.n_ublk * 8, b = ((int64_t)l * c.n_ublk + blk) * 8 + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  double v;
  v = warp_sum(nu_acc);
  if (lane == 0) part[UP_NU * nup + b] = v;
  if (elbo) {
    v = warp_sum(cat_acc);
    if (lane == 0) part[UP_CAT * nup + b] = v;
    v = warp_sum(t2_acc);
    if (lane == 0) part[UP_T2 * nup + b] = v;
  }
#pragma unroll
  for (int k = 0; k < K; ++k) {
    v = warp_sum(p0[k]);
    if (lane == 0) part[(UP_P0(K) + k) * nup + b] = v;
  }
  if (RMODE == VM_R_ALL) {  // the all-reporter statistics only need per-layer totals of delta
#pragma unroll
    for (int k = 0; k < K; ++k) {
      v = warp_sum(dsum[k]);
      if (lane == 0) part[(UP_DELTA + k) * nup + b] = v;
    }
  }
  } while (LIST == 2 && (blk += (int)gridDim.x) < (int)c.n_ublk);
}

// ---- the per-tie dense kernel: every owned tie, closed form, fp32 slab write + statistics partials -------------
// HBM-bound: writes 4*K bytes per tie, reads only the (L2-resident) tables and the special-tie patch data.
// A CTA owns a tile of tile_h rows x TW columns; its 8 warps are AUTONOMOUS (no block barrier in the row loop):
// warp w takes rows w, w+8, ...; for each row it sweeps the TW columns in NCH chunks of 128 (4 consecutive ties
// per lane, 128-bit stores), keeps the row sums in registers (one shuffle reduction per row), keeps the column
// sums of all its rows in registers, and finally overwrites the special ties of the row with their fp64-computed
// values (same warp, after __syncwarp: the sectors are still dirty in L2, so no extra DRAM traffic).  The tile
// pointers and row terms of the next row and the patch data of the current row are prefetched before the arithmetic.
// Column partials of the 8 warps are combined through shared memory once, at the end of the CTA.
// TW = 128*NCH depends on K so that the column accumulators (NCH*4*(K-1) registers) stay in registers.

// does a TMA dense kernel handle this (layer, column tile)?  (everything else is k_dense's)
template <int K>
__device__ __forceinline__ bool vm_fast_tile(const vm_ctx& c, int l, int ct) {
  return (((c.N * K) & 3) == 0) && ((int64_t)(ct + 1) * DenseCfg<K>::TW <= c.N) && c.r_mode != VM_R_CSR &&
         !vm_may_dead<K>(c, l);
}

// ---- lane <-> tie mapping inside a 128-tie chunk ------------------------------------------------------------------
// Measured on B200 (tools/write_bw.cu): a warp store instruction whose 32 lanes write 16 B each at a 32 B stride
// (every lane owning 32 contiguous bytes) reaches only 3.8 TB/s, while fully contiguous 512 B per instruction reaches
// 6.8-7.1 TB/s.  So the 4 ties of a lane are chosen such that EVERY 128-bit store instruction of the warp covers 512
// contiguous bytes: K=2 -> ties {2i, 2i+1, 64+2i, 64+2i+1};  K=4 -> ties {i, 32+i, 64+i, 96+i};  other K -> the natural
// {4i..4i+3} with a transpose through a per-warp shared-memory stage.
template <int K>
__device__ __forceinline__ int vm_tie_of(int lane, int t) {
  if (K == 2) return (t < 2) ? (2 * lane + t) : (64 + 2 * lane + (t - 2));
  if (K == 4) return 32 * t + lane;
  return 4 * lane + t;
}
template <int K>
__device__ __forceinline__ void vm_load_q4(const float* qrow_chunk, int lane, float* out) {
  if (K == 2) {
    const float2 a = *reinterpret_cast<const float2*>(qrow_chunk + 2 * lane);
    const float2 b = *reinterpret_cast<const float2*>(qrow_chunk + 64 + 2 * lane);
    out[0] = a.x; out[1] = a.y; out[2] = b.x; out[3] = b.y;
  } else if (K == 4) {
#pragma unroll
    for (int t = 0; t < 4; ++t) out[t] = qrow_chunk[32 * t + lane];
  } else {
    const float4 v = *reinterpret_cast<const float4*>(qrow_chunk + 4 * lane);
    out[0] = v.x; out[1] = v.y; out[2] = v.z; out[3] = v.w;
  }
}
// store the 4 ties of every lane (o[t*K+k]) of one chunk; `dst` = first float of the chunk (16-byte aligned)
template <int K>
__device__ __forceinline__ void vm_store_chunk(float* dst, int lane, const float* o, float* stage) {
  float4* d4 = reinterpret_cast<float4*>(dst);
  if (K == 2) {
    d4[lane] = make_float4(o[0], o[1], o[2], o[3]);
    d4[32 + lane] = make_float4(o[4], o[5], o[6], o[7]);
  } else if (K == 4) {
#pragma unroll
    for (int t = 0; t < 4; ++t) d4[32 * t + lane] = make_float4(o[4 * t], o[4 * t + 1], o[4 * t + 2], o[4 * t + 3]);
  } else if (K > 8) {  // many categories: natural layout (every lane owns 16*K contiguous bytes), no stage
#pragma unroll
    for (int v = 0; v < K; ++v) d4[K * lane + v] = make_float4(o[4 * v], o[4 * v + 1], o[4 * v + 2], o[4 * v + 3]);
  } else {
    float4* s4 = reinterpret_cast<float4*>(stage);
#pragma unroll
    for (int v = 0; v < K; ++v) s4[K * lane + v] = make_float4(o[4 * v], o[4 * v + 1], o[4 * v + 2], o[4 * v + 3]);
    __syncwarp();
#pragma unroll
    for (int v = 0; v < K; ++v) d4[32 * v + lane] = s4[32 * v + lane];
    __syncwarp();
  }
}
template <int K>
struct StageCfg {
  static constexpr int FLOATS = (K == 2 || K == 4 || K > 8) ? 4 : 128 * K;  // per-warp stage (unused for K = 2, 4, > 8)
};

// 4 ties of one lane. a[t][k] are the log2-odds; results in o[t*K+k].
template <int K, bool ELBO, bool MD>
__device__ __forceinline__ void dense_quad(const float (*a)[K], const bool* valid, float* o, float* rowacc,
                                           float (*colacc)[4], float* coldead_chunk, int lane, double& cat, float lp0,
                                           float lpk, float epsf) {
#pragma unroll
  for (int t = 0; t < 4; ++t) {
    float epsr;
    bool dead;
    vm_formula_rho<K>(a[t], MD, &o[t * K], epsr, dead);
#pragma unroll
    for (int k = 1; k < K; ++k) {
      colacc[k - 1][t] += o[t * K + k];
      rowacc[k] += o[t * K + k];
    }
    if (MD && dead && valid[t]) {
      rowacc[0] += 1.f;
      atomicAdd(&coldead_chunk[vm_tie_of<K>(lane, t)], 1.f);  // integer-valued: exact in any order
    }
    if (ELBO && valid[t]) cat += (double)vm_formula_cat<K>(&o[t * K], epsr, dead, lp0, lpk, epsf);
  }
}

// Generic dense kernel: any mask structure, ELBO partials, dead-row bookkeeping, partial tiles.
template <int K, bool ELBO, bool STORE, bool CSR>
__global__ void __launch_bounds__(VM_DENSE_THREADS) k_dense(const __grid_constant__ vm_ctx c, double* catpart, int skip_fast, int rt0, int rtn) {
  constexpr int NCH = DenseCfg<K>::NCH, TW = DenseCfg<K>::TW, NW = VM_DENSE_THREADS / 32;
  __shared__ __align__(16) float qs[K][TW];      // column terms of the tile (row 0: weight of k=0, dead check only)
  __shared__ __align__(16) float colbuf[K][TW];  // cross-warp column sums (row 0: dead counts)
  __shared__ __align__(16) float stage[NW][StageCfg<K>::FLOATS];
  __shared__ double sm_red[8];
  const int N = (int)c.N, nloc = (int)c.nloc, nct = (int)c.nct, nrt = (int)c.nrt;
  const int ct = blockIdx.x;
  const int l = blockIdx.y / rtn, rt = rt0 + (blockIdx.y - l * rtn);  // row tiles [rt0, rt0+rtn) of every layer
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  if (skip_fast && vm_fast_tile<K>(c, l, ct)) return;  // a TMA dense kernel has written this tile
  const int jt = ct * TW;
  const int i_lo = rt * (int)c.tile_h, i_hi = min(i_lo + (int)c.tile_h, nloc);
  const bool may_dead = vm_may_dead<K>(c, l);
  const bool vec_ok = (((int64_t)N * K) & 3) == 0;
  const double* lc = c.layer_consts + (int64_t)l * VM_LC_STRIDE(K);
  const float lp0 = (float)lc[VM_LC_LP0(K)], lpk = (float)lc[VM_LC_LPK(K)], epsf = (float)c.eps;
  float cc[K], dd[K];
#pragma unroll
  for (int k = 0; k < K; ++k) {
    cc[k] = (float)lc[VM_LC_C(k)];
    dd[k] = (float)lc[VM_LC_D(K, k)];
  }
  for (int idx = tid; idx < TW; idx += VM_DENSE_THREADS) {
    const int j = jt + idx;
#pragma unroll
    for (int k = 0; k < K; ++k) {
      qs[k][idx] = (!CSR && j < N) ? __ldg(&c.tab_q[((int64_t)l * N + j) * K + k]) : -INFINITY;
      colbuf[k][idx] = 0.f;
    }
  }
  __syncthreads();

  float colacc[NCH][K - 1][4];
#pragma unroll
  for (int ch = 0; ch < NCH; ++ch)
#pragma unroll
    for (int k = 0; k < K - 1; ++k)
#pragma unroll
      for (int t = 0; t < 4; ++t) colacc[ch][k][t] = 0.f;
  double cat = 0.0;

  for (int i = i_lo + warp; i < i_hi; i += NW) {
    const int64_t lrow = (int64_t)l * nloc + i;
    int ua = 0, ub = 0;
    if (STORE) {
      ua = __ldg(&c.utile_ptr[lrow * nct + ct]);
      ub = __ldg(&c.utile_ptr[lrow * nct + ct + 1]);
    }
    float p[K];
#pragma unroll
    for (int k = 0; k < K; ++k) p[k] = CSR ? 0.f : __ldg(&c.tab_p[lrow * K + k]);
    float rowacc[K];
#pragma unroll
    for (int k = 0; k < K; ++k) rowacc[k] = 0.f;
    float* rowdst = c.rho + lrow * N * K;
#pragma unroll
    for (int ch = 0; ch < NCH; ++ch) {
      const int jc = jt + ch * 128;  // first column of the chunk
      if (jc >= N) continue;         // warp-uniform
      bool valid[4];
      int jj[4];
      bool all_valid = true;
#pragma unroll
      for (int t = 0; t < 4; ++t) {
        jj[t] = jc + vm_tie_of<K>(lane, t);
        valid[t] = jj[t] < N;
        all_valid = all_valid && valid[t];
      }
      float a[4][K];
      if (CSR) {
#pragma unroll
        for (int t = 0; t < 4; ++t) {
          const float sv = valid[t] ? vm_csr_S32(c, l, lrow * N + jj[t]) : 0.f;
#pragma unroll
          for (int k = 0; k < K; ++k) a[t][k] = valid[t] ? __fmaf_rn(-sv, dd[k], cc[k]) : -INFINITY;
        }
      } else {
#pragma unroll
        for (int k = 0; k < K; ++k) {
          if (k == 0 && !may_dead) {
            a[0][0] = a[1][0] = a[2][0] = a[3][0] = 0.f;
            continue;
          }
          float qv[4];
          vm_load_q4<K>(&qs[k][ch * 128], lane, qv);
#pragma unroll
          for (int t = 0; t < 4; ++t) a[t][k] = __fadd_rn(p[k], qv[t]);
        }
      }
      float o[4 * K];
      if (may_dead)
        dense_quad<K, ELBO, true>(a, valid, o, rowacc, colacc[ch], &colbuf[0][ch * 128], lane, cat, lp0, lpk, epsf);
      else
        dense_quad<K, ELBO, false>(a, valid, o, rowacc, colacc[ch], &colbuf[0][ch * 128], lane, cat, lp0, lpk, epsf);
      if (STORE) {
        const bool chunk_full = jc + 128 <= N;  // warp-uniform
        if (vec_ok && chunk_full) {
          vm_store_chunk<K>(rowdst + (int64_t)jc * K, lane, o, stage[warp]);
        } else {
#pragma unroll
          for (int t = 0; t < 4; ++t)
            if (valid[t]) {
#pragma unroll
              for (int k = 0; k < K; ++k) rowdst[(int64_t)jj[t] * K + k] = o[t * K + k];
            }
        }
      }
    }
    // ---- row partials
    if (!CSR) {
#pragma unroll
      for (int k = 0; k < K; ++k) {
        if (k == 0 && !may_dead) continue;
        const float v = warp_sum(rowacc[k]);
        if (lane == 0) c.rowpart[(lrow * nct + ct) * K + k] = v;
      }
      if (!may_dead && lane == 0) c.rowpart[(lrow * nct + ct) * K] = 0.f;
    }
    // ---- patch the special ties of this row segment
    if (STORE) {
      __syncwarp();
      for (int u = ua + lane; u < ub; u += 32) {
        const int col = c.u_col[u];
#pragma unroll
        for (int k = 0; k < K; ++k) rowdst[(int64_t)col * K + k] = c.rho_u32[(int64_t)u * K + k];
      }
    }
  }
  // ---- column partials: combine the 8 warps in a fixed order
  if (!CSR) {
    for (int w = 0; w < NW; ++w) {
      if (warp == w) {
#pragma unroll
        for (int ch = 0; ch < NCH; ++ch)
#pragma unroll
          for (int k = 1; k < K; ++k)
#pragma unroll
            for (int t = 0; t < 4; ++t) colbuf[k][ch * 128 + vm_tie_of<K>(lane, t)] += colacc[ch][k - 1][t];
      }
      __syncthreads();
    }
    for (int idx = tid; idx < TW; idx += VM_DENSE_THREADS) {
      const int j = jt + idx;
      if (j < N) {
#pragma unroll
        for (int k = 0; k < K; ++k) c.colpart[(((int64_t)l * nrt + rt) * N + j) * K + k] = colbuf[k][idx];
      }
    }
  }
  if (ELBO) {
    const double v = block_sum<VM_DENSE_THREADS>(cat, sm_red);
    if (tid == 0) catpart[((int64_t)l * nrt + rt) * nct + ct] = v;
  }
}

// ---- fast (TMA) dense kernels: tile limit ---------------------------------------------------------------------------
// Same tiling and warp-autonomous structure as k_dense, for the common case: separable mask (ego / all), K <= 4,
// N*K % 4 == 0, column tile entirely inside the matrix, and no row of the layer can underflow completely (checked on
// the device; k_dense handles every tile they skip).  ~10 instructions per tie, branch-free chunk loop.
#define VM_FAST_MAX_TILE_H 128

// ---- TMA dense kernel ------------------------------------------------------------------------------------------------
// A row segment reaches HBM in ONE piece: the warp writes its TW ties into a per-warp shared-memory stage in the slab's own
// layout (conflict-free 128-bit shared stores), overwrites the special ties of the segment IN SHARED MEMORY, and one lane
// hands the whole segment (TW*K*4 bytes: 4 KB at K = 2) to the TMA engine with ONE bulk store
// (cp.async.bulk.global.shared::cta).  The slab then only ever sees full, contiguous writes: scattered 4-byte patch stores
// (two per special tie: 3e7 partial-sector L2 writes per launch at config 3, +30 % write requests) cost an STG.128 version
// of this kernel 0.11 ms of its 0.60 ms (profiles/r2_dense_experiments.txt).  Two stages per warp: the next row is computed
// while the engine still reads the previous one (cp.async.bulk.wait_group.read 1 before a stage is refilled).  The patch
// data of the NEXT row of the warp are requested (one special tie per lane, registers) before the current row is swept, so
// their latency -- several microseconds under a saturated store stream -- is covered by a whole row of work.
//
// SC (k_dense_sc, iterations without ELBO in vm_ctx.simple_mode): the special ties of a segment that take the shortcut
// are EVALUATED in the stage instead of patched from rho_u32 (vm_shortcut_tie), between filling the stage and the bulk
// store; the prefetched data are their 16/32-byte records `u_rec` and the row node's node-table entry.  Every other special
// tie of the segment (the special-tie kernel's list ties, and all special ties of a layer whose VM_LC_SIMPLE guard fails)
// keeps its closed form here; k_patch_rest copies their rho_u32 into the slab once the special-tie kernel, which runs
// next to this one, has written it.  The dense partials only ever count the closed form, so nothing else waits for it.
//
// STORE = false (VM_F_NO_STORE: the iteration writes no slab): statistics only -- no stage, no bulk store, no patch
// loads.  The SC variant still evaluates the shortcut ties (rho_u32, fixA, fixP, nu); the closed form their correction
// subtracts is recomputed with vm_formula_rho, which gives the very bits the chunk loop counted.
__device__ __forceinline__ void vm_bulk_store(void* gdst, const void* ssrc, uint32_t bytes) {
  asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(gdst),
               "r"((uint32_t)__cvta_generic_to_shared(ssrc)), "r"(bytes)
               : "memory");
  asm volatile("cp.async.bulk.commit_group;" ::: "memory");
}
template <int N>
__device__ __forceinline__ void vm_bulk_wait_read() {
  asm volatile("cp.async.bulk.wait_group.read %0;" ::"n"(N) : "memory");
}
__device__ __forceinline__ void vm_bulk_wait_all() { asm volatile("cp.async.bulk.wait_group 0;" ::: "memory"); }
__device__ __forceinline__ void vm_fence_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

// A fixed-point correction fq (|fq| <= 2^42) is accumulated in shared memory as TWO 32-bit words, fq = hi * 2^22 + lo with
// lo = the low 22 bits (unsigned) and hi = fq >> 22 (signed, |hi| <= 2^20): a node of a tile receives at most TW = 512
// terms, so neither word can overflow (512 * 2^22 = 2^31), the two native 32-bit adds need no carry -- hence no returned
// value to wait for: a 64-bit shared-memory atomic is a compare-and-swap spin loop (ATOMS.CAST.SPIN.64), and a carry taken
// from the returned old value exposed the atomic's latency twice per tie and category -- and the sum is exact.
__device__ __forceinline__ void vm_smem_add_split(unsigned int* w, long long v) {
  atomicAdd(&w[0], (unsigned int)((unsigned long long)v & 0x3fffffull));
  atomicAdd(&w[1], (unsigned int)(int)(v >> 22));
}
__device__ __forceinline__ unsigned long long vm_smem_split_value(const unsigned int* w) {
  return (unsigned long long)((long long)(int)w[1] * 4194304ll + (long long)w[0]);
}

#define VM_TMA_NBUF 2
template <int K, bool SC = false, bool STORE = true>
struct TmaSmem {
  static constexpr int TW = DenseCfg<K>::TW, NW = VM_DENSE_THREADS / 32, TH = VM_FAST_MAX_TILE_H;
  // row-segment stages (slab layout), 128-byte aligned (first member); a placeholder if nothing is stored
  float rowbuf[STORE ? NW : 1][STORE ? VM_TMA_NBUF : 1][STORE ? TW * K : 4];
  float qs[K - 1][TW];                    // column terms of the log2-odds
  union {
    float colbuf[K - 1][TW];                     // cross-warp column sums (after the row loop)
    unsigned int colfix[SC ? TW : 1][K - 1][2];  // SC, row loop: corrections of the column reporters (vm_smem_add_split)
  };
  float ps[K - 1][TH];                    // row terms
  int tp0[TH], tp1[TH];                   // special-tie range of every row segment
  float lam[SC ? 4 * K + 1 : 1];          // SC: G_lambda_k | G_lambda_k - G_lambda_0 | E[log lambda_k] log2e | G_nu | g_k
  double sm_red[8];
};

// the lane's 4 ties of chunk `ch` into the stage, in the slab's layout (16-byte shared stores, conflict-free)
template <int K>
__device__ __forceinline__ void vm_stage_chunk(float* sb_chunk, int lane, const float* o) {
  float4* d4 = reinterpret_cast<float4*>(sb_chunk);
  if (K == 2) {
    d4[lane] = make_float4(o[0], o[1], o[2], o[3]);
    d4[32 + lane] = make_float4(o[4], o[5], o[6], o[7]);
  } else if (K == 4) {
#pragma unroll
    for (int t = 0; t < 4; ++t) d4[32 * t + lane] = make_float4(o[4 * t], o[4 * t + 1], o[4 * t + 2], o[4 * t + 3]);
  } else {  // natural {4i..4i+3}: 4K contiguous floats per lane
#pragma unroll
    for (int v = 0; v < K; ++v) d4[K * lane + v] = make_float4(o[4 * v], o[4 * v + 1], o[4 * v + 2], o[4 * v + 3]);
  }
}

// ---- shortcut ties: the special ties whose posterior needs no fp64 and no entry list ---------------------------------
// (vm_ctx.simple_mode.)  A special tie u with u_px[u] > 0 takes the shortcut; its record u_rec[u] holds the column,
// X = u_px (total count of a SIMPLE tie / the count of a SINGLE tie's one report), xt = u_pxt (0 = SIMPLE; +-x^T = SINGLE,
// sign: reported by the row / the column node) and lo_k = u_lo = log2((pr_k+EPS)/(pr_0+EPS)).  With the per-node table
// nodetab[l,n] = (q_1..q_{K-1}, G_theta, E[log theta] log2e, active) written by k_tables, q_k = -E[theta_n] d_k:
//   log2 rho_k/rho_0 = q_k(i) + q_k(j) + lo_k + dat_k,
//   SIMPLE: dat_k = X (E[log lambda_k]-E[log lambda_0]) log2e
//   SINGLE: f_k = z1_k/(z1_k+z2), z1_k = G_theta_m G_lambda_k, z2 = G_nu x^T (model.py:686-696),
//           dat_k = x log2e [ (f_k-f_0) E[log theta_m] + f_k E[log lambda_k] - f_0 E[log lambda_0] ]
// every term O(1..30): fp32 does not cancel (the closed form's own p+q ~ -40 would).  The tie is accounted for exactly as
// the special-tie kernel would: fp32 posterior rho[K] (into the slab, and into rho_u32, which the gamma/phi passes gather),
// fq[k] = (posterior - closed form cf[k]) in fixed point for the per-reporter corrections, rho_k X of a SIMPLE tie into p0
// (its part of the next phi-shape sums, fixP), sum_k dz2_k rho_k = x z2 sum_k rho_k/(z1_k+z2) of a SINGLE tie
// (model.py:822-825) into nu (dev_flags[VM_FLAG_FIXNU]).  ni / nj: node-table entries of the row / column node; lam:
// TmaSmem::lam.
template <int K>
__device__ __forceinline__ void vm_shortcut_tie(const float* rec, const float* ni, const float* nj, const float* lam,
                                                const float* cf, float* rho, long long* fq, float& nu, float* p0) {
  const float X = rec[1];
  const float xt = rec[2];
  const bool single = xt != 0.f, rowrep = xt > 0.f;
  const float g = single ? (rowrep ? ni[K - 1] : nj[K - 1]) : 1.f;
  const float el = single ? (rowrep ? ni[K] : nj[K]) : 0.f;
  const float z2 = lam[3 * K] * fabsf(xt);
  float f[K], iden[K];
#pragma unroll
  for (int k = 0; k < K; ++k) {
    const float z1 = g * lam[k];
    iden[k] = vm_rcp(z1 + z2);
    f[k] = single ? z1 * iden[k] : 1.f;
  }
  const float t0 = z2 * g * iden[0];
  // log2-odds against k = 0, then a softmax with the maximum subtracted: for K >= 3 the odds of two categories can
  // both be astronomically large (a tie with a count of 20: 2^140) and only their RATIO matters -- clamping them (as
  // the closed form may, its odds being ~2^-40) would flatten it
  float a[K], amax = 0.f;
#pragma unroll
  for (int k = 1; k < K; ++k) {
    const float dat = single ? X * ((t0 * iden[k] * lam[K + k]) * el + (f[k] * lam[2 * K + k] - f[0] * lam[2 * K]))
                             : X * lam[3 * K + 1 + k];
    const float qk = nj[k - 1];
    a[k] = ni[k - 1] + qk + rec[2 + k] + dat;
    amax = fmaxf(amax, a[k]);
  }
  float es[K], s = vm_ex2(-amax);
  es[0] = s;
#pragma unroll
  for (int k = 1; k < K; ++k) {
    es[k] = vm_ex2(a[k] - amax);
    s += es[k];
  }
  const float inv = vm_rcp(s);
  rho[0] = es[0] * inv;
  float nu_t = rho[0] * iden[0];
#pragma unroll
  for (int k = 1; k < K; ++k) {
    rho[k] = es[k] * inv;
    nu_t += rho[k] * iden[k];
    fq[k] = __double2ll_rn(((double)rho[k] - (double)cf[k]) * VM_FIX_SCALE);
  }
  if (single) {
    nu += X * z2 * nu_t;
  } else {
#pragma unroll
    for (int k = 0; k < K; ++k) p0[k] += rho[k] * X;
  }
}

// floats per shortcut record u_rec: col, X, +-x^T, lo_1..lo_{K-1}, padding
template <int K>
struct ScRec {
  static constexpr int RS = (K == 2) ? 4 : 8;
};

// the first K + 2 floats of a shortcut record / node-table entry (col, X, +-x^T, lo_k | q_k, G_theta, E[log theta], active)
template <int K>
__device__ __forceinline__ void vm_load_rec(const float* p, float* v) {
  const float4 a = __ldg(reinterpret_cast<const float4*>(p));
  v[0] = a.x; v[1] = a.y; v[2] = a.z; v[3] = a.w;
  if (K == 3) v[4] = __ldg(p + 4);
  if (K == 4) {
    const float2 b = __ldg(reinterpret_cast<const float2*>(p + 4));
    v[4] = b.x; v[5] = b.y;
  }
}

#ifndef VM_TMA_PD
#define VM_TMA_PD 2  // rows of prefetch distance of the patch entries
#endif
template <int K, bool ELBO, bool SC, int PD, bool STORE = true>
__device__ __forceinline__ void dense_tma_body(const vm_ctx& c, double* catpart, int rt0, int rtn, unsigned char* smem) {
  constexpr int NCH = DenseCfg<K>::NCH, TW = DenseCfg<K>::TW, NW = VM_DENSE_THREADS / 32;
  constexpr int NT = NodeTab<K>::STRIDE, NV = SC ? K + 2 : K;  // floats per prefetched special tie
  static_assert(!(SC && ELBO), "the shortcut ties are evaluated on iterations without ELBO only");
  TmaSmem<K, SC, STORE>& S = *reinterpret_cast<TmaSmem<K, SC, STORE>*>(smem);
  const int N = (int)c.N, nloc = (int)c.nloc, nct = (int)c.nct, nrt = (int)c.nrt;
  const int ct = blockIdx.x;
  const int l = blockIdx.y / rtn, rt = rt0 + (blockIdx.y - l * rtn);  // row tiles [rt0, rt0+rtn) of every layer
  if (!vm_fast_tile<K>(c, l, ct)) return;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int jt = ct * TW;
  const int i_lo = rt * (int)c.tile_h;
  const int nrows = min((int)c.tile_h, nloc - i_lo);
  const double* lc = c.layer_consts + (int64_t)l * VM_LC_STRIDE(K);
  const float lp0 = (float)lc[VM_LC_LP0(K)], lpk = (float)lc[VM_LC_LPK(K)], epsf = (float)c.eps;
  // SC: does this layer take the shortcut?  (if not, k_patch_rest has all its special ties)
  const bool sc = SC && lc[VM_LC_SIMPLE(K)] != 0.0;
  // SC: statistics of the shortcut ties (see vm_shortcut_tie): fp32 per thread (~10 ties each), fp64 per CTA
  float nu = 0.f, p0[K];
#pragma unroll
  for (int k = 0; k < K; ++k) p0[k] = 0.f;
  double cat = 0.0;
  const float* patch_src = c.rho_u32;
  // ---- phase 0: tables of the tile, once per CTA
  for (int idx = tid; idx < TW; idx += VM_DENSE_THREADS) {
#pragma unroll
    for (int k = 1; k < K; ++k) {
      S.qs[k - 1][idx] = __ldg(&c.tab_q[((int64_t)l * N + jt + idx) * K + k]);
      if (SC) S.colfix[idx][k - 1][0] = S.colfix[idx][k - 1][1] = 0u;
      else S.colbuf[k - 1][idx] = 0.f;
    }
  }
  for (int r = tid; r < nrows; r += VM_DENSE_THREADS) {
    const int64_t lrow = (int64_t)l * nloc + i_lo + r;
#pragma unroll
    for (int k = 1; k < K; ++k) S.ps[k - 1][r] = __ldg(&c.tab_p[lrow * K + k]);
    if (SC || STORE) {
      S.tp0[r] = __ldg(&c.utile_ptr[lrow * nct + ct]);
      S.tp1[r] = (SC && !sc) ? S.tp0[r] : __ldg(&c.utile_ptr[lrow * nct + ct + 1]);
    }
  }
  if (SC && tid < K) {
    const double g0 = c.G_lambda[l * K], gkk = c.G_lambda[l * K + tid];
    S.lam[tid] = (float)gkk;
    S.lam[K + tid] = (float)(gkk - g0);
    S.lam[2 * K + tid] = (float)(c.Elog_lambda[l * K + tid] * VM_LOG2E);
    S.lam[3 * K + 1 + tid] = (float)lc[VM_LC_G(K, tid)];
    if (tid == 0) S.lam[3 * K] = (float)c.nu[VM_NU_G];
  }
  __syncthreads();
  float colacc[NCH][K - 1][4];
#pragma unroll
  for (int ch = 0; ch < NCH; ++ch)
#pragma unroll
    for (int k = 0; k < K - 1; ++k)
#pragma unroll
      for (int t = 0; t < 4; ++t) colacc[ch][k][t] = 0.f;
  // patch entries of this lane (special tie tp0[row] + lane) for the next PD rows of the warp, fetched PD rows ahead:
  // (column, value) -- or, SC, the tie's record and the lane's float of the row node's node-table entry
  int pq_col[PD];
  float pq_v[PD][NV], pq_rn[PD];
  auto fetch = [&](int row, int& col, float* v, float& rn) {
    col = 0;
    rn = 0.f;
#pragma unroll
    for (int k = 0; k < NV; ++k) v[k] = 0.f;
    if (row < nrows) {
      const int ua = S.tp0[row], n = S.tp1[row] - ua;
      if (SC) {
        if (n > 0) rn = __ldg(c.nodetab + ((int64_t)l * N + (int)c.row0 + i_lo + row) * NT + (lane & (NT - 1)));
        if (lane < n) vm_load_rec<K>(c.u_rec + (int64_t)(ua + lane) * ScRec<K>::RS, v);
      } else if (STORE && lane < n) {
        col = __ldg(&c.u_col[ua + lane]);
#pragma unroll
        for (int k = 0; k < K; ++k) v[k] = __ldg(&patch_src[(int64_t)(ua + lane) * K + k]);
      }
    }
  };
#pragma unroll
  for (int d = 0; d < PD; ++d)
    if (SC || STORE) fetch(warp + d * NW, pq_col[d], pq_v[d], pq_rn[d]);
  float prev[K];
  int64_t prev_idx = -1;
#pragma unroll
  for (int k = 1; k < K; ++k) prev[k] = 0.f;
  int buf = 0;
  for (int r = warp; r < nrows; r += NW) {
    const int64_t lrow = (int64_t)l * nloc + i_lo + r;
    // ---- request the patch entry of the row PD rows ahead
    int pn_col;
    float pn_v[NV], pn_rn;
    if (SC || STORE) fetch(r + PD * NW, pn_col, pn_v, pn_rn);
    float p[K];
#pragma unroll
    for (int k = 1; k < K; ++k) p[k] = S.ps[k - 1][r];
    float rowacc[K];
#pragma unroll
    for (int k = 1; k < K; ++k) rowacc[k] = 0.f;
    float* sb = S.rowbuf[warp][buf];
    if (STORE) {
      // the bulk store that last read this stage has finished reading it
      if (lane == 0) vm_bulk_wait_read<VM_TMA_NBUF - 1>();
      __syncwarp();
    }
#pragma unroll
    for (int ch = 0; ch < NCH; ++ch) {
      float qv[K][4];
#pragma unroll
      for (int k = 1; k < K; ++k) vm_load_q4<K>(&S.qs[k - 1][ch * 128], lane, qv[k]);
      float o[4 * K];
#pragma unroll
      for (int t = 0; t < 4; ++t) {
        // identical operation order to vm_formula_rho: s = ((0 + e1) + e2) + ..., inv = rcp(1 + s)
        float e[K], s = 0.f;
#pragma unroll
        for (int k = 1; k < K; ++k) {
          e[k] = vm_ex2(fminf(__fadd_rn(p[k], qv[k][t]), VM_CLAMP_LOG2));
          s = (k == 1) ? e[k] : __fadd_rn(s, e[k]);
        }
        const float inv = vm_rcp(__fadd_rn(1.f, s));
        o[t * K] = inv;
#pragma unroll
        for (int k = 1; k < K; ++k) {
          const float v = __fmul_rn(e[k], inv);
          o[t * K + k] = v;
          colacc[ch][k - 1][t] += v;
          rowacc[k] += v;
        }
        if (ELBO) cat += (double)vm_formula_cat<K>(&o[t * K], s, false, lp0, lpk, epsf);
      }
      if (STORE) vm_stage_chunk<K>(sb + ch * 128 * K, lane, o);
      if (ch < 5) {  // step `ch` of the previous row's reduction (same order as warp_sum: 16, 8, 4, 2, 1)
#pragma unroll
        for (int k = 1; k < K; ++k) prev[k] += __shfl_down_sync(0xffffffffu, prev[k], 16 >> ch);
      }
    }
#pragma unroll
    for (int st = NCH; st < 5; ++st) {
#pragma unroll
      for (int k = 1; k < K; ++k) prev[k] += __shfl_down_sync(0xffffffffu, prev[k], 16 >> st);
    }
    // ---- row partials of the previous row; this row's become `prev`
    if (prev_idx >= 0 && lane == 0) {
      c.rowpart[prev_idx] = 0.f;
#pragma unroll
      for (int k = 1; k < K; ++k) c.rowpart[prev_idx + k] = prev[k];
    }
    prev_idx = (lrow * nct + ct) * K;
#pragma unroll
    for (int k = 1; k < K; ++k) prev[k] = rowacc[k];
    // ---- overwrite the special ties of this row segment in the stage, then hand the segment to the TMA engine
    __syncwarp();
    const int ua = S.tp0[r], n = S.tp1[r] - ua;
    if constexpr (SC) {
      if (n > 0) {  // (warp-uniform)
        float ni[K + 2];
#pragma unroll
        for (int t = 0; t < K + 2; ++t) ni[t] = __shfl_sync(0xffffffffu, pq_rn[0], t);
        long long frow[K];  // corrections of the row reporter, k >= 1
#pragma unroll
        for (int k = 1; k < K; ++k) frow[k] = 0;
        for (int e = lane; e - lane < n; e += 32) {  // more than 32 special ties in the segment: rare
          float rec[K + 2];
          if (e < 32) {
#pragma unroll
            for (int t = 0; t < K + 2; ++t) rec[t] = pq_v[0][t];
          } else {
#pragma unroll
            for (int t = 0; t < K + 2; ++t) rec[t] = 0.f;
            if (e < n) vm_load_rec<K>(c.u_rec + (int64_t)(ua + e) * ScRec<K>::RS, rec);
          }
          if (rec[1] > 0.f) {  // a shortcut tie (lanes past the end hold X = 0)
            const int cj = (int)rec[0] - jt;
            float nj[K + 2];
            vm_load_rec<K>(c.nodetab + ((int64_t)l * N + jt + cj) * NT, nj);
            float* d = sb + cj * K;
            float cf[K], rho[K];
            long long fq[K];
            if (STORE) {
#pragma unroll
              for (int k = 1; k < K; ++k) cf[k] = d[k];  // the closed form the dense partials count for this tie
            } else {
              float a[K], epsr;
              bool dead;
              a[0] = 0.f;
#pragma unroll
              for (int k = 1; k < K; ++k) a[k] = __fadd_rn(p[k], S.qs[k - 1][cj]);
              vm_formula_rho<K>(a, false, cf, epsr, dead);
            }
            vm_shortcut_tie<K>(rec, ni, nj, S.lam, cf, rho, fq, nu, p0);
            const bool act_j = nj[K + 1] != 0.f;
#pragma unroll
            for (int k = 1; k < K; ++k) {
              if (act_j && fq[k] != 0) vm_smem_add_split(S.colfix[cj][k - 1], fq[k]);
              frow[k] += fq[k];
            }
            if (STORE) {
#pragma unroll
              for (int k = 0; k < K; ++k) d[k] = rho[k];
            }
            float* ru = c.rho_u32 + (int64_t)(ua + e) * K;
            if (K == 2) {
              *reinterpret_cast<float2*>(ru) = make_float2(rho[0], rho[1]);
            } else {
#pragma unroll
              for (int k = 0; k < K; ++k) ru[k] = rho[k];
            }
          }
        }
        if (ni[K + 1] != 0.f) {  // the row node is an active reporter: one atomic per category
#pragma unroll
          for (int k = 1; k < K; ++k) {
            long long v = frow[k];
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) v += __shfl_down_sync(0xffffffffu, v, o);
            if (lane == 0 && v != 0)
              atomicAdd(reinterpret_cast<unsigned long long*>(c.fixA) + ((int64_t)l * c.M + (int)c.row0 + i_lo + r) * K + k,
                        (unsigned long long)v);
          }
        }
      }
    } else if (STORE) {
      if (lane < n) {
        float* d = sb + (pq_col[0] - jt) * K;
#pragma unroll
        for (int k = 0; k < K; ++k) d[k] = pq_v[0][k];
      }
      for (int e = 32 + lane; e < n; e += 32) {  // more than 32 special ties in the segment (rare)
        const int col = __ldg(&c.u_col[ua + e]);
        float* d = sb + (col - jt) * K;
#pragma unroll
        for (int k = 0; k < K; ++k) d[k] = __ldg(&patch_src[(int64_t)(ua + e) * K + k]);
      }
    }
    if (STORE) {
      vm_fence_async_smem();
      __syncwarp();
      if (lane == 0) vm_bulk_store(c.rho + (lrow * N + jt) * K, sb, (uint32_t)(TW * K * sizeof(float)));
      buf = (buf + 1 == VM_TMA_NBUF) ? 0 : buf + 1;
    }
#pragma unroll
    for (int d = 0; d + 1 < PD; ++d) {
      pq_col[d] = pq_col[d + 1];
      pq_rn[d] = pq_rn[d + 1];
#pragma unroll
      for (int k = 0; k < NV; ++k) pq_v[d][k] = pq_v[d + 1][k];
    }
    pq_col[PD - 1] = pn_col;
    pq_rn[PD - 1] = pn_rn;
#pragma unroll
    for (int k = 0; k < NV; ++k) pq_v[PD - 1][k] = pn_v[k];
  }
  if (prev_idx >= 0) {  // the last row of this warp
#pragma unroll
    for (int k = 1; k < K; ++k) prev[k] = warp_sum(prev[k]);
    if (lane == 0) {
      c.rowpart[prev_idx] = 0.f;
#pragma unroll
      for (int k = 1; k < K; ++k) c.rowpart[prev_idx + k] = prev[k];
    }
  }
  if constexpr (SC) {
    // ---- corrections of the column reporters: one global atomic per touched node and category; then colfix's space
    // becomes colbuf
    __syncthreads();
    unsigned long long* fix_l = reinterpret_cast<unsigned long long*>(c.fixA) + (int64_t)l * c.M * K;
    for (int t = tid; t < TW * (K - 1); t += VM_DENSE_THREADS) {
      const unsigned long long v = vm_smem_split_value(&S.colfix[0][0][0] + 2 * t);
      if (v != 0ull) atomicAdd(fix_l + (int64_t)(jt + t / (K - 1)) * K + 1 + t % (K - 1), v);
    }
    __syncthreads();
    for (int idx = tid; idx < TW; idx += VM_DENSE_THREADS) {
#pragma unroll
      for (int k = 1; k < K; ++k) S.colbuf[k - 1][idx] = 0.f;
    }
    __syncthreads();
  }
  // ---- column partials: combine the 8 warps in a fixed order
  for (int w = 0; w < NW; ++w) {
    if (warp == w) {
#pragma unroll
      for (int ch = 0; ch < NCH; ++ch)
#pragma unroll
        for (int k = 1; k < K; ++k)
#pragma unroll
          for (int t = 0; t < 4; ++t) S.colbuf[k - 1][ch * 128 + vm_tie_of<K>(lane, t)] += colacc[ch][k - 1][t];
    }
    __syncthreads();
  }
  for (int idx = tid; idx < TW; idx += VM_DENSE_THREADS) {
    float* cp = c.colpart + (((int64_t)l * nrt + rt) * N + jt + idx) * K;
    cp[0] = 0.f;
#pragma unroll
    for (int k = 1; k < K; ++k) cp[k] = S.colbuf[k - 1][idx];
  }
  if (ELBO) {
    const double v = block_sum<VM_DENSE_THREADS>(cat, S.sm_red);
    if (tid == 0) catpart[((int64_t)l * nrt + rt) * nct + ct] = v;
  }
  if (sc) {
    // rho_k X of the SIMPLE ties (their part of the next phi-shape sums) and the nu statistic of the SINGLE ties
    const double vn = block_sum<VM_DENSE_THREADS>((double)nu, S.sm_red);
    if (tid == 0 && vn != 0.0)
      atomicAdd(reinterpret_cast<unsigned long long*>(c.dev_flags) + VM_FLAG_FIXNU,
                (unsigned long long)__double2ll_rn(vn * VM_FIXP_SCALE));
#pragma unroll
    for (int k = 0; k < K; ++k) {
      const double v = block_sum<VM_DENSE_THREADS>((double)p0[k], S.sm_red);
      if (tid == 0 && v != 0.0)
        atomicAdd(reinterpret_cast<unsigned long long*>(c.fixP) + l * K + k,
                  (unsigned long long)__double2ll_rn(v * VM_FIXP_SCALE));
    }
  }
  if (STORE && lane == 0) vm_bulk_wait_all();  // the stages must outlive the engine's reads
}

template <int K, bool ELBO, int PD = VM_TMA_PD, bool STORE = true>
__global__ void __launch_bounds__(VM_DENSE_THREADS, (K == 2 || K == 4) ? 3 : 2) k_dense_tma(const __grid_constant__ vm_ctx c, double* catpart, int rt0, int rtn) {
  extern __shared__ __align__(128) unsigned char vm_tma_smem[];
  dense_tma_body<K, ELBO, false, PD, STORE>(c, catpart, rt0, rtn, vm_tma_smem);
}
// the TMA dense kernel that also evaluates the shortcut ties (iterations without ELBO, vm_ctx.simple_mode).  Prefetch
// distance 1 row: at K = 2 the records of a second row do not fit in the 80 registers of 3 CTAs per SM.  At K = 4 its
// column-correction table leaves room for 2 CTAs per SM only.
template <int K, int PD = 1, bool STORE = true>
__global__ void __launch_bounds__(VM_DENSE_THREADS, (K == 2) ? 3 : 2) k_dense_sc(const __grid_constant__ vm_ctx c, int rt0, int rtn) {
  extern __shared__ __align__(128) unsigned char vm_tma_smem[];
  dense_tma_body<K, false, true, PD, STORE>(c, nullptr, rt0, rtn, vm_tma_smem);
}

// Special ties k_dense_sc left at their closed form, copied from rho_u32 into the slab: the list ties of the layers
// that take the shortcut (cx_*) and every special tie of the other layers.  (Ties of partial column tiles are rewritten
// with the value k_dense already wrote.)
template <int K>
__global__ void __launch_bounds__(256) k_patch_rest(const __grid_constant__ vm_ctx c) {
  const int l = blockIdx.y;
  const bool sc = c.layer_consts[(int64_t)l * VM_LC_STRIDE(K) + VM_LC_SIMPLE(K)] != 0.0;
  const int64_t lnt = (int64_t)c.nloc * c.nct;
  const int64_t p0 = sc ? c.cx_ptr[l] : c.utile_ptr[l * lnt], p1 = sc ? c.cx_ptr[l + 1] : c.utile_ptr[(l + 1) * lnt];
  for (int64_t p = p0 + (int64_t)blockIdx.x * blockDim.x + threadIdx.x; p < p1; p += (int64_t)gridDim.x * blockDim.x) {
    const int64_t u = sc ? c.cx_idx[p] : p;
    const int lrow = sc ? c.cx_lrow[p] : c.u_lrow[u], col = sc ? c.cx_col[p] : c.u_col[u];
    float* dst = c.rho + ((int64_t)lrow * c.N + col) * K;
#pragma unroll
    for (int k = 0; k < K; ++k) dst[k] = c.rho_u32[u * K + k];
  }
}

// ---- all-reporter mask: every special tie in fp32, entry-parallel (vm_ctx.all32_mode) ---------------------------------
// Drop-in for k_special<K, false, VM_R_ALL> on iterations without ELBO, for the layers flagged VM_LC_SIMPLE: same grid
// (n_ublk blocks of VM_SPECIAL_TIES_PER_BLOCK consecutive ties per layer), same per-warp block partials (nu, p0, delta),
// same rho_u32.  The fp64 kernel is instruction-bound there (config 4: 8.9e7 special ties with 1.8 entries on average,
// 2.2e9 warp instructions, 19 of 32 lanes active because a warp waits for its tie with the most entries: 4.1 ms,
// profiles/ncu_r2_c4_special.txt).  Here the work is per ENTRY: for each group of 256 consecutive ties the block's threads
// stride over the group's (contiguous) entries, each computing its entry's contribution to the log2-odds and to the nu
// statistic from a shared-memory reporter table -- coalesced 12-byte entry reads, every lane busy -- and stage it in
// shared memory; then one thread per tie sums its entries' staged values (fixed order), adds the prior and the S term,
// normalises and accumulates the statistics.  Groups with more entries than the stage holds go through it in slices.
// log2 rho_k/rho_0 = lo_k - S_all d_k + sum_e dat_k(e): every term O(1..30), fp32 does not cancel (see vm_shortcut_tie).
#define VM_A32_CAP 128  // staged entries per slice and WARP (a warp's 32 consecutive ties have ~58 entries at config 4)
// floats per staged entry: w_k = dz1_k (K), t_0 = dz1_0 E[log theta] and t_k = (dz1_k - dz1_0) E[log theta] (K),
// dz2_k (K); padded to 16 bytes
#define VM_A32_EF(K) ((3 * (K) + 3) / 4 * 4)
template <int K>
static inline size_t vm_all32_smem_bytes(int64_t M) {
  return ((size_t)2 * ((M + 3) / 4 * 4) + (size_t)8 * VM_A32_CAP * VM_A32_EF(K)) * sizeof(float);
}
template <int K>
__global__ void __launch_bounds__(256, (K <= 2) ? 4 : 3) k_all32(const __grid_constant__ vm_ctx c, double* part) {
  constexpr int EF = VM_A32_EF(K);
  extern __shared__ __align__(16) float a32_smem[];
  const int l = blockIdx.y, blk = blockIdx.x, tid = threadIdx.x;
  const int M = (int)c.M, Mp = (M + 3) / 4 * 4;
  float* s_G = a32_smem;        // [Mp] G_theta
  float* s_El = s_G + Mp;       // [Mp] E[log theta] log2e
  const int warp = tid >> 5, lane = tid & 31;
  float* s_ent = s_El + Mp + warp * (VM_A32_CAP * EF);  // this warp's stage [VM_A32_CAP * EF]
  const double* lc = c.layer_consts + (int64_t)l * VM_LC_STRIDE(K);
  if (lc[VM_LC_SIMPLE(K)] == 0.0) return;  // the fp64 special-tie kernel (LIST = 2) has this layer
  const int nloc = (int)c.nloc, nct = (int)c.nct;
  const int u0 = c.utile_ptr[(int64_t)l * nloc * nct], u1 = c.utile_ptr[(int64_t)(l + 1) * nloc * nct];
  const bool mut = c.mutuality != 0;
  for (int m = tid; m < M; m += 256) {
    const double2 ge = *reinterpret_cast<const double2*>(c.GE_theta + 2 * ((int64_t)l * M + m));
    s_G[m] = (float)ge.x;
    s_El[m] = (float)(ge.y * VM_LOG2E);
  }
  // Per-layer constants.  Those that multiply a tie's whole count -- E[log lambda_k], -S_all d_k -- stay in fp64 and are
  // applied once per tie to fp32 sums over its entries: rounded to fp32 they would shift the log-odds of EVERY tie of
  // the layer the same way (up to 5e-6 for a tie with 20 reports), an error that does not average out in the statistics.
  float Gl[K], dGl[K];
  double Ell[K], base[K];
  const double g0 = c.G_lambda[l * K], S_all = lc[VM_LC_SALL(K)];
#pragma unroll
  for (int k = 0; k < K; ++k) {
    Gl[k] = (float)c.G_lambda[l * K + k];
    dGl[k] = (float)(c.G_lambda[l * K + k] - g0);
    Ell[k] = c.Elog_lambda[l * K + k] * VM_LOG2E;
    base[k] = -S_all * lc[VM_LC_D(K, k)];  // k = 0: the S term of the log2 WEIGHT of category 0 (dead check)
  }
  const float Gnu = (float)c.nu[VM_NU_G];
  // the closed form the dense sweep counts for every tie of this layer (all-reporter mask: one value per layer)
  double cfv[K];
  {
    float a[K], cf[K], epsr;
    bool dead;
#pragma unroll
    for (int k = 0; k < K; ++k) a[k] = __fadd_rn(c.tab_p[((int64_t)l * nloc) * K + k], c.tab_q[((int64_t)l * c.N) * K + k]);
    vm_formula_rho<K>(a, false, cf, epsr, dead);
    double fk = 0.0;
#pragma unroll
    for (int k = 1; k < K; ++k) fk += (double)cf[k];
#pragma unroll
    for (int k = 0; k < K; ++k) cfv[k] = (k == 0) ? 1.0 - fk : (double)cf[k];
  }
  double nu_acc = 0.0, dsum[K], p0[K];
#pragma unroll
  for (int k = 0; k < K; ++k) dsum[k] = p0[k] = 0.0;
  __syncthreads();
  // Every warp is autonomous (no block barrier after the tables): it owns 128 consecutive ties of the block, 32 at a time;
  // the entry range of the NEXT 32 ties is requested before the current ones are processed.
  constexpr int TPW = VM_SPECIAL_TIES_PER_BLOCK / 8;  // ties per warp
  const int wbase = u0 + blk * VM_SPECIAL_TIES_PER_BLOCK + warp * TPW;
  int64_t n_p0 = 0, n_p1 = 0;
  if (wbase + lane < u1) {
    n_p0 = c.u_ptr[wbase + lane];
    n_p1 = c.u_ptr[wbase + lane + 1];
  }
#pragma unroll 1
  for (int it = 0; it < TPW / 32; ++it) {
    const int gbase = wbase + it * 32;
    const int ng = max(0, min(32, u1 - gbase));
    const int64_t p0v = n_p0, p1v = n_p1;
    if (it + 1 < TPW / 32 && gbase + 32 + lane < u1) {
      n_p0 = c.u_ptr[gbase + 32 + lane];
      n_p1 = c.u_ptr[gbase + 32 + lane + 1];
    }
    if (ng == 0) break;  // (warp-uniform; nothing follows for this warp)
    const int64_t e0 = __shfl_sync(0xffffffffu, p0v, 0);
    const int n_e = (int)(__shfl_sync(0xffffffffu, p1v, ng - 1) - e0);
    const int qlo = (lane < ng) ? (int)(p0v - e0) : 0, qhi = (lane < ng) ? (int)(p1v - e0) : 0;
    // per-tie constants of the fit, requested now, used after the entries
    const int u = gbase + lane;
    float lo[K], x0s = 0.f;
#pragma unroll
    for (int k = 0; k < K; ++k) lo[k] = 0.f;
    if (lane < ng) {
#pragma unroll
      for (int k = 0; k < K; ++k) lo[k] = c.u_lo[(int64_t)u * K + k];
      x0s = c.u_x0sum[u];
    }
    // (fp64 accumulators: a tie of this mask can have dozens of entries, and W_k is multiplied by |E[log lambda]| ~ 7)
    double W[K], T[K], dz[K];
#pragma unroll
    for (int k = 0; k < K; ++k) W[k] = T[k] = dz[k] = 0.0;
    for (int sl = 0; sl < n_e; sl += VM_A32_CAP) {
      const int ns = min(VM_A32_CAP, n_e - sl);
      // ---- phase 1: one lane per entry of the slice; the loads of two rounds (64 entries: more than a group's usual
      // 58) are issued together -- the kernel is latency-bound on exactly these loads
      for (int el0 = lane; el0 < ns; el0 += 64) {
        int mm[2];
        float xx[2], xt[2];
#pragma unroll
        for (int h = 0; h < 2; ++h) {
          const int el = el0 + 32 * h;
          const bool ok = el < ns;
          const int64_t e = e0 + sl + (ok ? el : 0);
          mm[h] = ok ? c.e_m[e] : 0;
          xx[h] = ok ? c.e_x[e] : 0.f;
          xt[h] = ok ? c.e_xT[e] : 0.f;
        }
#pragma unroll
        for (int h = 0; h < 2; ++h) {
          const int el = el0 + 32 * h;
          if (el >= ns) break;
          const int m = mm[h];
          const float x = xx[h], xT = xt[h];
          float o[EF];
#pragma unroll
          for (int q = 0; q < EF; ++q) o[q] = 0.f;
          const float elt = s_El[m];
          if (mut && xT != 0.f) {
            const float g = s_G[m];
            const float z2 = Gnu * xT;
            float iden[K];
#pragma unroll
            for (int k = 0; k < K; ++k) {
              const float z1 = g * Gl[k];
              iden[k] = vm_rcp(z1 + z2);
              o[k] = x * (z1 * iden[k]);        // dz1_k = x z1_k / (z1_k + z2)
              o[2 * K + k] = x * z2 * iden[k];  // dz2_k (model.py:693-696)
            }
            // dz1_k - dz1_0 = x z2 G_theta (G_lambda_k - G_lambda_0) / ((z1_k + z2)(z1_0 + z2)): the difference form
            const float t0 = x * z2 * g * iden[0];
            o[K] = o[0] * elt;
#pragma unroll
            for (int k = 1; k < K; ++k) o[K + k] = (t0 * iden[k] * dGl[k]) * elt;
          } else {  // no reciprocal report: dz1_k = x for every k, dz2 = 0
#pragma unroll
            for (int k = 0; k < K; ++k) o[k] = x;
            o[K] = x * elt;
          }
          float4* dst = reinterpret_cast<float4*>(s_ent + el * EF);
#pragma unroll
          for (int q = 0; q < EF / 4; ++q) dst[q] = make_float4(o[4 * q], o[4 * q + 1], o[4 * q + 2], o[4 * q + 3]);
        }
      }
      __syncwarp();
      // ---- phase 2: one lane per tie sums its entries of the slice (ascending: fixed order)
      const int qa = max(qlo, sl), qb = min(qhi, sl + ns);
      for (int q = qa; q < qb; ++q) {
        const float* v = s_ent + (q - sl) * EF;
#pragma unroll
        for (int k = 0; k < K; ++k) {
          W[k] += (double)v[k];
          T[k] += (double)v[K + k];
          dz[k] += (double)v[2 * K + k];
        }
      }
      __syncwarp();
    }
    // ---- the tie: softmax with the maximum subtracted, statistics, store
    if (lane < ng) {
      // log2 rho_k/rho_0 = lo_k - S_all d_k + T_k + E[log lambda_k] W_k - E[log lambda_0] W_0: the K-1 sums and the
      // subtraction of the maximum in fp64 (a few operations per tie), so that the exponent that matters reaches ex2 with
      // full relative precision
      const double w0 = Ell[0] * W[0];
      double a[K], amax = 0.0;
      a[0] = 0.0;
#pragma unroll
      for (int k = 1; k < K; ++k) {
        a[k] = (double)lo[k] + base[k] + T[k] + (Ell[k] * W[k] - w0);
        amax = fmax(amax, a[k]);
      }
      // the largest log2 WEIGHT of the tie: below the reference's underflow threshold the whole row stays 0 (Q3)
      const bool dead = (double)lo[0] + base[0] + T[0] + w0 + amax < (double)VM_DEAD_LOG2;
      float es[K], ssum = 0.f;
#pragma unroll
      for (int k = 0; k < K; ++k) {
        es[k] = vm_ex2((float)(a[k] - amax));
        ssum += es[k];
      }
      const float inv = dead ? 0.f : vm_rcp(ssum);
      if (dead) {  // (rare) as the fp64 kernel: flag it, and take its E0 entries' x out of the constant g0
        c.dev_flags[VM_FLAG_DEAD] = 1;
        for (int64_t e = e0 + qlo; e < e0 + qhi; ++e)
          if (!mut || c.e_xT[e] == 0.f)
            atomicAdd(reinterpret_cast<unsigned long long*>(c.fixG) + (int64_t)l * M + c.e_m[e],
                      (unsigned long long)(-__double2ll_rn((double)c.e_x[e] * VM_FIX_SCALE)));
      }
      float rho[K];
#pragma unroll
      for (int k = 0; k < K; ++k) {
        rho[k] = es[k] * inv;
        nu_acc += (double)rho[k] * dz[k];
        p0[k] += (double)(rho[k] * x0s);
        dsum[k] += (double)rho[k] - cfv[k];
      }
      float* ru = c.rho_u32 + (int64_t)u * K;
      if (K == 2) {
        *reinterpret_cast<float2*>(ru) = make_float2(rho[0], rho[1]);
      } else {
#pragma unroll
        for (int k = 0; k < K; ++k) ru[k] = rho[k];
      }
    }
  }
  // per-WARP partials, the layout k_special writes (k_sums_stage1 / k_stats_all read them)
  const int64_t nup = c.L * c.n_ublk * 8, b = ((int64_t)l * c.n_ublk + blk) * 8 + warp;
  double v = warp_sum(nu_acc);
  if (lane == 0) part[UP_NU * nup + b] = v;
#pragma unroll
  for (int k = 0; k < K; ++k) {
    v = warp_sum(p0[k]);
    if (lane == 0) part[(UP_P0(K) + k) * nup + b] = v;
    v = warp_sum(dsum[k]);
    if (lane == 0) part[(UP_DELTA + k) * nup + b] = v;
  }
}

// ---- statistics of the new rho: A[l,m,k] = sum of rho_k over the ties reported by (l,m) ------------------------
// column partials of the dense kernel summed over the row tiles (coalesced: consecutive threads = consecutive (m,k))
template <int K>
__global__ void k_col_reduce(const __grid_constant__ vm_ctx c) {
  const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= c.L * c.M * K) return;
  const int64_t lm = t / K;
  const int k = (int)(t - lm * K);
  const int l = (int)(lm / c.M), m = (int)(lm - (int64_t)l * c.M);
  double s = 0.0;
  for (int64_t rt = 0; rt < c.nrt; ++rt) s += (double)c.colpart[((l * c.nrt + rt) * c.N + m) * K + k];
  c.colsum[t] = s;
}

// ego mask: row sums + column sums of the closed form (dense partials) + the special-tie corrections.
// One warp per reporter; fixed summation order.
template <int K>
__global__ void __launch_bounds__(256) k_stats_ego(const __grid_constant__ vm_ctx c, int init) {
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int64_t lm = (int64_t)blockIdx.x * 8 + warp;
  if (lm >= c.L * c.M) return;
  double* out = c.red3 + lm * K;
  if (!c.rep[lm]) {
    if (lane < K) out[lane] = 0.0;
    return;
  }
  const int l = (int)(lm / c.M), m = (int)(lm - (int64_t)l * c.M);
  const int N = (int)c.N, nloc = (int)c.nloc, nct = (int)c.nct;
  const bool local = m >= c.row0 && m < c.row0 + nloc;
  const int64_t lrow = (int64_t)l * nloc + (m - c.row0);
  double f[K], d[K];
#pragma unroll
  for (int k = 0; k < K; ++k) f[k] = d[k] = 0.0;
  if (!init) {
    if (local)
      for (int t = lane; t < nct; t += 32) {
#pragma unroll
        for (int k = 0; k < K; ++k) f[k] += (double)c.rowpart[(lrow * nct + t) * K + k];
      }
    if (lane == 0) {
#pragma unroll
      for (int k = 0; k < K; ++k) f[k] += c.colsum[lm * K + k];
      if (local) {  // the (m,m) tie is in the row AND the column sums
        float a[K], g[K], epsr;
        bool dead;
        vm_tie_logodds<K>(c, l, lrow, m, a);
        vm_formula_rho<K>(a, vm_may_dead<K>(c, l), g, epsr, dead);
        const double w = c.ego_diag ? 1.0 : 2.0;
#pragma unroll
        for (int k = 1; k < K; ++k) f[k] -= w * (double)g[k];
        if (dead) f[0] -= w;
      }
    }
  }
  // special-tie corrections: accumulated by k_special / k_init_delta in fixed point
  if (lane == 0) {
    double rest = 0.0;
#pragma unroll
    for (int k = 1; k < K; ++k) {
      d[k] = (double)c.fixA[lm * K + k] * VM_FIX_INV;
      rest += d[k];
    }
    d[0] = (double)c.fixA[lm * K] * VM_FIX_INV - rest;
  }
#pragma unroll
  for (int k = 0; k < K; ++k) {
    f[k] = warp_sum(f[k]);
    d[k] = warp_sum(d[k]);
  }
  if (lane == 0) {
    const double nties = (local ? (double)N : 0.0) + (double)nloc - (local ? (c.ego_diag ? 1.0 : 2.0) : 0.0);
    double f0 = nties - (init ? 0.0 : f[0]);
#pragma unroll
    for (int k = 1; k < K; ++k) f0 -= f[k];
    out[0] = f0 + d[0];
#pragma unroll
    for (int k = 1; k < K; ++k) out[k] = f[k] + d[k];
  }
}

// all-reporter mask: A[l,m,:] is the same for every m = per-layer totals.
template <int K>
__global__ void __launch_bounds__(1024) k_stats_all(const __grid_constant__ vm_ctx c, int init, const double* upart) {
  __shared__ double sm[32];
  __shared__ double tot[K];
  const int l = blockIdx.x;
  const int64_t nrow = c.nloc * c.nct, nup = c.L * c.n_ublk * 8, nwl = c.n_ublk * 8;
  double f[K], d[K];
#pragma unroll
  for (int k = 0; k < K; ++k) f[k] = d[k] = 0.0;
  if (!init)
    for (int64_t t = threadIdx.x; t < nrow; t += 1024) {
#pragma unroll
      for (int k = 0; k < K; ++k) f[k] += (double)c.rowpart[((int64_t)l * nrow + t) * K + k];
    }
  for (int64_t b = threadIdx.x; b < nwl; b += 1024) {
#pragma unroll
    for (int k = 0; k < K; ++k) d[k] += upart[(UP_DELTA + k) * nup + (int64_t)l * nwl + b];
  }
  double fs[K], ds[K];
#pragma unroll
  for (int k = 0; k < K; ++k) {
    fs[k] = block_sum<1024>(f[k], sm);
    ds[k] = block_sum<1024>(d[k], sm);
  }
  if (threadIdx.x == 0) {
    double f0 = (double)c.nloc * (double)c.N - (init ? 0.0 : fs[0]);
#pragma unroll
    for (int k = 1; k < K; ++k) f0 -= fs[k];
    tot[0] = f0 + ds[0];
#pragma unroll
    for (int k = 1; k < K; ++k) tot[k] = fs[k] + ds[k];
  }
  __syncthreads();
  for (int64_t t = threadIdx.x; t < c.M * K; t += 1024) c.red3[(int64_t)l * c.M * K + t] = tot[t % K];
}

// general mask: gather the (patched) dense slab through the per-reporter CSC.
template <int K>
__global__ void __launch_bounds__(256) k_stats_csc(const __grid_constant__ vm_ctx c, int init) {
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int64_t lm = (int64_t)blockIdx.x * 8 + warp;
  if (lm >= c.L * c.M) return;
  double f[K];
#pragma unroll
  for (int k = 0; k < K; ++k) f[k] = 0.0;
  for (int64_t p = c.c_ptr[lm] + lane; p < c.c_ptr[lm + 1]; p += 32) {
    const int64_t tie = c.c_tie[p];
#pragma unroll
    for (int k = 0; k < K; ++k) f[k] += (double)c.rho[tie * K + k];
  }
#pragma unroll
  for (int k = 0; k < K; ++k) f[k] = warp_sum(f[k]);
  if (lane == 0) {
#pragma unroll
    for (int k = 0; k < K; ++k) c.red3[lm * K + k] = f[k];
  }
}

// initial statistics (rho = pr_rho, model.py:602): delta = rho_u - onehot per special tie
template <int K>
__global__ void __launch_bounds__(256) k_init_delta(const __grid_constant__ vm_ctx c, double* part) {
  // same (layer, block, warp) decomposition as k_special, so that the partials land in the same slots
  const int l = blockIdx.y;
  const int nloc = (int)c.nloc, nct = (int)c.nct;
  const int u0 = c.utile_ptr[(int64_t)l * nloc * nct], u1 = c.utile_ptr[(int64_t)(l + 1) * nloc * nct];
  double p0[K];
#pragma unroll
  for (int k = 0; k < K; ++k) p0[k] = 0.0;
  for (int it = 0; it < VM_SPECIAL_TIES_PER_BLOCK / 256; ++it) {
    const int u = u0 + blockIdx.x * VM_SPECIAL_TIES_PER_BLOCK + it * 256 + threadIdx.x;
    const bool valid = u < u1;
    double d[K];
#pragma unroll
    for (int k = 0; k < K; ++k) d[k] = 0.0;
    int i = 0, j = 0, lrow = 0;
    double ti = 0.0, tj = 0.0;
    if (valid) {
      const double x0s = (double)c.u_x0sum[u];
#pragma unroll
      for (int k = 0; k < K; ++k) {
        const double r = c.rho_u[(size_t)u * K + k];
        d[k] = r - (k == 0 ? 1.0 : 0.0);
        c.delta_u[(size_t)u * K + k] = d[k];
        c.rho_u32[(size_t)u * K + k] = (float)r;
        p0[k] += r * x0s;
      }
      if (c.r_mode == VM_R_EGO) {
        lrow = c.u_lrow[u];
        i = lrow - l * nloc + (int)c.row0;
        j = c.u_col[u];
        // activity flags from the mask itself (the caches may not be final yet)
        ti = (i < (int)c.M && c.rep[(int64_t)l * c.M + i]) ? 1.0 : 0.0;
        tj = (j < (int)c.M && c.rep[(int64_t)l * c.M + j]) ? 1.0 : 0.0;
      }
    }
    if (c.r_mode == VM_R_EGO)
      vm_fix_accumulate<K>(reinterpret_cast<unsigned long long*>(c.fixA) + (int64_t)l * c.M * K, c.ego_diag != 0, valid,
                           lrow, i, j, ti, tj, d, 0);
  }
  const int64_t nup = c.L * c.n_ublk * 8, b = ((int64_t)l * c.n_ublk + blockIdx.x) * 8 + (threadIdx.x >> 5);
#pragma unroll
  for (int k = 0; k < K; ++k) {
    const double v = warp_sum(p0[k]);
    if ((threadIdx.x & 31) == 0) part[(UP_P0(K) + k) * nup + b] = v;
  }
}
// per-layer totals of delta_u, for the all-reporter initial statistics
__global__ void __launch_bounds__(256) k_init_delta_all(const __grid_constant__ vm_ctx c, double* upart) {
  __shared__ double sm[8];
  const int l = blockIdx.y;
  const int64_t u0 = c.utile_ptr[(int64_t)l * c.nloc * c.nct], u1 = c.utile_ptr[(int64_t)(l + 1) * c.nloc * c.nct];
  const int64_t nup = c.L * c.n_ublk * 8;
  for (int k = 0; k < (int)c.K; ++k) {
    double acc = 0.0;
    for (int r = 0; r < VM_SPECIAL_TIES_PER_BLOCK / 256; ++r) {
      const int64_t u = u0 + (int64_t)blockIdx.x * VM_SPECIAL_TIES_PER_BLOCK + r * 256 + threadIdx.x;
      if (u < u1) acc += c.delta_u[u * c.K + k];
    }
    const double v = block_sum<256>(acc, sm);
    if (threadIdx.x < 8)  // warp-partial layout of k_special: the block total goes to warp slot 0
      upart[(UP_DELTA + k) * nup + ((int64_t)l * c.n_ublk + blockIdx.x) * 8 + threadIdx.x] = threadIdx.x == 0 ? v : 0.0;
  }
}

// ELBO eta part: B = sum over X entries whose transposed position is reported of x * sum_k rho_k[transposed tie]
// (model.py:1269-1290); sum_k rho_k is 1 for a live tie and 0 for a fully-underflowed one (Q3).  The kernel sums
// the x of the DEAD positions (B = b_all - that); it exits at once when no tie can have underflowed.
template <int K>
__global__ void __launch_bounds__(256) k_elbo_b(const __grid_constant__ vm_ctx c, double* part) {
  __shared__ double sm[8];
  bool any = c.dev_flags[VM_FLAG_DEAD] != 0 || c.may_dead != 0;
  for (int l = 0; l < (int)c.L && !any; ++l) any = c.layer_consts[(int64_t)l * VM_LC_STRIDE(K) + VM_LC_DEAD(K)] != 0.0;
  if (!any) {
    if (threadIdx.x == 0) part[blockIdx.x] = 0.0;
    return;
  }
  double acc = 0.0;
  for (int64_t t = (int64_t)blockIdx.x * 256 + threadIdx.x; t < c.IT; t += (int64_t)gridDim.x * 256) {
    const int u = c.t_u[t];
    bool alive = true;
    if (u >= 0) {
      float s = 0.f;
#pragma unroll
      for (int k = 0; k < K; ++k) s += c.rho_u32[(int64_t)u * K + k];
      alive = s > 0.f;
    } else {
      const int64_t lrow = c.t_lrow[t];
      const int l = (int)(lrow / c.nloc);
      if (vm_may_dead<K>(c, l)) {
        float a[K], g[K], epsr;
        bool dead;
        vm_tie_logodds<K>(c, l, lrow, c.t_col[t], a);
        vm_formula_rho<K>(a, true, g, epsr, dead);
        alive = !dead;
      }
    }
    if (!alive) acc += (double)c.t_x[t];
  }
  const double v = block_sum<256>(acc, sm);
  if (threadIdx.x == 0) part[blockIdx.x] = v;
}

// second pass over the scalar partials, in two stages (one block cannot stream the ~1e5 per-warp partials fast enough):
// stage 1: grid (VM_S1_BLOCKS, L), block (bx, l) reduces its slice of layer l's per-warp partials of k_special /
// k_init_delta: nu, cat, t2 and p0[k] -> s1[((l*VM_S1_BLOCKS + bx)*(3+K)) + slot]
#define VM_S1_BLOCKS 64
#define VM_F_LISTED 256  // internal: this rho update ran the special-tie kernel in list mode (see launch_special)
__global__ void __launch_bounds__(256) k_sums_stage1(const __grid_constant__ vm_ctx c, int flags, const double* upart,
                                                     double* s1) {
  __shared__ double sm[8];
  const int l = blockIdx.y, K = (int)c.K;
  const bool elbo = flags & VM_F_ELBO, init = flags & VM_F_INIT;
  const int64_t nwl = c.n_ublk * 8, nup = c.L * nwl;
  // a layer whose special-tie kernel ran in list mode only wrote the partials of its first n_cxblk blocks
  const bool listed = (flags & VM_F_LISTED) && c.layer_consts[(int64_t)l * VM_LC_STRIDE(K) + VM_LC_SIMPLE(K)] != 0.0;
  const int64_t nuse = listed ? min(nwl, c.n_cxblk * 8) : nwl;
  const int64_t per = (nwl + VM_S1_BLOCKS - 1) / VM_S1_BLOCKS;
  const int64_t q0 = (int64_t)l * nwl + (int64_t)blockIdx.x * per, q1 = min(q0 + per, (int64_t)l * nwl + nuse);
  double* out = s1 + ((int64_t)l * VM_S1_BLOCKS + blockIdx.x) * (3 + K);
  for (int slot = 0; slot < 3 + K; ++slot) {
    const bool used = slot >= 3 ? true : (init ? false : (slot == UP_NU ? true : elbo));
    const int64_t src = slot >= 3 ? (UP_P0(K) + (slot - 3)) : slot;
    double v = 0.0;
    if (used)
      for (int64_t q = q0 + threadIdx.x; q < q1; q += 256) v += upart[src * nup + q];
    v = block_sum<256>(v, sm);
    if (threadIdx.x == 0) out[slot] = v;
  }
}

// stage 2: nu, cat, t2 (special-tie partials), cat (dense blocks), B, and phi0[l,k]
__global__ void __launch_bounds__(256) k_sums_reduce(const __grid_constant__ vm_ctx c, int flags, const double* s1,
                                                     const double* catpart, int64_t n_cat, const double* bpart,
                                                     int64_t n_b) {
  __shared__ double sm[8];
  const int K = (int)c.K, L = (int)c.L;
  const bool elbo = flags & VM_F_ELBO;
  double acc[3] = {0.0, 0.0, 0.0}, b = 0.0;
  for (int t = threadIdx.x; t < L * VM_S1_BLOCKS; t += 256) {
    acc[0] += s1[(int64_t)t * (3 + K) + UP_NU];
    acc[1] += s1[(int64_t)t * (3 + K) + UP_CAT];
    acc[2] += s1[(int64_t)t * (3 + K) + UP_T2];
  }
  if (elbo) {
    for (int64_t q = threadIdx.x; q < n_cat; q += 256) acc[1] += catpart[q];
    for (int64_t q = threadIdx.x; q < n_b; q += 256) b += bpart[q];
  }
  const double nu = block_sum<256>(acc[0], sm);
  const double cat = block_sum<256>(acc[1], sm);
  const double t2 = block_sum<256>(acc[2], sm);
  b = block_sum<256>(b, sm);
  if (threadIdx.x == 0) {
    double* ex = c.red3 + c.L * c.M * c.K;
    // + the SINGLE ties the shortcut kernel evaluated this iteration (0 on every other iteration)
    ex[VM_R3_NU] = nu + ((c.simple_mode && !(flags & VM_F_INIT)) ? (double)c.dev_flags[VM_FLAG_FIXNU] * (1.0 / VM_FIXP_SCALE) : 0.0);
    ex[VM_R3_CAT] = cat;
    ex[VM_R3_T2] = t2;
    ex[VM_R3_B] = elbo ? c.b_all - b : 0.0;
  }
  // phi0[l,k] = sum over this rank's special ties of layer l of rho_k * u_x0sum
  for (int l = 0; l < L; ++l)
    for (int k = 0; k < K; ++k) {
      double v = (threadIdx.x < VM_S1_BLOCKS) ? s1[((int64_t)l * VM_S1_BLOCKS + threadIdx.x) * (3 + K) + 3 + k] : 0.0;
      v = block_sum<256>(v, sm);
      if (threadIdx.x == 0) {
        // + the simple ties the shortcut kernel evaluated this iteration (0 on every other iteration)
        if (c.simple_mode && !(flags & VM_F_INIT)) v += (double)c.fixP[l * K + k] * (1.0 / VM_FIXP_SCALE);
        c.phi0[l * K + k] = v;
      }
    }
}

// =====================================================================================================
// phase finish
// =====================================================================================================
#define VM_EP_BLOCKS 64
// partial sums of the A-weighted Poisson-mean term and of the gamma ELBO terms of theta (model.py:957-965, 997-1002)
template <int K>
__global__ void __launch_bounds__(256) k_elbo_partial(const __grid_constant__ vm_ctx c, double* part) {
  __shared__ double sm[8];
  double t1 = 0.0, g = 0.0;
  const int64_t LM = c.L * c.M;
  for (int64_t lm = (int64_t)blockIdx.x * 256 + threadIdx.x; lm < LM; lm += (int64_t)gridDim.x * 256) {
    const int l = (int)(lm / c.M);
    double s = 0.0;
#pragma unroll
    for (int k = 0; k < K; ++k) s += c.E_lambda[l * K + k] * c.red3[lm * K + k];
    t1 += c.E_theta[lm] * s;
    g += vm_gamma_elbo_term(c.alpha_theta[lm], c.beta_theta[lm], c.gamma_shp[lm], c.gamma_rte[lm]);
  }
  t1 = block_sum<256>(t1, sm);
  g = block_sum<256>(g, sm);
  if (threadIdx.x == 0) {
    part[2 * blockIdx.x] = t1;
    part[2 * blockIdx.x + 1] = g;
  }
}

// `_update_nu` (model.py:820-830), nu part of the cache (model.py:684), and `__ELBO` assembly (model.py:948-1019).
__global__ void __launch_bounds__(256) k_finish(const __grid_constant__ vm_ctx c, int flags, const double* part,
                                                int n_part) {
  __shared__ double sm[8];
  const int64_t LMK = c.L * c.M * c.K;
  const double* ex = c.red3 + LMK;
  double t1 = 0.0, g = 0.0;
  if (flags & VM_F_ELBO)
    for (int q = threadIdx.x; q < n_part; q += 256) {
      t1 += part[2 * q];
      g += part[2 * q + 1];
    }
  t1 = block_sum<256>(t1, sm);
  g = block_sum<256>(g, sm);
  if (threadIdx.x != 0) return;
  double* nu = c.nu;
  if (c.mutuality && !(flags & VM_F_INIT)) nu[VM_NU_SHP] = c.alpha_eta + ex[VM_R3_NU];
  nu[VM_NU_G_STALE] = nu[VM_NU_G];
  nu[VM_NU_E] = nu[VM_NU_SHP] / nu[VM_NU_RTE];
  if (c.mutuality) nu[VM_NU_G] = exp(vm_digamma(nu[VM_NU_SHP]) - log(nu[VM_NU_RTE]));
  if (flags & VM_F_ELBO) {
    double gl = 0.0;
    for (int64_t t = 0; t < c.L * c.K; ++t)
      gl += vm_gamma_elbo_term(c.alpha_lambda[t], c.beta_lambda[t], c.phi_shp[t], c.phi_rte[t]);
    const double ge = vm_gamma_elbo_term(c.alpha_eta, c.beta_eta, nu[VM_NU_SHP], nu[VM_NU_RTE]);
    const double tb = c.mutuality ? nu[VM_NU_E] * ex[VM_R3_B] : 0.0;
    double* o = c.elbo_out;
    o[1] = -t1;
    o[2] = -tb;
    o[3] = ex[VM_R3_T2];
    o[4] = g;
    o[5] = gl;
    o[6] = ge;
    o[7] = ex[VM_R3_CAT];
    o[0] = -t1 - tb + ex[VM_R3_T2] + g + gl + ge + ex[VM_R3_CAT];
  }
}

// =====================================================================================================
// posterior consumers / utilities
// =====================================================================================================
__global__ void k_fill_onehot(float* rho, int64_t T, int K) {
  for (int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; t < T * K; t += (int64_t)gridDim.x * blockDim.x)
    rho[t] = (t % K == 0) ? 1.f : 0.f;
}
__global__ void k_patch_special(const __grid_constant__ vm_ctx c) {
  const int64_t u = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (u >= c.U) return;
  float* dst = c.rho + ((int64_t)c.u_lrow[u] * c.N + c.u_col[u]) * c.K;
  for (int k = 0; k < (int)c.K; ++k) dst[k] = (float)c.rho_u[u * c.K + k];
}
// rho_max (model.py:1148-1149): argmax_k r[k], the first maximum wins (mode 0) / fixed threshold on rho[...,1]
// (model.py:1155-1166, utils.py:207-217, mode 1).  Shared by the dense (k_infer) and the sparse (k_edges) consumers.
__device__ __forceinline__ int vm_infer_label(const float* r, int K, int mode, float thr) {
  if (mode == 0) {
    int best = 0;
    float bv = r[0];
    for (int k = 1; k < K; ++k)
      if (r[k] > bv) {
        bv = r[k];
        best = k;
      }
    return best;
  }
  return r[1] >= thr ? 1 : 0;
}
__global__ void k_infer(const float* rho, int64_t T, int K, int mode, float thr, uint8_t* out) {
  for (int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; t < T; t += (int64_t)gridDim.x * blockDim.x)
    out[t] = (uint8_t)vm_infer_label(rho + t * K, K, mode, thr);
}

// ---- sparse consumers (vm_edges_count / vm_edges_emit) ----------------------------------------------------------------
// qmax[l*K+k] = max_j tab_q[l,j,k], one CTA per (k, l); NaN when the layer has a NaN entry (then no row of it is skipped:
// every comparison with NaN is false).
__global__ void __launch_bounds__(256) k_edges_qmax(const float* __restrict__ tab_q, int64_t N, int K, float* qmax) {
  __shared__ float sm[8];
  const int k = blockIdx.x, l = blockIdx.y;
  float m = -INFINITY;
  bool nan = false;
  for (int64_t j = threadIdx.x; j < N; j += blockDim.x) {
    const float v = tab_q[((int64_t)l * N + j) * K + k];
    m = fmaxf(m, v);
    nan |= v != v;
  }
  nan = __syncthreads_or(nan);
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) m = fmaxf(m, __shfl_down_sync(0xffffffffu, m, o));
  if ((threadIdx.x & 31) == 0) sm[threadIdx.x >> 5] = m;
  __syncthreads();
  if (threadIdx.x == 0) {
    for (int w = 1; w < 8; ++w) m = fmaxf(m, sm[w]);
    qmax[l * K + k] = nan ? __int_as_float(0x7fc00000) : m;
  }
}

// Can no tie of this row's closed form have a nonzero label?  With a_k = fl(p_k + q_k) for the tie's column and the layer's
// column maximum qmax_k >= q_k, rounding is monotone: a_k <= fl(p_k + qmax_k) =: b_k.  Then (vm_formula_rho: r_k =
// ex2(a_k), s = sum r_k, inv = rcp(1+s), out = (inv, r_k*inv); ex2/rcp.approx are within 2 ulp, far inside the margins):
//  ARGMAX:    b_k < -1 for every k >= 1 gives r_k < 1/2 (1+2^-21) < 1, so out_k = fl(r_k*inv) <= fl(inv) = out_0: never
//             strictly greater, the label stays 0.  A dead tie (all zeros) is label 0 too.
//  THRESHOLD: thr > 0 and b_1 < log2(thr) - 1 gives r_1 < thr/2 (1+2^-21) and inv <= 1 (1+2^-23), so out_1 < thr.  A dead
//             tie is 0 < thr.
//  SAMPLE:    b_k < -30 for every k >= 1 gives r_k < 2^-30 (1+2^-21), out_k < 2^-29.9 inv: K-1 <= 31 such terms are each
//             below half an ulp of inv (inv >= 1/2 since s < 2^-25), so the fp32 sum of vm_sample_label equals p[0] = inv > 0
//             and every draw lands in category 0 (see there).  Only when the layer cannot be dead: a dead tie sums to 0 and
//             goes to the LAST category, an edge.
template <int K>
__device__ __forceinline__ bool vm_edges_row_skip(const float* p, const float* qmax, int what, float thr, float thr_bound,
                                                  bool may_dead) {
  if (what == VM_EDGES_THRESHOLD) return thr > 0.f && __fadd_rn(p[1], qmax[1]) < thr_bound;
  if (what == VM_EDGES_SAMPLE && may_dead) return false;
  const float bound = what == VM_EDGES_ARGMAX ? -1.f : -30.f;
  bool s = true;
#pragma unroll
  for (int k = 1; k < K; ++k) s = s && __fadd_rn(p[k], qmax[k]) < bound;
  return s;
}

template <int K>
__device__ __forceinline__ int vm_edge_label(const float* o, int what, float thr, int64_t n_trials, uint64_t gt, uint2 key) {
  if (what == VM_EDGES_SAMPLE) return vm_sample_label(o, K, n_trials, gt, key);
  return vm_infer_label(o, K, what, thr);  // VM_EDGES_ARGMAX / _THRESHOLD = vm_infer's modes 0 / 1
}

// One step of 256 ties (one per thread, in order): the block-wide exclusive prefix of (label != 0) places this thread's
// edge; returns the row's running count.  Every thread of the block calls it.
__device__ __forceinline__ int64_t vm_edges_put(int lab, int64_t key, int64_t pos, bool emit, const vm_edges_args& a,
                                                int* s_warp) {
  const bool pred = lab != 0;
  const unsigned b = __ballot_sync(0xffffffffu, pred);
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  if (lane == 0) s_warp[w] = __popc(b);
  __syncthreads();
  int off = __popc(b & ((1u << lane) - 1u)), tot = 0;
#pragma unroll
  for (int q = 0; q < 8; ++q) {
    const int v = s_warp[q];
    off += q < w ? v : 0;
    tot += v;
  }
  __syncthreads();
  if (emit && pred) {
    a.o_key[pos + off] = key;
    a.o_val[pos + off] = (uint8_t)lab;
  }
  return pos + tot;
}

// Count (emit = 0) or write (emit = 1) the edges of the local rows, one CTA of 256 threads per row (rows strided over the
// grid), columns in chunks of 256.  Implicit source: the closed form of vm_materialize_rows, and the row's special ties
// (utile_ptr[lrow*nct] .. utile_ptr[(lrow+1)*nct], ascending in column) from rho_u32, found chunk by chunk by a moving
// pointer -- at most 256 of them fall into a chunk of 256 columns; a row that vm_edges_row_skip rules out only walks its
// special ties.  Slab source: ctx->rho.
template <int K>
__global__ void __launch_bounds__(256) k_edges(const __grid_constant__ vm_ctx c, const __grid_constant__ vm_edges_args a,
                                               int emit, float thr, float thr_bound) {
  __shared__ int s_u[256];
  __shared__ int s_warp[8];
  const int N = (int)c.N, tid = threadIdx.x, what = (int)a.what;
  const bool implicit = a.source == VM_EDGES_IMPLICIT;
  const uint2 key = make_uint2((uint32_t)a.seed, (uint32_t)(a.seed >> 32));
  const int64_t rows = c.L * c.nloc;
  for (int64_t lrow = blockIdx.x; lrow < rows; lrow += gridDim.x) {
    const int l = (int)(lrow / c.nloc);
    const int64_t g0 = ((int64_t)l * N + (lrow - (int64_t)l * c.nloc + c.row0)) * N;  // global id of the row's column 0
    int64_t pos = emit ? a.row_off[lrow] : 0;
    int us = 0, ue = 0;
    bool may_dead = false, skip = false;
    if (implicit) {
      us = c.utile_ptr[lrow * c.nct];
      ue = c.utile_ptr[(lrow + 1) * c.nct];
      may_dead = vm_may_dead<K>(c, l);
      skip = vm_edges_row_skip<K>(c.tab_p + lrow * K, a.workspace + (int64_t)l * K, what, thr, thr_bound, may_dead);
    }
    if (skip) {
      for (int u0 = us; u0 < ue; u0 += 256) {
        const int u = u0 + tid;
        int lab = 0, col = 0;
        if (u < ue) {
          float o[K];
          col = c.u_col[u];
#pragma unroll
          for (int k = 0; k < K; ++k) o[k] = c.rho_u32[(int64_t)u * K + k];
          lab = vm_edge_label<K>(o, what, thr, a.n_trials, (uint64_t)(g0 + col), key);
        }
        pos = vm_edges_put(lab, g0 + col, pos, emit, a, s_warp);
      }
    } else {
      int up = us;
      for (int j0 = 0; j0 < N; j0 += 256) {
        const int j = j0 + tid;
        int su = -1;
        if (implicit) {
          s_u[tid] = -1;
          __syncthreads();
          const int u = up + tid;
          const bool in = u < ue && c.u_col[u] < j0 + 256;
          if (in) s_u[c.u_col[u] - j0] = u;
          up += __syncthreads_count(in);
          su = s_u[tid];
        }
        int lab = 0;
        if (j < N) {
          float o[K];
          if (!implicit) {
#pragma unroll
            for (int k = 0; k < K; ++k) o[k] = c.rho[(lrow * N + j) * K + k];
          } else if (su >= 0) {
#pragma unroll
            for (int k = 0; k < K; ++k) o[k] = c.rho_u32[(int64_t)su * K + k];
          } else {
            float lo[K], epsr;
            bool dead;
            vm_tie_logodds<K>(c, l, lrow, j, lo);
            vm_formula_rho<K>(lo, may_dead, o, epsr, dead);
          }
          lab = vm_edge_label<K>(o, what, thr, a.n_trials, (uint64_t)(g0 + j), key);
        }
        pos = vm_edges_put(lab, g0 + j, pos, emit, a, s_warp);
      }
    }
    if (!emit && tid == 0) a.row_count[lrow] = pos;
  }
}
// The posterior the last rho update left, for the local rows [lrow0, lrow0+nrows) (lrow = l*nloc + i), into `out` in the
// slab's layout -- bit for bit what a storing iteration writes: the closed form from the row/column tables with the
// layer's dead-row switch (the dense kernels' arithmetic), then the special ties of each row segment overwritten from
// rho_u32.  One CTA per (row, column tile), rows strided over gridDim.y; store-bound.
template <int K>
__global__ void __launch_bounds__(256) k_materialize_rows(const __grid_constant__ vm_ctx c, int64_t lrow0, int64_t nrows,
                                                          float* out) {
  const int ct = blockIdx.x, N = (int)c.N;
  const int j0 = ct * (int)c.tile_w, j1 = min(j0 + (int)c.tile_w, N);
  for (int64_t r = blockIdx.y; r < nrows; r += gridDim.y) {
    const int64_t lrow = lrow0 + r;
    const int l = (int)(lrow / c.nloc);
    const bool may_dead = vm_may_dead<K>(c, l);
    float* dst = out + r * N * K;
    for (int j = j0 + (int)threadIdx.x; j < j1; j += blockDim.x) {
      float a[K], o[K], epsr;
      bool dead;
      vm_tie_logodds<K>(c, l, lrow, j, a);
      vm_formula_rho<K>(a, may_dead, o, epsr, dead);
#pragma unroll
      for (int k = 0; k < K; ++k) dst[(int64_t)j * K + k] = o[k];
    }
    __syncthreads();
    const int64_t seg = lrow * c.nct + ct;
    for (int64_t u = c.utile_ptr[seg] + threadIdx.x; u < c.utile_ptr[seg + 1]; u += blockDim.x) {
      const int col = c.u_col[u];
#pragma unroll
      for (int k = 0; k < K; ++k) dst[(int64_t)col * K + k] = c.rho_u32[u * K + k];
    }
    __syncthreads();
  }
}

// The posterior at given ties (vm_rho_at): one thread per query, grid-stride.  key[q] = (l*N+i)*N+j; a key outside
// [0, L*N*N) or outside this rank's rows [row0, row0+nloc) is skipped and out[q*K..] is not written.  Implicit source: the
// special ties of the tie's (row, column tile) segment are sorted by column (at most tile_w of them): a binary search
// finds the tie there (rho_u32), else the closed form of k_materialize_rows -- the same bits.  Slab source: ctx->rho.
template <int K>
__global__ void __launch_bounds__(256) k_rho_at(const __grid_constant__ vm_ctx c, int implicit, int64_t n,
                                                const int64_t* __restrict__ key, float* __restrict__ out) {
  const int64_t N = c.N, T = c.L * N * N;
  for (int64_t q = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; q < n; q += (int64_t)gridDim.x * blockDim.x) {
    const int64_t g = key[q];
    if (g < 0 || g >= T) continue;
    const int64_t li = g / N, j = g - li * N, l = li / N, i = li - l * N;
    if (i < c.row0 || i >= c.row0 + c.nloc) continue;
    const int64_t lrow = l * c.nloc + i - c.row0;
    float o[K];
    if (!implicit) {
#pragma unroll
      for (int k = 0; k < K; ++k) o[k] = c.rho[(lrow * N + j) * K + k];
    } else {
      const int64_t seg = lrow * c.nct + j / c.tile_w;
      // 64-bit: the indices reach U < 2^31, where lo + hi would overflow an int
      const int64_t end = c.utile_ptr[seg + 1];
      int64_t lo = c.utile_ptr[seg], hi = end;
      while (lo < hi) {
        const int64_t mid = (lo + hi) >> 1;
        if (c.u_col[mid] < j) lo = mid + 1;
        else hi = mid;
      }
      if (lo < end && c.u_col[lo] == j) {
#pragma unroll
        for (int k = 0; k < K; ++k) o[k] = c.rho_u32[lo * K + k];
      } else {
        float a[K], epsr;
        bool dead;
        vm_tie_logodds<K>(c, (int)l, lrow, (int)j, a);
        vm_formula_rho<K>(a, vm_may_dead<K>(c, (int)l), o, epsr, dead);
      }
    }
#pragma unroll
    for (int k = 0; k < K; ++k) out[q * K + k] = o[k];
  }
}

// =====================================================================================================
// host-side launchers
// =====================================================================================================
static inline int64_t cdiv(int64_t a, int64_t b) { return (a + b - 1) / b; }
static inline int64_t imin64(int64_t a, int64_t b) { return a < b ? a : b; }

// blkpart regions (doubles)
static inline double* region_u(const vm_ctx* c) { return c->blkpart; }  // special-tie block partials
static inline int64_t n_upart(const vm_ctx* c) { return c->L * c->n_ublk * 8; }  // one partial per warp
static inline double* region_cat(const vm_ctx* c) { return c->blkpart + n_upart(c) * UP_SLOTS(c->K); }
static inline int64_t n_catpart(const vm_ctx* c) { return c->nct * c->L * c->nrt; }
static inline double* region_b(const vm_ctx* c) { return region_cat(c) + n_catpart(c); }
#define VM_B_BLOCKS 128
static inline double* region_ep(const vm_ctx* c) { return region_b(c) + VM_B_BLOCKS; }
static inline double* region_s1(const vm_ctx* c) { return region_ep(c) + 2 * VM_EP_BLOCKS; }  // L*VM_S1_BLOCKS*(3+K)

// an entry point that writes or reads the dense slab needs one: only VM_F_NO_STORE iterations run without (vm_ctx.rho =
// NULL), and not under the general mask, whose statistics gather the slab
static int slab_check(const vm_ctx* c, int flags) {
  if (!(flags & VM_F_NO_STORE)) return c->rho != nullptr ? 0 : VM_EINVAL;
  return c->r_mode == VM_R_CSR ? VM_ENOTSUP : 0;
}

static int check_ctx(const vm_ctx* c) {
  if (!c) return VM_EINVAL;
  if (c->K < 2 || c->K > VM_MAX_K) return VM_EINVAL;
  if (c->tile_w != vm_dense_tile_w_host(c->K) || c->tile_h < 1) return VM_EINVAL;
  if (c->nct != cdiv(c->N, c->tile_w) || c->nrt != cdiv(c->nloc, c->tile_h)) return VM_EINVAL;
  if (c->r_mode < 0 || c->r_mode > 2) return VM_EINVAL;
  if (c->L * c->nrt > 65535 || c->L > 65535) return VM_EINVAL;
  return 0;
}

#define VM_CASE(k, ...)        \
  case k: {                    \
    constexpr int K = k;       \
    __VA_ARGS__;               \
  } break;
#define DISPATCH_K(KV, ...)                       \
  switch (KV) {                                   \
    VM_DISPATCH_CASES(VM_CASE, __VA_ARGS__)       \
    default:                                      \
      return VM_EINVAL;                           \
  }

// does this rho update use the fast dense kernel (for the tiles that qualify on the device)?
template <int K>
static bool dense_fast_eligible(const vm_ctx* c) {
  return K <= 4 && c->r_mode != VM_R_CSR && ((c->N * K) & 3) == 0 && c->N >= c->tile_w &&
         c->tile_h <= VM_FAST_MAX_TILE_H;
}
// ... and do the fast dense kernel / the list mode of the special-tie kernel handle the simple special ties in it?
template <int K>
static bool simple_iteration(const vm_ctx* c, int flags) {
  return c->simple_mode != 0 && c->r_mode == VM_R_EGO && !(flags & VM_F_ELBO) && dense_fast_eligible<K>(c);
}

// dynamic shared memory of the TMA dense kernels (opt-in above 48 KB)
template <int K>
static cudaError_t fast_setup_all() {
  if constexpr (K <= 4) {  // the TMA kernels are only instantiated (and eligible) for K <= 4
    cudaError_t e;
    if ((e = cudaFuncSetAttribute(k_dense_tma<K, false>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                  (int)sizeof(TmaSmem<K>))) != cudaSuccess) return e;
    if ((e = cudaFuncSetAttribute(k_dense_tma<K, true>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                  (int)sizeof(TmaSmem<K>))) != cudaSuccess) return e;
    return cudaFuncSetAttribute(k_dense_sc<K>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(TmaSmem<K, true>));
  } else {
    return cudaSuccess;
  }
}

// the special-tie kernel in list mode, on the iterations whose shortcut ties k_dense_sc evaluates: LIST = 1 walks the list
// of the other special ties of the layers that take the shortcut (its grid covers that list only; k_sums_stage1 reads as
// many partial slots), LIST = 2 has every special tie of the layers that cannot
template <int K>
static void launch_listed(const vm_ctx* c, cudaStream_t s) {
  if constexpr (K <= 4) {  // (simple_iteration is never true for larger K)
    if (c->n_ublk <= 0) return;
    const dim3 gridl((unsigned)(c->n_cxblk > 0 ? c->n_cxblk : 1), (unsigned)c->L);
    k_special<K, false, VM_R_EGO, 1><<<gridl, 256, 0, s>>>(*c, region_u(c));
    const dim3 grid2((unsigned)imin64(c->n_ublk, 148 * 2), (unsigned)c->L);
    k_special<K, false, VM_R_EGO, 2><<<grid2, 256, 0, s>>>(*c, region_u(c));
  }
}

// the TMA dense kernel of one rho update: k_dense_sc on the iterations whose shortcut ties it evaluates (`sc`), else
// k_dense_tma.  STORE = false (VM_F_NO_STORE): their statistics-only variants, which need no shared-memory opt-in.
template <int K, bool STORE>
static void launch_tma(const vm_ctx* c, bool sc, bool elbo, dim3 grid, cudaStream_t st, int rt0, int rtn) {
  if constexpr (K <= 4) {
    static_assert(sizeof(TmaSmem<K, true, false>) <= 48 * 1024, "no opt-in for the statistics-only kernels");
    constexpr size_t smem = sizeof(TmaSmem<K, false, STORE>), smem_sc = sizeof(TmaSmem<K, true, STORE>);
    double* cp = region_cat(c);
    if (sc) k_dense_sc<K, 1, STORE><<<grid, VM_DENSE_THREADS, smem_sc, st>>>(*c, rt0, rtn);
    else if (elbo) k_dense_tma<K, true, VM_TMA_PD, STORE><<<grid, VM_DENSE_THREADS, smem, st>>>(*c, cp, rt0, rtn);
    else k_dense_tma<K, false, VM_TMA_PD, STORE><<<grid, VM_DENSE_THREADS, smem, st>>>(*c, cp, rt0, rtn);
  }
}

// `sums_flags` >= 0: the scalar-sum kernels that only depend on the special-tie kernels (k_elbo_b, k_sums_stage1) also go
// to the aux stream, under the dense kernel; *sums_done tells the caller whether they were launched here.
// `sc` (simple_iteration): the dense kernel is k_dense_sc, and the list-mode special-tie kernels are launched here, on the
// aux stream ahead of the sums and the partial tiles, so that they run under it; k_patch_rest follows the join when the
// iteration stores the slab.
template <int K>
static int launch_dense(const vm_ctx* c, int flags, cudaStream_t st, int rt0, int rtn, int sums_flags = -1,
                        bool* sums_done = nullptr, bool sc = false) {
  if (sums_done) *sums_done = false;
  if (rtn <= 0) return 0;
  const dim3 grid((unsigned)c->nct, (unsigned)(c->L * rtn));
  const bool elbo = flags & VM_F_ELBO, store = !(flags & VM_F_NO_STORE), csr = c->r_mode == VM_R_CSR;
  double* cp = region_cat(c);
  const bool fast = dense_fast_eligible<K>(c);
  if (fast) {
    const cudaError_t e = fast_setup_all<K>();
    if (e != cudaSuccess) return (int)e;
  }
  // The general kernel only has the tiles the fast one leaves (the partial last column tile: 157 of 6280 CTAs at config 3,
  // each a serial sweep of its rows, 32 us): it goes to the caller's aux stream, forked from and joined back into `st`,
  // so that it runs under the fast kernel instead of after it.  The two write disjoint tiles and disjoint partial slots.
  // The fork/join events are the caller's (vm_ctx.ev_fork / ev_join, created once per engine); without them a pair is
  // created and destroyed here.
  cudaStream_t aux = (cudaStream_t)c->aux_stream;
  const bool side = fast && aux != nullptr && aux != st;
  cudaStream_t sg = side ? aux : st;
  cudaEvent_t ev_fork = (cudaEvent_t)c->ev_fork, ev_join = (cudaEvent_t)c->ev_join;
  bool own_events = false;
  if (side && (ev_fork == nullptr || ev_join == nullptr)) {
    ev_fork = ev_join = nullptr;
    if (cudaEventCreateWithFlags(&ev_fork, cudaEventDisableTiming) != cudaSuccess ||
        cudaEventCreateWithFlags(&ev_join, cudaEventDisableTiming) != cudaSuccess) {
      const cudaError_t e = cudaGetLastError();
      if (ev_fork) cudaEventDestroy(ev_fork);
      return (int)e;
    }
    own_events = true;
  }
  if (side) {
    cudaEventRecord(ev_fork, st);
    cudaStreamWaitEvent(aux, ev_fork, 0);
    if (sc) launch_listed<K>(c, aux);
    if (sums_flags >= 0) {
      if ((flags & VM_F_ELBO) && c->mutuality) k_elbo_b<K><<<VM_B_BLOCKS, 256, 0, aux>>>(*c, region_b(c));
      k_sums_stage1<<<dim3(VM_S1_BLOCKS, (unsigned)c->L), 256, 0, aux>>>(*c, sums_flags, region_u(c), region_s1(c));
      if (sums_done) *sums_done = true;
    }
  } else if (sc) {
    launch_listed<K>(c, st);
  }
  const auto launch_fast = [&] {
    if (store) launch_tma<K, true>(c, sc, elbo, grid, st, rt0, rtn);
    else launch_tma<K, false>(c, sc, elbo, grid, st, rt0, rtn);
  };
  if (fast && !side) launch_fast();
#define LD(E, S, C) k_dense<K, E, S, C><<<grid, VM_DENSE_THREADS, 0, sg>>>(*c, cp, fast ? 1 : 0, rt0, rtn)
  if (csr) {  // always stores (slab_check)
    if (elbo) LD(true, true, true); else LD(false, true, true);
  } else if (elbo) {
    if (store) LD(true, true, false); else LD(true, false, false);
  } else {
    if (store) LD(false, true, false); else LD(false, false, false);
  }
#undef LD
  if (side) {
    launch_fast();
    cudaEventRecord(ev_join, aux);
    cudaStreamWaitEvent(st, ev_join, 0);
    if (own_events) {
      cudaEventDestroy(ev_fork);  // destruction is deferred by the runtime until the events have completed
      cudaEventDestroy(ev_join);
    }
  }
  if constexpr (K <= 4) {
    if (sc && store && c->n_ublk > 0) {
      const dim3 gridp((unsigned)imin64(c->n_ublk * (VM_SPECIAL_TIES_PER_BLOCK / 256), 148 * 8), (unsigned)c->L);
      k_patch_rest<K><<<gridp, 256, 0, st>>>(*c);
    }
  }
  return 0;
}

template <int K>
static int launch_special(const vm_ctx* c, int flags, cudaStream_t st) {
  const int64_t gridx = c->n_ublk;
  if (gridx <= 0) return 0;
  const dim3 grid((unsigned)gridx, (unsigned)c->L);
  const bool elbo = flags & VM_F_ELBO;
#define LS(E, M) k_special<K, E, M><<<grid, 256, 0, st>>>(*c, region_u(c))
  if (c->r_mode == VM_R_EGO) {
    if (elbo) LS(true, VM_R_EGO); else LS(false, VM_R_EGO);
  } else if (c->r_mode == VM_R_ALL && c->all32_mode != 0 && !elbo) {
    // layers whose guard holds: every special tie in fp32, entry-parallel; the others: the fp64 kernel (strided grid)
    const size_t smb = vm_all32_smem_bytes<K>(c->M);
    k_all32<K><<<grid, 256, smb, st>>>(*c, region_u(c));
    const dim3 grid2((unsigned)imin64(gridx, 148 * 2), (unsigned)c->L);
    k_special<K, false, VM_R_ALL, 2><<<grid2, 256, 0, st>>>(*c, region_u(c));
  } else if (c->r_mode == VM_R_ALL) {
    if (elbo) LS(true, VM_R_ALL); else LS(false, VM_R_ALL);
  } else {
    if (elbo) LS(true, VM_R_CSR); else LS(false, VM_R_CSR);
  }
#undef LS
  return 0;
}

// special-tie kernels, then the dense kernel, of one rho update.  On iterations whose shortcut ties the dense kernel
// evaluates (simple_iteration), the list-mode special-tie kernels run next to it instead, on the aux stream (launch_dense).
// (Running an unpatched dense kernel next to a separate shortcut kernel was measured in round 2 and lost: each wants the
// registers and warp slots the other holds, profiles/r2_dense_experiments.txt.)
template <int K>
static int launch_rho_kernels(const vm_ctx* c, int flags, cudaStream_t st, bool* sums_done) {
  const bool sc = simple_iteration<K>(c, flags);
  int rc;
  if (!sc && (rc = launch_special<K>(c, flags, st))) return rc;
  return launch_dense<K>(c, flags, st, 0, (int)c->nrt, flags | (sc ? VM_F_LISTED : 0), sums_done, sc);
}

template <int K>
static int launch_stats(const vm_ctx* c, int init, cudaStream_t st) {
  const int64_t LM = c->L * c->M;
  if (c->r_mode == VM_R_EGO) {
    if (!init) k_col_reduce<K><<<(unsigned)cdiv(LM * K, 256), 256, 0, st>>>(*c);
    k_stats_ego<K><<<(unsigned)cdiv(LM, 8), 256, 0, st>>>(*c, init);
  } else if (c->r_mode == VM_R_ALL) {
    k_stats_all<K><<<(unsigned)c->L, 1024, 0, st>>>(*c, init, region_u(c));
  } else {
    k_stats_csc<K><<<(unsigned)cdiv(LM, 8), 256, 0, st>>>(*c, init);
  }
  return 0;
}


static int tu_materialize_prior(const vm_ctx* c, void* stream) {
  int rc = check_ctx(c);
  if (rc) return rc;
  if ((rc = slab_check(c, 0))) return rc;
  cudaStream_t st = (cudaStream_t)stream;
  const int64_t T = c->L * c->nloc * c->N;
  k_fill_onehot<<<(unsigned)imin64(cdiv(T * c->K, 256), 148 * 16), 256, 0, st>>>(c->rho, T, (int)c->K);
  VM_CHECK_LAUNCH();
  if (c->U > 0) k_patch_special<<<(unsigned)cdiv(c->U, 256), 256, 0, st>>>(*c);
  VM_CHECK_LAUNCH();
  return 0;
}

static int tu_refresh_cache(const vm_ctx* c, void* stream) {
  int rc = check_ctx(c);
  if (rc) return rc;
  const int64_t n = c->L * (c->M > c->K ? c->M : c->K);
  k_refresh_cache<<<(unsigned)cdiv(n, 256), 256, 0, (cudaStream_t)stream>>>(*c);
  VM_CHECK_LAUNCH();
  return 0;
}

static int tu_init_stats(const vm_ctx* c, void* stream) {
  int rc = check_ctx(c);
  if (rc) return rc;
  cudaStream_t st = (cudaStream_t)stream;
  {  // function attributes are set here, outside any stream capture
    cudaError_t e = cudaSuccess;
    DISPATCH_K(c->K, e = fast_setup_all<K>());
    if (e != cudaSuccess) return (int)e;
    if (c->all32_mode) {
      DISPATCH_K(c->K, e = cudaFuncSetAttribute(k_all32<K>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                                (int)vm_all32_smem_bytes<K>(c->M)));
      if (e != cudaSuccess) return (int)e;
    }
  }
  if (c->r_mode == VM_R_EGO) {
    cudaMemsetAsync(c->fixA, 0, (size_t)(c->L * c->M * c->K) * sizeof(int64_t), st);
    VM_CHECK_LAUNCH();
  }
  cudaMemsetAsync(c->fixG, 0, (size_t)(c->L * c->M) * sizeof(int64_t), st);
  VM_CHECK_LAUNCH();
  DISPATCH_K(c->K, (k_init_delta<K><<<dim3((unsigned)c->n_ublk, (unsigned)c->L), 256, 0, st>>>(*c, region_u(c))));
  VM_CHECK_LAUNCH();
  if (c->r_mode == VM_R_ALL) {
    k_init_delta_all<<<dim3((unsigned)c->n_ublk, (unsigned)c->L), 256, 0, st>>>(*c, region_u(c));
    VM_CHECK_LAUNCH();
  }
  if (c->r_mode == VM_R_CSR) {  // gather needs the slab
    rc = tu_materialize_prior(c, stream);
    if (rc) return rc;
  }
  DISPATCH_K(c->K, launch_stats<K>(c, 1, st));
  VM_CHECK_LAUNCH();
  // scalar sums = 0, phi0 from the prior
  k_sums_stage1<<<dim3(VM_S1_BLOCKS, (unsigned)c->L), 256, 0, st>>>(*c, VM_F_INIT, region_u(c), region_s1(c));
  VM_CHECK_LAUNCH();
  k_sums_reduce<<<1, 256, 0, st>>>(*c, VM_F_INIT, region_s1(c), nullptr, 0, nullptr, 0);
  VM_CHECK_LAUNCH();
  return 0;
}

static int tu_phase_gamma(const vm_ctx* c, void* stream) {
  int rc = check_ctx(c);
  if (rc) return rc;
  cudaStream_t st = (cudaStream_t)stream;
  if (c->gamma_ts) {  // tie-sorted pass (few reporters)
    const size_t smb = (size_t)c->M * sizeof(double) + (size_t)8 * c->M * 3 * sizeof(unsigned int);
    DISPATCH_K(c->K, (k_gamma_partial_ts<K><<<dim3((unsigned)c->n_phichunk, (unsigned)c->L), 256, smb, st>>>(*c, c->blkpart)));
    VM_CHECK_LAUNCH();
    k_gamma_reduce_ts<<<(unsigned)cdiv(c->L * c->M, 8), 256, 0, st>>>(*c, c->blkpart);
    VM_CHECK_LAUNCH();
    return 0;
  }
  if (c->n_gchunk > 0) {
    DISPATCH_K(c->K, (k_gamma_partial<K><<<(unsigned)cdiv(c->n_gchunk, 8), 256, 0, st>>>(*c, c->blkpart)));
    VM_CHECK_LAUNCH();
  }
  k_gamma_reduce<<<(unsigned)cdiv(c->L * c->M, 8), 256, 0, st>>>(*c, c->blkpart);
  VM_CHECK_LAUNCH();
  return 0;
}

static int tu_phase_phi(const vm_ctx* c, void* stream) {
  int rc = check_ctx(c);
  if (rc) return rc;
  cudaStream_t st = (cudaStream_t)stream;
  DISPATCH_K(c->K, (k_gamma_finish<K><<<dim3((unsigned)cdiv(c->M, VM_GF_THREADS), (unsigned)c->L), VM_GF_THREADS, 0, st>>>(*c)));
  VM_CHECK_LAUNCH();
  DISPATCH_K(c->K, (k_phi_partial<K><<<dim3((unsigned)c->n_phichunk, (unsigned)c->L), 256, 0, st>>>(*c, c->blkpart)));
  VM_CHECK_LAUNCH();
  DISPATCH_K(c->K, (k_phi_reduce<K><<<(unsigned)c->L, 256, 0, st>>>(*c, c->blkpart)));
  VM_CHECK_LAUNCH();
  return 0;
}

static int tu_phase_rho(const vm_ctx* c, int flags, void* stream) {
  int rc = check_ctx(c);
  if (rc) return rc;
  if ((rc = slab_check(c, flags))) return rc;
  cudaStream_t st = (cudaStream_t)stream;
  DISPATCH_K(c->K, (k_phi_finish<K><<<(unsigned)c->L, 256, 0, st>>>(*c)));
  VM_CHECK_LAUNCH();
  if (c->r_mode != VM_R_CSR) {
    DISPATCH_K(c->K, (k_tables<K><<<(unsigned)cdiv(c->L * c->N, 256), 256, 0, st>>>(*c)));
    VM_CHECK_LAUNCH();
  }
  bool sums_done = false;
  DISPATCH_K(c->K, rc = launch_rho_kernels<K>(c, flags, st, &sums_done));
  if (rc) return rc;
  VM_CHECK_LAUNCH();
  DISPATCH_K(c->K, launch_stats<K>(c, 0, st));
  VM_CHECK_LAUNCH();
  if (!sums_done) {
    if ((flags & VM_F_ELBO) && c->mutuality) {
      DISPATCH_K(c->K, (k_elbo_b<K><<<VM_B_BLOCKS, 256, 0, st>>>(*c, region_b(c))));
      VM_CHECK_LAUNCH();
    }
    bool listed = false;
    DISPATCH_K(c->K, listed = simple_iteration<K>(c, flags));
    k_sums_stage1<<<dim3(VM_S1_BLOCKS, (unsigned)c->L), 256, 0, st>>>(*c, flags | (listed ? VM_F_LISTED : 0), region_u(c),
                                                                      region_s1(c));
    VM_CHECK_LAUNCH();
  }
  k_sums_reduce<<<1, 256, 0, st>>>(*c, flags, region_s1(c), region_cat(c), n_catpart(c), region_b(c),
                                   c->mutuality ? VM_B_BLOCKS : 0);
  VM_CHECK_LAUNCH();
  return 0;
}

static int tu_dense_only(const vm_ctx* c, int flags, void* stream) {
  int rc = check_ctx(c);
  if (rc) return rc;
  if ((rc = slab_check(c, flags))) return rc;
  DISPATCH_K(c->K, rc = launch_dense<K>(c, flags, (cudaStream_t)stream, 0, (int)c->nrt));
  if (rc) return rc;
  VM_CHECK_LAUNCH();
  return 0;
}

static int tu_phase_finish(const vm_ctx* c, int flags, void* stream) {
  int rc = check_ctx(c);
  if (rc) return rc;
  cudaStream_t st = (cudaStream_t)stream;
  if (c->A != c->red3) {
    cudaMemcpyAsync(c->A, c->red3, (size_t)(c->L * c->M * c->K) * sizeof(double), cudaMemcpyDeviceToDevice, st);
    VM_CHECK_LAUNCH();
  }
  const int nb = (int)imin64(VM_EP_BLOCKS, cdiv(c->L * c->M, 256));
  if (flags & VM_F_ELBO) {
    DISPATCH_K(c->K, (k_elbo_partial<K><<<nb, 256, 0, st>>>(*c, region_ep(c))));
    VM_CHECK_LAUNCH();
  }
  k_finish<<<1, 256, 0, st>>>(*c, flags, region_ep(c), nb);
  VM_CHECK_LAUNCH();
  return 0;
}

static int tu_iteration(const vm_ctx* c, int flags, void* stream) {
  int rc;
  if (c && (rc = slab_check(c, flags))) return rc;  // before any phase has changed the state
  if ((rc = tu_phase_gamma(c, stream))) return rc;
  if ((rc = tu_phase_phi(c, stream))) return rc;
  if ((rc = tu_phase_rho(c, flags, stream))) return rc;
  return tu_phase_finish(c, flags, stream);
}

static int tu_run(const vm_ctx* c, int n_iter, int flags, int last_flags, void* stream) {
  int rc;
  if (c && n_iter > 0 && ((rc = slab_check(c, last_flags)) || (n_iter > 1 && (rc = slab_check(c, flags))))) return rc;
  for (int it = 0; it < n_iter; ++it) {
    rc = tu_iteration(c, it == n_iter - 1 ? last_flags : flags, stream);
    if (rc) return rc;
  }
  return 0;
}

static int tu_infer(const vm_ctx* c, int mode, double threshold, uint8_t* out, void* stream) {
  int rc = check_ctx(c);
  if (rc) return rc;
  if (mode == 1 && c->K < 2) return VM_EINVAL;
  if ((rc = slab_check(c, 0))) return rc;
  const int64_t T = c->L * c->nloc * c->N;
  k_infer<<<(unsigned)imin64(cdiv(T, 256), 148 * 16), 256, 0, (cudaStream_t)stream>>>(c->rho, T, (int)c->K, mode,
                                                                                          (float)threshold, out);
  VM_CHECK_LAUNCH();
  return 0;
}


static int tu_materialize_rows(const vm_ctx* c, int64_t lrow0, int64_t nrows, float* out, void* stream) {
  int rc = check_ctx(c);
  if (rc) return rc;
  if (!out || lrow0 < 0 || nrows < 0 || lrow0 + nrows > c->L * c->nloc) return VM_EINVAL;
  if (c->r_mode == VM_R_CSR) return VM_ENOTSUP;  // no row/column tables: the general mask's posterior lives in the slab
  if (nrows == 0) return 0;
  const dim3 grid((unsigned)c->nct, (unsigned)imin64(nrows, 65535));
  DISPATCH_K(c->K, (k_materialize_rows<K><<<grid, 256, 0, (cudaStream_t)stream>>>(*c, lrow0, nrows, out)));
  VM_CHECK_LAUNCH();
  return 0;
}

// vm_edges_count (emit = 0) / vm_edges_emit (emit = 1); every argument is checked before anything is launched
static int tu_edges(const vm_ctx* c, const vm_edges_args* a, int emit, void* stream) {
  int rc = check_ctx(c);
  if (rc) return rc;
  if (!a || a->what < VM_EDGES_ARGMAX || a->what > VM_EDGES_SAMPLE) return VM_EINVAL;
  if (a->source != VM_EDGES_SLAB && a->source != VM_EDGES_IMPLICIT) return VM_EINVAL;
  if (a->what == VM_EDGES_SAMPLE && a->n_trials < 1) return VM_EINVAL;
  if (emit ? (!a->row_off || !a->o_key || !a->o_val) : !a->row_count) return VM_EINVAL;
  const bool implicit = a->source == VM_EDGES_IMPLICIT;
  if (implicit ? !a->workspace : !c->rho) return VM_EINVAL;
  if (implicit && c->r_mode == VM_R_CSR) return VM_ENOTSUP;  // no row/column tables (as vm_materialize_rows)
  const int64_t rows = c->L * c->nloc;
  if (rows <= 0) return 0;
  cudaStream_t st = (cudaStream_t)stream;
  if (implicit && !emit) {
    k_edges_qmax<<<dim3((unsigned)c->K, (unsigned)c->L), 256, 0, st>>>(c->tab_q, c->N, (int)c->K, a->workspace);
    VM_CHECK_LAUNCH();
  }
  const float thr = (float)a->threshold;  // as vm_infer
  const float thr_bound = thr > 0.f ? (float)(log2((double)thr) - 1.0) : 0.f;
  const unsigned grid = (unsigned)imin64(rows, 148 * 8);
  DISPATCH_K(c->K, (k_edges<K><<<grid, 256, 0, st>>>(*c, *a, emit, thr, thr_bound)));
  VM_CHECK_LAUNCH();
  return 0;
}

// vm_rho_at; every argument is checked before anything is launched
static int tu_rho_at(const vm_ctx* c, int64_t source, int64_t n, const int64_t* key, float* out, void* stream) {
  int rc = check_ctx(c);
  if (rc) return rc;
  if (n < 0 || (n > 0 && (!key || !out))) return VM_EINVAL;
  if (source != VM_EDGES_SLAB && source != VM_EDGES_IMPLICIT) return VM_EINVAL;
  const bool implicit = source == VM_EDGES_IMPLICIT;
  if (!implicit && !c->rho) return VM_EINVAL;
  if (implicit && c->r_mode == VM_R_CSR) return VM_ENOTSUP;  // no row/column tables (as vm_materialize_rows)
  if (n == 0) return 0;
  const unsigned grid = (unsigned)imin64(cdiv(n, 256), 148 * 16);
  DISPATCH_K(c->K, (k_rho_at<K><<<grid, 256, 0, (cudaStream_t)stream>>>(*c, (int)implicit, n, key, out)));
  VM_CHECK_LAUNCH();
  return 0;
}

}  // namespace

extern "C" const vm_tu_api* VM_PASTE(vm_tu_api_, VM_TU_ID)(void) {
  using namespace VM_PASTE(vmtu, VM_TU_ID);
  static const vm_tu_api api = {tu_materialize_prior, tu_refresh_cache, tu_init_stats, tu_phase_gamma, tu_phase_phi,
                                tu_phase_rho,         tu_dense_only,    tu_phase_finish, tu_iteration, tu_run, tu_infer,
                                tu_materialize_rows,  tu_edges,         tu_rho_at};
  return &api;
}
