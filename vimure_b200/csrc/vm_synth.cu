// vimure_b200 -- device-side synthetic reports (SURVEY.md section 8, row f2).
//
// Samples the observed network X of the reference's `_build_X` (`synthetic.py:138-209`) for ONE node-row block, sparsely
// and without a sequential RNG, under three reporter masks: the self-reporter (ego) mask (`vm_synth_ego`, mask
// `synthetic.py:1184-1204`), the all-reporter mask (`vm_synth_all`, flag_self_reporter=False) and an explicit list of
// (l, i, j, m) entries (`vm_synth_masked`).  Every draw is a pure function of (seed, layer, reporter m, pair {a, b}) --
// `pair_draw` below, shared by every kernel -- so any rank can evaluate any (reporter, pair), all ranks that do agree bit
// for bit, and every mask gives the same count for the same (seed, layer, reporter, pair).  A rank therefore generates
// exactly the entries it needs -- X[l,i,j,m] with i in its rows, plus (optionally) the reciprocal entries X[l,j,i,m] whose
// row j lives on another rank -- with nothing exchanged.
//
// Law (per layer l, reporter m with reliability theta_lm, pair {a, b}; lambda_ab = Y_lab if Y_lab > 0 else 0.01):
//   a fair coin picks the first direction; x_first ~ Poisson((theta lambda_first + eta theta lambda_second)/(1-eta^2)),
//   x_second ~ Poisson(theta lambda_second + eta x_first)                                (synthetic.py:170-190)
//   the self tie (a,a): the same two-step draw with both directions equal to (a,a) -- the reference's loop visits it with
//   i == j, so the second assignment overwrites the first: x ~ Poisson(theta 0.01 + eta Poisson(theta 0.01/(1-eta))).
//   The all-reporter and explicit masks draw the self tie (l,a,a) of every reporter m with this law and m's theta.
// Pairs without a true tie in either direction have the tiny base mean theta*0.01 both ways: for them a single uniform
// decides "both counts are zero" (98-99 % of the candidates) before anything else is computed.
//
// Counters (Philox4x32-10, key = (seed, layer)): a reporter on the pair (m in {a, b}, n the other node) uses
// (m, n, class, 0x5eed) and the coin means "the first direction is m->n"; a reporter off the pair uses
// (min(a,b), max(a,b), 3 + class, m) and the coin means "the first direction is min->max".  class: 0 = base pair,
// 1 = a true tie in either direction, 2 = self tie.  The two counter spaces are disjoint (third word < 3 vs >= 3).
//
// The stream is NOT numpy's: parity is always checked on identical inputs, never on regenerated ones; the law is
// checked by moments (tests/test_synth_law.py, tests/test_gpu_synth_masks.py) against the reference generator's.
#include <cuda_runtime.h>
#include <math.h>
#include <stdint.h>

#include "vimure_b200.h"

namespace {

__device__ __forceinline__ uint4 philox4x32(uint4 ctr, uint2 key) {
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
// uniform on (0,1) from 32 random bits
__device__ __forceinline__ double u01(uint32_t r) { return ((double)r + 0.5) * (1.0 / 4294967296.0); }

// Poisson(mu) by inversion of one uniform (means here are O(1): a handful of steps); conditioned on >= 1 if `zt`
__device__ __forceinline__ int poisson_inv(double mu, double u, bool zt) {
  if (mu <= 0.0) return zt ? 1 : 0;
  double p = exp(-mu);
  if (zt) u = p + u * (1.0 - p);  // uniform on (P(0), 1)
  double F = p;
  int k = 0;
  while (u > F && k < 4096) {
    ++k;
    p *= mu / (double)k;
    F += p;
    if (p < 1e-300) break;
  }
  return (zt && k == 0) ? 1 : k;
}

// lambda of the directed tie (l,a,b): its true value Y_lab, or 0 when there is no true tie
__device__ __forceinline__ int y_lookup(const int64_t* __restrict__ yk, const int32_t* __restrict__ yv, int64_t nY,
                                        int64_t key) {
  int64_t lo = 0, hi = nY;
  while (lo < hi) {
    const int64_t mid = (lo + hi) >> 1;
    if (yk[mid] < key) lo = mid + 1;
    else hi = mid;
  }
  return (lo < nY && yk[lo] == key) ? yv[lo] : 0;
}

// average interactions of a tie whose ground truth is category y: the caller's table, or the reference generator's
// default (0.01 for "no tie", y itself otherwise; synthetic.py:140-157)
__device__ __forceinline__ double lam_of(const vm_synth& s, int l, int y) {
  if (s.lam) return s.lam[(int64_t)l * s.K + (y < (int)s.K ? y : (int)s.K - 1)];
  return y > 0 ? (double)y : 0.01;
}

struct Emit {
  const vm_synth s;
  __device__ __forceinline__ bool owns(int r) const { return r >= s.row0 && r < s.row0 + s.nloc; }
  __device__ __forceinline__ void operator()(int l, int i, int j, int m, int x) const {
    if (x <= 0) return;
    const bool own = owns(i);
    const bool tr = s.emit_transposed && !own && owns(j);
    if (!own && !tr) return;
    const unsigned long long p = atomicAdd(reinterpret_cast<unsigned long long*>(s.counter), 1ull);
    if ((int64_t)p >= s.cap) return;  // counted, not stored: the caller sees counter > cap and retries with more room
    s.o_l[p] = l;
    s.o_i[p] = i;
    s.o_j[p] = j;
    s.o_m[p] = m;
    s.o_x[p] = x;
  }
};

// ---- the per-draw law ----------------------------------------------------------------------------------------------
__device__ __forceinline__ uint2 philox_key(const vm_synth& s, int l) {
  return make_uint2((uint32_t)s.seed ^ 0x243F6A88u, (uint32_t)(s.seed >> 32) + (uint32_t)l * 0x9E3779B9u);
}

// the Philox counter of reporter m's draw of class `cls` on a pair {m, n} she is part of
__device__ __forceinline__ uint4 ctr_on(int m, int n, uint32_t cls) {
  return make_uint4((uint32_t)m, (uint32_t)n, cls, 0x5eedu);
}
// the Philox counter of reporter m's draw on the pair {a, b} of class `cls` (see the header comment); (p, q) is the
// direction the coin's "true" refers to
__device__ __forceinline__ uint4 pair_ctr(int m, int a, int b, uint32_t cls, int& p, int& q) {
  if (m == a || m == b) {
    p = m;
    q = m == a ? b : a;
    return ctr_on(p, q, cls);
  }
  p = min(a, b);
  q = max(a, b);
  return make_uint4((uint32_t)p, (uint32_t)q, 3u + cls, (uint32_t)m);
}

// reporter-dependent constants of the base law (class 0) and of the self tie: mean theta*lambda_0 and the probabilities
// of "first > 0" and "first = 0, second > 0"
struct BaseLaw {
  double mu, mm, a, b;
};
__device__ __forceinline__ BaseLaw base_law(const vm_synth& s, int l, double th) {
  BaseLaw w;
  w.mu = th * lam_of(s, l, 0);
  w.mm = w.mu / (1.0 - s.eta);
  w.a = -expm1(-w.mm);
  w.b = exp(-w.mm) * (-expm1(-w.mu));
  return w;
}

// class 2, the self tie: x ~ Poisson(mu + eta Poisson(mm))
__device__ __forceinline__ int self_draw(const BaseLaw& w, double eta, uint4 r) {
  const int y = poisson_inv(w.mm, u01(r.x), false);
  return poisson_inv(w.mu + eta * (double)y, u01(r.y), false);
}

// class 0: false (one uniform) when both counts are zero, else (x_pq, x_qp)
__device__ __forceinline__ bool base_draw(const BaseLaw& w, double eta, uint4 r, int& x_pq, int& x_qp) {
  const double u0 = u01(r.x);
  if (!(u0 < w.a + w.b)) return false;
  const bool first_pos = u0 < w.a;
  const int x1 = first_pos ? poisson_inv(w.mm, u01(r.y), true) : 0;
  const int x2 = first_pos ? poisson_inv(w.mu + eta * (double)x1, u01(r.z), false) : poisson_inv(w.mu, u01(r.z), true);
  const bool coin = (r.w & 1u) != 0;  // first direction is p->q
  x_pq = coin ? x1 : x2;
  x_qp = coin ? x2 : x1;
  return true;
}

// class 1: a true tie in either direction, lam_pq / lam_qp the average interactions of the two directions
__device__ __forceinline__ void edge_draw(double th, double eta, double lam_pq, double lam_qp, uint4 r, int& x_pq,
                                          int& x_qp) {
  const bool coin = (r.w & 1u) != 0;  // first direction is p->q
  const double l1 = coin ? lam_pq : lam_qp, l2 = coin ? lam_qp : lam_pq;
  const int x1 = poisson_inv((th * l1 + eta * th * l2) / (1.0 - eta * eta), u01(r.x), false);
  const int x2 = poisson_inv(th * l2 + eta * (double)x1, u01(r.y), false);
  x_pq = coin ? x1 : x2;
  x_qp = coin ? x2 : x1;
}

// ---- pair_draw: reporter m's two counts on the pair {a, b} (x_ab = a->b, x_ba = b->a; both x_aa for a self tie) ------
// Every kernel below evaluates its draws through these functions, so that every mask gives the same count for the same
// (seed, layer, reporter, pair).  The ego and all-reporter kernels split the classes over two kernels (`base` skips the
// pairs that carry a true tie, found only once a base draw is positive); `pair_draw` is the general form.
__device__ __forceinline__ int self_of(const vm_synth& s, int l, int m, int a, const BaseLaw& w) {
  int p, q;
  return self_draw(w, s.eta, philox4x32(pair_ctr(m, a, a, 2u, p, q), philox_key(s, l)));
}
__device__ __forceinline__ bool base_of(const vm_synth& s, int l, int m, int a, int b, const BaseLaw& w, int& x_ab,
                                        int& x_ba) {
  int p, q, x_pq = 0, x_qp = 0;
  const uint4 ctr = pair_ctr(m, a, b, 0u, p, q);
  if (!base_draw(w, s.eta, philox4x32(ctr, philox_key(s, l)), x_pq, x_qp)) return false;
  x_ab = p == a ? x_pq : x_qp;
  x_ba = p == a ? x_qp : x_pq;
  return true;
}
__device__ __forceinline__ void edge_of(const vm_synth& s, int l, int m, int a, int b, int yab, int yba, double th,
                                        int& x_ab, int& x_ba) {
  int p, q, x_pq, x_qp;
  const uint4 r = philox4x32(pair_ctr(m, a, b, 1u, p, q), philox_key(s, l));
  const bool fwd = p == a;
  edge_draw(th, s.eta, lam_of(s, l, fwd ? yab : yba), lam_of(s, l, fwd ? yba : yab), r, x_pq, x_qp);
  x_ab = fwd ? x_pq : x_qp;
  x_ba = fwd ? x_qp : x_pq;
}
__device__ __forceinline__ void pair_draw(const vm_synth& s, int l, int m, int a, int b, int& x_ab, int& x_ba) {
  const double th = s.theta[(int64_t)l * s.M + m];
  x_ab = x_ba = 0;
  if (a == b) {
    x_ab = x_ba = self_of(s, l, m, a, base_law(s, l, th));
    return;
  }
  const int yab = y_lookup(s.y_key, s.y_val, s.nY, ((int64_t)l * s.N + a) * s.N + b);
  const int yba = y_lookup(s.y_key, s.y_val, s.nY, ((int64_t)l * s.N + b) * s.N + a);
  if (yab > 0 || yba > 0) edge_of(s, l, m, a, b, yab, yba, th, x_ab, x_ba);
  else base_of(s, l, m, a, b, base_law(s, l, th), x_ab, x_ba);
}

// the pair {a, b} carries a true tie in either direction
__device__ __forceinline__ bool has_tie(const vm_synth& s, int l, int a, int b) {
  return y_lookup(s.y_key, s.y_val, s.nY, ((int64_t)l * s.N + a) * s.N + b) > 0 ||
         y_lookup(s.y_key, s.y_val, s.nY, ((int64_t)l * s.N + b) * s.N + a) > 0;
}

// ---- ego kernel A: every owned tie (l, i, j), reporters m in {i, j}; pairs WITHOUT a true tie, and the self ties -----
__global__ void __launch_bounds__(256) k_synth_base(const __grid_constant__ vm_synth s) {
  const Emit emit{s};
  const int64_t T = s.L * s.nloc * s.N;
  for (int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; t < T; t += (int64_t)gridDim.x * blockDim.x) {
    const int64_t lrow = t / s.N;
    const int j = (int)(t - lrow * s.N), l = (int)(lrow / s.nloc), i = (int)(lrow - (int64_t)l * s.nloc + s.row0);
    if (i == j) {
      if (i >= s.M) continue;
      emit(l, i, i, i, self_of(s, l, i, i, base_law(s, l, s.theta[(int64_t)l * s.M + i])));
      continue;
    }
#pragma unroll
    for (int side = 0; side < 2; ++side) {
      const int m = side == 0 ? i : j, n = side == 0 ? j : i;
      if (m >= s.M) continue;
      // base_of(s, l, m, i, j, ..) with the endpoint m known: the counter of ctr_on(m, n, 0) directly
      int x_mn = 0, x_nm = 0;
      const BaseLaw w = base_law(s, l, s.theta[(int64_t)l * s.M + m]);
      if (!base_draw(w, s.eta, philox4x32(ctr_on(m, n, 0u), philox_key(s, l)), x_mn, x_nm)) continue;
      if (has_tie(s, l, i, j)) continue;  // a pair with a true tie is sampled by kernel B instead
      // this thread's tie is i->j: x = count in that direction, x^T the other one
      const int x = side == 0 ? x_mn : x_nm, xT = side == 0 ? x_nm : x_mn;
      emit(l, i, j, m, x);
      if (s.emit_transposed && !emit.owns(j)) emit(l, j, i, m, xT);
    }
  }
}

// decode the true tie q of y_key; false when it is a self tie or the reciprocated pair's (max, min) entry, which the
// kernels skip (the generators never produce a true self tie; a pair whose both directions are true ties is handled from
// its (min, max) entry)
__device__ __forceinline__ bool true_pair(const vm_synth& s, int64_t q, int& l, int& a, int& b, int& yab, int& yba) {
  const int64_t key = s.y_key[q], lr = key / s.N;
  b = (int)(key - lr * s.N);
  l = (int)(lr / s.N);
  a = (int)(lr - (int64_t)l * s.N);
  if (a == b) return false;
  yab = s.y_val[q];
  yba = y_lookup(s.y_key, s.y_val, s.nY, ((int64_t)l * s.N + b) * s.N + a);
  return !(yba > 0 && a > b);
}

// ---- ego kernel B: pairs WITH a true tie in either direction, one thread per (true tie, reporter side) ----------------
__global__ void __launch_bounds__(256) k_synth_edges(const __grid_constant__ vm_synth s) {
  const Emit emit{s};
  for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < 2 * s.nY; e += (int64_t)gridDim.x * blockDim.x) {
    int l, a, b, yab, yba;
    if (!true_pair(s, e >> 1, l, a, b, yab, yba)) continue;
    const int side = (int)(e & 1);
    const int m = side == 0 ? a : b;
    if (m >= s.M) continue;
    if (!emit.owns(a) && !emit.owns(b)) continue;
    int x_ab, x_ba;
    edge_of(s, l, m, a, b, yab, yba, s.theta[(int64_t)l * s.M + m], x_ab, x_ba);
    emit(l, a, b, m, x_ab);
    emit(l, b, a, m, x_ba);
  }
}

// ---- all-reporter kernel A: every owned tie (l, i, j) of layer blockIdx.y, every reporter m < M; pairs WITHOUT a true
// tie, and the self ties.  The reporters' base-law constants are staged in shared memory, RCH reporters at a time.
constexpr int RCH = 256;
__global__ void __launch_bounds__(256) k_synth_all_base(const __grid_constant__ vm_synth s) {
  __shared__ BaseLaw law[RCH];
  const Emit emit{s};
  const int l = (int)blockIdx.y;
  const int64_t T = s.nloc * s.N;
  for (int64_t m0 = 0; m0 < s.M; m0 += RCH) {
    const int nm = (int)min((int64_t)RCH, s.M - m0);
    __syncthreads();
    for (int k = threadIdx.x; k < nm; k += blockDim.x) law[k] = base_law(s, l, s.theta[(int64_t)l * s.M + m0 + k]);
    __syncthreads();
    for (int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; t < T; t += (int64_t)gridDim.x * blockDim.x) {
      const int i = (int)(t / s.N + s.row0), j = (int)(t % s.N);
      if (i == j) {
        for (int k = 0; k < nm; ++k) emit(l, i, i, (int)m0 + k, self_of(s, l, (int)m0 + k, i, law[k]));
        continue;
      }
      const bool tr = s.emit_transposed && !emit.owns(j);
      int tie = -1;  // looked up at the first positive base draw: most pairs have none
      for (int k = 0; k < nm; ++k) {
        const int m = (int)m0 + k;
        int x = 0, xT = 0;
        if (!base_of(s, l, m, i, j, law[k], x, xT)) continue;
        if (tie < 0) tie = has_tie(s, l, i, j) ? 1 : 0;
        if (tie) break;  // sampled by kernel B instead
        emit(l, i, j, m, x);
        if (tr) emit(l, j, i, m, xT);
      }
    }
  }
}

// ---- all-reporter kernel B: pairs WITH a true tie in either direction, one thread per (true tie, reporter) -------------
__global__ void __launch_bounds__(256) k_synth_all_edges(const __grid_constant__ vm_synth s) {
  const Emit emit{s};
  const int64_t E = s.nY * s.M;
  for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < E; e += (int64_t)gridDim.x * blockDim.x) {
    const int64_t q = e / s.M;
    const int m = (int)(e - q * s.M);
    int l, a, b, yab, yba;
    if (!true_pair(s, q, l, a, b, yab, yba)) continue;
    if (!emit.owns(a) && !emit.owns(b)) continue;
    int x_ab, x_ba;
    edge_of(s, l, m, a, b, yab, yba, s.theta[(int64_t)l * s.M + m], x_ab, x_ba);
    emit(l, a, b, m, x_ab);
    emit(l, b, a, m, x_ba);
  }
}

// ---- explicit mask: one thread per entry (l, i, j, m), X[l,i,j,m] = pair_draw(l, m, i, j)'s i->j count ---------------
__global__ void __launch_bounds__(256) k_synth_masked(const __grid_constant__ vm_synth s,
                                                      const __grid_constant__ vm_synth_mask mk) {
  const Emit emit{s};
  for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < mk.n; e += (int64_t)gridDim.x * blockDim.x) {
    const int l = mk.l[e], i = mk.i[e], j = mk.j[e], m = mk.m[e];
    if (l < 0 || l >= s.L || i < 0 || i >= s.N || j < 0 || j >= s.N || m < 0 || m >= s.M) continue;
    if (!emit.owns(i) && !(s.emit_transposed && emit.owns(j))) continue;
    int x_ij, x_ji;
    pair_draw(s, l, m, i, j, x_ij, x_ji);
    emit(l, i, j, m, x_ij);
  }
}

bool synth_args_ok(const vm_synth* s) {
  return s && s->L >= 1 && s->N >= 1 && s->M >= 1 && s->nloc >= 0 && s->row0 >= 0 && s->row0 + s->nloc <= s->N &&
         s->eta >= 0.0 && s->eta < 1.0 && s->cap >= 0 && s->counter && s->theta && s->nY >= 0 &&
         (s->nY == 0 || (s->y_key && s->y_val)) && s->N < ((int64_t)1 << 31) && s->M < ((int64_t)1 << 31) &&
         s->L < ((int64_t)1 << 31) && (s->cap == 0 || (s->o_l && s->o_i && s->o_j && s->o_m && s->o_x));
}

unsigned grid_for(int64_t work) {
  int64_t nb = (work + 255) / 256;
  if (nb > 148 * 64) nb = 148 * 64;
  return (unsigned)nb;
}

}  // namespace

extern "C" int64_t vm_synth_size(void) { return (int64_t)sizeof(vm_synth); }
extern "C" int64_t vm_synth_mask_size(void) { return (int64_t)sizeof(vm_synth_mask); }

extern "C" int vm_synth_ego(const vm_synth* s, void* stream) {
  if (!s || s->L < 1 || s->N < 1 || s->M < 1 || s->M > s->N || s->nloc < 0 || s->row0 < 0 || s->row0 + s->nloc > s->N ||
      s->eta < 0.0 || s->eta >= 1.0 || s->cap < 0 || !s->counter || !s->theta || (s->nY > 0 && (!s->y_key || !s->y_val)))
    return VM_EINVAL;
  if (s->N >= (int64_t)1 << 31) return VM_EINVAL;
  cudaStream_t st = (cudaStream_t)stream;
  cudaError_t e = cudaMemsetAsync(s->counter, 0, sizeof(int64_t), st);
  if (e != cudaSuccess) return (int)e;
  const int64_t T = s->L * s->nloc * s->N;
  if (T > 0) {
    k_synth_base<<<grid_for(T), 256, 0, st>>>(*s);
    if ((e = cudaGetLastError()) != cudaSuccess) return (int)e;
  }
  if (s->nY > 0) {
    k_synth_edges<<<grid_for(2 * s->nY), 256, 0, st>>>(*s);
    if ((e = cudaGetLastError()) != cudaSuccess) return (int)e;
  }
  return 0;
}

extern "C" int vm_synth_all(const vm_synth* s, void* stream) {
  if (!synth_args_ok(s) || s->L > 65535) return VM_EINVAL;
  cudaStream_t st = (cudaStream_t)stream;
  cudaError_t e = cudaMemsetAsync(s->counter, 0, sizeof(int64_t), st);
  if (e != cudaSuccess) return (int)e;
  const int64_t T = s->nloc * s->N;
  if (T > 0) {
    int64_t nb = (T + 255) / 256;
    const int64_t most = (148 * 64 + s->L - 1) / s->L;
    if (nb > most) nb = most;
    k_synth_all_base<<<dim3((unsigned)nb, (unsigned)s->L), 256, 0, st>>>(*s);
    if ((e = cudaGetLastError()) != cudaSuccess) return (int)e;
  }
  if (s->nY > 0 && s->nloc > 0) {
    k_synth_all_edges<<<grid_for(s->nY * s->M), 256, 0, st>>>(*s);
    if ((e = cudaGetLastError()) != cudaSuccess) return (int)e;
  }
  return 0;
}

extern "C" int vm_synth_masked(const vm_synth* s, const vm_synth_mask* mask, void* stream) {
  if (!synth_args_ok(s) || !mask || mask->n < 0 || (mask->n > 0 && (!mask->l || !mask->i || !mask->j || !mask->m)))
    return VM_EINVAL;
  cudaStream_t st = (cudaStream_t)stream;
  cudaError_t e = cudaMemsetAsync(s->counter, 0, sizeof(int64_t), st);
  if (e != cudaSuccess) return (int)e;
  if (mask->n > 0 && s->nloc > 0) {
    k_synth_masked<<<grid_for(mask->n), 256, 0, st>>>(*s, *mask);
    if ((e = cudaGetLastError()) != cudaSuccess) return (int)e;
  }
  return 0;
}
