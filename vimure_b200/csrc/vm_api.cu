// vimure_b200 -- the extern "C" entry points of include/vimure_b200.h.
// The kernels are instantiated per K in several translation units (csrc/vm_kernels.cu compiled once per TU by
// vimure_b200/build.py); every entry point routes to the TU that owns ctx->K through its function table.
#include <stdio.h>

#include "vm_common.cuh"
#include "vm_tu_list.h"  // generated: declarations of vm_tu_api_<id>() and vm_tu_for_K()

static const vm_tu_api* tu(const vm_ctx* c) {
  if (!c || c->K < 2 || c->K > VM_MAX_K) return nullptr;
  return vm_tu_for_K((int)c->K);
}
#define VM_ROUTE(call)              \
  const vm_tu_api* t = tu(c);       \
  if (!t) return VM_EINVAL;         \
  return t->call

extern "C" int64_t vm_ctx_size(void) { return (int64_t)sizeof(vm_ctx); }
extern "C" int64_t vm_abi_version(void) { return VM_ABI_VERSION; }
extern "C" int64_t vm_dense_tile_w(int64_t K) { return vm_dense_tile_w_host(K); }

extern "C" int vm_materialize_prior(const vm_ctx* c, void* stream) { VM_ROUTE(materialize_prior(c, stream)); }
extern "C" int vm_refresh_cache(const vm_ctx* c, void* stream) { VM_ROUTE(refresh_cache(c, stream)); }
extern "C" int vm_init_stats(const vm_ctx* c, void* stream) { VM_ROUTE(init_stats(c, stream)); }
extern "C" int vm_phase_gamma(const vm_ctx* c, void* stream) { VM_ROUTE(phase_gamma(c, stream)); }
extern "C" int vm_phase_phi(const vm_ctx* c, void* stream) { VM_ROUTE(phase_phi(c, stream)); }
extern "C" int vm_phase_rho(const vm_ctx* c, int flags, void* stream) { VM_ROUTE(phase_rho(c, flags, stream)); }
extern "C" int vm_dense_only(const vm_ctx* c, int flags, void* stream) { VM_ROUTE(dense_only(c, flags, stream)); }
extern "C" int vm_phase_finish(const vm_ctx* c, int flags, void* stream) { VM_ROUTE(phase_finish(c, flags, stream)); }
extern "C" int vm_iteration(const vm_ctx* c, int flags, void* stream) { VM_ROUTE(iteration(c, flags, stream)); }
extern "C" int vm_run(const vm_ctx* c, int n_iter, int flags, int last_flags, void* stream) {
  VM_ROUTE(run(c, n_iter, flags, last_flags, stream));
}
extern "C" int vm_infer(const vm_ctx* c, int mode, double threshold, uint8_t* out, void* stream) {
  VM_ROUTE(infer(c, mode, threshold, out, stream));
}
extern "C" int vm_materialize_rows(const vm_ctx* c, int64_t lrow0, int64_t nrows, float* out, void* stream) {
  VM_ROUTE(materialize_rows(c, lrow0, nrows, out, stream));
}

// ---- rho_mean on the slab (model.py:1151-1153): sum_k k rho_k, 4 bytes per tie back instead of an fp64 copy of rho -----
__global__ void __launch_bounds__(256) k_infer_mean(const float* __restrict__ rho, int64_t T, int K, float* __restrict__ out) {
  for (int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; t < T; t += (int64_t)gridDim.x * blockDim.x) {
    const float* r = rho + t * K;
    float s = 0.f;
    for (int k = 1; k < K; ++k) s += (float)k * r[k];
    out[t] = s;
  }
}
extern "C" int vm_infer_mean(const vm_ctx* c, float* out, void* stream) {
  if (!c || !out || c->K < 2 || c->K > VM_MAX_K || !c->rho) return VM_EINVAL;
  const int64_t T = c->L * c->nloc * c->N;
  if (T <= 0) return 0;
  int64_t nb = (T + 255) / 256;
  if (nb > 148 * 32) nb = 148 * 32;
  k_infer_mean<<<(unsigned)nb, 256, 0, (cudaStream_t)stream>>>(c->rho, T, (int)c->K, out);
  cudaError_t e = cudaGetLastError();
  return e == cudaSuccess ? 0 : (int)e;
}

// ---- posterior sampling on the slab (model.py:1062-1096): one thread per owned tie, vm_sample_label -------------
__global__ void __launch_bounds__(256) k_sample(const float* __restrict__ rho, int64_t nloc, int64_t N, int64_t row0,
                                                int64_t T, int K, int64_t n_trials, uint64_t seed,
                                                uint8_t* __restrict__ out) {
  const uint2 key = make_uint2((uint32_t)seed, (uint32_t)(seed >> 32));
  for (int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; t < T; t += (int64_t)gridDim.x * blockDim.x) {
    const int64_t lrow = t / N, j = t - lrow * N, l = lrow / nloc, i = lrow - l * nloc + row0;
    const uint64_t gt = (uint64_t)((l * N + i) * N + j);
    out[t] = (uint8_t)vm_sample_label(rho + t * K, K, n_trials, gt, key);
  }
}
extern "C" int vm_sample(const vm_ctx* c, int64_t n_trials, uint64_t seed, uint8_t* out, void* stream) {
  if (!c || !out || c->K < 2 || c->K > VM_MAX_K || n_trials < 1 || !c->rho) return VM_EINVAL;
  const int64_t T = c->L * c->nloc * c->N;
  if (T <= 0) return 0;
  int64_t nb = (T + 255) / 256;
  if (nb > 148 * 32) nb = 148 * 32;
  k_sample<<<(unsigned)nb, 256, 0, (cudaStream_t)stream>>>(c->rho, c->nloc, c->N, c->row0, T, (int)c->K, n_trials, seed, out);
  cudaError_t e = cudaGetLastError();
  return e == cudaSuccess ? 0 : (int)e;
}

extern "C" int64_t vm_edges_size(void) { return (int64_t)sizeof(vm_edges_args); }
extern "C" int vm_edges_count(const vm_ctx* c, const vm_edges_args* a, void* stream) { VM_ROUTE(edges(c, a, 0, stream)); }
extern "C" int vm_edges_emit(const vm_ctx* c, const vm_edges_args* a, void* stream) { VM_ROUTE(edges(c, a, 1, stream)); }
extern "C" int vm_rho_at(const vm_ctx* c, int64_t source, int64_t n, const int64_t* key, float* out, void* stream) {
  VM_ROUTE(rho_at(c, source, n, key, out, stream));
}

__global__ void k_test_special(const double* x, double* dg, double* lg, int64_t n) {
  const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= n) return;
  dg[t] = vm_digamma(x[t]);
  lg[t] = lgamma(x[t]);
}
extern "C" int vm_test_special(const double* x, double* dg, double* lg, int64_t n, void* stream) {
  if (n <= 0) return 0;
  k_test_special<<<(unsigned)((n + 255) / 256), 256, 0, (cudaStream_t)stream>>>(x, dg, lg, n);
  cudaError_t e = cudaGetLastError();
  return e == cudaSuccess ? 0 : (int)e;
}
