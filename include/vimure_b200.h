/*
 * vimure_b200 -- C ABI of the B200-native CAVI hot path of VIMuRe (`VimureModel.fit`).
 *
 * The reference (latentnetworks/vimure) is pure Python: it has no FFI/plugin seam, the drop-in
 * boundary is the Python class `vimure.model.VimureModel` (reference `src/python/vimure/model.py:28-448`).
 * This header is the LOWER face of that boundary: what the Python host (`vimure_b200/model.py`)
 * binds with ctypes, and what any other host (R via .C/.Call, C++) would bind instead.
 * Each entry point names the reference routine(s) it replaces.
 *
 * Conventions
 *   - every function returns 0 on success, a positive cudaError_t, or a negative VM_E* code;
 *     nothing throws, nothing is allocated or kept by the library: the caller owns every buffer
 *     (device pointers, normally PyTorch tensors) and passes them in `vm_ctx`;
 *   - `stream` is a cudaStream_t passed as void*; all work is enqueued on it, no host sync;
 *   - one host thread per GPU/rank; no global state;
 *   - `vm_ctx` contains only 8-byte fields (int64_t / double / pointers) so that its layout is
 *     padding-free and trivially mirrored from ctypes; `vm_ctx_size()` lets the host verify it.
 *
 * Tie indexing.  A rank owns the node rows [row0, row0+nloc) of every layer (row-block sharding,
 * SURVEY.md section 8e).  Local row  lrow = l*nloc + (i-row0);  local tie = lrow*N + j;  the dense
 * posterior slab `rho` is float32 [L][nloc][N][K] (same order as the reference's (L,N,N,K) array).
 */
#ifndef VIMURE_B200_H
#define VIMURE_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define VM_ABI_VERSION 17

/* reporter-mask structure (how R[l,i,j,m] is represented) */
#define VM_R_EGO 0 /* reporter m == node m reports row m and column m (vimure synthetic.py:1184-1204, _io.py:229-242) */
#define VM_R_ALL 1 /* every reporter reports every tie (R == 1, model.py:207-211) */
#define VM_R_CSR 2 /* general mask: explicit per-tie CSR + per-reporter CSC */

/* flags for vm_phase_rho / vm_phase_finish / vm_iteration */
#define VM_F_ELBO 1      /* also produce the ELBO (model.py:948-1019) */
#define VM_F_NO_STORE 2  /* write no dense rho slab this iteration: the dense kernels run statistics-only (no stage,
                            no store, no patches) and vm_ctx.rho may be NULL.  Every other kernel and every number is
                            that of a storing iteration; the tables (tab_p, tab_q, layer_consts) and rho_u32 the
                            iteration leaves behind ARE the posterior (vm_materialize_rows evaluates it).  Not with
                            VM_R_CSR, whose statistics gather the slab: VM_ENOTSUP before any phase runs. */
#define VM_F_INIT 4      /* vm_phase_finish only: consume the initial statistics, do not update nu */

/* error codes (negative) */
#define VM_EINVAL (-1)    /* bad argument / unsupported K */
#define VM_ENOTSUP (-2)   /* combination not implemented */

/* slots of the small fp64 vector `nu` */
#define VM_NU_SHP 0
#define VM_NU_RTE 1
#define VM_NU_G 2       /* exp(psi(nu_shp)-log(nu_rte)) to be used by the NEXT iteration's cache */
#define VM_NU_E 3       /* nu_shp/nu_rte */
#define VM_NU_G_STALE 4 /* the G_exp_nu used during the last iteration (what the reference leaves in self.G_exp_nu, Q2) */
#define VM_NU_LEN 8

/* slots appended after A[L*M*K] in the `red3` statistics vector (the all-reduced payload) */
#define VM_R3_NU 0   /* sum_I sum_k dz2*rho_new         (model.py:822-825) */
#define VM_R3_CAT 1  /* categorical ELBO term           (model.py:1306-1313) */
#define VM_R3_T2 2   /* sum_I x log(EPS + ...)          (model.py:967-995) */
#define VM_R3_B 3    /* sum_J x^T_J sum_k rho_k         (model.py:1286-1290, the eta part) */
#define VM_R3_EXTRA 4

/* slots of dev_flags */
#define VM_FLAG_DEAD 0
#define VM_FLAG_FIXNU 1

/* maximum K compiled in.  K = number of categories of a report; when the caller does not pass K the reference defaults to
   max(X)+1 (model.py:179-196), which for count data easily exceeds 8 -- hence 32, although every BASELINE config has
   K <= 3.  The kernels are templates on K, one translation unit per group of K (vimure_b200/build.py); K > 4 only
   instantiates the general kernels. */
#define VM_MAX_K 32
/* special ties handled by one block of the special-tie kernel (n_ublk = ceil(max per layer / this)) */
#ifndef VM_SPECIAL_TIES_PER_BLOCK /* (a timing variant may be built with a multiple of it: tools/ab_libs.py) */
#define VM_SPECIAL_TIES_PER_BLOCK 1024
#endif

typedef struct vm_ctx {
  /* ---- dimensions ---- */
  int64_t L, N, M, K;
  int64_t row0, nloc;       /* this rank's node-row block */
  int64_t r_mode;           /* VM_R_* */
  int64_t ego_diag;         /* EGO: the mask contains the (m,m) tie of reporter m */
  int64_t mutuality;        /* model.py:39-65 */
  int64_t may_dead;         /* 1 = always check closed-form rows for complete underflow (else decided per layer on device) */
  int64_t U;                /* special ties owned (union of X ties, all diagonal ties) */
  int64_t I;                /* X entries whose tie is owned */
  int64_t IT;               /* X entries whose TRANSPOSED tie is owned and reported (ELBO eta term) */
  int64_t tile_w, tile_h;   /* dense tiling; tile_w must be vm_dense_tile_w(K) */
  int64_t nct, nrt;         /* ceil(N/tile_w), ceil(nloc/tile_h) */
  int64_t n_gchunk;         /* reporter chunks (gamma pass) */
  int64_t phi_chunk;        /* entries per block in the phi pass */
  int64_t n_phichunk;       /* max over layers of ceil(entries_in_layer/phi_chunk) */
  int64_t n_ublk;           /* blocks per layer of the special-tie kernel */
  void* aux_stream;         /* cudaStream_t owned by the caller */
  void* ev_fork;            /* two cudaEvent_t (timing disabled) owned by the caller, used to fork the aux stream from and */
  void* ev_join;            /*   join it back into the main one; NULL: the library creates and destroys a pair per launch */
  double eps;               /* EPS, model.py:215-218 */
  double alpha_eta, beta_eta;
  double b_all;             /* sum of t_x: the eta part of the ELBO when no tie has underflowed completely */

  /* ---- special ties, sorted by (lrow, col) ---- */
  const int32_t* u_lrow;    /* [U] */
  const int32_t* u_col;     /* [U] */
  const int64_t* u_ptr;     /* [U+1] range of entries of the tie */
  const double* u_logpr;    /* [U*K] log(pr_rho+EPS) (model.py:559) */
  const int32_t* u_cnt;     /* [U] number of X entries of the tie (0 for a bare diagonal tie) */
  const int32_t* u_m0;      /* [U] reporter / count / reciprocal count of the tie's FIRST X entry, stored inline so that */
  const float* u_x0;        /* [U]   the special-tie kernel needs no dependent load for single-entry ties */
  const float* u_xT0;       /* [U] */
  const int32_t* utile_ptr; /* [L*nloc*nct+1] first special tie of each (lrow, column tile) */

  /* ---- shortcut ties: special ties whose posterior needs neither fp64 nor the entry list ----
     Ego mask, K <= 4, off the diagonal, in a full column tile, and either
       SIMPLE: none of the tie's X entries has a reciprocal report (x^T = 0, or mutuality off).  Its Poisson allocation is
               dz1_k = x whatever the parameters and the E[log theta] of its reporters is common to every k, so
                  log2 rho_k/rho_0 = lo_k - S (E[lambda_k]-E[lambda_0]) log2e + X (E[log lambda_k]-E[log lambda_0]) log2e,
               lo_k = log2((pr_k+EPS)/(pr_0+EPS)), X = sum of its x: the separable form of a tie without data plus a
               per-tie constant and a per-layer multiple of X;  or
       SINGLE: exactly ONE X entry, which has a reciprocal report (x^T > 0) and whose reporter is the row node or the
               column node (always the case for entries inside an ego mask).  With f_k = z1_k/(z1_k+z2),
               z1_k = G_theta_m G_lambda_k, z2 = G_nu x^T  (model.py:686-696):
                  ln rho_k/rho_0 = ln2 lo_k - S (E[lambda_k]-E[lambda_0])
                                   + x [ (f_k-f_0) E[log theta_m] + f_k E[log lambda_k] - f_0 E[log lambda_0] ],
               every term O(1..30).
     On iterations that do not evaluate the ELBO the dense kernel itself (k_dense_sc: in fp32, from one 16/32-byte
     record per tie (u_rec) and the per-node table, no entry list, no fp64 transcendental) evaluates these ties --
     posterior into rho_u32 (and the slab, if stored), (posterior - closed form) into the fixed-point per-reporter corrections, the
     SINGLE ties' part of the nu statistic (x z2 sum_k rho_k/(z1_k+z2), model.py:822-825) -- and the fp64 special-tie
     kernel only visits the others (`cx_idx`, `cx_*`); every other iteration runs the special-tie kernel over all special
     ties in fp64, as does any layer for which k_phi_finish cannot rule out a completely underflowed tie or an fp32 range
     problem (layer constant VM_LC_SIMPLE). */
  int64_t simple_mode;      /* 1 = enabled (EGO mask, K <= 4, fast dense kernel eligible, serial special/dense launch) */
  int64_t n_cx;             /* special ties that take no shortcut */
  int64_t n_cxblk;          /* blocks per layer of the special-tie kernel in list mode: ceil(max per-layer count / 1024) */
  const int32_t* cx_idx;    /* [n_cx] their indices, ascending */
  const int64_t* cx_ptr;    /* [L+1] range of cx_idx of every layer */
  /* compacted copies of the per-tie arrays for those ties (coalesced reads in the list mode of the special-tie kernel) */
  const int32_t* cx_lrow;   /* [n_cx] */
  const int32_t* cx_col;
  const int32_t* cx_cnt;
  const int32_t* cx_m0;
  const float* cx_x0;
  const float* cx_xT0;
  const float* cx_x0sum;
  const double* cx_logpr;   /* [n_cx*K] */
  const float* u_px;        /* [U] X of a shortcut tie (sum of its x; the one report's x for a SINGLE tie), 0 = no shortcut */
  const float* u_pxt;       /* [U] 0 for a SIMPLE tie; SINGLE: +x^T if the entry's reporter is the row node, -x^T if it is
                               the column node */
  const float* u_rec;       /* [U*RS] one record per special tie for the shortcut kernel, RS = 4 floats at K = 2, 8 at K = 3, 4:
                               (col as a float, u_px, u_pxt, lo_1..lo_{K-1}, padding), lo_k = log2((pr_k+EPS)/(pr_0+EPS))
                               -- constant over a fit (built by the host from u_col / u_px / u_pxt and the prior) */
  float* nodetab;           /* [L*N*stride] per node: q_1..q_{K-1} (= -E[theta] d_k), G_theta, E[log theta] log2e, active;
                               stride = 4 floats at K = 2, 8 at K = 3, 4 (written by k_tables) */
  const double* simple_consts; /* [3+K] over the shortcut ties: min log(pr_0+EPS); max X; max x^T; min log(pr_k+EPS), k < K */
  /* ---- all-reporter mask: fp32 evaluation of EVERY special tie on iterations without ELBO (k_all32) ----
     With the all-reporter mask S is a per-layer constant, most ties carry reports (69 % at config 4) and a tie has
     several entries, so the work is per ENTRY: the kernel computes each entry's contribution to the log2-odds
       log2 rho_k/rho_0 = lo_k - S_all (E[lambda_k]-E[lambda_0]) log2e + sum over the tie's entries of dat_k(entry)
     (dat_k as for a SINGLE tie above, or x (E[log lambda_k]-E[log lambda_0]) log2e for an entry without a reciprocal
     report) entry-parallel from a shared-memory reporter table, then one thread per tie sums its entries and normalises.
     Same outputs and block partials as the special-tie kernel, which still runs every special tie in fp64 on ELBO
     iterations and for layers whose VM_LC_SIMPLE guard (fp32 range, closed-form rows alive) fails.  A tie whose every
     log-weight lies below the reference's underflow threshold is detected per tie (its log2 weight of category 0 is
     carried along) and zeroed as the fp64 kernel does.  simple_consts then covers all special ties. */
  int64_t all32_mode;       /* 1 = enabled (ALL mask, K <= 4, M <= 4096, counts and priors in fp32 range) */
  int64_t gamma_ts;         /* 1 = the gamma pass walks the TIE-sorted entries (f_*) with per-reporter accumulators in shared
                               memory instead of the reporter-sorted copies (g_*): with few reporters (all-reporter mask,
                               M <= 256, K <= 8) every reporter's entries are spread over all ties, so the reporter-sorted pass reads
                               a whole 32-byte sector per 8-byte posterior (7.8 GB per pass at config 4 instead of 2.6) */
  const float* u_lo;        /* [U*K] per special tie: log2(pr_0+EPS), then lo_k = log2((pr_k+EPS)/(pr_0+EPS)), k = 1..K-1
                               (built by the host; the first value only serves the complete-underflow check) */
  int64_t* fixP;            /* [L*K] fixed point 2^-30: sum over the simple ties of rho_k X (their part of phi0) */

  /* ---- X entries, sorted by tie ---- */
  const int32_t* e_u;       /* [I] special-tie index */
  const int32_t* e_m;       /* [I] reporter */
  const float* e_x;         /* [I] X[l,i,j,m] */
  const float* e_xT;        /* [I] X[l,j,i,m], pre-paired (replaces data_T_vals, model.py:152-161) */
  const uint8_t* e_flags;   /* [I] bit0: (l,i,j,m) is in R */
  /* The gamma / phi passes only visit the entries WITH a reciprocal report (x^T > 0, "E1"): for the others the Poisson
     allocation is dz1_k = x whatever the parameters, so their contribution is a pack-time constant (g0) for gamma and
     sum_ties rho_k * u_x0sum for phi (accumulated by the special-tie kernel into phi0).  I1 = number of E1 entries. */
  int64_t I1;
  const int32_t* f_u;       /* [I1] E1 entries sorted by tie: special-tie index, reporter, x, x^T */
  const int32_t* f_m;
  const float* f_x;
  const float* f_xT;
  const int64_t* lay_eptr;  /* [L+1] E1 entry range of each layer (phi pass) */
  const double* g0;         /* [L*M] sum of x over the E0 entries of reporter (l,m) */
  const float* u_x0sum;     /* [U] sum of x over the E0 entries of the special tie */
  const int64_t* g_chunk_ptr; /* [n_gchunk+1] ranges in reporter-sorted order */
  const int32_t* g_chunk_lm;  /* [n_gchunk] reporter id l*M+m */
  const int32_t* g_u;         /* [I1] reporter-sorted E1 entries (coalesced gamma pass) */
  const float* g_x;           /* [I1] */
  const float* g_xT;          /* [I1] */
  const int64_t* g_lm_cptr;   /* [L*M+1] chunk range of each reporter */

  /* ---- transposed-position list (ELBO eta term) ---- */
  const int32_t* t_u;       /* [IT] special index of the transposed tie, or -1 */
  const int32_t* t_lrow;    /* [IT] */
  const int32_t* t_col;     /* [IT] */
  const float* t_x;         /* [IT] x * multiplicity in R */

  /* ---- reporter mask ---- */
  const uint8_t* rep;       /* EGO: [L*M] reporter is active */
  const int64_t* r_ptr;     /* CSR: [L*nloc*N+1] */
  const int32_t* r_m;       /* CSR: reporter of each mask entry */
  const float* r_val;       /* CSR: R.vals (used by the rho update only, Q4) */
  const int64_t* c_ptr;     /* CSC: [L*M+1] */
  const int64_t* c_tie;     /* CSC: local tie of each mask entry */

  /* ---- priors (model.py:238-317), broadcast to full arrays ---- */
  const double* alpha_theta; /* [L*M] */
  const double* beta_theta;  /* [L*M] */
  const double* alpha_lambda; /* [L*K] */
  const double* beta_lambda;  /* [L*K] */

  /* ---- variational state (fp64) ---- */
  double* gamma_shp;        /* [L*M] */
  double* gamma_rte;        /* [L*M] */
  double* phi_shp;          /* [L*K] */
  double* phi_rte;          /* [L*K] */
  double* nu;               /* [VM_NU_LEN] */
  double* G_theta;          /* [L*M] exp(psi(shp)-log(rte)) */
  double* E_theta;          /* [L*M] shp/rte */
  double* Elog_theta;       /* [L*M] psi(shp)-log(rte) */
  double* G_lambda;         /* [L*K] */
  double* E_lambda;         /* [L*K] */
  double* Elog_lambda;      /* [L*K] */
  double* GE_theta;         /* [L*M*2] (G_theta, Elog_theta) interleaved: one 16-byte gather per X entry */
  double* A;                /* [L*M*K] sum of rho_k over the ties reported by (l,m) */
  double* rho_u;            /* [U*K] posterior of the special ties, fp64 (as of the last update by the special-tie kernel) */
  float* rho_u32;           /* [U*K] fp32 posterior of the special ties: patch source of the dense slab and what the gamma /
                               phi passes gather (written by the special-tie kernel and by the shortcut-tie kernel) */
  double* delta_u;          /* [U*K] rho_u - formula value */
  float* rho;               /* [L*nloc*N*K] dense posterior slab, or NULL: then every iteration must pass VM_F_NO_STORE,
                               and the entry points that read or write the slab return VM_EINVAL */

  /* ---- workspaces ---- */
  double* layer_consts;     /* [L*(3*K+5)] per layer: c_k, d_k (log2 domain), S_all, log-prior consts, dead flag,
                               simple-tie flag, g_k */
  float* tab_p;             /* [L*nloc*K] row part of the log2-odds */
  float* tab_q;             /* [L*N*K] column part */
  float* rowpart;           /* [L*nloc*nct*K] */
  float* colpart;           /* [L*nrt*N*K] */
  double* er_node;          /* [L*N] EGO: E[theta] of node n acting as reporter (0 if not an active reporter) */
  double* colsum;           /* [L*M*K] column partials reduced over the row tiles */
  int64_t* dev_flags;       /* [8] [0]: a special tie underflowed completely in the last rho update;
                               [VM_FLAG_FIXNU]: fixed point 2^-30, nu statistic of the SINGLE ties the shortcut kernel evaluated */
  int64_t* fixG;            /* [L*M] fixed-point correction of g0: -x of the E0 entries of special ties that underflowed */
  double* phi0;             /* [L*K] sum over special ties of rho_k * u_x0sum (E0 part of the next phi-shape sums) */
  int64_t* fixA;            /* [L*M*K] EGO: per-reporter sums of (special - closed form), fixed point 2^-42, accumulated
                               with integer atomics (order-independent => bit-reproducible); slot k=0 holds only the
                               residual count (live special) - (live closed form) */
  double* gfpart;           /* [L*ceil(M/256)*(K+4)] block partials of k_gamma_finish for k_phi_finish */
  double* blkpart;          /* [max(n_ublk, nct*L*nrt, L*n_phichunk*K, n_gchunk, ...)*4] */
  double* red1;             /* [L*M] gamma-shape sums (all-reduced by the host between phases when sharded) */
  double* red2;             /* [L*K] phi-shape sums */
  double* red3;             /* [L*M*K + VM_R3_EXTRA] */
  double* elbo_out;         /* [8]: [0]=ELBO, [1..] its terms */
} vm_ctx;

/* sizeof(vm_ctx) and ABI version, for the host-side mirror to verify */
int64_t vm_ctx_size(void);
int64_t vm_abi_version(void);
/* column-tile width of the dense kernel for a given K (the packer builds `utile_ptr` for this width) */
int64_t vm_dense_tile_w(int64_t K);

/* theta/lambda/nu caches (G_*, E_*, Elog_*) from the current shapes/rates: `_update_cache` (model.py:676-684) and the
 * cache part of `_initialize_priors` (model.py:596-605). Call once after injecting the initial state. */
int vm_refresh_cache(const vm_ctx* c, void* stream);

/* Initial statistics from rho = pr_rho (model.py:602): fills delta_u from rho_u, and red3[A] with this
 * rank's share of A. Follow with (all-reduce red3 and) vm_phase_finish(VM_F_INIT). */
int vm_init_stats(const vm_ctx* c, void* stream);

/* Phase 1 -- replaces `_update_cache` + `_sp_uttkrp_theta` (model.py:662-696, 832-859):
 * red1[l,m] = sum over owned X entries of (l,m) of sum_k rho_k * dz1_k. */
int vm_phase_gamma(const vm_ctx* c, void* stream);

/* Phase 2 -- finishes `_update_gamma` (model.py:698-727) from red1 and A, refreshes the theta cache, then
 * `_sp_uttkrp_lambda` (model.py:861-887): red2[l,k] = sum over owned X entries of rho_k * dz1_k. */
int vm_phase_phi(const vm_ctx* c, void* stream);

/* Phase 3 -- finishes `_update_phi` (model.py:729-761) from red2 and A, then `_update_rho` +
 * `_sp_uttkrp_rho` (model.py:763-818, 889-923) for every owned tie: special ties in fp64, all ties by
 * the per-tie dense kernel (writes the fp32 slab unless VM_F_NO_STORE; the statistics are the same bits either way),
 * and this rank's share of the statistics of the NEW rho into red3: A, the nu sum (model.py:820-830) and, with
 * VM_F_ELBO, the ELBO sums. */
int vm_phase_rho(const vm_ctx* c, int flags, void* stream);

/* Measurement hook: launches ONLY the per-tie dense kernel of phase 3 (tables and special ties as left by the last
 * vm_phase_rho), so that its duration can be timed in isolation for the roofline figure. The statistics are unchanged
 * and the slab is rewritten with the same values. */
int vm_dense_only(const vm_ctx* c, int flags, void* stream);

/* Phase 4 -- consumes (all-reduced) red3: A <- red3, `_update_nu` (model.py:820-830), refreshes the nu cache,
 * and with VM_F_ELBO assembles `__ELBO` (model.py:948-1019) into elbo_out[0]. */
int vm_phase_finish(const vm_ctx* c, int flags, void* stream);

/* One full `_update_CAVI` (model.py:623-660) on a single rank = the four phases back to back. */
int vm_iteration(const vm_ctx* c, int flags, void* stream);

/* n_iter iterations back to back; the LAST one runs with `last_flags` (the others with `flags`). */
int vm_run(const vm_ctx* c, int n_iter, int flags, int last_flags, void* stream);

/* Writes rho = pr_rho into the dense slab (one-hot + special ties), model.py:602. */
int vm_materialize_prior(const vm_ctx* c, void* stream);

/* The posterior the last rho update left (the implicit one of a VM_F_NO_STORE iteration, or the slab's own values), for
 * the local rows [lrow0, lrow0+nrows), lrow = l*nloc + (i-row0), into `out` (float32 [nrows][N][K], the slab's layout):
 * bit-identical to what a storing iteration writes into those rows of the slab.  Reads tab_p, tab_q, layer_consts,
 * utile_ptr, u_col and rho_u32 only; VM_ENOTSUP under the general mask (VM_R_CSR). */
int vm_materialize_rows(const vm_ctx* c, int64_t lrow0, int64_t nrows, float* out, void* stream);

/* Posterior consumers on the dense slab (model.py:1148-1166, utils.py:207-217):
 * out[t] = argmax_k rho[t,k] (mode 0) or rho[t,1] >= threshold (mode 1), uint8, [L*nloc*N]. */
int vm_infer(const vm_ctx* c, int mode, double threshold, uint8_t* out, void* stream);

/* rho_mean (model.py:1151-1153): out[t] = sum_k k rho[t,k], float32, [L*nloc*N]. */
int vm_infer_mean(const vm_ctx* c, float* out, void* stream);

/* `sample_inferred_model` on the dense slab (model.py:1062-1096): out[t] = argmax_k of the counts of n_trials draws from
 * Categorical(rho[t,:]) (numpy: multinomial(n_trials, rho).argmax(-1)), uint8, [L*nloc*N].  Counter-based RNG (Philox4x32-10)
 * keyed by `seed` and the GLOBAL tie id: reproducible, independent of launch geometry and of the sharding.  The stream is
 * not numpy's (the reference draws with numpy.random.default_rng(seed)). */
int vm_sample(const vm_ctx* c, int64_t n_trials, uint64_t seed, uint8_t* out, void* stream);

/* ---- sparse consumers: the ties of the inferred network whose label is nonzero, as an edge list ------------------------
 * The labels of vm_infer (VM_EDGES_ARGMAX: mode 0; VM_EDGES_THRESHOLD: mode 1) and vm_sample (VM_EDGES_SAMPLE), bit for bit,
 * without any (L, nloc, N)-sized buffer.  Two passes over the local rows lrow = l*nloc + (i-row0), no host synchronisation
 * inside either:
 *   vm_edges_count: row_count[lrow] = number of ties of the row whose label is nonzero;
 *   vm_edges_emit:  with row_off = the caller's exclusive prefix sum of row_count, o_key[row_off[lrow] + r] = (l*N+i)*N+j
 *                   (the global flat id) and o_val[...] = label (>= 1) of the r-th such tie of the row, ascending in j: the
 *                   output is sorted by key, and equals np.nonzero of the dense consumer's output.
 * `source` says where the posterior is read: VM_EDGES_SLAB = ctx->rho (any mask); VM_EDGES_IMPLICIT = what
 * vm_materialize_rows evaluates (tab_p, tab_q, layer_consts, utile_ptr, u_col, rho_u32; VM_ENOTSUP under VM_R_CSR).  With
 * the implicit source, vm_edges_count first writes the per-layer column maxima of tab_q into `workspace`, which
 * vm_edges_emit reads: rows whose closed form provably has label 0 at every column then only visit their special ties.
 * VM_EINVAL before any launch for a NULL required pointer, an unknown `what` / `source`, n_trials < 1 (SAMPLE), or the slab
 * source without a slab. */
#define VM_EDGES_ARGMAX 0
#define VM_EDGES_THRESHOLD 1
#define VM_EDGES_SAMPLE 2
#define VM_EDGES_SLAB 0
#define VM_EDGES_IMPLICIT 1
typedef struct vm_edges_args {
  int64_t what, source;      /* VM_EDGES_ARGMAX / _THRESHOLD / _SAMPLE;  VM_EDGES_SLAB / _IMPLICIT */
  double threshold;          /* VM_EDGES_THRESHOLD: label = rho_1 >= (float)threshold */
  int64_t n_trials;          /* VM_EDGES_SAMPLE, >= 1 */
  uint64_t seed;             /* VM_EDGES_SAMPLE: the Philox key of vm_sample */
  int64_t* row_count;        /* [L*nloc], written by vm_edges_count */
  const int64_t* row_off;    /* [L*nloc], exclusive prefix sum of row_count, read by vm_edges_emit */
  int64_t* o_key;            /* [sum of row_count], written by vm_edges_emit */
  uint8_t* o_val;            /* [sum of row_count], written by vm_edges_emit */
  float* workspace;          /* [L*K], written by vm_edges_count, read by vm_edges_emit (implicit source) */
} vm_edges_args;
int64_t vm_edges_size(void);
int vm_edges_count(const vm_ctx* c, const vm_edges_args* a, void* stream);
int vm_edges_emit(const vm_ctx* c, const vm_edges_args* a, void* stream);

/* rho at given ties: out[q*K + k] = posterior of the tie key[q] = (l*N+i)*N+j, for every key of this rank's rows;
 * the outputs of other keys are not written.  source = VM_EDGES_SLAB (ctx->rho, any mask) or VM_EDGES_IMPLICIT
 * (what vm_materialize_rows evaluates; VM_ENOTSUP under VM_R_CSR).  Bit for bit the value the slab / vm_materialize_rows
 * holds for that tie.  n = 0 launches nothing.
 * One thread per query, in any order, duplicates allowed; a key outside [0, L*N*N) or outside the rows [row0, row0+nloc)
 * is skipped, so that on a sharded fit every rank answers the keys of its own rows into a zero-filled buffer and one
 * sum over the ranks combines them exactly.  The implicit source finds a special tie by a binary search of u_col within
 * its (row, column tile) segment of utile_ptr.  VM_EINVAL before any launch for n < 0, a NULL key / out with n > 0, an
 * unknown source, or the slab source without a slab. */
int vm_rho_at(const vm_ctx* c, int64_t source, int64_t n, const int64_t* key, float* out, void* stream);

/* ---- data packing (replaces the data preparation of `__check_fit_params`, model.py:147-176, and utils.py:73-84) --------
 * From the COO list of reports (device arrays) to every packed array `vm_ctx` points to, for one node-row block and a
 * structured reporter mask (VM_R_EGO / VM_R_ALL; a general COO mask is packed by the host-side packer): entries outside
 * the block's needs are dropped, ONE radix sort by (l,i,j,m) puts the reports in tie order, a binary search pairs each
 * with its reciprocal X[l,j,i,m], head flags + prefix sums give the special ties (+ the diagonal ties of an ego mask),
 * their dense-tile pointers, classes (shortcut / not), the E0/E1 split, the reporter-sorted copies and chunk tables of
 * the gamma pass and the transposed-position list of the ELBO.  No host synchronisation inside; the caller allocates
 * every output by the upper bounds below and reads `counts` (device int64[16]) once the stream has drained:
 *   counts[0..8] = U, I, I1, IT, n_cx, n_gchunk, max special ties per layer, max E1 entries per layer, max cx per layer
 *   counts[9] != 0: duplicate entries; counts[10] != 0: subscripts outside the shape;
 *   counts[11] = sum of the counts of the owned entries; counts[12] = b_all (integer).
 * Capacities: cap_e >= n_in; cap_u >= n_in + L*nloc (ego) ; cap_g >= n_in/256 + L*M + 1. */
typedef struct vm_pack_args {
  int64_t L, N, M, K, row0, nloc, tile_h;
  int64_t r_mode, ego_diag;  /* VM_R_EGO / VM_R_ALL; EGO: the mask contains the (m,m) ties */
  int64_t mutuality, split_e0;
  int64_t simple, single;    /* classify SIMPLE / SINGLE shortcut ties (see vm_ctx.simple_mode) */
  int64_t n_in;              /* reports given */
  const int32_t* x_l; const int32_t* x_i; const int32_t* x_j; const int32_t* x_m; const int32_t* x_v;
  const uint8_t* rep;        /* EGO: [L*M] reporter is active */
  int64_t cap_e, cap_u, cap_g;
  int32_t* e_u; int32_t* e_m; float* e_x; float* e_xT; uint8_t* e_flags;
  int32_t* e_src;            /* [cap_e] position of the owned entry in the caller's list */
  int32_t* f_u; int32_t* f_m; float* f_x; float* f_xT;
  int32_t* g_u; float* g_x; float* g_xT;
  int32_t* u_lrow; int32_t* u_col; int32_t* u_cnt; int32_t* u_m0;
  float* u_x0; float* u_xT0; float* u_x0sum; float* u_px; float* u_pxt;
  int64_t* u_ptr;            /* [cap_u+1] */
  uint8_t* u_has_x; uint8_t* u_reported;
  int64_t* u_gflat;          /* [cap_u] global flat id (l*N+i)*N+j of the tie (for injecting a prior keyed by tie) */
  int32_t* utile_ptr;        /* [L*nloc*nct+1] */
  int32_t* cx_idx; int64_t* cx_ptr; int32_t* cx_lrow; int32_t* cx_col; int32_t* cx_cnt; int32_t* cx_m0;
  float* cx_x0; float* cx_xT0; float* cx_x0sum;
  int64_t* lay_eptr;         /* [L+1] */
  double* g0;                /* [L*M] */
  int64_t* g_chunk_ptr;      /* [cap_g+1] */
  int32_t* g_chunk_lm;       /* [cap_g] */
  int64_t* g_lm_cptr;        /* [L*M+1] */
  int32_t* t_u; int32_t* t_lrow; int32_t* t_col; float* t_x;
  int64_t* counts;           /* [16] device */
  void* workspace; int64_t workspace_bytes;
} vm_pack_args;
int64_t vm_pack_size(void);
int64_t vm_pack_workspace_bytes(const vm_pack_args* p);
int vm_pack(const vm_pack_args* p, void* stream);

/* ---- device-side synthetic reports (the "next" row f2 of SURVEY.md section 8) ----------------------------------------
 * Samples the observed network X of the reference's `_build_X` under the self-reporter (ego) mask
 * (synthetic.py:138-209; mask synthetic.py:1184-1204) for ONE node-row block [row0, row0+nloc), sparsely, with a
 * counter-based RNG keyed by (seed, layer, reporter, partner): every rank generates exactly the entries of its own rows
 * (plus, with emit_transposed, the reciprocal entries X[l,j,i,m] whose row j it does not own, so that its shard pairs
 * without any exchange), and all ranks agree on every entry.  Output: unordered COO (o_l,o_i,o_j,o_m,o_x); *counter = the
 * number of entries produced -- if it exceeds `cap` the arrays hold only the first `cap` and the caller retries with more room. */
typedef struct vm_synth {
  int64_t L, N, M, K;
  int64_t row0, nloc;
  int64_t emit_transposed;   /* also emit X[l,j,i,m] for owned (i,j) when row j is not owned */
  uint64_t seed;
  double eta;                /* mutuality of the reports, in [0,1) */
  const double* theta;       /* [L*M] reporter reliabilities */
  const double* lam;         /* [L*K] average interactions per ground-truth category (lam[l,0]: no tie), or NULL for the
                                reference generator's default 0.01, 1, 2, .. (synthetic.py:140-157) */
  const int64_t* y_key;      /* [nY] sorted keys (l*N+i)*N+j of the true ties Y (ground truth, a few per node) */
  const int32_t* y_val;      /* [nY] Y_lij >= 1 */
  int64_t nY;
  int64_t cap;               /* capacity of the output arrays */
  int32_t* o_l; int32_t* o_i; int32_t* o_j; int32_t* o_m; int32_t* o_x;
  int64_t* counter;          /* [1] device */
} vm_synth;
int64_t vm_synth_size(void);
int vm_synth_ego(const vm_synth* s, void* stream);

/* Special functions exposed for testing the device implementations against scipy. */
int vm_test_special(const double* x, double* out_digamma, double* out_lgamma, int64_t n, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* VIMURE_B200_H */
