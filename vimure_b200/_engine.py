"""Host-side driver of the CUDA CAVI kernels: owns the device buffers (PyTorch tensors = plumbing),
fills the `vm_ctx` of include/vimure_b200.h and calls the extern "C" launchers.

One engine = one rank's shard (node-row block) of one fit.  An iteration that does not store the slab (VM_F_NO_STORE)
leaves the posterior implicit in the row/column tables and the special ties' rho_u32, bit-identical to what a storing
one writes.  With `slab=False` the engine holds no dense posterior slab: every iteration runs so, and the consumers
evaluate the posterior block by block (`vm_materialize_rows`).  With `group` set, the three statistics vectors
(red1: gamma-shape sums, red2: phi-shape sums, red3: A + nu + ELBO sums) are all-reduced with
torch.distributed (NCCL over NVLink on the GPU box) between the phases -- the only exchange the path needs
(SURVEY.md section 8e).  There is no CPU fallback: without CUDA the constructor raises.
"""
import ctypes

import numpy as np
import torch

from . import _capi
from ._pack_native import dense_fast_eligible


def _packing_const():
    from ._pack_native import SPECIAL_TIES_PER_BLOCK

    return SPECIAL_TIES_PER_BLOCK


# rows of posterior the consumers of a slab-free engine materialise at a time: at most this many bytes
IMPLICIT_BLOCK_BYTES = 256 << 20

# the buffers that hold the implicit posterior of a slab-free engine (what `vm_materialize_rows` reads besides the packed
# data)
IMPLICIT_STATE = ("tab_p", "tab_q", "layer_consts", "rho_u32")


class CaviEngine:
    def __init__(self, packed, priors, mutuality=True, eps=1e-12, group=None, may_dead=False, slab=True, all32=True,
                 gamma_ts=True):
        """`all32` and `gamma_ts` permit the fp32 special-tie kernel and the tie-sorted gamma pass of an all-reporter
        mask where the problem allows them; `False` keeps the fp64 special-tie kernel / the reporter-sorted gamma pass,
        the references the tests compare them against."""
        P = self.P = packed
        if not torch.cuda.is_available():
            raise RuntimeError("vimure_b200 needs a CUDA device: the CAVI kernels have no CPU fallback")
        self.lib = _capi.load()
        self.C = _capi.consts()
        self.group = group
        L, N, M, K, nloc = P.L, P.N, P.M, P.K, P.nloc
        if not (2 <= K <= self.C["VM_MAX_K"]):
            raise ValueError("vimure_b200 supports 2 <= K <= %d (got K=%d)" % (self.C["VM_MAX_K"], K))
        dev = self.dev = P.t["u_lrow"].device
        if dev.type != "cuda":
            raise RuntimeError("packed data must live on a CUDA device")
        self.mutuality = bool(mutuality)
        self.slab = bool(slab)
        if not self.slab and P.r_mode == 2:
            raise ValueError("a fit without the dense slab needs an ego or all-reporter mask (the general mask's "
                             "statistics gather the slab)")
        if self.mutuality and not P.mutuality:
            raise ValueError("the data were packed for mutuality=False (no entry visits the gamma/phi passes)")
        f64 = dict(dtype=torch.float64, device=dev)
        f32 = dict(dtype=torch.float32, device=dev)

        def bcast(v, shape):
            return torch.as_tensor(np.broadcast_to(np.asarray(v, dtype=np.float64), shape).copy(), **f64).contiguous()

        self.alpha_theta = bcast(priors["alpha_theta"], (L, M))
        self.beta_theta = bcast(priors["beta_theta"], (L, M))
        self.alpha_lambda = bcast(priors["alpha_lambda"], (L, K))
        self.beta_lambda = bcast(priors["beta_lambda"], (L, K))
        self.alpha_eta, self.beta_eta = float(priors["alpha_eta"]), float(priors["beta_eta"])

        z = lambda *s: torch.zeros(*s, **f64)  # noqa: E731
        self.gamma_shp, self.gamma_rte = z(L, M), z(L, M)
        self.phi_shp, self.phi_rte = z(L, K), z(L, K)
        self.nu = z(self.C["VM_NU_LEN"])
        self.G_theta, self.E_theta, self.Elog_theta = z(L, M), z(L, M), z(L, M)
        self.G_lambda, self.E_lambda, self.Elog_lambda = z(L, K), z(L, K), z(L, K)
        self.GE_theta = z(L, M, 2)
        U = P.U
        self.u_logpr = z(max(U, 1), K)
        self.rho_u = z(max(U, 1), K)
        self.rho_u32 = torch.zeros(max(U, 1), K, **f32)
        self.delta_u = z(max(U, 1), K)
        self.rho = torch.empty(L, nloc, N, K, **f32) if self.slab else None
        self.rho_valid = False
        self.block_rows = max(1, IMPLICIT_BLOCK_BYTES // (N * K * 4))  # consumers of a slab-free engine
        # workspaces
        self.layer_consts = z(L * (3 * K + 5))
        self.tab_p = torch.zeros(L * nloc * K, **f32)
        self.tab_q = torch.zeros(L * N * K, **f32)
        self.rowpart = torch.zeros(L * nloc * P.nct * K, **f32)
        self.colpart = torch.zeros(L * P.nrt * N * K, **f32)
        self.er_node = z(L * N)
        self.colsum = z(L * M * K)
        self.dev_flags = torch.zeros(8, dtype=torch.int64, device=dev)
        self.fixA = torch.zeros(L * M * K, dtype=torch.int64, device=dev)
        self.fixG = torch.zeros(L * M, dtype=torch.int64, device=dev)
        self.phi0 = z(L * K)
        # simple special ties (see include/vimure_b200.h): patch source of the fast dense kernel, their phi0 part
        self.simple_mode = bool(P.simple_ok)
        self.u_rec = torch.zeros(max(U, 1) if self.simple_mode else 1, 4 if K == 2 else 8, **f32)
        stride = 4 if K == 2 else (8 if K <= 6 else K + 2)
        self.nodetab = torch.zeros(L * N * stride if self.simple_mode else 4, **f32)
        self.fixP = torch.zeros(L * K, dtype=torch.int64, device=dev)
        self.simple_consts = z(3 + K)
        # all-reporter mask: every special tie in fp32 on iterations without ELBO (k_all32, see the header)
        self.all32_mode = bool(all32 and P.r_mode == 1 and K <= 4 and M <= 4096 and U > 0 and P.split_e0)
        self.u_lo = torch.zeros(max(U, 1) * K if self.all32_mode else 1, **f32)
        self.gfpart = z(L * ((M + 255) // 256) * (K + 4))
        # fork/join events of the aux stream, created once (vm_ctx.ev_fork / ev_join)
        self._ev_fork, self._ev_join = torch.cuda.Event(), torch.cuda.Event()
        self._ev_fork.record()
        self._ev_join.record()
        self.cx_logpr = z(max(P.n_cx, 1) if self.simple_mode else 1, K)
        assert _packing_const() == self.C["VM_SPECIAL_TIES_PER_BLOCK"]
        # tie-sorted gamma pass (vm_ctx.gamma_ts): few reporters, counts small enough for its 2^-30 fixed point
        self.gamma_ts = bool(gamma_ts and P.r_mode == 1 and K <= 8 and M <= 256 and P.I1 > 0
                             and float(P.t["f_x"].max()) < 2.0 ** 19)
        n_blk = max(P.n_gchunk, L * P.n_phichunk * K, (L * P.n_phichunk * M) if self.gamma_ts else 0,
                    L * P.n_ublk * 8 * (3 + 2 * K) + P.nct * L * P.nrt + 128 + 2 * 64 + L * 64 * (3 + K)) + 64
        self.blkpart = z(n_blk)
        self.red1, self.red2 = z(L * M), z(L * K)
        self.red3 = z(L * M * K + self.C["VM_R3_EXTRA"])
        self.elbo_out = z(8)
        self._dummy = torch.zeros(8, dtype=torch.int64, device=dev)

        Ctx = _capi.ctx_class()
        c = self.ctx = Ctx()
        for name in ("L", "N", "M", "K", "row0", "nloc", "U", "I", "I1", "IT", "tile_w", "tile_h", "nct", "nrt", "n_gchunk",
                     "phi_chunk", "n_phichunk", "n_ublk", "n_cx", "n_cxblk", "r_mode", "ego_diag"):
            setattr(c, name, int(getattr(P, name)))
        c.mutuality = int(self.mutuality)
        c.may_dead = int(bool(may_dead))
        c.eps = float(eps)
        c.alpha_eta, c.beta_eta = self.alpha_eta, self.beta_eta
        c.b_all = float(P.b_all)
        c.simple_mode = int(self.simple_mode)
        c.all32_mode = int(self.all32_mode)
        c.gamma_ts = int(self.gamma_ts)
        # the aux stream carries the general dense kernel (partial column tiles) under the fast one (see launch_dense)
        self.aux_stream = torch.cuda.Stream(device=dev)
        c.aux_stream = self.aux_stream.cuda_stream
        self._keep = []

        def ptr(t):
            self._keep.append(t)
            return t.data_ptr() if t.numel() else self._dummy.data_ptr()

        for name in ("u_lrow", "u_col", "u_ptr", "u_cnt", "u_m0", "u_x0", "u_xT0", "utile_ptr", "e_u", "e_m", "e_x", "e_xT",
                     "e_flags", "f_u", "f_m", "f_x", "f_xT", "lay_eptr", "g0", "u_x0sum", "g_chunk_ptr", "g_chunk_lm", "g_u", "g_x", "g_xT", "g_lm_cptr", "t_u", "t_lrow",
                     "t_col", "t_x", "rep", "r_ptr", "r_m", "r_val", "c_ptr", "c_tie", "cx_idx", "cx_ptr", "cx_lrow", "cx_col", "cx_cnt",
                     "cx_m0", "cx_x0", "cx_xT0", "cx_x0sum", "u_px", "u_pxt"):
            setattr(c, name, ptr(P.t[name]) if name in P.t else self._dummy.data_ptr())
        for name in ("u_logpr", "alpha_theta", "beta_theta", "alpha_lambda", "beta_lambda", "gamma_shp", "gamma_rte",
                     "phi_shp", "phi_rte", "nu", "G_theta", "E_theta", "Elog_theta", "G_lambda", "E_lambda",
                     "Elog_lambda", "GE_theta", "rho_u", "rho_u32", "delta_u", "layer_consts", "tab_p", "tab_q",
                     "rowpart", "colpart", "er_node", "colsum", "dev_flags", "fixA", "fixG", "phi0", "blkpart", "red1", "red2", "red3",
                     "elbo_out", "u_rec", "nodetab", "fixP", "simple_consts", "cx_logpr", "gfpart", "u_lo"):
            setattr(c, name, ptr(getattr(self, name)))
        c.rho = ptr(self.rho) if self.slab else None
        c.A = self.red3.data_ptr()  # A aliases the (all-reduced) statistics vector
        c.ev_fork, c.ev_join = self._ev_fork.cuda_event, self._ev_join.cuda_event
        self._cref = ctypes.byref(c)
        self.n_launch = 0
        self._graphs = None  # flags -> captured CUDA graph of one iteration (small, launch-bound problems)
        self._capture_stream = None

    # ------------------------------------------------------------------ helpers
    def _stream(self):
        return ctypes.c_void_p(torch.cuda.current_stream(self.dev).cuda_stream)

    def _allreduce(self, t):
        if self.group is not None:
            torch.distributed.all_reduce(t, group=self.group if self.group is not True else None)

    def kernels_per_iteration(self, elbo=False, store=True):
        """Number of kernels of this library launched by one iteration (for bench.py's gpu_launches).
        gamma: partial, reduce | phi: gamma_finish, phi_partial, phi_reduce | rho: phi_finish, [tables], special,
        [dense_fast], dense, [col_reduce], stats, [elbo_b], sums_reduce | finish: [elbo_partial], finish."""
        P = self.P
        csr, ego = P.r_mode == 2, P.r_mode == 0
        fast = dense_fast_eligible(P.K, P.r_mode, P.N, P.tile_w, P.tile_h)
        n = 2 + 3 + 1 + (0 if csr else 1) + 1 + (1 if fast else 0) + 1 + (1 if ego else 0) + 1 + 2 + 1
        if elbo:
            n += 1 + (1 if self.mutuality else 0)
        elif self.simple_mode and fast:
            # the special-tie kernel is launched twice (layers that take the shortcut / that cannot) + k_patch_rest, which
            # only a stored slab needs
            n += 2 if store else 1
        elif self.all32_mode:
            n += 1  # k_all32 + the fp64 special-tie kernel for the layers whose guard fails
        return n

    # ------------------------------------------------------------------ state
    def set_state(self, gamma_shp, gamma_rte, phi_shp, phi_rte, nu_shp, nu_rte, pr_u, eps):
        """Inject the initial variational state (what `_initialize_priors`, model.py:561-605, draws) and the prior of
        the special ties; computes the caches and the initial statistics A from rho = pr_rho."""
        P = self.P
        f64 = dict(dtype=torch.float64, device=self.dev)
        self.gamma_shp.copy_(torch.as_tensor(np.asarray(gamma_shp, dtype=np.float64), **f64).reshape(P.L, P.M))
        self.gamma_rte.copy_(torch.as_tensor(np.asarray(gamma_rte, dtype=np.float64), **f64).reshape(P.L, P.M))
        self.phi_shp.copy_(torch.as_tensor(np.asarray(phi_shp, dtype=np.float64), **f64).reshape(P.L, P.K))
        self.phi_rte.copy_(torch.as_tensor(np.asarray(phi_rte, dtype=np.float64), **f64).reshape(P.L, P.K))
        nu = np.zeros(self.C["VM_NU_LEN"])
        nu[self.C["VM_NU_SHP"]], nu[self.C["VM_NU_RTE"]] = float(nu_shp), float(nu_rte)
        self.nu.copy_(torch.as_tensor(nu, **f64))
        if P.U:
            pr = (pr_u.to(**f64) if torch.is_tensor(pr_u) else torch.as_tensor(pr_u, **f64)).reshape(P.U, P.K)
            self.rho_u.copy_(pr)
            torch.add(pr, float(eps), out=self.u_logpr)  # log(pr_rho + EPS), model.py:559, without temporaries
            self.u_logpr.log_()
            if self.simple_mode:
                # constants of the shortcut ties: lo_k = log2((pr_k+EPS)/(pr_0+EPS)); prior of the others compacted
                sm = P.t["u_simple"] | P.t["u_single"]
                lp = self.u_logpr
                if P.n_cx:
                    torch.index_select(lp, 0, P.t["cx_idx"].to(torch.int64), out=self.cx_logpr)
                # per-tie record of the shortcut kernel: (col, X, +-x^T, lo_1..lo_{K-1})
                rec = self.u_rec
                rec[:, 0] = P.t["u_col"].to(torch.float32)  # exact below 2^24 nodes
                rec[:, 1] = P.t["u_px"]
                rec[:, 2] = P.t["u_pxt"]
                rec[:, 3:2 + P.K] = ((lp[:, 1:] - lp[:, :1]) * 1.4426950408889634).to(torch.float32)
                big = torch.full_like(lp[:, 0], 1e300)
                self.simple_consts[0] = torch.where(sm, lp[:, 0], big).min().clamp(max=0.0)
                self.simple_consts[1] = P.t["u_px"].max().to(torch.float64)
                self.simple_consts[2] = P.t["u_pxt"].abs().max().to(torch.float64)
                self.simple_consts[3:] = torch.where(sm[:, None], lp, big[:, None]).min(dim=0)[0].clamp(max=0.0)
            if self.all32_mode:
                lp = self.u_logpr
                ulo = self.u_lo.view(P.U, P.K)
                ulo[:, 0] = (lp[:, 0] * 1.4426950408889634).to(torch.float32)
                ulo[:, 1:] = ((lp[:, 1:] - lp[:, :1]) * 1.4426950408889634).to(torch.float32)
                # guard constants over ALL special ties: min log(pr_0+EPS); largest total count of a tie; largest x^T
                xt = torch.zeros(P.U, dtype=torch.float32, device=self.dev)
                if P.I:
                    xt.index_add_(0, P.t["e_u"].to(torch.int64), P.t["e_x"])
                self.simple_consts[0] = lp[:, 0].min().clamp(max=0.0)
                self.simple_consts[1] = xt.max().to(torch.float64)
                self.simple_consts[2] = (P.t["e_xT"].abs().max() if P.I else torch.zeros((), device=self.dev)).to(torch.float64)
                self.simple_consts[3:] = lp.min(dim=0)[0].clamp(max=0.0)
        st = self._stream()
        _capi.check(self.lib.vm_refresh_cache(self._cref, st), "vm_refresh_cache")
        _capi.check(self.lib.vm_init_stats(self._cref, st), "vm_init_stats")
        self._allreduce(self.red3)
        _capi.check(self.lib.vm_phase_finish(self._cref, self.C["VM_F_INIT"], st), "vm_phase_finish")
        self.rho_valid = False
        self.rho_is_prior = True

    # ------------------------------------------------------------------ iterations
    def _flags(self, store=True, elbo=False):
        """vm_* flags of an iteration that stores the slab if `store` (an engine without a slab never does) and
        evaluates the ELBO if `elbo`."""
        F = self.C
        return (0 if store and self.slab else F["VM_F_NO_STORE"]) | (F["VM_F_ELBO"] if elbo else 0)

    def iterate(self, n=1, elbo_last=False, store=True, store_last=True):
        """Run n CAVI iterations; the last one also evaluates the ELBO if `elbo_last`.  Only the iterations with `store`
        (the last one: `store or store_last`) write the slab; every statistic is the same either way.
        Returns nothing; read `elbo()` after an ELBO iteration (one D2H scalar)."""
        if n <= 0:
            return
        nost = self.C["VM_F_NO_STORE"]
        base, last = self._flags(store), self._flags(store or store_last, elbo_last)
        st = self._stream()
        if self._graphs is not None:
            for it in range(n):
                self._graph(last if it == n - 1 else base).replay()
        elif self.group is None:
            _capi.check(self.lib.vm_run(self._cref, int(n), base, last, st), "vm_run")
        else:
            for it in range(n):
                self._sharded_iteration(last if it == n - 1 else base)
        self.n_launch += (n - 1) * self.kernels_per_iteration(False, not (base & nost)) + \
            self.kernels_per_iteration(elbo_last, not (last & nost))
        self.rho_valid = not (last & nost)
        self.rho_is_prior = False

    def _sharded_iteration(self, flags):
        """One iteration of a row-block shard: the four phases with the three statistics all-reduces between them."""
        st = self._stream()
        _capi.check(self.lib.vm_phase_gamma(self._cref, st), "vm_phase_gamma")
        self._allreduce(self.red1)
        _capi.check(self.lib.vm_phase_phi(self._cref, st), "vm_phase_phi")
        self._allreduce(self.red2)
        _capi.check(self.lib.vm_phase_rho(self._cref, int(flags), st), "vm_phase_rho")
        self._allreduce(self.red3)
        _capi.check(self.lib.vm_phase_finish(self._cref, int(flags), st), "vm_phase_finish")

    def enable_graphs(self):
        """Replay one captured CUDA graph per iteration instead of ~17 launches.  On a sharded fit the graph holds the
        whole iteration INCLUDING the three NCCL all-reduces (every rank captures the same sequence), so that nothing
        waits for the host between the phases.  Returns False, and leaves the engine on eager launches, for a sharded fit
        whose backend is not NCCL.  An engine on which this is never called runs eagerly (`fit(graphs=False)`)."""
        # only NCCL collectives are stream operations that a graph can hold (gloo reduces on the host)
        if self.group is not None and torch.distributed.get_backend() != "nccl":
            return False
        if self._graphs is None:
            self._graphs = {}
        return self._graphs is not None

    def prepare_graphs(self, store=True):
        """Capture the graphs `iterate(..., elbo_last=True, store=store, store_last=True)` replays, up front (a capture
        synchronises the device: do it before several engines start to run side by side on their own streams)."""
        if self._graphs is not None:
            for flags in (self._flags(store), self._flags(elbo=True)):
                self._graph(flags)

    def _graph(self, flags):
        g = self._graphs.get(flags)
        if g is None:
            import time

            t_cap = time.time()
            # Explicit capture_begin/capture_end on a side stream instead of the `torch.cuda.graph` context manager: that
            # one runs gc.collect() and torch.cuda.empty_cache() on entry (hundreds of ms once the caching allocator holds
            # many blocks), which a capture that allocates nothing does not need.  Capture only: nothing executes, the
            # state does not advance.
            g = torch.cuda.CUDAGraph()
            cur = torch.cuda.current_stream(self.dev)
            if self._capture_stream is None:
                self._capture_stream = torch.cuda.Stream(device=self.dev)
            side = self._capture_stream
            side.wait_stream(cur)
            with torch.cuda.stream(side):
                g.capture_begin(capture_error_mode="thread_local")
                rc = 0
                try:
                    if self.group is None:
                        rc = self.lib.vm_iteration(self._cref, int(flags), self._stream())
                    else:
                        self._sharded_iteration(flags)
                finally:
                    g.capture_end()
                _capi.check(rc, "vm_iteration (capture)")
            cur.wait_stream(side)
            self._graphs[flags] = g
            self.capture_s = getattr(self, "capture_s", 0.0) + time.time() - t_cap
        return g

    # single phases, for tests that emulate several ranks on one GPU
    def phase(self, name, flags=0):
        st = self._stream()
        fn = getattr(self.lib, "vm_phase_" + name)
        flags = int(flags) | self._flags()
        if name in ("rho", "finish"):
            _capi.check(fn(self._cref, flags, st), "vm_phase_" + name)
        else:
            _capi.check(fn(self._cref, st), "vm_phase_" + name)
        if name == "rho":
            self.rho_valid = not (flags & self.C["VM_F_NO_STORE"])
            self.rho_is_prior = False

    def dense_only(self, flags=0):
        """Launch only the per-tie dense kernel (measurement hook, see vm_dense_only)."""
        _capi.check(self.lib.vm_dense_only(self._cref, int(flags) | self._flags(), self._stream()), "vm_dense_only")
        self.n_launch += 1

    def elbo(self):
        return float(self.elbo_out[0].item())

    def elbo_terms(self):
        return self.elbo_out.cpu().numpy()

    # ------------------------------------------------------------------ results
    def params(self):
        """Small posterior parameters as numpy (one D2H each; a few KB .. MB)."""
        C = self.C
        nu = self.nu.cpu().numpy()
        return dict(
            gamma_shp=self.gamma_shp.cpu().numpy().copy(), gamma_rte=self.gamma_rte.cpu().numpy().copy(),
            phi_shp=self.phi_shp.cpu().numpy().copy(), phi_rte=self.phi_rte.cpu().numpy().copy(),
            nu_shp=np.float64(nu[C["VM_NU_SHP"]]), nu_rte=np.float64(nu[C["VM_NU_RTE"]]),
            G_exp_theta=self.G_theta.cpu().numpy().copy(), G_exp_lambda=self.G_lambda.cpu().numpy().copy(),
            G_exp_nu=np.float64(nu[C["VM_NU_G_STALE"]]),
        )

    def rho_slab(self, state=None):
        """The dense posterior slab of this rank, float32 (L, nloc, N, K), on the device.  Without a slab it is evaluated
        into a new tensor (from `state`, a `snapshot()`, if given)."""
        if not self.slab:
            old = self._use_slab(state)
            try:
                return self.materialize_rows(0, self.P.L * self.P.nloc).view(self.P.L, self.P.nloc, self.P.N, self.P.K)
            finally:
                self._restore(old)
        if not self.rho_valid:
            if getattr(self, "rho_is_prior", False):
                _capi.check(self.lib.vm_materialize_prior(self._cref, self._stream()), "vm_materialize_prior")
                self.n_launch += 2
                self.rho_valid = True
            else:
                raise RuntimeError("the dense rho slab was not stored in the last iteration (store=False)")
        return self.rho

    def materialize_rows(self, lrow0, nrows, out=None):
        """The posterior of local rows [lrow0, lrow0+nrows) (lrow = l*nloc + i) as the slab holds it after the last rho
        update: float32 (nrows, N, K) on the device (`vm_materialize_rows`)."""
        P = self.P
        if out is None:
            out = torch.empty(nrows, P.N, P.K, dtype=torch.float32, device=self.dev)
        _capi.check(self.lib.vm_materialize_rows(self._cref, int(lrow0), int(nrows), ctypes.c_void_p(out.data_ptr()),
                                                 self._stream()), "vm_materialize_rows")
        self.n_launch += 1
        return out

    def snapshot(self):
        """Copy of the implicit posterior of a slab-free engine (row/column tables, layer constants, rho_u32: O(N + U)
        floats) -- what a storing engine would clone its slab for.  `infer(..., slab=snapshot)` etc. read it."""
        assert not self.slab
        self._check_posterior()
        return {name: getattr(self, name).clone() for name in IMPLICIT_STATE}

    def _check_posterior(self):
        if getattr(self, "rho_is_prior", True):
            raise RuntimeError("no posterior yet: a fit without the dense slab has none before its first iteration")

    def _use_slab(self, slab):
        """Point the consumers at `slab` (a copy of an earlier restart's posterior: a slab tensor, or a `snapshot()` of a
        slab-free engine) instead of the engine's own; returns what `_restore` puts back."""
        if not self.slab:
            if slab is None:
                self._check_posterior()
                return {}
            old = {name: getattr(self.ctx, name) for name in IMPLICIT_STATE}
            for name in IMPLICIT_STATE:
                setattr(self.ctx, name, slab[name].data_ptr())
            return old
        old = {"rho": self.ctx.rho}
        if slab is None:
            self.rho_slab()
        else:
            self.ctx.rho = slab.data_ptr()
        return old

    def _restore(self, old):
        for name, v in old.items():
            setattr(self.ctx, name, v)

    def _consume(self, fn, out, what, *args):
        """Run the slab consumer `fn(ctx, *args, out)`: on the slab, or, without one, row block by row block on a
        materialised block, through a view of the ctx that covers the block only (L = 1, nloc = its rows; the row offset
        l*N + row0 + i0 keeps the global tie ids (l*N+i)*N+j that key vm_sample's stream)."""
        if self.slab:
            _capi.check(fn(self._cref, *args, ctypes.c_void_p(out.data_ptr()), self._stream()), what)
            self.n_launch += 1
            return out
        P = self.P
        rb = min(P.nloc, self.block_rows)
        buf = torch.empty(rb, P.N, P.K, dtype=torch.float32, device=self.dev)
        view = _capi.ctx_class()()
        ctypes.memmove(ctypes.byref(view), self._cref, ctypes.sizeof(view))
        for l in range(P.L):
            for i0 in range(0, P.nloc, rb):
                n = min(rb, P.nloc - i0)
                self.materialize_rows(l * P.nloc + i0, n, buf)
                view.L, view.nloc, view.nrt = 1, n, -(-n // P.tile_h)
                view.row0 = l * P.N + P.row0 + i0
                view.rho = buf.data_ptr()
                _capi.check(fn(ctypes.byref(view), *args, ctypes.c_void_p(out[l, i0].data_ptr()), self._stream()), what)
                self.n_launch += 1
        return out

    def infer(self, mode=0, threshold=0.5, slab=None):
        """argmax_k rho (mode 0) or rho[...,1] >= threshold (mode 1) on the device: uint8 (L, nloc, N)."""
        old = self._use_slab(slab)
        try:
            P = self.P
            out = torch.empty(P.L, P.nloc, P.N, dtype=torch.uint8, device=self.dev)
            return self._consume(self.lib.vm_infer, out, "vm_infer", int(mode), float(threshold))
        finally:
            self._restore(old)

    def infer_mean(self, slab=None):
        """sum_k k rho_k (reference `rho_mean`, model.py:1151-1153) on the device: float32 (L, nloc, N)."""
        old = self._use_slab(slab)
        try:
            P = self.P
            out = torch.empty(P.L, P.nloc, P.N, dtype=torch.float32, device=self.dev)
            return self._consume(self.lib.vm_infer_mean, out, "vm_infer_mean")
        finally:
            self._restore(old)

    def infer_edges(self, mode=0, threshold=0.5, slab=None):
        """The ties of `infer(mode, threshold, slab)` whose label is nonzero, as an edge list of this rank's rows: (keys
        int64 (l*N+i)*N+j ascending, labels uint8) on the device, without any (L, nloc, N) buffer (`vm_edges_*`)."""
        return self._edges(self.C["VM_EDGES_THRESHOLD"] if mode == 1 else self.C["VM_EDGES_ARGMAX"], slab,
                           threshold=float(threshold))

    def sample_edges(self, n_trials=1, seed=0, slab=None):
        """The ties of `sample(n_trials, seed, slab)` whose label is nonzero: (keys int64 ascending, labels uint8) on the
        device, this rank's rows."""
        return self._edges(self.C["VM_EDGES_SAMPLE"], slab, n_trials=int(n_trials), seed=int(seed) & (2**64 - 1))

    def _implicit_source(self, slab):
        """Where the per-tie consumers (`_edges`, `rho_at`) read the posterior: from the tables (implicit source) whenever
        they describe the posterior being consumed -- this engine's own after an iteration, slab or not, or a `snapshot()`
        -- and from a slab for a cloned slab of an earlier restart, the prior, and the general mask (which has no tables)."""
        return not self.slab or (slab is None and not getattr(self, "rho_is_prior", False) and self.P.r_mode != 2)

    def _edges(self, what, slab, **kw):
        """One vm_edges_count, the row offsets (one cumsum), one D2H read of the total, one vm_edges_emit.  The posterior is
        read where it is cheapest to evaluate (`_implicit_source`)."""
        C, P = self.C, self.P
        old = self._use_slab(slab)  # the dense consumers' preconditions (and the prior's slab, when that is the posterior)
        try:
            implicit = self._implicit_source(slab)
            rows = P.L * P.nloc
            i64 = dict(dtype=torch.int64, device=self.dev)
            off = torch.zeros(rows + 1, **i64)
            cnt = torch.empty(rows, **i64)
            ws = torch.empty(P.L * P.K, dtype=torch.float32, device=self.dev)
            a = _capi.edges_class()(what=what, source=C["VM_EDGES_IMPLICIT"] if implicit else C["VM_EDGES_SLAB"],
                                    row_count=cnt.data_ptr(), workspace=ws.data_ptr(), **kw)
            st = self._stream()
            _capi.check(self.lib.vm_edges_count(self._cref, ctypes.byref(a), st), "vm_edges_count")
            torch.cumsum(cnt, 0, out=off[1:])
            total = int(off[-1])
            keys = torch.empty(max(total, 1), **i64)
            vals = torch.empty(max(total, 1), dtype=torch.uint8, device=self.dev)
            a.row_off, a.o_key, a.o_val = off.data_ptr(), keys.data_ptr(), vals.data_ptr()
            _capi.check(self.lib.vm_edges_emit(self._cref, ctypes.byref(a), st), "vm_edges_emit")
            self.n_launch += 2 + int(implicit)
            return keys[:total], vals[:total]
        finally:
            self._restore(old)

    def rho_at(self, keys, slab=None):
        """The posterior at the ties `keys` (int64 device tensor of global ids (l*N+i)*N+j, any order, duplicates allowed)
        as the slab holds it: float32 (n, K) on the device (`vm_rho_at`), read from the source `_edges` reads.  Only the
        keys of this rank's rows are answered; the rows of the others are zero."""
        if not torch.is_tensor(keys) or keys.dtype != torch.int64 or keys.device != self.dev:
            raise ValueError("rho_at takes an int64 tensor of tie keys on the engine's device (%s)" % self.dev)
        keys = keys.reshape(-1).contiguous()
        old = self._use_slab(slab)
        try:
            C, n = self.C, keys.numel()
            out = torch.zeros(n, self.P.K, dtype=torch.float32, device=self.dev)
            source = C["VM_EDGES_IMPLICIT"] if self._implicit_source(slab) else C["VM_EDGES_SLAB"]
            _capi.check(self.lib.vm_rho_at(self._cref, source, n, ctypes.c_void_p(keys.data_ptr()),
                                           ctypes.c_void_p(out.data_ptr()), self._stream()), "vm_rho_at")
            self.n_launch += int(n > 0)
            return out
        finally:
            self._restore(old)

    def sample(self, n_trials=1, seed=0, slab=None):
        """argmax of the counts of `n_trials` categorical draws per tie (reference `sample_inferred_model`,
        model.py:1086-1088) on the device: uint8 (L, nloc, N).  Philox stream keyed by (seed, global tie id)."""
        old = self._use_slab(slab)
        try:
            P = self.P
            out = torch.empty(P.L, P.nloc, P.N, dtype=torch.uint8, device=self.dev)
            return self._consume(self.lib.vm_sample, out, "vm_sample", int(n_trials),
                                 ctypes.c_uint64(int(seed) & (2**64 - 1)))
        finally:
            self._restore(old)
