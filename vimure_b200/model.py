"""Inference model: a drop-in for `vimure.model.VimureModel` whose CAVI loop runs on a B200.

Upper face (unchanged from the reference, `src/python/vimure/model.py:28-448, 1062-1214`):
    VimureModel(undirected=False, mutuality=True, convergence_tol=0.1, decision=1, verbose=False)
    .fit(X, theta_prior=(0.1, 0.1), lambda_prior=(10., 10.), eta_prior=(0.5, 1.), rho_prior=None, seed=None,
         R=, K=, EPS=, bias0=, max_iter=, num_realisations=, alpha_lambda=, beta_lambda=, alpha_theta=, beta_theta=)
    .get_inferred_model(method, threshold) / .get_posterior_estimates() / .sample_inferred_model(N, seed)
and the posterior attributes rho, gamma_shp, gamma_rte, phi_shp, phi_rte, nu_shp, nu_rte, G_exp_*, *_f, trace, maxL.

Lower face: the extern "C" launchers of include/vimure_b200.h (through `_engine.CaviEngine`).  The host
code here only normalises the inputs, draws the initial state with the reference's RNG stream, drives the
iteration / convergence loop (`model.py:386-437, 1021-1056`) and copies the small posteriors back.

Extra, optional `fit` keywords (a superset of the reference's):
    init_state : dict with gamma_shp, gamma_rte, phi_shp, phi_rte, nu_shp and pr_ties (n,3) / pr_vals (n,K):
                 inject the initial state of the first realisation instead of drawing it (parity tests);
    init       : "reference" (bit-compatible RNG stream: consumes L*N*N*K draws like model.py:470),
                 "fast" (draws only for the ties that need them), or "auto" (reference when L*N*N*K <= 5e7);
    device     : CUDA device (default: current);
    distributed: "auto" | True | False -- shard the ties by node-row blocks over torch.distributed ranks;
    presharded : (sharded fits) X holds only THIS rank's entries instead of the whole list on every rank (sharded
                 ingestion); K must then be given.  True: every X[l,i,j,m] whose row i is in the rank's block AND every
                 reciprocal X[l,j,i,m] of those (each rank uploads, sorts and pairs about 2/G of the entries).
                 "rows": only the entries of the rank's own rows (1/G of the entries over PCIe); the reciprocal entries a
                 rank needs come from the rank that owns them, device to device (one all-to-all over NVLink);
    concurrent_realisations: "auto" | True | False -- run the `num_realisations` restarts (model.py:386-437) side by
                 side, one CUDA stream + one state per restart over the shared packed data, instead of one after the
                 other.  Same seeds, same trace, same best restart; "auto" = when an iteration is launch-bound
                 (L*N*N*K <= 2e7) and the restarts' posterior slabs fit together;
    store_rho  : True (default) -- keep the dense posterior slab rho (float32, 4*L*N*N*K bytes) on the device;
                 False -- write it at the ELBO iterations only (the other iterations run statistics-only kernels);
                 "never" -- never allocate it: the posterior stays implicit in O(N) row/column tables and the special
                 ties' posteriors, and `rho`, `rho_f`, `get_inferred_model`, `get_posterior_estimates` and
                 `sample_inferred_model` evaluate it block by block on demand; it lets a sparse network whose slab
                 exceeds the GPU's memory be fitted.  With False and "never", parameters, trace and every output are
                 bit-identical to the default.  Both need an ego or all-reporter mask (ValueError otherwise: the general
                 mask's statistics gather the slab).
"""
import os
import time
import warnings

import numpy as np
import pandas as pd
import torch
from scipy.stats import poisson
from sklearn.base import BaseEstimator, TransformerMixin

from . import _packing, masks
from ._engine import CaviEngine
from ._log import setup_logging
from .sptensor import is_sparse_like, sptensor
from .utils import get_optimal_threshold, match_arg

INF = 1e10
DEFAULT_EPS = 1e-12
DEFAULT_BIAS0 = 0.0
DEFAULT_MAX_ITER = 500
DEFAULT_NUM_REALISATIONS = 1
AUTO_REFERENCE_INIT_LIMIT = 5e7
GRAPH_LIMIT = 2e7  # below this many rho entries an iteration is launch-bound (restarts are then run side by side)
CONCURRENT_SLAB_BYTES = 8e9  # restarts run side by side only while their posterior slabs fit together in this many bytes


class VimureModel(TransformerMixin, BaseEstimator):
    """
    **ViMuRe** -- B200-native.

    Fit a probabilistic generative model to double sampled networks. It returns reliability parameters for the
    reporters (theta), average interactions for the links (lambda) and the estimate of the true and unknown
    network (rho). The inference is performed with a Variational Inference approach (CAVI).
    """

    def __init__(self, *, undirected: bool = False, mutuality: bool = True, convergence_tol: float = 0.1,
                 decision: int = 1, verbose: bool = False):
        # reference model.py:39-71
        self.undirected = undirected
        if undirected:
            warnings.warn("Overriding mutuality to False because the network is undirected")
            self.mutuality = False
        else:
            self.mutuality = mutuality
        self.convergence_tol = convergence_tol
        self.decision = decision
        self.verbose = verbose
        self.logger = setup_logging("vm.model.VimureModel", verbose)

    # ------------------------------------------------------------------ input normalisation
    def _check_fit_params(self, X, lambda_prior, theta_prior, eta_prior, rho_prior, seed, **extra_params):
        """Host-side restatement of `__check_fit_params` (reference model.py:79-325): same coercions, same
        warnings and ValueErrors, but X/R end up as COO arrays + a structured mask instead of sktensor objects."""
        available = ["R", "EPS", "K", "bias0", "max_iter", "alpha_lambda", "beta_lambda", "alpha_theta", "beta_theta",
                     "alpha_teta", "beta_teta", "num_realisations", "init_state", "init", "device", "distributed",
                     "store_rho", "tile_h", "graphs", "concurrent_realisations", "presharded"]
        for p in extra_params:
            if p not in available:
                self.logger.warning("Ignoring unrecognised parameter %s." % p)

        R_in = extra_params.get("R", None)
        K_in = extra_params.get("K", None)
        have_R = "R" in extra_params

        if isinstance(X, pd.DataFrame):  # reference model.py:107-124
            from .io import read_from_edgelist

            net_obj = read_from_edgelist(X)
            X = net_obj.X
            self.nodeNames = net_obj.nodeNames
            self.layerNames = net_obj.layerNames
            R_in, have_R = net_obj.R, True
            if K_in is None:
                K_in = net_obj.K

        # ---- X -> COO
        if is_sparse_like(X):
            shape = tuple(int(d) for d in X.shape)
            # no copies here: the packer moves each index array to the device in the narrowest integer type
            subs = tuple(np.asarray(s) for s in X.subs) if len(X.vals) else tuple(np.zeros(0, np.int64) for _ in range(4))
            vals = np.asarray(X.vals)
            for s_ in subs:
                if s_.dtype.kind not in "iu":
                    raise ValueError("Subscripts must be integers")
        elif isinstance(X, np.ndarray):
            Xd = np.asarray(X)
            if Xd.ndim != 4:
                raise ValueError("X has to be a tensor of dimensions L x N x N x M")
            if not Xd.dtype == np.dtype(int).type:
                Xd = Xd.astype(int)  # preprocess(), utils.py:241-242
            shape = Xd.shape
            nz = np.nonzero(Xd)
            subs = tuple(nz)
            vals = Xd[nz]
        else:
            raise ValueError("X must be a DataFrame, a numpy array or a sparse tensor with .subs/.vals/.shape")
        if len(shape) != 4 or shape[1] != shape[2]:
            raise ValueError("X has to be a tensor of dimensions L x N x N x M")
        self.L, self.N, self.M = int(shape[0]), int(shape[1]), int(shape[3])
        self.X = sptensor(tuple(subs), vals, shape=shape)
        self.subs_nz = self.X.subs
        self.sumX = None  # sum of all counts: from the packer (one rank) or a host sum (several), see fit

        # ---- K (model.py:179-196)
        if K_in is None:
            self.K = int(np.max(vals)) + 1
            warnings.warn(f"Parameter K was None. Defaulting to: {self.K}", UserWarning)
        else:
            self.K = int(K_in)

        # ---- R (model.py:199-213)
        if not have_R or R_in is None:
            msg = "Reporters Mask was not informed (parameter R). "
            msg += "The model will assume that every reporter can report on any tie."
            warnings.warn(msg, UserWarning)
            self.R = masks.AllMask(self.L, self.N, self.M)
        else:
            try:
                self.R = masks.from_input(R_in, self.L, self.N, self.M)
            except ValueError as e:
                self.logger.error(str(e))
                raise

        self.EPS = float(extra_params["EPS"]) if "EPS" in extra_params else DEFAULT_EPS
        self.bias0 = float(extra_params["bias0"]) if "bias0" in extra_params else DEFAULT_BIAS0
        self.max_iter = int(extra_params["max_iter"]) if "max_iter" in extra_params else DEFAULT_MAX_ITER
        self.num_realisations = (int(extra_params["num_realisations"]) if "num_realisations" in extra_params
                                 else DEFAULT_NUM_REALISATIONS)

        # ---- theta priors (model.py:238-266)
        if "alpha_theta" in extra_params or "beta_theta" in extra_params:
            self.alpha_theta = extra_params["alpha_theta"]
            self.beta_theta = extra_params["beta_theta"]
            if self.alpha_theta.shape != (self.L, self.M):
                msg = "alpha_theta matrix is not valid."
                msg += " When using this parameter, make sure to inform a %d x %d matrix."
                self.logger.error(msg)
                raise ValueError(msg % (self.L, self.M))
            if self.beta_theta.shape != (self.L, self.M):
                msg = "beta_theta matrix is not valid. When using this parameter, make sure to inform a %d x %d matrix."
                self.logger.error(msg)
                raise ValueError(msg % (self.L, self.M))
        else:
            if type(theta_prior) is not tuple or len(theta_prior) != 2:
                msg = "theta_prior must be a 2D tuple!"
                self.logger.error(msg)
                raise ValueError(msg)
            self.alpha_theta, self.beta_theta = theta_prior

        # ---- lambda priors (model.py:271-310)
        if "alpha_lambda" in extra_params or "beta_lambda" in extra_params:
            self.alpha_lambda = extra_params["alpha_lambda"]
            self.beta_lambda = extra_params["beta_lambda"]
            for nm, arr in (("alpha_lambda", self.alpha_lambda), ("beta_lambda", self.beta_lambda)):
                if arr.shape != (self.L, self.K):
                    msg = nm + " matrix is not valid (dimensions = %d x %d)."
                    msg += "When using this parameter, make sure to pass a %d x %d matrix."
                    msg = msg % (arr.shape[0], arr.shape[1], self.L, self.K)
                    self.logger.error(msg)
                    raise ValueError(msg)
        else:
            if type(lambda_prior) is not tuple or len(lambda_prior) != 2:
                msg = "lambda_prior must be a 2D tuple!"
                self.logger.error(msg)
                raise ValueError(msg)
            self.alpha_lambda, self.beta_lambda = lambda_prior

        if type(eta_prior) is not tuple or len(eta_prior) != 2:
            msg = "eta_prior must be a 2D tuple!"
            self.logger.error(msg)
            raise ValueError(msg)
        self.alpha_mutuality, self.beta_mutuality = eta_prior

        if rho_prior is not None and rho_prior.shape != (self.L, self.N, self.N):
            msg = "rho_prior has to have shape equal to (L, N, N)!"
            self.logger.error(msg)
            raise ValueError(msg)
        self.rho_prior = rho_prior

        self._change_seed(seed)

    def _change_seed(self, seed):
        self.seed = seed
        self.prng = np.random.RandomState(seed)

    # ------------------------------------------------------------------ fit
    def fit(self, X, theta_prior=(0.1, 0.1), lambda_prior=(10.0, 10.0), eta_prior=(0.5, 1.0), rho_prior=None,
            seed: int = None, **extra_params):
        """Fit the model (reference model.py:327-448).  Returns self."""
        t_fit = time.time()
        self._check_fit_params(X, lambda_prior=lambda_prior, theta_prior=theta_prior, eta_prior=eta_prior,
                               rho_prior=rho_prior, seed=seed, **extra_params)
        t_check = time.time() - t_fit
        dev = extra_params.get("device", None)
        if not torch.cuda.is_available():
            raise RuntimeError("vimure_b200.VimureModel.fit needs a CUDA device (B200); there is no CPU fallback")
        dev = torch.device("cuda", torch.cuda.current_device()) if dev is None else torch.device(dev)
        store_rho = extra_params.get("store_rho", True)
        if isinstance(store_rho, str) and store_rho != "never":
            raise ValueError('store_rho must be True, False or "never"')
        self._slab = not isinstance(store_rho, str)
        self._store_rho = self._slab and bool(store_rho)
        if not self._store_rho and self.R.kind not in ("ego", "all"):
            raise ValueError('store_rho=%r needs an ego or all-reporter mask: the statistics of a general reporter '
                             'mask gather the dense posterior slab' % (store_rho,))

        # ---- sharding (row blocks over ranks, SURVEY.md section 8e)
        dist_opt = extra_params.get("distributed", "auto")
        world, rank, group = 1, 0, None
        if dist_opt is True or (dist_opt == "auto" and torch.distributed.is_available()
                                and torch.distributed.is_initialized()):
            world, rank = torch.distributed.get_world_size(), torch.distributed.get_rank()
            group = True if world > 1 else None
        self._world, self._rank = world, rank
        row0, nloc = shard_rows(self.N, world, rank)
        if world > 1:
            # Every rank must draw the same initial gamma/phi/nu and derive the same restart seeds, or the replicated
            # parameters diverge and the ranks leave the loop at different iterations (a hang in the next all-reduce).
            # With seed=None the reference seeds from the OS; here rank 0 does and the others adopt its choice.
            self.prng = np.random.RandomState(_agree_int(
                int(np.random.SeedSequence().generate_state(1)[0] % (2**31 - 1)) if seed is None else int(seed), dev))

        self.timings = {"check_params": t_check}
        with torch.cuda.device(dev):
            t0 = time.time()
            # entries without a reciprocal report have a parameter-free Poisson allocation (dz1 = x) unless a prior is so
            # small that exp(E[log theta/lambda]) can underflow to exactly 0 (then model.py:692 applies): psi(0.01) ~ -100
            split_e0 = (not self.mutuality) or (float(np.min(self.alpha_theta)) >= 0.01 and
                                                float(np.min(self.alpha_lambda)) >= 0.01)
            presharded = extra_params.get("presharded", False) if world > 1 else False
            x_subs, x_vals = self.X.subs, self.X.vals
            if presharded == "rows":
                x_subs, x_vals = _exchange_reciprocals(x_subs, x_vals, self.N, world, rank, dev)
            self._packed = P = _packing.pack(x_subs, x_vals, self.L, self.N, self.M, self.K, self.R, dev,
                                             row0=row0, nloc=nloc, tile_h=int(extra_params.get("tile_h", 128)),
                                             mutuality=self.mutuality, split_e0=split_e0)
            # nu_rte = beta + sum X (model.py:593-595): the packer already summed the counts of the rows it owns
            if world == 1 and getattr(P, "sumX", None) is not None:
                self.sumX = float(P.sumX)
            elif not presharded:
                self.sumX = float(self.X.vals.sum())
            if presharded:
                # the sum of all counts (nu_rte = beta + sum X, model.py:593-595) from the ranks' own rows
                if "K" not in extra_params or extra_params["K"] is None:
                    raise ValueError("presharded=True needs K (a rank cannot see max(X))")
                t = torch.tensor([float(P.sumX_owned or 0.0)], dtype=torch.float64, device=dev)
                torch.distributed.all_reduce(t)
                self.sumX = float(t.item())
            if self.undirected:  # model.py:127-132: X must be symmetric in (i, j)
                asym = int(not bool(torch.all(P.t["e_xT"] == P.t["e_x"])))
                if world > 1:  # every rank raises, or none does
                    asym = _agree_int(asym, dev, op="max")
                if asym:
                    msg = "If undirected is True, the given network has to be symmetric wrt l and m!"
                    self.logger.error(msg)
                    raise ValueError(msg)
            if os.environ.get("VM_PACK_TRACE") == "1":
                torch.cuda.synchronize(dev)
                self.timings["pack"] = time.time() - t0
            priors = dict(alpha_theta=self.alpha_theta, beta_theta=self.beta_theta, alpha_lambda=self.alpha_lambda,
                          beta_lambda=self.beta_lambda, alpha_eta=self.alpha_mutuality, beta_eta=self.beta_mutuality)
            self._engine = eng = CaviEngine(P, priors, mutuality=self.mutuality, eps=self.EPS, group=group,
                                            slab=self._slab)
            if extra_params.get("graphs", True):
                # one graph replay per iteration instead of ~17 launches: decisive for launch-bound sizes, and still 1.6 %
                # at config 3 (1.377 -> 1.355 ms per iteration, B200); sharded fits capture their all-reduces too
                eng.enable_graphs()
            torch.cuda.synchronize(dev)
            self.pack_time = self.timings["pack+engine"] = time.time() - t0

            maxL = -INF
            trace = []
            self._rho_f_dev = None
            self._engine_f = None
            injected = extra_params.get("init_state", None)
            init_mode = extra_params.get("init", "auto")
            conc = extra_params.get("concurrent_realisations", "auto")
            small = float(self.L) * self.N * self.N * self.K <= GRAPH_LIMIT
            if conc == "auto":
                conc = small and float(self.L) * nloc * self.N * self.K * 4 * self.num_realisations <= CONCURRENT_SLAB_BYTES
            if conc and self.num_realisations > 1 and group is None:
                maxL, trace = self._fit_concurrent(P, priors, dev, injected, init_mode,
                                                   use_graphs=extra_params.get("graphs", True))
                cols = ["realisation", "seed", "iter", "elbo", "runtime", "reached_convergence"]
                self.trace = pd.DataFrame(trace, columns=cols)
                self.maxL = maxL
                self.timings["fit_total"] = time.time() - t_fit
                return self
            for r in range(self.num_realisations):
                bias0 = DEFAULT_BIAS0 if r < 5 else (r - 4) * self.bias0  # model.py:390-394
                t1 = time.time()
                if injected is not None and r == 0:
                    st = self._state_from_injection(injected)
                else:
                    st = self._draw_initial_state(bias0, init_mode)
                self.timings["draw_init"] = self.timings.get("draw_init", 0.0) + time.time() - t1
                t1 = time.time()
                eng.set_state(st["gamma_shp"], st["gamma_rte"], st["phi_shp"], st["phi_rte"], st["nu_shp"],
                              st["nu_rte"], st["pr_u"], self.EPS)
                self._pr_u = st["pr_u"]
                torch.cuda.synchronize(dev)
                self.timings["init_state"] = self.timings.get("init_state", 0.0) + time.time() - t1
                t_loop = time.time()

                coincide, it, reached, elbo = 0, 1, False, -INF
                while not reached and it <= self.max_iter:
                    # batch the iterations up to (and including) the next ELBO evaluation: no host sync in between
                    nxt = it
                    while not (nxt == 1 or nxt % 10 == 0 or nxt == self.max_iter):
                        nxt += 1
                    n = nxt - it + 1
                    torch.cuda.synchronize(dev)
                    t_start = time.time()
                    eng.iterate(n, elbo_last=True, store=self._store_rho, store_last=True)
                    new_elbo = eng.elbo()  # the one D2H scalar (also syncs)
                    if world > 1:  # identical on every rank by construction; rank 0's value decides all the same
                        new_elbo = _agree_float(new_elbo, dev)
                    runtime = (time.time() - t_start) / n
                    # `_check_for_convergence`, model.py:1036-1056
                    if np.isnan(new_elbo):
                        raise ValueError("ELBO is NaN!!!!")
                    old_L, elbo = elbo, new_elbo
                    coincide = coincide + 1 if abs(elbo - old_L) < self.convergence_tol else 0
                    if coincide > self.decision:
                        reached = True
                    if self.verbose:
                        self.logger.debug(f"Realisation {r:2} | Iter {nxt:4} | ELBO value: {elbo:6.12f} | "
                                          f"Reached convergence: {reached}")
                    it = nxt + 1
                    if (it - 1) % 10 == 0:  # model.py:423-426
                        trace.append((r, self.seed, it - 1, elbo, runtime, reached))
                self.n_iter_ = it - 1
                self.timings["cavi_loop"] = self.timings.get("cavi_loop", 0.0) + time.time() - t_loop
                self.timings["graph_capture"] = getattr(eng, "capture_s", 0.0)  # (part of cavi_loop)
                t1 = time.time()
                self._fetch_params()
                if maxL < elbo:
                    self._update_optimal_parameters()
                    maxL = elbo
                self.timings["fetch_results"] = self.timings.get("fetch_results", 0.0) + time.time() - t1
                new_seed = self.prng.randint(1, 500) if self.seed is None else self.seed + self.prng.randint(1, 500)
                self._change_seed(new_seed)

        cols = ["realisation", "seed", "iter", "elbo", "runtime", "reached_convergence"]
        self.trace = pd.DataFrame(trace, columns=cols)
        self.maxL = maxL
        self.timings["fit_total"] = time.time() - t_fit
        return self

    def _fit_concurrent(self, P, priors, dev, injected, init_mode, use_graphs):
        """The `num_realisations` restarts of reference model.py:386-437, run side by side (SURVEY.md section 8 f3).

        The reference's restarts are independent given their initial states, and its RNG is only consumed while a state
        is drawn (model.py:458-605) and when the next seed is derived (model.py:431-435) -- never inside the CAVI loop.
        So the states are drawn first, in the reference's order, and the loops then advance together: restart r owns a
        CUDA stream and an engine (state, special-tie posterior, dense slab) over the SHARED packed data; all restarts
        that are still running are launched up to their next ELBO evaluation before any ELBO is read back."""
        R = self.num_realisations
        states, seeds = [], []
        t1 = time.time()
        for r in range(R):
            bias0 = DEFAULT_BIAS0 if r < 5 else (r - 4) * self.bias0  # model.py:390-394
            st = self._state_from_injection(injected) if (injected is not None and r == 0) else \
                self._draw_initial_state(bias0, init_mode)
            states.append(st)
            seeds.append(self.seed)
            new_seed = self.prng.randint(1, 500) if self.seed is None else self.seed + self.prng.randint(1, 500)
            self._change_seed(new_seed)
        self.timings["draw_init"] = time.time() - t1

        t1 = time.time()
        engines = [self._engine] + [CaviEngine(P, priors, mutuality=self.mutuality, eps=self.EPS, slab=self._slab)
                                    for _ in range(R - 1)]
        streams = [torch.cuda.Stream(device=dev) for _ in range(R)]
        torch.cuda.synchronize(dev)  # the engines' buffers were zero-filled on the current stream
        for eng, st, s in zip(engines, states, streams):
            with torch.cuda.stream(s):
                eng.set_state(st["gamma_shp"], st["gamma_rte"], st["phi_shp"], st["phi_rte"], st["nu_shp"],
                              st["nu_rte"], st["pr_u"], self.EPS)
        torch.cuda.synchronize(dev)
        if use_graphs:
            for eng in engines:  # capture before anything runs asynchronously
                if eng.enable_graphs():
                    eng.prepare_graphs(store=self._store_rho)
        self.timings["init_state"] = time.time() - t1

        t_loop = time.time()
        run = [dict(coincide=0, it=1, reached=False, elbo=-INF, rows=[]) for _ in range(R)]
        active = list(range(R))
        while active:
            torch.cuda.synchronize(dev)
            t_start = time.time()
            batch = {}
            for r in active:
                it = nxt = run[r]["it"]
                while not (nxt == 1 or nxt % 10 == 0 or nxt == self.max_iter):
                    nxt += 1
                batch[r] = (nxt, nxt - it + 1)
                with torch.cuda.stream(streams[r]):
                    engines[r].iterate(nxt - it + 1, elbo_last=True, store=self._store_rho, store_last=True)
            for r in active:
                with torch.cuda.stream(streams[r]):
                    new_elbo = engines[r].elbo()
                nxt, n = batch[r]
                runtime = (time.time() - t_start) / n
                q = run[r]
                if np.isnan(new_elbo):
                    raise ValueError("ELBO is NaN!!!!")
                old_L, q["elbo"] = q["elbo"], new_elbo  # `_check_for_convergence`, model.py:1036-1056
                q["coincide"] = q["coincide"] + 1 if abs(q["elbo"] - old_L) < self.convergence_tol else 0
                if q["coincide"] > self.decision:
                    q["reached"] = True
                if self.verbose:
                    self.logger.debug(f"Realisation {r:2} | Iter {nxt:4} | ELBO value: {new_elbo:6.12f} | "
                                      f"Reached convergence: {q['reached']}")
                q["it"] = nxt + 1
                if nxt % 10 == 0:  # model.py:423-426
                    q["rows"].append((r, seeds[r], nxt, new_elbo, runtime, q["reached"]))
            active = [r for r in active if not run[r]["reached"] and run[r]["it"] <= self.max_iter]
        torch.cuda.synchronize(dev)
        self.timings["cavi_loop"] = time.time() - t_loop

        maxL, trace, best = -INF, [], None
        for r in range(R):  # the reference's bookkeeping, in the reference's order
            trace.extend(run[r]["rows"])
            if maxL < run[r]["elbo"]:
                maxL, best = run[r]["elbo"], r
        self.n_iter_ = run[R - 1]["it"] - 1
        self._pr_u = states[R - 1]["pr_u"]
        if best is not None:
            self._engine = engines[best]
            self._fetch_params()
            self._update_optimal_parameters(clone_rho=False)  # every restart keeps its own slab: nothing to copy
        self._engine = engines[R - 1]  # `rho`, `gamma_shp`, ... without _f are the LAST restart's (model.py:925-942)
        self._fetch_params()
        self._engine_f = engines[best] if best is not None else None
        # (without a slab the best engine's own tables are rho_f: nothing to materialise)
        self._rho_f_dev = engines[best].rho_slab() if (best is not None and best != R - 1 and self._slab) else None
        self._rho_f_cache = None
        return maxL, trace

    # ------------------------------------------------------------------ initial state
    def _special_tie_info(self):
        P = self._packed
        flat = P.t["u_gflat"].cpu().numpy()
        keep = (P.t["u_has_x"] & P.t["u_reported"]).cpu().numpy()  # ties that keep a random prior (model.py:536-556)
        return flat, keep

    def _draw_initial_state(self, bias0, init_mode):
        """`_set_rho_prior` + `_initialize_priors` (model.py:458-605) for the special ties only, consuming the
        reference's RNG stream in the reference's order when init == "reference"."""
        L, N, M, K = self.L, self.N, self.M, self.K
        P = self._packed
        U = P.U
        if init_mode == "auto":
            init_mode = "reference" if float(L) * N * N * K <= AUTO_REFERENCE_INIT_LIMIT else "fast"
        if init_mode not in ("reference", "fast"):
            raise ValueError("init must be 'reference', 'fast' or 'auto'")
        if init_mode == "fast" and self.rho_prior is None and not self.undirected:
            # device-side draw: only the ties that keep a random prior, nothing crosses PCIe
            dev = P.t["u_lrow"].device
            gen = torch.Generator(device=dev)
            gen.manual_seed(int(self.prng.randint(0, 2**31 - 1)))
            # in place, no host synchronisation: one draw per special tie, then the ties that keep the one-hot prior
            # (no X entry / not reported, model.py:536-556) are overwritten
            drop = ~(P.t["u_has_x"] & P.t["u_reported"])
            pr_u = torch.rand((U, K), generator=gen, dtype=torch.float64, device=dev)
            pr_u.mul_(0.01).add_(1.0)
            pr_u[:, 0] += bias0
            pr_u /= pr_u.sum(dim=-1, keepdim=True)
            pr_u.masked_fill_(drop[:, None], 0.0)
            pr_u[:, 0].masked_fill_(drop, 1.0)
            st = dict(pr_u=pr_u)
            self._draw_small_params(st)
            return st
        flat, keep = self._special_tie_info()
        pr_u = np.zeros((U, K))
        pr_u[:, 0] = 1.0
        kidx = np.nonzero(keep)[0]
        if self.rho_prior is None:
            if init_mode == "reference":
                want = flat[kidx]
                if self.undirected:  # also the transposed ties' draws (model.py:477-478)
                    l_ = want // (N * N)
                    i_ = (want // N) % N
                    j_ = want % N
                    wt = (l_ * N + j_) * N + i_
                    allw, inv = np.unique(np.concatenate([want, wt]), return_inverse=True)
                    d = _packing.reference_prior_draws(self.prng, L, N, K, allw)
                    u = 1 + 0.01 * d[inv[: len(want)]]
                    ut = 1 + 0.01 * d[inv[len(want):]]
                    u[:, 0] += bias0
                    ut[:, 0] += bias0
                    pr = (u + ut) / 2.0
                else:
                    pr = 1 + 0.01 * _packing.reference_prior_draws(self.prng, L, N, K, want)
                    pr[:, 0] += bias0
            else:
                # one draw of the host stream whatever the number of ties this rank owns, then a counter-based uniform
                # keyed by the GLOBAL tie (undirected: by the unordered pair, so that (i,j) and (j,i) get the same
                # prior, model.py:477-478, even when they live on different ranks)
                key0 = int(self.prng.randint(0, 2**31 - 1))
                tie = flat[kidx]
                if self.undirected:
                    l_ = tie // (N * N)
                    i_ = (tie // N) % N
                    j_ = tie % N
                    tie = (l_ * N + np.minimum(i_, j_)) * N + np.maximum(i_, j_)
                pr = 1 + 0.01 * _keyed_uniform(key0, tie, K)
                pr[:, 0] += bias0
            pr /= pr.sum(axis=-1)[:, None]
            pr_u[kidx] = pr
        else:
            # model.py:485-500: poisson pmf + uniform noise on the non-zeros of rho_prior; zero elsewhere
            rp = np.asarray(self.rho_prior)
            sub_nz = rp.nonzero()
            nz_flat = (sub_nz[0] * N + sub_nz[1]) * N + sub_nz[2]
            vals_nz = rp[sub_nz]
            dense_pr = np.zeros((len(nz_flat), K))
            for k in range(K):
                dense_pr[:, k] = poisson.pmf(k, vals_nz) + 1.0 * self.prng.rand(len(nz_flat))
            if self.undirected:
                pos = np.searchsorted(nz_flat, (sub_nz[0] * N + sub_nz[2]) * N + sub_nz[1])
                pos = np.minimum(pos, len(nz_flat) - 1)
                has_t = nz_flat[pos] == (sub_nz[0] * N + sub_nz[2]) * N + sub_nz[1]
                tr = np.where(has_t[:, None], dense_pr[pos], 0.0)
                dense_pr = (dense_pr + tr) / 2.0
            dense_pr /= dense_pr.sum(axis=-1)[:, None]
            pr_u[kidx] = 0.0
            if len(nz_flat):
                pos = np.minimum(np.searchsorted(nz_flat, flat[kidx]), len(nz_flat) - 1)
                hit = nz_flat[pos] == flat[kidx]
                pr_u[kidx[hit]] = dense_pr[pos[hit]]
        st = dict(pr_u=pr_u)
        self._draw_small_params(st)
        return st

    def _draw_small_params(self, st):
        """`_initialize_priors` (reference model.py:570-600): gamma/phi shapes and rates, nu."""
        L, M, K = self.L, self.M, self.K
        rs = self.prng.random_sample
        st["gamma_shp"] = self.alpha_theta * rs(size=(L, M)) + self.alpha_theta
        st["phi_shp"] = self.alpha_lambda * rs(size=(L, K)) + self.alpha_lambda
        st["gamma_rte"] = self.beta_theta * rs(size=(L, M)) + self.beta_theta
        st["phi_rte"] = self.beta_lambda * rs(size=(L, K)) + self.beta_lambda
        if self.mutuality:
            st["nu_shp"] = self.alpha_mutuality * rs(1)[0] + self.alpha_mutuality
            st["nu_rte"] = self.beta_mutuality + self.sumX
        else:
            st["nu_shp"], st["nu_rte"] = 0.000001, 1.0
        return st

    def _state_from_injection(self, inj):
        L, N, K = self.L, self.N, self.K
        P = self._packed
        flat, _ = self._special_tie_info()
        pr_u = np.zeros((P.U, K))
        pr_u[:, 0] = 1.0
        ties = np.asarray(inj.get("pr_ties", np.zeros((0, 3), dtype=np.int64))).astype(np.int64)
        if len(ties):
            tf = (ties[:, 0] * N + ties[:, 1]) * N + ties[:, 2]
            order = np.argsort(tf)
            tf, vals = tf[order], np.asarray(inj["pr_vals"], dtype=np.float64)[order]
            pos = np.minimum(np.searchsorted(tf, flat), len(tf) - 1)
            hit = tf[pos] == flat
            pr_u[hit] = vals[pos[hit]]
            # every injected tie owned by this rank must be a special tie
            own = (ties[:, 1] >= P.row0) & (ties[:, 1] < P.row0 + P.nloc)
            if int(hit.sum()) != int(own.sum()):
                raise ValueError("init_state: a prior was given for a tie that carries no X entry")
        st = dict(pr_u=pr_u)
        for k in ("gamma_shp", "gamma_rte", "phi_shp", "phi_rte"):
            st[k] = np.asarray(inj[k], dtype=np.float64)
        if self.mutuality:
            st["nu_shp"] = float(inj["nu_shp"])
            st["nu_rte"] = float(inj.get("nu_rte", self.beta_mutuality + self.sumX))
        else:
            st["nu_shp"], st["nu_rte"] = 0.000001, 1.0
        return st

    # ------------------------------------------------------------------ results
    def _fetch_params(self):
        p = self._engine.params()
        self.gamma_shp, self.gamma_rte = p["gamma_shp"], p["gamma_rte"]
        self.phi_shp, self.phi_rte = p["phi_shp"], p["phi_rte"]
        self.nu_shp, self.nu_rte = p["nu_shp"], p["nu_rte"]
        self.G_exp_theta, self.G_exp_lambda, self.G_exp_nu = p["G_exp_theta"], p["G_exp_lambda"], p["G_exp_nu"]
        if not self.mutuality:
            self.G_exp_nu = 0.0
        self._rho_cache = None
        self._pr_rho_cache = None

    def _update_optimal_parameters(self, clone_rho=True):
        """reference model.py:925-942"""
        import scipy.special as sp

        self.gamma_shp_f = np.copy(self.gamma_shp)
        self.gamma_rte_f = np.copy(self.gamma_rte)
        self.phi_shp_f = np.copy(self.phi_shp)
        self.phi_rte_f = np.copy(self.phi_rte)
        self.nu_shp_f = np.copy(self.nu_shp)
        self.nu_rte_f = np.copy(self.nu_rte)
        self.G_exp_theta_f = np.exp(sp.psi(self.gamma_shp_f) - np.log(self.gamma_rte_f))
        self.G_exp_lambda_f = np.exp(sp.psi(self.phi_shp_f) - np.log(self.phi_rte_f))
        self.G_exp_nu_f = np.exp(sp.psi(self.nu_shp_f) - np.log(self.nu_rte_f))
        # rho_f stays on the device; a copy is needed only when further realisations will overwrite the slab (without a
        # slab: the tables and special-tie posteriors it is evaluated from)
        if self.num_realisations > 1 and clone_rho:
            self._rho_f_dev = self._engine.rho_slab().clone() if self._engine.slab else self._engine.snapshot()
        else:
            self._rho_f_dev = None
        self._rho_f_cache = None

    def _gather_rho(self, slab):
        """Device slab (L, nloc, N, K) float32 -> full host array (L, N, N, K) float64."""
        if self._world > 1:
            slab = self._all_gather_rows(slab)
        return slab.cpu().numpy().astype(np.float64)

    @property
    def rho(self):
        """Posterior of the last realisation, (L, N, N, K) float64 -- materialised on the host on first access."""
        if getattr(self, "_rho_cache", None) is None:
            self._rho_cache = self._gather_rho(self._engine.rho_slab())
        return self._rho_cache

    @property
    def rho_f(self):
        """Posterior of the best realisation (reference model.py:937)."""
        if getattr(self, "_rho_f_cache", None) is None:
            eng_f = self._engine_of_rho_f()
            if self._rho_f_dev is None and eng_f is self._engine:
                self._rho_f_cache = self.rho
            else:
                self._rho_f_cache = self._gather_rho(self._rho_f_slab())
        return self._rho_f_cache

    def _rho_f_slab(self):
        eng_f = self._engine_of_rho_f()
        if self._rho_f_dev is None:
            return eng_f.rho_slab()
        return eng_f.rho_slab(self._rho_f_dev) if isinstance(self._rho_f_dev, dict) else self._rho_f_dev

    @property
    def pr_rho(self):
        """Prior of the last realisation as the reference's dense (L, N, N, K) array (model.py:558)."""
        if getattr(self, "_pr_rho_cache", None) is None:
            if self._world > 1:
                raise NotImplementedError("pr_rho is only materialised on single-rank fits")
            pr = np.zeros((self.L, self.N, self.N, self.K))
            pr[..., 0] = 1.0
            flat, _ = self._special_tie_info()
            pr_u = self._pr_u.cpu().numpy() if torch.is_tensor(self._pr_u) else self._pr_u
            pr.reshape(-1, self.K)[flat] = pr_u
            self._pr_rho_cache = pr
        return self._pr_rho_cache

    @property
    def logpr_rho(self):
        return np.log(self.pr_rho + self.EPS)

    @property
    def data_T_vals(self):
        """X[l,j,i,m] for every non-zero X[l,i,j,m], in the caller's COO order (reference model.py:159-161)."""
        if not self.mutuality:
            return None
        if self._world > 1:
            raise NotImplementedError("data_T_vals is only materialised on single-rank fits")
        P = self._packed
        out = np.zeros(len(self.X.vals), dtype=int)
        out[P.entry_src.cpu().numpy()] = P.t["e_xT"].cpu().numpy().astype(int)
        return out

    @property
    def data_T(self):
        l, i, j, m = self.X.subs
        if not self.mutuality:
            return sptensor(tuple(np.array([], dtype="int8") for _ in range(4)), [], shape=self.X.shape)
        return sptensor((l, j, i, m), self.X.vals, shape=self.X.shape)

    # ------------------------------------------------------------------ inferred model (model.py:1062-1214)
    def _consume(self, what, *args):
        """Run a posterior consumer (`infer`, `infer_mean`, `sample` of the engine) on the device slab that IS rho_f --
        the best restart's own when the restarts ran side by side, the last restart's, or the device copy kept when an
        earlier restart won -- and assemble the (L, N, N) result on the host: 1 byte (4 for rho_mean) per tie crosses
        PCIe instead of an fp64 copy of rho.  On a sharded fit every rank consumes its row block and the blocks are
        all-gathered (collective: every rank must call)."""
        eng, slab = self._rho_f_source()
        out = getattr(eng, what)(*args, slab=slab)
        if self._world > 1:
            out = self._all_gather_rows(out)
        return out.cpu().numpy()

    def _rho_f_source(self):
        """(engine, slab argument of its consumers) that read rho_f: see `_consume`."""
        eng = getattr(self, "_engine_f", None) or self._engine
        slab = None if (getattr(self, "_engine_f", None) is not None or self._rho_f_dev is None) else self._rho_f_dev
        return eng, slab

    def _consume_edges(self, what, dtype, *args):
        """Run a sparse consumer (`infer_edges`, `sample_edges` of the engine) on rho_f, chosen as in `_consume`, and return
        the ties whose label is nonzero as an sptensor (L, N, N) with subs (l, i, j), sorted, and `dtype` values.  On a
        sharded fit every rank extracts its own rows and the edge lists are all-gathered (collective: every rank must
        call); a rank's rows cover every layer, so the gathered lists are merged by key."""
        eng, slab = self._rho_f_source()
        keys, vals = getattr(eng, what)(*args, slab=slab)
        if self._world > 1:
            keys, vals = self._all_gather_edges(keys, vals)
        keys, vals = keys.cpu().numpy(), vals.cpu().numpy()
        l, r = np.divmod(keys, np.int64(self.N) * self.N)
        i, j = np.divmod(r, np.int64(self.N))
        return sptensor((l, i, j), vals.astype(dtype), shape=(self.L, self.N, self.N))

    def _all_gather_edges(self, keys, vals):
        """Every rank's (keys, labels), merged by key on every rank (collective): the counts first, then one padded
        all_gather of each -- on the device with NCCL, on the host with gloo (as `_all_gather_rows`)."""
        import torch.distributed as dist

        if dist.get_backend() != "nccl":
            keys, vals = keys.cpu(), vals.cpu()
        n = torch.tensor([keys.numel()], dtype=torch.int64, device=keys.device)
        ns = [torch.empty_like(n) for _ in range(self._world)]
        dist.all_gather(ns, n)
        ns = [int(v) for v in torch.cat(ns).cpu()]
        cap = max(max(ns), 1)
        parts = []
        for t in (keys, vals):
            pad = torch.zeros(cap, dtype=t.dtype, device=t.device)
            pad[:t.numel()] = t
            got = [torch.empty_like(pad) for _ in range(self._world)]
            dist.all_gather(got, pad)
            parts.append(torch.cat([g[:c] for g, c in zip(got, ns)]))
        keys, order = torch.sort(parts[0])
        return keys, parts[1][order]

    def _all_gather_rows(self, t):
        """Concatenate the ranks' row blocks (dim 1) of a per-tie tensor; every rank gets the whole (collective).  NCCL
        gathers device tensors; gloo (CPU tests, ranks sharing one GPU) gathers on the host."""
        host = torch.distributed.get_backend() != "nccl"
        if host:
            t = t.cpu()
        shape = list(t.shape)
        parts = []
        for r in range(self._world):
            shape[1] = shard_rows(self.N, self._world, r)[1]
            parts.append(torch.empty(shape, dtype=t.dtype, device=t.device))
        torch.distributed.all_gather(parts, t.contiguous())
        return torch.cat(parts, dim=1)

    def _engine_of_rho_f(self):
        """The engine whose consumers read rho_f (see `_consume`; pass `slab=self._rho_f_dev` when that is not None)."""
        return self._rho_f_source()[0]

    def sample_inferred_model(self, N=1, seed=None, rng="auto", sparse=False):
        """Sample Y trials from the rho distribution (reference model.py:1062-1096): a list of N arrays (L, N, N), each the
        argmax of the counts of N categorical draws per tie.

        rng = "numpy": the reference's generator (`default_rng(seed + i).multinomial`) on the host, which materialises
        rho_f as float64 -- 8 bytes * L*N*N*K; rng = "device": the `vm_sample` kernel on the fp32 slab (Philox stream
        keyed by seed and tie: same law, different stream, 1 byte per tie comes back); "auto": numpy while
        L*N*N*K <= 5e7, else device.

        sparse=True: a list of `sptensor` (L, N, N) holding the ties whose label is nonzero, equal to `sptensor.fromarray`
        of the device draws for the same seeds, evaluated tie by tie on the device without any N*N-sized buffer (the
        device generator only: "auto" means "device", "numpy" raises)."""
        if seed is None:
            seed = self.seed
        if rng not in ("auto", "numpy", "device"):
            raise ValueError("rng must be 'auto', 'numpy' or 'device'")
        if sparse:
            if rng == "numpy":
                raise ValueError('sample_inferred_model(sparse=True) draws on the device: rng="numpy" materialises rho_f')
            return [self._consume_edges("sample_edges", "int", N, int(seed) + i) for i in range(0, N)]
        if rng == "auto":
            rng = "device" if float(self.L) * self.N * self.N * self.K > AUTO_REFERENCE_INIT_LIMIT else "numpy"
        if rng == "device":
            return [self._consume("sample", N, int(seed) + i).astype("int") for i in range(0, N)]

        def sampleY(seed):
            pnrg = np.random.default_rng(seed)
            pv = self.rho_f / self.rho_f.sum(axis=-1, keepdims=True)  # float32 storage: renormalise for numpy's check
            Y = pnrg.multinomial(n=N, pvals=pv, size=(self.L, self.N, self.N))
            return Y.argmax(axis=-1)

        return [sampleY(seed + i) for i in range(0, N)]

    def _inferred_method(self, method, threshold):
        """Resolve `get_inferred_model`'s method (model.py:1099-1188): (the engine's infer arguments (mode, threshold), or
        None for rho_mean; the dtype of the result)."""
        OPTIONS = ["rho_max", "rho_mean", "fixed_threshold", "heuristic_threshold"]
        try:
            method = match_arg(method, OPTIONS)[0]
        except IndexError:
            raise ValueError("'method' should be one of {}.".format(", ".join(['"' + x + '"' for x in OPTIONS])))

        if (not self.mutuality and method != "rho_max") or (self.K > 2 and "threshold" in method):
            msg = ("threshold methods is incompatible with VIMuRe's mutuality=False "
                   'or for data with more than 2 categories. Using "rho_max" method.')
            warnings.warn(msg, UserWarning)
            method = "rho_max"

        if method == "rho_max":
            return (0, 0.5), "int"
        if method == "rho_mean":  # np.dot(rho_f, range(K)), model.py:1151-1153
            return None, np.float64
        if method == "fixed_threshold":
            if (threshold is None) or (threshold > 1) or (threshold < 0):
                raise ValueError('For method="fixed_threshold", you must set the threshold to a value in [0,1].')
            return (1, float(threshold)), np.float64
        # heuristic_threshold: 0.54 * G_exp_nu - 0.01 (utils.py:200-204; reads G_exp_nu, not G_exp_nu_f)
        return (1, float(get_optimal_threshold(self))), "int"

    def get_inferred_model(self, method="rho_max", threshold=None, sparse=False):
        """Estimate Y from rho_f: rho_max | rho_mean | fixed_threshold | heuristic_threshold (model.py:1099-1188).
        Every method runs on the device slab (float32 storage: a posterior that sits within ~1e-7 of a threshold, or two
        categories that tie to that precision, can come out differently from a float64 evaluation).

        sparse=True: an `sptensor` (L, N, N) of the ties whose estimate is nonzero, equal to `sptensor.fromarray` of the
        dense result (same subs, values and dtype), evaluated tie by tie on the device without any N*N-sized buffer --
        the form to ask for on large networks.  Not for rho_mean, whose every tie is nonzero (ValueError)."""
        args, dtype = self._inferred_method(method, threshold)
        if args is None:
            if sparse:
                raise ValueError('get_inferred_model("rho_mean") has no sparse form: the posterior mean of every tie is '
                                 "nonzero")
            return self._consume("infer_mean").astype(dtype)
        if sparse:
            return self._consume_edges("infer_edges", dtype, *args)
        return self._consume("infer", *args).astype(dtype)

    def rho_f_at(self, subs):
        """The posterior rho_f at given ties: subs = (l, i, j), three 1-D integer arrays of equal length (the first three
        subscripts of an `sptensor`, such as the edges `get_inferred_model(..., sparse=True)` returns) -> float64 (n, K),
        equal to `rho_f[l, i, j]`.  Evaluated tie by tie on the device (`vm_rho_at`) wherever rho_f lives -- the best
        restart's engine, a snapshot or a cloned slab (see `_consume`) -- without any N*N-sized buffer: only the keys go to
        the device and n*K floats come back; the form to ask for on networks whose rho_f does not fit.  On a sharded fit
        every rank answers the ties of its own rows and one all-reduce combines them (collective: every rank must call with
        the same subs).  ValueError, before any device work, for anything but three integer arrays of equal length within
        the shape (L, N, N); empty integer arrays give (0, K)."""
        if not isinstance(subs, (tuple, list)) or len(subs) != 3:
            raise ValueError("rho_f_at takes subs = (l, i, j): three 1-D integer arrays")
        subs = [np.asarray(s) for s in subs]
        if any(s.ndim != 1 for s in subs) or len({s.size for s in subs}) != 1:
            raise ValueError("rho_f_at: l, i, j must be 1-D arrays of equal length")
        if any(not np.issubdtype(s.dtype, np.integer) for s in subs):
            raise ValueError("rho_f_at: the subscripts must be integer arrays")
        if subs[0].size == 0:
            return np.zeros((0, self.K))
        l, i, j = (s.astype(np.int64) for s in subs)
        for s, hi, name in ((l, self.L, "l"), (i, self.N, "i"), (j, self.N, "j")):
            if s.min() < 0 or s.max() >= hi:
                raise ValueError("rho_f_at: %s out of range [0, %d)" % (name, hi))
        eng, slab = self._rho_f_source()
        keys = torch.as_tensor((l * self.N + i) * self.N + j, device=eng.dev)
        out = eng.rho_at(keys, slab=slab)  # this rank's rows, zeros elsewhere
        if self._world > 1:
            # every key belongs to exactly one rank and x + 0 = x: the sum is exact.  NCCL on the device, gloo on the host
            if torch.distributed.get_backend() != "nccl":
                out = out.cpu()
            torch.distributed.all_reduce(out)
        return out.cpu().numpy().astype(np.float64)

    def get_posterior_estimates(self):
        """Posterior estimates nu, theta, lambda, rho (reference model.py:1191-1214)."""
        return {"nu": self.G_exp_nu_f, "theta": self.G_exp_theta_f, "lambda": self.G_exp_lambda_f, "rho": self.rho_f}


def _agree_int(v, dev, op="bcast"):
    """Rank 0's integer (op="bcast") or the maximum over the ranks (op="max"), on every rank."""
    t = torch.tensor([int(v)], dtype=torch.int64, device=dev)
    if op == "max":
        torch.distributed.all_reduce(t, op=torch.distributed.ReduceOp.MAX)
    else:
        torch.distributed.broadcast(t, src=0)
    return int(t.item())


def _exchange_reciprocals(subs, vals, N, world, rank, dev):
    """Sharded ingestion from the entries of a rank's OWN rows (`presharded="rows"`): the entry X[l,i,j,m] is also needed by
    the rank that owns row j (it pairs X[l,j,i,m] with it and lists it for the eta part of the ELBO), so every rank sends
    each of its entries to the owner of its column node -- one variable-size all-to-all, device to device -- and packs
    its own entries followed by what it received.  Returns (4 index tensors, value tensor), int32, on `dev`."""
    import torch.distributed as dist

    cols = [torch.as_tensor(np.ascontiguousarray(np.asarray(a).astype(np.int32, copy=False))) for a in (*subs, vals)]
    own = torch.stack([c.to(dev, non_blocking=True) for c in cols], dim=1)  # (n, 5): l, i, j, m, x
    bounds = torch.tensor([shard_rows(N, world, r)[0] for r in range(1, world)], dtype=torch.int32, device=dev)
    dest = torch.bucketize(own[:, 2].contiguous(), bounds, right=True)  # owner of the column node j
    away = dest != rank
    d_away = dest[away]
    order = torch.argsort(d_away, stable=True)
    send = own[away][order].contiguous()
    n_send = torch.bincount(d_away, minlength=world).to(torch.int64)
    if dist.get_backend() == "nccl":
        n_recv = torch.empty_like(n_send)
        dist.all_to_all_single(n_recv, n_send)
        ns, nr = [int(v) for v in n_send.cpu()], [int(v) for v in n_recv.cpu()]
        recv = torch.empty((sum(nr), 5), dtype=torch.int32, device=dev)
        dist.all_to_all_single(recv, send, output_split_sizes=nr, input_split_sizes=ns)
    else:  # gloo (CPU tests, ranks sharing a GPU): gather everything on the host and keep what is addressed to this rank
        host = (send.cpu(), d_away[order].cpu())
        parts = [None] * world
        dist.all_gather_object(parts, host)
        recv = torch.cat([p_[0][p_[1] == rank] for p_ in parts], dim=0).to(dev)
    both = torch.cat([own, recv], dim=0)
    return tuple(both[:, d].contiguous() for d in range(4)), both[:, 4].contiguous()


def _agree_float(v, dev):
    t = torch.tensor([float(v)], dtype=torch.float64, device=dev)
    torch.distributed.broadcast(t, src=0)
    return float(t.item())


def _keyed_uniform(key, ids, K):
    """Counter-based uniforms in [0, 1): (len(ids), K) doubles, a pure function of (key, id, k) -- splitmix64 finaliser.
    Used where the draw must not depend on how the ties are distributed over ranks."""
    ids = np.asarray(ids, dtype=np.uint64)
    with np.errstate(over="ignore"):
        x = (ids[:, None] * np.uint64(K) + np.arange(K, dtype=np.uint64)[None, :]) + \
            np.uint64(key) * np.uint64(0x9E3779B97F4A7C15) + np.uint64(0x9E3779B97F4A7C15)
        x ^= x >> np.uint64(30)
        x *= np.uint64(0xBF58476D1CE4E5B9)
        x ^= x >> np.uint64(27)
        x *= np.uint64(0x94D049BB133111EB)
        x ^= x >> np.uint64(31)
    return (x >> np.uint64(11)).astype(np.float64) * (1.0 / 9007199254740992.0)


def shard_rows(N, world, rank):
    """Node-row block [row0, row0+nloc) of `rank` (balanced, contiguous)."""
    base, rem = divmod(int(N), int(world))
    row0 = rank * base + min(rank, rem)
    return row0, base + (1 if rank < rem else 0)
