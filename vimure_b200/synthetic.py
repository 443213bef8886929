"""Sparse synthetic generators for large networks.

The reference's generators (`synthetic.py:63-352, 548-571, 848-940`) follow the laws below but materialise
dense (L,N,N,M) arrays and loop over every (reporter, tie) in python, so they stop around N ~ 500.  These
generators sample the SAME laws sparsely (only the non-zero counts are ever created), which is what the
N = 20k .. 64k benchmark configurations need.  They do not reproduce the reference's RNG stream: parity is
always checked on identical inputs, never on regenerated ones.

Laws
  Y (StandardSBM, synthetic.py:548-571): Y_ij ~ Poisson(c * w[g_i, g_j]), equal-size groups, assortative
      w (within p1, between 0.1*p1), c such that sum = N*avg_degree; no self ties; cut at K-1.
  Y (Multitensor / "GMReciprocity", synthetic.py:848-940): pairs i<j, a fair coin picks the first direction,
      first ~ Poisson(M), second ~ Poisson(M0 + eta*first), M = (M0 + eta*M0^T)/(1-eta^2),
      sum(M0) = ExpM*(1-eta), ExpM = N*avg_degree/2.
  X (`_build_X` with the self-reporter mask, synthetic.py:138-209): theta_lm ~ Gamma(sh, sc);
      lambda_lij = Y_lij if Y_lij > 0 else 0.01; for reporter m and every pair {m,n} a fair coin picks the first
      direction, first ~ Poisson((th*lam_ab + eta*th*lam_ba)/(1-eta^2)), second ~ Poisson(th*lam_ba + eta*first).
      The device generators (`device_reports`) draw the same law for any reporter and pair, under the self-reporter,
      the all-reporter or an explicit mask.
"""
import numpy as np

from . import masks
from .masks import AllMask, EgoMask
from .sptensor import sptensor

LAMBDA_0 = 0.01


def _ztp(prng, mu):
    """Zero-truncated Poisson(mu), vectorised (exact: 1 + Poisson(mu - t), t = -log(1 - u(1-e^-mu)))."""
    u = prng.random_sample(mu.shape)
    t = -np.log1p(-u * (-np.expm1(-mu)))
    return 1 + prng.poisson(np.maximum(mu - t, 0.0))


class SparseSyntheticNetwork:
    """Ground truth Y (COO) + observed X (COO) + ego reporter mask, generated sparsely."""

    def __init__(self, N=100, M=None, L=1, K=2, C=2, avg_degree=10.0, eta=None, structure="assortative", seed=10):
        self.N, self.L, self.K, self.C = int(N), int(L), int(K), int(C)
        self.M = self.N if M is None else int(M)
        if self.M > self.N:
            raise ValueError("M <= N is required (reporter m is node m)")
        self.avg_degree, self.eta_Y, self.structure, self.seed = float(avg_degree), eta, structure, seed
        self.prng = np.random.RandomState(seed)
        self._build_Y()

    # ------------------------------------------------------------------ Y
    def _groups(self):
        size = max(1, self.N // self.C)
        return np.minimum(np.arange(self.N) // size, self.C - 1)

    def _build_Y(self):
        N, C, L, K = self.N, self.C, self.L, self.K
        g = self._groups()
        members = [np.nonzero(g == c)[0] for c in range(C)]
        sizes = np.array([len(m) for m in members], dtype=float)
        p1 = self.avg_degree * C / N
        if self.structure == "assortative":
            w = p1 * 0.1 * np.ones((C, C))
            np.fill_diagonal(w, p1)
        else:
            w = p1 * np.ones((C, C))
            np.fill_diagonal(w, 0.1 * p1)
        npairs = np.outer(sizes, sizes) - np.diag(sizes)  # ordered pairs without the diagonal
        out = []
        for l in range(L):
            if self.eta_Y is None:
                c = N * self.avg_degree / (w * npairs).sum()
                rate = c * w  # per ordered pair
                li, lj, lv = [], [], []
                for a in range(C):
                    for b in range(C):
                        n = self.prng.poisson(rate[a, b] * sizes[a] * sizes[b])
                        i = members[a][self.prng.randint(0, len(members[a]), n)]
                        j = members[b][self.prng.randint(0, len(members[b]), n)]
                        keep = i != j
                        li.append(i[keep])
                        lj.append(j[keep])
                i, j = np.concatenate(li), np.concatenate(lj)
                key, cnt = np.unique(i.astype(np.int64) * N + j, return_counts=True)
                i, j, v = key // N, key % N, cnt
            else:
                eta = float(self.eta_Y)
                ExpM = N * self.avg_degree / 2.0
                c = ExpM * (1.0 - eta) / (w * npairs).sum()
                M0 = c * w
                Mfull = M0 / (1.0 - eta)  # w symmetric => (M0 + eta*M0^T)/(1-eta^2)
                fi, fj, fv = [], [], []
                # "first" draws that are positive: every ordered pair is first with prob 1/2
                for a in range(C):
                    for b in range(C):
                        n = self.prng.poisson(0.5 * (-np.expm1(-Mfull[a, b])) * sizes[a] * sizes[b])
                        i = members[a][self.prng.randint(0, len(members[a]), n)]
                        j = members[b][self.prng.randint(0, len(members[b]), n)]
                        keep = i != j
                        fi.append(i[keep])
                        fj.append(j[keep])
                        fv.append(_ztp(self.prng, np.full(int(keep.sum()), Mfull[a, b])))
                i1, j1, v1 = np.concatenate(fi), np.concatenate(fj), np.concatenate(fv)
                key1, first_idx = np.unique(np.minimum(i1, j1).astype(np.int64) * N + np.maximum(i1, j1), return_index=True)
                i1, j1, v1 = i1[first_idx], j1[first_idx], v1[first_idx]
                v2 = self.prng.poisson(M0[g[j1], g[i1]] + eta * v1)  # the reciprocated direction
                # pairs whose first draw was zero: second ~ Poisson(M0), positive with prob ~M0
                si, sj, sv = [], [], []
                for a in range(C):
                    for b in range(C):
                        n = self.prng.poisson(np.exp(-Mfull[a, b]) * (-np.expm1(-M0[a, b])) * 0.5 * sizes[a] * sizes[b])
                        i = members[a][self.prng.randint(0, len(members[a]), n)]
                        j = members[b][self.prng.randint(0, len(members[b]), n)]
                        keep = i != j
                        si.append(i[keep])
                        sj.append(j[keep])
                        sv.append(_ztp(self.prng, np.full(int(keep.sum()), M0[a, b])))
                i3, j3, v3 = np.concatenate(si), np.concatenate(sj), np.concatenate(sv)
                k3 = np.minimum(i3, j3).astype(np.int64) * N + np.maximum(i3, j3)
                new = ~np.isin(k3, key1)
                i3, j3, v3 = i3[new], j3[new], v3[new]
                _, u3 = np.unique(k3[new], return_index=True)
                i = np.concatenate([i1, j1, i3[u3]])
                j = np.concatenate([j1, i1, j3[u3]])
                v = np.concatenate([v1, v2, v3[u3]])
                pos = v > 0
                i, j, v = i[pos], j[pos], v[pos]
            v = np.minimum(v, K - 1)
            out.append(np.stack([np.full(len(i), l), i, j, v]))
        y = np.concatenate(out, axis=1).astype(np.int64)
        self.Y_subs, self.Y_vals = y[:3], y[3]
        self.Y = sptensor(tuple(self.Y_subs), self.Y_vals, shape=(L, N, N))

    # ------------------------------------------------------------------ X
    def build_X(self, mutuality=0.5, sh_theta=2.0, sc_theta=0.5, seed=None, theta=None, lambda_diff=None):
        """Observed reports under the self-reporter (ego) mask.  Returns self (sets X, R, theta)."""
        N, M, L = self.N, self.M, self.L
        prng = np.random.RandomState(self.seed if seed is None else seed)
        eta = float(mutuality)
        if eta < 0 or eta >= 1:
            raise ValueError("The mutuality parameter has to be in [0, 1)!")
        if theta is None:
            theta = prng.gamma(shape=sh_theta, scale=sc_theta, size=(L, M))
        self.theta = theta
        subs, vals = [], []

        def emit(l, i, j, m, x):
            pos = x > 0
            subs.append(np.stack([np.full(int(pos.sum()), l), i[pos], j[pos], m[pos]]))
            vals.append(x[pos])

        for l in range(L):
            sel = self.Y_subs[0] == l
            yi, yj, yv = self.Y_subs[1][sel], self.Y_subs[2][sel], self.Y_vals[sel].astype(float)
            lam_edge = yv if lambda_diff is None else np.full(len(yv), LAMBDA_0 + lambda_diff)
            ykey = yi * N + yj
            ysort = np.argsort(ykey)
            ykey_s, ylam_s = ykey[ysort], lam_edge[ysort]

            def lam(i, j):
                k = i * N + j
                if len(ykey_s) == 0:
                    return np.full(len(k), LAMBDA_0)
                p = np.minimum(np.searchsorted(ykey_s, k), len(ykey_s) - 1)
                return np.where(ykey_s[p] == k, ylam_s[p], LAMBDA_0)

            th = theta[l]
            # ---- pairs {m, n} that carry a true tie in either direction: sampled directly
            em = np.concatenate([yi, yj])
            en = np.concatenate([yj, yi])
            ok = em < M
            pk = np.unique(em[ok] * N + en[ok])
            em, en = pk // N, pk % N
            edge_pairs = pk
            t = th[em]
            l_ab, l_ba = lam(em, en), lam(en, em)
            coin = prng.random_sample(len(em)) < 0.5
            a_i = np.where(coin, em, en)
            a_j = np.where(coin, en, em)
            l_first = np.where(coin, l_ab, l_ba)
            l_second = np.where(coin, l_ba, l_ab)
            x1 = prng.poisson((t * l_first + eta * t * l_second) / (1.0 - eta * eta))
            x2 = prng.poisson(t * l_second + eta * x1)
            emit(l, a_i, a_j, em, x1)
            emit(l, a_j, a_i, em, x2)
            # ---- all the other pairs: base mean mu = theta*LAMBDA_0 in both directions, positives sampled sparsely
            mu = th * LAMBDA_0
            mm = mu / (1.0 - eta)
            a = -np.expm1(-mm)
            b = np.exp(-mm) * (-np.expm1(-mu))
            npos = prng.binomial(N - 1, a + b)
            rm = np.repeat(np.arange(M), npos)
            rn = prng.randint(0, N - 1, len(rm))
            rn = rn + (rn >= rm)
            pk = np.unique(rm.astype(np.int64) * N + rn)
            pk = pk[~np.isin(pk, edge_pairs)]
            rm, rn = pk // N, pk % N
            mu_r, mm_r, a_r, b_r = mu[rm], mm[rm], a[rm], b[rm]
            first_pos = prng.random_sample(len(rm)) < a_r / (a_r + b_r)
            x1 = np.where(first_pos, _ztp(prng, mm_r), 0)
            x2 = np.where(first_pos, prng.poisson(mu_r + eta * x1), _ztp(prng, mu_r))
            coin = prng.random_sample(len(rm)) < 0.5
            a_i = np.where(coin, rm, rn)
            a_j = np.where(coin, rn, rm)
            emit(l, a_i, a_j, rm, x1)
            emit(l, a_j, a_i, rm, x2)
            # ---- the (m, m) self ties (allowed by the mask, lambda = LAMBDA_0)
            md = np.arange(M)
            xd = prng.poisson(mu + eta * prng.poisson(mm))
            emit(l, md, md, md, xd)
        s = np.concatenate(subs, axis=1).astype(np.int64)
        v = np.concatenate(vals).astype(np.int64)
        self.X = sptensor(tuple(s), v, shape=(L, N, N, M))
        self.R = EgoMask(L, N, M, diag=True)
        self.mutuality = eta
        return self


    # ------------------------------------------------------------------ X on the device
    def build_X_device(self, mutuality=0.5, sh_theta=2.0, sc_theta=0.5, seed=None, theta=None, device="cuda", row0=0,
                       nloc=None, emit_transposed=False, flag_self_reporter=True, Rinput=None):
        """Device-side `build_X` (the `vm_synth_*` kernels of include/vimure_b200.h): the same law, sampled with a
        counter-based RNG keyed by (seed, layer, reporter, pair), for the node-row block [row0, row0+nloc) only.

        The mask follows the reference's arguments: `Rinput` (anything `masks.from_input` accepts, or a ReporterMask) when
        given, else the self-reporter mask (`flag_self_reporter=True`) or the all-reporter mask (False); see
        `device_reports` for how each is generated.

        Returns (subs, vals): int32 tensors (4, n) and (n,) ON THE DEVICE -- the entries X[l,i,j,m] with i in the block and,
        with `emit_transposed`, the reciprocal entries X[l,j,i,m] whose row the block does not own (so that the shard can
        be paired without an exchange).  Every rank that evaluates an entry gets the same value, whatever its block.
        Also sets self.theta, self.R (the EgoMask, AllMask or CooMask used), self.mutuality (not self.X: use
        `sptensor(tuple(subs.cpu()), vals.cpu(), ...)`)."""
        sd = self.seed if seed is None else seed
        eta = float(mutuality)
        if eta < 0 or eta >= 1:
            raise ValueError("The mutuality parameter has to be in [0, 1)!")
        R = _report_mask(Rinput, flag_self_reporter, self.L, self.N, self.M)
        if theta is None:
            theta = np.random.RandomState(sd).gamma(shape=sh_theta, scale=sc_theta, size=(self.L, self.M))
        self.theta = theta
        subs, vals = device_reports(self.L, self.N, self.M, self.K, self.Y_subs, self.Y_vals, theta, eta, sd, device=device,
                                    row0=row0, nloc=nloc, emit_transposed=emit_transposed, mask=R)
        self.R = R
        self.mutuality = eta
        return subs, vals


def _report_mask(Rinput, flag_self_reporter, L, N, M):
    """The reporter mask of the reference's `build_X(Rinput=..., flag_self_reporter=...)`, as a ReporterMask."""
    if Rinput is not None:
        return masks.from_input(Rinput, L, N, M)
    return EgoMask(L, N, M, diag=True) if flag_self_reporter else AllMask(L, N, M)


def _full_ego(R):
    return isinstance(R, EgoMask) and R.diag and bool(np.all(R.rep))


def device_reports(L, N, M, K, Y_subs, Y_vals, theta, eta, seed, lam=None, device="cuda", row0=0, nloc=None,
                   emit_transposed=False, mask=None):
    """Reports X for a given ground truth Y (COO), reliabilities theta (L, M), mutuality eta and, optionally, a table lam
    (L, K) of average interactions per ground-truth category (default: 0.01, 1, 2, ..), sampled on the device
    (include/vimure_b200.h).  Returns int32 device tensors (subs (4, n), vals (n,)).

    mask: None or a full EgoMask(diag=True) -> `vm_synth_ego`; any other EgoMask -> `vm_synth_ego`, filtered on the
    device by rep[l, m] and diag; AllMask -> `vm_synth_all`; anything else `masks.from_input` accepts -> `vm_synth_masked`
    over its distinct entries (`masked_reports`).  Every mask gives the same count for the same (seed, layer, reporter,
    pair), so a mask's reports are those of a larger mask restricted to its entries."""
    R = None if mask is None else masks.from_input(mask, L, N, M)
    args = (L, N, M, K, Y_subs, Y_vals, theta, eta, seed, lam, device, row0, nloc, emit_transposed)
    if R is None or isinstance(R, EgoMask):
        subs, vals = _generate("vm_synth_ego", *args)
        if R is None or _full_ego(R):
            return subs, vals
        import torch

        keep = torch.as_tensor(R.rep.astype(bool), device=subs.device)[subs[0].long(), subs[3].long()]
        if not R.diag:
            keep &= subs[1] != subs[2]
        return subs[:, keep], vals[keep]
    if isinstance(R, AllMask):
        return _generate("vm_synth_all", *args)
    sel = R.vals != 0
    return masked_reports(L, N, M, K, Y_subs, Y_vals, theta, eta, seed, R.subs[:, sel], lam=lam, device=device, row0=row0,
                          nloc=nloc, emit_transposed=emit_transposed)


def masked_reports(L, N, M, K, Y_subs, Y_vals, theta, eta, seed, entries, lam=None, device="cuda", row0=0, nloc=None,
                   emit_transposed=False):
    """Reports X under an explicit mask `entries` (4, n) = (l, i, j, m), duplicates allowed: `vm_synth_masked` over the
    distinct entries, X[l,i,j,m] = reporter m's i->j count on the pair {i, j} (as every other generator draws it).
    ValueError, before any device work, for an entry outside (L, N, N, M).  Returns int32 device tensors as
    `device_reports`."""
    import torch

    e = np.asarray(entries)
    if e.ndim != 2 or e.shape[0] != 4:
        raise ValueError("entries must be (4, n): l, i, j, m")
    e = e.astype(np.int64)
    if e.shape[1]:
        lo, hi = e.min(axis=1), e.max(axis=1)
        if np.any(lo < 0) or np.any(hi >= np.array([L, N, N, M])):
            raise ValueError("mask entries outside the shape (L, N, N, M) = (%d, %d, %d, %d)" % (L, N, N, M))
    if L * N * N * M >= 2 ** 63:
        raise ValueError("L*N*N*M must stay below 2^63")
    dev = torch.device(device)
    if dev.type != "cuda":
        raise RuntimeError("masked_reports needs a CUDA device")
    t = torch.from_numpy(np.ascontiguousarray(e)).to(dev)
    key = torch.unique(((t[0] * N + t[1]) * N + t[2]) * M + t[3])
    del t
    rest = torch.div(key, M, rounding_mode="floor")
    m = (key - rest * M).to(torch.int32)
    lij = torch.div(rest, N, rounding_mode="floor")
    j = (rest - lij * N).to(torch.int32)
    l = torch.div(lij, N, rounding_mode="floor")
    i = (lij - l * N).to(torch.int32)
    l = l.to(torch.int32)
    del key, rest, lij
    return _generate("vm_synth_masked", L, N, M, K, Y_subs, Y_vals, theta, eta, seed, lam, device, row0, nloc,
                     emit_transposed, mask=(l, i, j, m))


def _generate(entry, L, N, M, K, Y_subs, Y_vals, theta, eta, seed, lam, device, row0, nloc, emit_transposed, mask=None):
    """One `vm_synth_*` entry point, counted then filled: returns int32 device tensors (subs (4, n), vals (n,))."""
    import ctypes

    import torch

    from . import _capi

    nloc = N - row0 if nloc is None else int(nloc)
    dev = torch.device(device)
    if dev.type != "cuda":
        raise RuntimeError("device_reports needs a CUDA device (host counterpart: SparseSyntheticNetwork.build_X)")
    lib = _capi.load()
    Y_subs = np.asarray(Y_subs).astype(np.int64)
    ykey = (Y_subs[0] * N + Y_subs[1]) * N + Y_subs[2]
    o = np.argsort(ykey, kind="stable")
    yk = torch.from_numpy(np.ascontiguousarray(ykey[o])).to(dev)
    yv = torch.from_numpy(np.ascontiguousarray(np.asarray(Y_vals)[o]).astype(np.int32)).to(dev)
    th = torch.from_numpy(np.ascontiguousarray(theta, dtype=np.float64)).to(dev)
    lam_t = None if lam is None else torch.from_numpy(np.ascontiguousarray(lam, dtype=np.float64).reshape(L, K)).to(dev)
    counter = torch.zeros(1, dtype=torch.int64, device=dev)
    S = _capi.synth_class()()
    S.L, S.N, S.M, S.K, S.row0, S.nloc = int(L), int(N), int(M), int(K), int(row0), nloc
    S.emit_transposed = int(bool(emit_transposed))
    S.seed = int(seed) & (2**64 - 1)
    S.eta = float(eta)
    S.theta, S.y_key, S.y_val, S.nY = th.data_ptr(), yk.data_ptr(), yv.data_ptr(), int(yk.numel())
    S.lam = None if lam_t is None else lam_t.data_ptr()
    S.counter = counter.data_ptr()
    stream = ctypes.c_void_p(torch.cuda.current_stream(dev).cuda_stream)
    fn = getattr(lib, entry)
    extra = ()
    if mask is not None:
        Mk = _capi.synth_mask_class()()
        Mk.l, Mk.i, Mk.j, Mk.m = (int(t.data_ptr()) for t in mask)
        Mk.n = int(mask[0].numel())
        extra = (ctypes.byref(Mk),)
    # pass 1 counts (cap = 0: nothing is stored), pass 2 fills arrays of exactly that size
    S.cap = 0
    _capi.check(fn(ctypes.byref(S), *extra, stream), entry + " (count)")
    n = int(counter.item())
    out = torch.empty((5, max(n, 1)), dtype=torch.int32, device=dev)
    S.cap = n
    S.o_l, S.o_i, S.o_j, S.o_m, S.o_x = (out[d].data_ptr() for d in range(5))
    _capi.check(fn(ctypes.byref(S), *extra, stream), entry + " (fill)")
    if int(counter.item()) != n:
        raise RuntimeError("%s: the two passes disagree (%d vs %d entries)" % (entry, int(counter.item()), n))
    return out[:4, :n], out[4, :n]


class PosteriorSyntheticNetwork:
    """Generates data (Y, X) from the posterior estimates of a fitted model: the counterpart of the reference's
    `vimure.synthetic.PosteriorSyntheticNetwork` (synthetic.py:964-1177) under the ego, all-reporter or an explicit
    reporter mask, without an fp64 host copy of rho and without dense (L,N,N) or (L,N,N,M) arrays.

    build_Y : Y_lij ~ Categorical(rho_f[l,i,j,:]) (one draw; `model.sample_inferred_model(N=1, seed=seed_Y)`: numpy's
              stream like the reference for small problems, the device kernel for large ones -- as an edge list
              evaluated on the device, so it works without the posterior slab at any N).
    build_X : theta ~ Gamma(gamma_shp_f, 1/gamma_rte_f), lambda ~ Gamma(phi_shp_f, 1/phi_rte_f), eta ~ Gamma(nu_shp_f,
              1/nu_rte_f) drawn with RandomState(seed_X) in the reference's order (synthetic.py:1040-1042); a tie of
              category k >= 1 gets lambda[l,k], every other tie lambda[0,0] (synthetic.py:1044-1048); the reports follow
              `_build_X`'s law (synthetic.py:1063-1098) under the mask of `Rinput` / `flag_self_reporter`, sampled by the
              device generator (`device_reports`).  Also the union / intersection baselines (synthetic.py:1139-1172)."""

    def __init__(self, model, seed_Y):
        self.model, self.seed_Y = model, seed_Y
        self.theta_shp, self.theta_rte = model.gamma_shp_f, model.gamma_rte_f
        self.lambda_shp, self.lambda_rte = model.phi_shp_f, model.phi_rte_f
        self.mutuality_shp, self.mutuality_rte = model.nu_shp_f, model.nu_rte_f
        self.L, self.N, self.K = model.L, model.N, model.K
        self.M = self.theta_shp.shape[1]

    def build_Y(self, rng="auto"):
        from .model import AUTO_REFERENCE_INIT_LIMIT

        device = rng == "device" or (rng == "auto" and float(self.L) * self.N * self.N * self.K > AUTO_REFERENCE_INIT_LIMIT)
        if device:  # the device sampler's draws as an edge list: no (L, N, N) array
            Ys = self.model.sample_inferred_model(N=1, seed=self.seed_Y, sparse=True)[0]
            self.Y_subs = np.stack(Ys.subs).astype(np.int64)
            self.Y_vals = np.minimum(Ys.vals, self.K - 1).astype(np.int64)
        else:
            Y = np.asarray(self.model.sample_inferred_model(N=1, seed=self.seed_Y, rng=rng)[0])
            Y = np.minimum(Y, self.K - 1)
            subs = np.nonzero(Y)
            self.Y_subs = np.stack(subs).astype(np.int64)
            self.Y_vals = Y[subs].astype(np.int64)
        self.Y = sptensor(tuple(self.Y_subs), self.Y_vals, shape=(self.L, self.N, self.N))
        return self

    def build_X(self, Rinput=None, flag_self_reporter=True, cutoff_X=False, Q=None, seed_X=None, device="cuda"):
        """Reports under `Rinput` (anything `masks.from_input` accepts) when given, else under the self-reporter mask
        (`flag_self_reporter=True`) or the all-reporter mask (False).  Sets X, R (the EgoMask, AllMask or CooMask sampled,
        so that `VimureModel().fit(X, R=R, ...)` takes them as they are), theta, lambda_k, mutuality and the baselines."""
        import torch

        R = _report_mask(Rinput, flag_self_reporter, self.L, self.N, self.M)
        for nm in ("theta_rte", "lambda_rte", "mutuality_rte"):
            if np.any(np.asarray(getattr(self, nm)) == 0):
                raise ValueError(nm + " has some zero entries!")
        if seed_X is None:
            seed_X = 90
        self.seed_X = seed_X
        prng = np.random.RandomState(seed_X)
        theta = prng.gamma(shape=self.theta_shp, scale=1.0 / self.theta_rte, size=(self.L, self.M))
        lambda_k = prng.gamma(shape=self.lambda_shp, scale=1.0 / self.lambda_rte, size=(self.L, self.K))
        mutuality = prng.gamma(shape=self.mutuality_shp, scale=1.0 / self.mutuality_rte, size=1)[0]
        if not (0.0 <= mutuality < 1.0):
            raise ValueError("the drawn mutuality (%g) is outside [0, 1)" % mutuality)
        lam = np.array(lambda_k, dtype=np.float64)
        lam[:, 0] = lambda_k[0, 0]  # every tie without a positive category gets lambda_k[0, 0] (synthetic.py:1044)
        subs_d, vals_d = device_reports(self.L, self.N, self.M, self.K, self.Y_subs, self.Y_vals, theta, mutuality, seed_X,
                                        lam=lam, device=device, mask=R)
        # baselines (synthetic.py:1139-1172): ties reported by anybody / by exactly two reports, from int64 tie keys
        s64 = subs_d[:3].long()
        ties, cnt = torch.unique((s64[0] * self.N + s64[1]) * self.N + s64[2], return_counts=True)
        inter = ties[cnt == 2]
        del s64
        subs, vals = subs_d.cpu().numpy().astype(np.int64), vals_d.cpu().numpy().astype(np.int64)
        del subs_d, vals_d
        if cutoff_X:
            vals = np.minimum(vals, (self.K if Q is None else Q) - 1)
        self.X = sptensor(tuple(subs), vals, shape=(self.L, self.N, self.N, self.M))
        self.R = R
        self.theta, self.lambda_k, self.mutuality = theta, lambda_k, mutuality
        shape3 = (self.L, self.N, self.N)
        for name, k in (("X_union", ties), ("X_intersection", inter)):
            k = k.cpu().numpy()
            l, r = np.divmod(k, np.int64(self.N) * self.N)
            i, j = np.divmod(r, np.int64(self.N))
            setattr(self, name, sptensor((l, i, j), np.ones(len(k), dtype=np.int8), shape=shape3))
        return self


def StandardSBM(N=100, M=None, L=1, K=2, C=2, avg_degree=2.0, structure="assortative", seed=10):
    """Sparse counterpart of `vimure.synthetic.StandardSBM` (call `.build_X(...)` afterwards)."""
    return SparseSyntheticNetwork(N=N, M=M, L=L, K=K, C=C, avg_degree=avg_degree, eta=None, structure=structure, seed=seed)


def Multitensor(N=100, M=None, L=1, K=2, C=2, avg_degree=2.0, eta=0.5, structure="assortative", seed=10):
    """Sparse counterpart of `vimure.synthetic.Multitensor` ("GMReciprocity")."""
    return SparseSyntheticNetwork(N=N, M=M, L=L, K=K, C=C, avg_degree=avg_degree, eta=eta, structure=structure, seed=seed)


def dense_reporting_X(net, M, mutuality=0.5, sh_theta=2.0, sc_theta=0.5, seed=None):
    """Every one of M reporters reports every ordered pair (flag_self_reporter=False, synthetic.py:211-231),
    sampled sparsely.  Returns (X sptensor, theta); the mask is AllMask."""
    N, L = net.N, net.L
    prng = np.random.RandomState(net.seed if seed is None else seed)
    eta = float(mutuality)
    theta = prng.gamma(shape=sh_theta, scale=sc_theta, size=(L, M))
    subs, vals = [], []
    npairs = N * (N - 1) // 2
    for l in range(L):
        sel = net.Y_subs[0] == l
        yi, yj, yv = net.Y_subs[1][sel], net.Y_subs[2][sel], net.Y_vals[sel].astype(float)
        ykey = yi * N + yj
        o = np.argsort(ykey)
        ykey_s, ylam_s = ykey[o], yv[o]

        def lam(i, j):
            k = i * N + j
            p = np.minimum(np.searchsorted(ykey_s, k), max(len(ykey_s) - 1, 0))
            return np.where(ykey_s[p] == k, ylam_s[p], LAMBDA_0) if len(ykey_s) else np.full(len(k), LAMBDA_0)

        ei, ej = np.minimum(yi, yj), np.maximum(yi, yj)
        ek = np.unique(ei * N + ej)
        ei, ej = ek // N, ek % N
        for m in range(M):
            t = theta[l, m]
            # pairs with a true tie
            l_ab, l_ba = lam(ei, ej), lam(ej, ei)
            coin = prng.random_sample(len(ei)) < 0.5
            a_i, a_j = np.where(coin, ei, ej), np.where(coin, ej, ei)
            lf, ls = np.where(coin, l_ab, l_ba), np.where(coin, l_ba, l_ab)
            x1 = prng.poisson((t * lf + eta * t * ls) / (1 - eta * eta))
            x2 = prng.poisson(t * ls + eta * x1)
            # the other pairs
            mu = t * LAMBDA_0
            mm = mu / (1 - eta)
            a = -np.expm1(-mm)
            b = np.exp(-mm) * (-np.expm1(-mu))
            n = prng.binomial(npairs, a + b)
            pi = prng.randint(0, N, n)
            pj = prng.randint(0, N, n)
            keep = pi != pj
            pi, pj = pi[keep], pj[keep]
            pk = np.unique(np.minimum(pi, pj).astype(np.int64) * N + np.maximum(pi, pj))
            pk = pk[~np.isin(pk, ek)]
            pi, pj = pk // N, pk % N
            fp = prng.random_sample(len(pi)) < a / (a + b)
            y1 = np.where(fp, _ztp(prng, np.full(len(pi), mm)), 0)
            y2 = np.where(fp, prng.poisson(mu + eta * y1), _ztp(prng, np.full(len(pi), mu)))
            coin = prng.random_sample(len(pi)) < 0.5
            b_i, b_j = np.where(coin, pi, pj), np.where(coin, pj, pi)
            for (i, j, x) in ((a_i, a_j, x1), (a_j, a_i, x2), (b_i, b_j, y1), (b_j, b_i, y2)):
                pos = x > 0
                subs.append(np.stack([np.full(int(pos.sum()), l), i[pos], j[pos], np.full(int(pos.sum()), m)]))
                vals.append(x[pos])
    s = np.concatenate(subs, axis=1).astype(np.int64)
    v = np.concatenate(vals).astype(np.int64)
    return sptensor(tuple(s), v, shape=(L, N, N, M)), theta
