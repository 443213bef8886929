"""Row-block shards of one fit against the fp64 oracle and the single-rank engine.

A sharded fit packs and iterates the node rows [row0, row0 + nloc) on each rank and all-reduces the three statistics
vectors between the phases (red1 after gamma, red2 after phi, red3 after rho).  Every kernel that reads row0, nloc or a
per-rank count runs a different case on a shard than on one rank.  Here W ranks are emulated on one GPU: W engines, one
per `shard_rows(N, W, r)`, run the phases one by one and the statistics vectors are summed by hand in between (what the
NCCL all-reduce does).  The production cadence (ELBO on the first iteration, then iterations without it, a
statistics-only iteration, a storing one) makes the fast kernels -- the shortcut ties of k_dense_sc, k_all32, the
tie-sorted gamma pass -- run sharded.  A multi-process fit on the all-reporter mask closes the file."""
import os
import socket
import sys
import warnings

import numpy as np
import pytest

from tests.test_gpu_implicit import STATE
from tests.test_gpu_scaled import PRIORS, _cuda

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

PARAMS = ("gamma_shp", "gamma_rte", "phi_shp", "phi_rte", "nu_shp")
# computed on every shard from the same reduced sums: bit-identical across shards
SHARED = ("gamma_shp", "gamma_rte", "phi_shp", "phi_rte", "nu", "elbo_out")
RTOL, RTOL_ELBO, RTOL_RHO = 1e-5, 1e-6, 2e-5  # against the oracle
# k_all32 at K >= 3 on these all-reporter problems: the fp32 posterior cannot follow the free-running fp64 trajectory within
# the tolerances (tests/test_gpu_every_k.py, test_all_mask_boundary_k: the problem's conditioning amplifies the fp32
# rounding of rho about x10 per iteration).  As there, the free-running oracle is held to the tolerances for the first
# steps (the ELBO iteration and two k_all32 iterations; the third reaches 3.7e-5 on rho at K = 3, 4.5e-5 at K = 4, on one
# rank as on several); from then on the oracle restarts every step from the single-rank engine's state, which isolates
# the error of one iteration, with the rho tolerance of that test.
FREE_STEPS_ALL32, RTOL_RHO_ALL32 = 3, 3e-5
# against the single-rank engine: the reduction order differs (parameters ~1e-8 apart), which a few ulp of an fp32 tie
# reflect; the smallest probabilities (log rho ~ -30) amplify it most, hence the absolute floor of the slab comparison
RTOL_ONE, RTOL_ONE_SLAB, ATOL_ONE_SLAB = 1e-6, 5e-6, 1e-15


def _drop_rows(subs, vals, row0, nloc):
    """Every report that touches a node of [row0, row0 + nloc), as row or as column, removed."""
    inside = lambda a: (a >= row0) & (a < row0 + nloc)  # noqa: E731
    keep = ~(inside(subs[1]) | inside(subs[2]))
    return subs[:, keep], vals[keep]


def _ego_net(kind, N, L, K, seed, avg_degree=10, M=None):
    import vimure_b200.synthetic as syn

    if kind == "gm":
        net = syn.Multitensor(N=N, M=M, L=L, K=K, C=2, avg_degree=avg_degree, eta=0.5, seed=seed)
    else:
        net = syn.StandardSBM(N=N, M=M, L=L, K=K, C=2, avg_degree=avg_degree, seed=seed)
    net = net.build_X(mutuality=0.5, seed=seed + 10)
    return np.stack(net.X.subs).astype(np.int64), np.asarray(net.X.vals).astype(np.int64)


def _all_net(N, M, L, K, seed=5):
    import vimure_b200.synthetic as syn

    y = syn.StandardSBM(N=N, M=M, L=L, K=K, C=2, avg_degree=8, seed=seed)
    X, _ = syn.dense_reporting_X(y, M=M, mutuality=0.4, seed=seed + 1)
    return np.stack(X.subs).astype(np.int64), np.asarray(X.vals).astype(np.int64)


def all_k2_l2_problem():
    """The all-reporter problem of the case `all_k2_l2_w3` (also fitted by two processes below)."""
    return _all_net(600, 16, 2, 2)


def _case(name):
    """(subs, vals, L, N, M, K, mask, oracle spec, W, tile_h, shard whose rows carry no reports or None)."""
    import vimure_b200 as vm
    from vimure_b200.model import shard_rows

    ego = lambda L, N, M=None, rep=None, diag=True: (  # noqa: E731
        vm.masks.EgoMask(L, N, N if M is None else M, rep=rep, diag=diag),
        {"kind": "ego", "rep": np.ones((L, N if M is None else M), np.uint8) if rep is None else rep, "diag": diag})
    allm = lambda L, N, M: (vm.masks.AllMask(L, N, M), {"kind": "all", "dense_input": True})  # noqa: E731
    empty = None
    if name == "ego_k3_l4_w8":
        L, N, K, W, tile_h = 4, 1100, 3, 8, 128
        s, v = _ego_net("gm", N, L, K, seed=7)
        M = N
        mask, spec = ego(L, N)
    elif name == "ego_k3_n1024_w8":
        L, N, K, W, tile_h = 2, 1024, 3, 8, 128
        s, v = _ego_net("gm", N, L, K, seed=9)
        M = N
        mask, spec = ego(L, N)
    elif name == "ego_k2_w8_small":
        L, N, K, W, tile_h = 1, 640, 2, 8, 128
        s, v = _ego_net("sbm", N, L, K, seed=11)
        M = N
        mask, spec = ego(L, N)
    elif name == "ego_k4_l2_w2":
        L, N, K, W, tile_h = 2, 600, 4, 2, 64
        s, v = _ego_net("gm", N, L, K, seed=13, avg_degree=12)
        M = N
        mask, spec = ego(L, N)
    elif name == "ego_subset_nodiag_w3":
        L, N, K, M, W, tile_h = 2, 600, 2, 60, 3, 64
        s, v = _ego_net("sbm", N, L, K, seed=15, avg_degree=8, M=M)
        rep = np.zeros((L, M), dtype=np.uint8)
        rep[:, ::2] = 1
        keep = (s[3] < M) & (rep[s[0], np.minimum(s[3], M - 1)] == 1) & (s[1] != s[2])
        s, v = s[:, keep], v[keep]
        mask, spec = ego(L, N, M, rep=rep, diag=False)
    elif name == "all_k2_l2_w3":
        L, N, K, M, W, tile_h = 2, 600, 2, 16, 3, 64
        s, v = all_k2_l2_problem()
        mask, spec = allm(L, N, M)
    elif name == "all_k3_w3":
        L, N, K, M, W, tile_h = 1, 600, 3, 40, 3, 64
        s, v = _all_net(N, M, L, K, seed=21)
        mask, spec = allm(L, N, M)
    elif name == "all_k4_w2":
        L, N, K, M, W, tile_h = 1, 300, 4, 16, 2, 64
        s, v = _all_net(N, M, L, K, seed=23)
        mask, spec = allm(L, N, M)
    elif name == "coo_w2":
        from tests.test_gpu_every_k import _coo_problem

        pb = _coo_problem(3, seed=3)
        s, v, L, N, M, K, mask, spec = (pb[k] for k in ("subs", "vals", "L", "N", "M", "K", "mask", "spec"))
        W, tile_h = 2, 32
    elif name == "empty_shard_ego":
        L, N, K, W, tile_h, empty = 1, 1100, 2, 3, 128, 1
        s, v = _ego_net("sbm", N, L, K, seed=17)
        s, v = _drop_rows(s, v, *shard_rows(N, W, empty))
        s, v = s[:, s[1] != s[2]], v[s[1] != s[2]]
        M = N
        mask, spec = ego(L, N, diag=False)
    elif name == "empty_shard_all":
        L, N, K, M, W, tile_h, empty = 1, 600, 2, 16, 3, 64, 2
        s, v = _all_net(N, M, L, K, seed=25)
        s, v = _drop_rows(s, v, *shard_rows(N, W, empty))
        mask, spec = allm(L, N, M)
    elif name == "mixed_guard":
        L, N, K, W, tile_h = 1, 1100, 2, 3, 128
        s, v = _ego_net("sbm", N, L, K, seed=19)
        # one SIMPLE tie (one report, none reciprocal) with a count of 250 in shard 0's rows: that rank's guard constant
        # X_max fails the underflow bound for the layer, the other ranks' (counts of a few tens at most) do not.  (At 400
        # the oracle's unnormalised exp(log rho) of that tie overflows, as the reference's does.)
        i, j = 5, 300
        pair = ((s[1] == i) & (s[2] == j)) | ((s[1] == j) & (s[2] == i))
        s = np.concatenate([s[:, ~pair], np.array([[0], [i], [j], [i]])], axis=1)
        v = np.concatenate([v[~pair], [250]])
        M = N
        mask, spec = ego(L, N)
    else:
        raise KeyError(name)
    return dict(subs=np.asarray(s, dtype=np.int64), vals=np.asarray(v, dtype=np.int64), L=L, N=N, M=M, K=K, mask=mask,
                spec=spec, W=W, tile_h=tile_h, empty=empty)


CASES = ["ego_k3_l4_w8", "ego_k3_n1024_w8", "ego_k2_w8_small", "ego_k4_l2_w2", "ego_subset_nodiag_w3", "all_k2_l2_w3",
         "all_k3_w3", "all_k4_w2", "coo_w2", "empty_shard_ego", "empty_shard_all", "mixed_guard"]


def _build(c, seed=3):
    """W shards (a storing engine and a slab-free twin each, except for the general mask, which needs the slab), the
    single-rank engine and the oracle, all from one initial state.  The special ties' priors are keyed by the global tie
    id: drawn once on the single-rank packing, looked up per shard."""
    _cuda()
    from oracle.cavi_numpy import OracleCAVI
    from vimure_b200 import _packing
    from vimure_b200._engine import CaviEngine
    from vimure_b200.model import shard_rows

    L, N, M, K, W = c["L"], c["N"], c["M"], c["K"], c["W"]
    subs, vals, mask = c["subs"], c["vals"], c["mask"]
    rs = np.random.RandomState(seed).random_sample
    st = dict(gamma_shp=0.1 * rs((L, M)) + 0.1, phi_shp=10.0 * rs((L, K)) + 10.0, gamma_rte=0.1 * rs((L, M)) + 0.1,
              phi_rte=10.0 * rs((L, K)) + 10.0, nu_shp=0.5 * rs(1)[0] + 0.5)
    nu_rte = PRIORS["beta_eta"] + float(vals.sum())

    def pack(row0, nloc):
        return _packing.pack(subs, vals, L, N, M, K, mask, "cuda", row0=row0, nloc=nloc, tile_h=c["tile_h"])

    P1 = pack(0, None)
    flat1 = P1.t["u_gflat"].cpu().numpy()
    keep1 = (P1.t["u_has_x"] & P1.t["u_reported"]).cpu().numpy()
    assert np.all(np.diff(flat1) > 0)
    pr1 = np.zeros((P1.U, K))
    pr1[:, 0] = 1.0
    pr = 1 + 0.01 * rs((int(keep1.sum()), K))
    pr1[keep1] = pr / pr.sum(axis=1)[:, None]

    def engine(P, slab=True):
        flat = P.t["u_gflat"].cpu().numpy()
        pos = np.searchsorted(flat1, flat)
        assert np.array_equal(flat1[pos], flat)  # a shard's special ties are the single rank's in its rows
        assert np.array_equal(keep1[pos], (P.t["u_has_x"] & P.t["u_reported"]).cpu().numpy())
        e = CaviEngine(P, PRIORS, mutuality=True, eps=1e-12, slab=slab)
        e.set_state(st["gamma_shp"], st["gamma_rte"], st["phi_shp"], st["phi_rte"], st["nu_shp"], nu_rte,
                    pr1[pos], 1e-12)
        return e

    one = engine(P1)
    shards = [pack(*shard_rows(N, W, r)) for r in range(W)]
    engs = [engine(P) for P in shards]
    twins = [engine(P, slab=False) for P in shards] if mask.kind != "coo" else []
    o = OracleCAVI(L, N, M, K, subs, vals, c["spec"], mutuality=True, **PRIORS)
    ties = np.stack([flat1 // (N * N), (flat1 // N) % N, flat1 % N], axis=1)[keep1]
    o.set_state(st["gamma_shp"], st["gamma_rte"], st["phi_shp"], st["phi_rte"], st["nu_shp"],
                o.default_pr_rho(ties, pr1[keep1]))
    return one, engs, twins, o


def _allreduce(group, attr):
    tot = sum(getattr(e, attr) for e in group)
    for e in group:
        getattr(e, attr).copy_(tot)


def _step(group, flags):
    for name, red in (("gamma", "red1"), ("phi", "red2"), ("rho", "red3")):
        for e in group:
            e.phase(name, flags)  # (the gamma and phi phases take no flags)
        _allreduce(group, red)
    for e in group:
        e.phase("finish", flags)


def _assert_case_paths(name, c, one, engs):
    """Each case runs the path it was built for."""
    from vimure_b200._pack_native import dense_fast_eligible

    P1, W, N, K = one.P, c["W"], c["N"], c["K"]
    fast = dense_fast_eligible(K, P1.r_mode, N, P1.tile_w, P1.tile_h)
    nl = [e.P.nloc for e in engs]
    assert sum(nl) == N and engs[0].P.row0 == 0 and all(e.P.row0 > 0 for e in engs[1:])
    if name.startswith("ego") or name in ("empty_shard_ego", "mixed_guard"):
        assert fast and all(e.simple_mode for e in engs) and one.simple_mode
    if name.startswith("all") or name == "empty_shard_all":
        assert fast and one.all32_mode and one.gamma_ts
    if name == "ego_k3_l4_w8":
        assert N % P1.tile_w and all(c["tile_h"] < n < 2 * c["tile_h"] for n in nl)  # one full row tile + a partial one
        assert all(0 < e.P.n_cx < e.P.U for e in engs)  # list-mode special-tie kernel next to the shortcut ties
    elif name == "ego_k3_n1024_w8":
        assert N % P1.tile_w == 0 and all(n == c["tile_h"] for n in nl)
    elif name == "ego_k2_w8_small":
        assert all(n < c["tile_h"] for n in nl)
    elif name == "ego_k4_l2_w2":
        assert P1.tile_w == 256
    elif name == "ego_subset_nodiag_w3":
        assert engs[-1].P.row0 >= c["M"] and engs[-1].P.I > 0 and not engs[-1].P.ego_diag
    elif name in ("all_k2_l2_w3", "all_k3_w3", "all_k4_w2"):
        assert all(e.all32_mode and e.gamma_ts for e in engs)
        if name == "all_k3_w3":  # ties the fp64 special-tie kernel sweeps warp-cooperatively
            assert all(int(e.P.t["u_cnt"].max()) > 8 for e in engs)
    elif name == "coo_w2":
        assert P1.r_mode == 2 and not fast and all(e.P.I1 > 0 for e in engs)
    elif name == "empty_shard_ego":
        # the rank's special ties are its (unreported) diagonal ties: no entry, nothing for the gamma / phi passes, no
        # shortcut tie
        z = engs[c["empty"]]
        assert z.P.I == 0 and z.P.I1 == 0 and z.P.U == z.P.nloc and z.P.n_cx == z.P.U
        assert all(e.P.I1 > 0 for r, e in enumerate(engs) if r != c["empty"])
    elif name == "empty_shard_all":
        z = engs[c["empty"]]
        assert z.P.U == 0 and z.P.I1 == 0 and not z.all32_mode and not z.gamma_ts
        assert all(e.all32_mode and e.gamma_ts for r, e in enumerate(engs) if r != c["empty"])


def _expected_simple(name, c, e, r):
    """The per-layer VM_LC_SIMPLE flag rank r is built to compute: the fp32 paths on every rank that runs them, except
    shard 0 of `mixed_guard`, whose own count-250 tie fails the guard (a rank decides from its own special ties)."""
    on = (e.simple_mode and e.P.r_mode == 0) or (e.all32_mode and e.P.r_mode == 1)
    flags = np.full(c["L"], 1.0 if on else 0.0)
    if name == "mixed_guard" and r == 0:
        flags[0] = 0.0
    return flags


def _rho_at_oracle(o, flat):
    N = o.N
    return o.rho[flat // (N * N), (flat // N) % N, flat % N]


@pytest.mark.parametrize("name", CASES)
def test_shards_match_the_oracle_and_the_single_rank(name):
    torch = _cuda()
    c = _case(name)
    one, engs, twins, o = _build(c)
    _assert_case_paths(name, c, one, engs)
    L, N, K = c["L"], c["N"], c["K"]
    F = one.C
    lcs = 3 * K + 5
    # the mixed-guard case runs one layer in fp64 on one rank and in fp32 on the others, while the single rank runs it in
    # fp64 everywhere: the shards then differ from the single rank by the fp32 evaluation of the shortcut ties
    rtol_one = 5e-6 if name == "mixed_guard" else RTOL_ONE
    rtol_one_slab = 1e-5 if name == "mixed_guard" else RTOL_ONE_SLAB
    for group in (engs, twins):
        if group:
            _allreduce(group, "red3")  # the initial statistics were computed per shard
    # (the general mask has no statistics-only iteration: its statistics gather the stored slab, VM_ENOTSUP)
    nost = ("store", 0) if c["mask"].kind == "coo" else ("statistics only", F["VM_F_NO_STORE"])
    cadence = [("ELBO", F["VM_F_ELBO"])] + [("fast", 0)] * 3 + [("ELBO", F["VM_F_ELBO"]), nost, ("store", 0)]
    restart = one.all32_mode and K >= 3
    for step, (what, fl) in enumerate(cadence):
        tag = f"{name} step {step} ({what})"
        free = not restart or step < FREE_STEPS_ALL32  # against the free-running oracle
        rtol_rho = RTOL_RHO if free else RTOL_RHO_ALL32
        if not free:
            tag += ", oracle restarted from the single rank's state"
            q = one.params()
            o.gamma_shp, o.gamma_rte, o.phi_shp, o.phi_rte = (q[k] for k in ("gamma_shp", "gamma_rte", "phi_shp", "phi_rte"))
            o.nu_shp = float(q["nu_shp"])
            o.rho = one.materialize_rows(0, L * N).view(L, N, N, K).cpu().numpy().astype(np.float64)
        _step(engs, fl)
        if twins:
            _step(twins, fl)
        one.iterate(1, elbo_last=bool(fl & F["VM_F_ELBO"]), store=not (fl & F["VM_F_NO_STORE"]),
                    store_last=not (fl & F["VM_F_NO_STORE"]))
        o.iterate()
        for e in engs[1:]:
            for k in SHARED:
                assert torch.equal(getattr(e, k), getattr(engs[0], k)), f"{k} differs across shards: {tag}"
        p, q = engs[0].params(), one.params()
        for k in PARAMS:
            np.testing.assert_allclose(p[k], getattr(o, k), rtol=RTOL, err_msg=f"{k} vs oracle: {tag}")
            np.testing.assert_allclose(p[k], q[k], rtol=rtol_one, err_msg=f"{k} vs single rank: {tag}")
        if fl & F["VM_F_ELBO"]:
            np.testing.assert_allclose(engs[0].elbo(), o.elbo(), rtol=RTOL_ELBO, err_msg=tag)
            np.testing.assert_allclose(engs[0].elbo(), one.elbo(), rtol=RTOL_ELBO, err_msg=tag)
        flat1 = one.P.t["u_gflat"].cpu().numpy()
        ru1 = one.rho_u32.cpu().numpy().astype(np.float64)
        np.testing.assert_allclose(ru1, _rho_at_oracle(o, flat1), rtol=rtol_rho, atol=1e-30,
                                   err_msg=f"rho_u32 of the single rank: {tag}")
        for r, e in enumerate(engs):
            if e.P.U:
                flat = e.P.t["u_gflat"].cpu().numpy()
                ru = e.rho_u32.cpu().numpy().astype(np.float64)
                np.testing.assert_allclose(ru, ru1[np.searchsorted(flat1, flat)], rtol=rtol_one_slab, atol=ATOL_ONE_SLAB,
                                           err_msg=f"rho_u32 of shard {r} vs single rank: {tag}")
                np.testing.assert_allclose(ru, _rho_at_oracle(o, flat), rtol=rtol_rho, atol=1e-30,
                                           err_msg=f"rho_u32 of shard {r}: {tag}")
            lc = e.layer_consts.cpu().numpy().reshape(L, lcs)[:, 2 * K + 4]
            assert np.array_equal(lc, _expected_simple(name, c, e, r)), f"VM_LC_SIMPLE of shard {r}: {lc}, {tag}"
        for r, (e, t) in enumerate(zip(engs, twins)):
            for k in STATE:
                assert torch.equal(getattr(e, k), getattr(t, k)), f"{k} of shard {r} without a slab: {tag}"
    if name == "mixed_guard":
        lc1 = one.layer_consts.cpu().numpy().reshape(L, lcs)[:, 2 * K + 4]
        assert lc1[0] == 0.0  # the single rank sees the count-250 tie too

    # ---- the slabs
    slab = torch.cat([e.rho_slab() for e in engs], dim=1)
    a = slab.cpu().numpy().astype(np.float64)
    np.testing.assert_allclose(a, o.rho, rtol=rtol_rho, atol=1e-30, err_msg=f"{name}: slab vs oracle")
    np.testing.assert_allclose(a, one.rho_slab().cpu().numpy(), rtol=rtol_one_slab, atol=ATOL_ONE_SLAB,
                               err_msg=f"{name}: slab vs single rank")
    for r, (e, t) in enumerate(zip(engs, twins)):
        n = e.P.L * e.P.nloc
        assert torch.equal(t.materialize_rows(0, n), e.rho_slab().view(n, N, K)), f"{name}: shard {r} materialised"

    # ---- the consumers, shard by shard
    rng = np.random.RandomState(1)
    keys = np.unique(np.concatenate([rng.randint(0, L * N * N, 20000), one.P.t["u_gflat"].cpu().numpy()]))
    kd = torch.as_tensor(keys, device=engs[0].dev)
    want = _rho_at_oracle(o, keys)
    row = (keys // N) % N
    # (a tie whose top two posteriors lie within the comparison's tolerance of each other can flip: 0.4999994 / 0.5000006
    # is 0.5 / 0.5 in fp32)
    top = np.sort(o.rho, axis=-1)
    clear = (top[..., -1] - top[..., -2]) >= np.maximum(1e-6, 2 * rtol_rho * top[..., -1])
    lab = np.zeros((L, N, N), dtype=np.int64)
    for r, e in enumerate(engs):
        got = e.rho_at(kd).cpu().numpy().astype(np.float64)
        own = (row >= e.P.row0) & (row < e.P.row0 + e.P.nloc)
        assert not got[~own].any(), f"{name}: shard {r} answered keys of other rows"
        np.testing.assert_allclose(got[own], want[own], rtol=rtol_rho, atol=1e-30, err_msg=f"{name}: rho_at, shard {r}")
        ek, ev = e.infer_edges(0)
        ek, ev = ek.cpu().numpy(), ev.cpu().numpy()
        ei = (ek // N) % N
        assert np.all((ei >= e.P.row0) & (ei < e.P.row0 + e.P.nloc)), f"{name}: shard {r} emitted edges of other rows"
        lab.reshape(-1)[ek] = ev
    mine = np.argmax(a, axis=-1)
    bad = np.flatnonzero(lab != mine)
    assert not bad.size, f"{name}: edges vs the slab's argmax at {bad.size} ties, first {bad[:5]}: {lab.flat[bad[:5]]} " \
                         f"vs {mine.flat[bad[:5]]}"
    ref = np.argmax(o.rho, axis=-1)
    bad = np.flatnonzero(clear & (lab != ref))
    assert not bad.size, f"{name}: edges vs the oracle's argmax at {bad.size} ties, first {bad[:5]}: " \
                         f"{lab.flat[bad[:5]]} vs {ref.flat[bad[:5]]}, oracle {o.rho.reshape(-1, K)[bad[:5]]}, " \
                         f"slab {a.reshape(-1, K)[bad[:5]]}"
    torch.cuda.synchronize()


# ---------------------------------------------------------------------------------------------------- multi-process fit

def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


FIT = dict(K=2, seed=11, max_iter=12, num_realisations=1, init="reference")


def _fit(X, mask, **kw):
    import vimure_b200 as vm

    m = vm.VimureModel(mutuality=True, convergence_tol=0.0)
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        m.fit(X, R=mask, **FIT, **kw)
    return m


def _rho_keys(L, N, n=10000):
    rng = np.random.RandomState(2)
    return rng.randint(0, L, n), rng.randint(0, N, n), rng.randint(0, N, n)


def _fit_record(m, L, N):
    e = m._engine
    return dict(params={k: np.array(getattr(m, k)) for k in PARAMS}, maxL=float(m.maxL),
                rho=m.rho_f_at(_rho_keys(L, N)), world=m._world, modes=(e.all32_mode, e.gamma_ts),
                graphs=bool(e._graphs))


def _all_mask_worker(rank, world, port, ngpu, out):
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    sys.path.insert(0, ROOT)
    import torch
    import torch.distributed as dist

    dev = rank if ngpu >= world else 0
    torch.cuda.set_device(dev)
    if ngpu >= world:
        dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", dev))
    else:
        dist.init_process_group("gloo", rank=rank, world_size=world)
    res = {}
    try:
        import vimure_b200 as vm
        from vimure_b200.model import shard_rows

        L, N, M = 2, 600, 16
        s, v = all_k2_l2_problem()
        mask = vm.masks.AllMask(L, N, M)
        res["all"] = _fit_record(_fit(vm.sptensor.sptensor(tuple(s), v, shape=(L, N, N, M)), mask), L, N)
        row0, nloc = shard_rows(N, world, rank)
        own = (s[1] >= row0) & (s[1] < row0 + nloc)
        Xs = vm.sptensor.sptensor(tuple(s[:, own]), v[own], shape=(L, N, N, M))
        res["rows"] = _fit_record(_fit(Xs, mask, presharded="rows"), L, N)
        res["ok"] = True
    except Exception:  # noqa: BLE001
        import traceback

        res["ok"] = False
        res["error"] = traceback.format_exc()[-2000:]
    out.put((rank, res))
    dist.destroy_process_group()


def test_two_rank_fit_on_the_all_reporter_mask():
    """`VimureModel.fit` by two ranks on the all-reporter mask (k_all32 and the tie-sorted gamma pass on every rank; with
    two devices NCCL and the captured sharded graph, with one gloo and eager launches), from the whole list and from each
    rank's own rows (presharded="rows"), against a single-rank fit from the same seed."""
    torch = _cuda()
    import torch.multiprocessing as mp
    import vimure_b200 as vm

    L, N, M = 2, 600, 16
    s, v = all_k2_l2_problem()
    ref = _fit(vm.sptensor.sptensor(tuple(s), v, shape=(L, N, N, M)), vm.masks.AllMask(L, N, M))
    eng = ref._engine
    assert eng.all32_mode and eng.gamma_ts and ref._world == 1
    want = _fit_record(ref, L, N)
    ngpu, world = torch.cuda.device_count(), 2
    ctx = mp.get_context("spawn")
    out = ctx.Queue()
    port = _free_port()
    ps = [ctx.Process(target=_all_mask_worker, args=(r, world, port, ngpu, out)) for r in range(world)]
    for p in ps:
        p.start()
    results = dict(out.get(timeout=900) for _ in ps)
    for p in ps:
        p.join(timeout=120)
    for rank in range(world):
        res = results[rank]
        assert res["ok"], res.get("error")
        for mode in ("all", "rows"):
            got, tag = res[mode], f"rank {rank}, {mode}"
            assert got["world"] == world and got["modes"] == (True, True), tag
            assert got["graphs"] == (ngpu >= world), tag  # NCCL replays the captured sharded iteration
            for k in PARAMS:
                np.testing.assert_allclose(got["params"][k], want["params"][k], rtol=1e-6, err_msg=f"{k}: {tag}")
            np.testing.assert_allclose(got["maxL"], want["maxL"], rtol=1e-8, err_msg=tag)
            np.testing.assert_allclose(got["rho"], want["rho"], rtol=5e-6, atol=1e-30, err_msg=tag)
