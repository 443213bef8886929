"""Scaled-down versions of BASELINE configs 3-5 against the CPU oracle, and size-independent properties at the
full config-3 size (N = 20 000), all through the C ABI."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

PRIORS = dict(alpha_theta=0.1, beta_theta=0.1, alpha_lambda=10.0, beta_lambda=10.0, alpha_eta=0.5, beta_eta=1.0)


def _cuda():
    import torch

    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")
    return torch


def _engine_and_oracle(net, mask, spec, K, mutuality=True, seed=3, tile_h=64, row0=0, nloc=None, simple=True, all32=True):
    _cuda()
    from oracle.cavi_numpy import OracleCAVI
    from vimure_b200 import _packing
    from vimure_b200._engine import CaviEngine

    L, N, M = net.X.shape[0], net.X.shape[1], net.X.shape[3]
    subs = np.stack(net.X.subs)
    P = _packing.pack(subs, net.X.vals, L, N, M, K, mask, "cuda", row0=row0, nloc=nloc, tile_h=tile_h,
                      mutuality=mutuality, simple=simple)
    eng = CaviEngine(P, PRIORS, mutuality=mutuality, eps=1e-12, all32=all32)
    prng = np.random.RandomState(seed)
    rs = prng.random_sample
    st = dict(gamma_shp=0.1 * rs((L, M)) + 0.1, phi_shp=10.0 * rs((L, K)) + 10.0, gamma_rte=0.1 * rs((L, M)) + 0.1,
              phi_rte=10.0 * rs((L, K)) + 10.0, nu_shp=0.5 * rs(1)[0] + 0.5)
    keep = (P.t["u_has_x"] & P.t["u_reported"]).cpu().numpy()
    pr_u = np.zeros((P.U, K))
    pr_u[:, 0] = 1.0
    pr = 1 + 0.01 * rs((int(keep.sum()), K))
    pr_u[keep] = pr / pr.sum(axis=1)[:, None]
    nu_rte = PRIORS["beta_eta"] + float(net.X.vals.sum())
    eng.set_state(st["gamma_shp"], st["gamma_rte"], st["phi_shp"], st["phi_rte"], st["nu_shp"] if mutuality else 1e-6,
                  nu_rte if mutuality else 1.0, pr_u, 1e-12)
    o = None
    if spec is not None:
        o = OracleCAVI(L, N, M, K, subs, net.X.vals, spec, mutuality=mutuality, **PRIORS)
        flat = P.t["u_gflat"].cpu().numpy()[keep]
        ties = np.stack([flat // (N * N), (flat // N) % N, flat % N], axis=1)
        o.set_state(st["gamma_shp"], st["gamma_rte"], st["phi_shp"], st["phi_rte"], st["nu_shp"],
                    o.default_pr_rho(ties, pr_u[keep]))
    return eng, o, P


def _compare(eng, o, iters):
    for it in range(iters):
        eng.iterate(1, elbo_last=True)
        o.iterate()
        p = eng.params()
        np.testing.assert_allclose(p["gamma_shp"], o.gamma_shp, rtol=1e-5, err_msg=f"it{it}")
        np.testing.assert_allclose(p["gamma_rte"], o.gamma_rte, rtol=1e-5, err_msg=f"it{it}")
        np.testing.assert_allclose(p["phi_shp"], o.phi_shp, rtol=1e-5, err_msg=f"it{it}")
        np.testing.assert_allclose(p["phi_rte"], o.phi_rte, rtol=1e-5, err_msg=f"it{it}")
        if o.mutuality:
            np.testing.assert_allclose(p["nu_shp"], o.nu_shp, rtol=1e-5, err_msg=f"it{it}")
        np.testing.assert_allclose(eng.elbo(), o.elbo(), rtol=1e-6, err_msg=f"it{it}")
    rho = eng.rho_slab().cpu().numpy().astype(np.float64)
    np.testing.assert_allclose(rho, o.rho, rtol=2e-5, atol=1e-30)


def test_config3_scaled_sbm_ego_k2():
    """config 3 law (StandardSBM, ego-only, K=2) at N=1100: two column tiles (one partial), several row tiles."""
    import vimure_b200.synthetic as syn

    net = syn.StandardSBM(N=1100, L=1, K=2, C=2, avg_degree=10, seed=10).build_X(mutuality=0.5, seed=20)
    spec = {"kind": "ego", "rep": np.ones((1, 1100), dtype=np.uint8), "diag": True}
    eng, o, _ = _engine_and_oracle(net, net.R, spec, 2)
    _compare(eng, o, 4)


def test_config4_scaled_dense_reporting():
    """config 4 law (every reporter reports every tie, L=2, K=2) at N=300, M=16: the reporter-reduction heavy case."""
    import vimure_b200 as vm
    import vimure_b200.synthetic as syn

    y = syn.StandardSBM(N=300, M=16, L=2, K=2, C=2, avg_degree=8, seed=5)
    X, theta = syn.dense_reporting_X(y, M=16, mutuality=0.4, seed=6)

    class Net:
        pass

    net = Net()
    net.X = X
    eng, o, _ = _engine_and_oracle(net, vm.masks.AllMask(2, 300, 16), {"kind": "all", "dense_input": True}, 2)
    _compare(eng, o, 4)


@pytest.mark.parametrize("case", ["k2_m16", "k3_m40_nomut_layer"])
def test_all_reporter_mask_fp32_special_ties(case):
    """All-reporter mask: on iterations without ELBO every special tie is evaluated in fp32, entry-parallel (k_all32,
    include/vimure_b200.h: vm_ctx.all32_mode).  Against the oracle (usual tolerances, after runs of such iterations, slab
    included) and against the same engine on the fp64 special-tie kernel (all32=False)."""
    torch = _cuda()
    import vimure_b200 as vm
    import vimure_b200.synthetic as syn

    if case == "k2_m16":
        L, N, M, K, mut = 2, 300, 16, 2, 0.4
    else:  # more reporters than a tie group's stage slice would hold per tie is not needed: several entries per tie, K = 3
        L, N, M, K, mut = 1, 200, 40, 3, 0.5
    y = syn.StandardSBM(N=N, M=M, L=L, K=K, C=2, avg_degree=8, seed=5)
    X, theta = syn.dense_reporting_X(y, M=M, mutuality=mut, seed=6)

    class Net:
        pass

    net = Net()
    net.X = X
    mask = vm.masks.AllMask(L, N, M)
    eng, o, P = _engine_and_oracle(net, mask, {"kind": "all", "dense_input": True}, K)
    assert eng.all32_mode
    ref, _, _ = _engine_and_oracle(net, mask, None, K, all32=False)
    assert not ref.all32_mode

    def check(tag):
        p, q = eng.params(), ref.params()
        for k in ("gamma_shp", "gamma_rte", "phi_shp", "phi_rte"):
            np.testing.assert_allclose(p[k], getattr(o, k), rtol=1e-5, err_msg=f"{k} vs oracle {tag}")
            np.testing.assert_allclose(p[k], q[k], rtol=5e-6, err_msg=f"{k} vs fp64 path {tag}")
        np.testing.assert_allclose(p["nu_shp"], o.nu_shp, rtol=1e-5, err_msg=tag)
        np.testing.assert_allclose(p["nu_shp"], q["nu_shp"], rtol=5e-6, err_msg=tag)
        a = eng.rho_slab().cpu().numpy().astype(np.float64)
        np.testing.assert_allclose(a, o.rho, rtol=2e-5, atol=1e-30, err_msg=tag)
        np.testing.assert_allclose(a, ref.rho_slab().cpu().numpy(), rtol=2e-5, atol=1e-30, err_msg=tag)

    for e in (eng, ref):
        e.iterate(3)  # iterations without ELBO: the fp32 kernel
    for _ in range(3):
        o.iterate()
    lc = eng.layer_consts.cpu().numpy().reshape(L, 3 * K + 5)
    assert (lc[:, 2 * K + 4] == 1.0).all()  # every layer's guard holds
    check("after 3 fp32 iterations")
    for e in (eng, ref):
        e.iterate(3, elbo_last=True)
    for _ in range(3):
        o.iterate()
    np.testing.assert_allclose(eng.elbo(), o.elbo(), rtol=1e-6)
    np.testing.assert_allclose(eng.elbo(), ref.elbo(), rtol=1e-7)
    check("after an ELBO iteration")
    for e in (eng, ref):
        e.iterate(2)
    for _ in range(2):
        o.iterate()
    check("fp32 iterations after an ELBO iteration")
    torch.cuda.synchronize()


def test_config5_scaled_gm_l2_k3():
    """config 5 law (Multitensor/GMReciprocity, ego-only, K=3, several layers) at N=640, L=2 (N % 4 == 0: fast kernel)."""
    import vimure_b200.synthetic as syn

    net = syn.Multitensor(N=640, L=2, K=3, C=2, avg_degree=10, eta=0.5, seed=7).build_X(mutuality=0.5, seed=8)
    spec = {"kind": "ego", "rep": np.ones((2, 640), dtype=np.uint8), "diag": True}
    eng, o, _ = _engine_and_oracle(net, net.R, spec, 3)
    _compare(eng, o, 4)


def test_k4_and_k5_paths():
    """K=4 (strided lane mapping) and K=5 (generic kernel only) against the oracle."""
    import vimure_b200.synthetic as syn

    for K, N in ((4, 520), (5, 260)):
        net = syn.Multitensor(N=N, L=1, K=K, C=2, avg_degree=12, eta=0.3, seed=K).build_X(mutuality=0.3, seed=K + 1)
        spec = {"kind": "ego", "rep": np.ones((1, N), dtype=np.uint8), "diag": True}
        eng, o, _ = _engine_and_oracle(net, net.R, spec, K)
        _compare(eng, o, 3)


def test_full_size_properties_config3():
    """N = 20 000 (4e8 ties): properties that do not need the oracle."""
    torch = _cuda()
    import vimure_b200.synthetic as syn

    N, K = 20000, 2
    net = syn.StandardSBM(N=N, L=1, K=K, C=2, avg_degree=10, seed=10).build_X(mutuality=0.5, seed=20)
    runs = []
    for rep in range(2):
        eng, _, P = _engine_and_oracle(net, net.R, None, K)
        eng.iterate(3, elbo_last=True)
        p = eng.params()
        runs.append((p, eng.elbo()))
        if rep == 0:
            # (i) the reporter statistic conserves the number of reported ties: sum_k A[l,m,k] = 2N-1
            A = eng.red3[: N * K].cpu().numpy().reshape(N, K)
            np.testing.assert_allclose(A.sum(axis=1), 2 * N - 1, rtol=0, atol=1e-6)
            # (ii) every stored tie is a probability vector; special ties carry their fp64-computed posterior
            slab = eng.rho_slab()
            rows = torch.randint(0, N, (64,), device=slab.device)
            s = slab[0, rows].sum(dim=-1)
            assert float((s - 1).abs().max()) < 1e-6
            u = torch.randint(0, P.U, (100000,), device=slab.device)
            got = slab[0, P.t["u_lrow"][u].long(), P.t["u_col"][u].long()]
            assert torch.equal(got, eng.rho_u32[u])
            # (iii) the ELBO is finite
            assert np.isfinite(eng.elbo())
        del eng
        torch.cuda.empty_cache()
    # (iv) bit-reproducible run to run (deterministic two-pass reductions + integer atomics)
    for k in ("gamma_shp", "gamma_rte", "phi_shp", "phi_rte", "nu_shp"):
        assert np.array_equal(runs[0][0][k], runs[1][0][k]), k
    assert runs[0][1] == runs[1][1]


@pytest.mark.parametrize("case", ["sbm_k2", "gm_l2_k3", "nomut_k2", "subset_k4"])
def test_simple_special_ties_in_the_dense_kernel(case):
    """On iterations without ELBO the shortcut kernel (k_shortcut) evaluates the special ties that have no reciprocal report
    (fp32, include/vimure_b200.h: vm_ctx.simple_mode) and the special-tie kernel only walks the others.  Against the
    oracle (the usual tolerances, after runs of such iterations) and against the same engine with the shortcut off."""
    torch = _cuda()
    import vimure_b200 as vm
    import vimure_b200.synthetic as syn

    mutuality = True
    if case == "sbm_k2":  # two full column tiles + a partial one
        L, N, K = 1, 1100, 2
        net = syn.StandardSBM(N=N, L=L, K=K, C=2, avg_degree=10, seed=10).build_X(mutuality=0.5, seed=20)
        mask, rep, diag = net.R, np.ones((L, N), dtype=np.uint8), True
    elif case == "gm_l2_k3":
        L, N, K = 2, 640, 3
        net = syn.Multitensor(N=N, L=L, K=K, C=2, avg_degree=8, eta=0.5, seed=3).build_X(mutuality=0.5, seed=4)
        mask, rep, diag = net.R, np.ones((L, N), dtype=np.uint8), True
    elif case == "nomut_k2":  # mutuality off: every tie with a report is simple
        L, N, K, mutuality = 1, 600, 2, False
        net = syn.StandardSBM(N=N, L=L, K=K, C=2, avg_degree=6, seed=5).build_X(mutuality=0.3, seed=6)
        mask, rep, diag = net.R, np.ones((L, N), dtype=np.uint8), True
    else:  # reporters are a subset of the nodes, no diagonal entries in the mask
        L, N, K, M = 2, 520, 4, 60
        net = syn.StandardSBM(N=N, M=M, L=L, K=K, C=2, avg_degree=6, seed=7).build_X(mutuality=0.4, seed=8)
        rep = np.zeros((L, M), dtype=np.uint8)
        rep[:, ::2] = 1
        s = np.stack(net.X.subs)
        keep = (s[3] < M) & (rep[s[0], np.minimum(s[3], M - 1)] == 1)
        net.X = vm.sptensor.sptensor(tuple(s[:, keep]), np.asarray(net.X.vals)[keep], shape=(L, N, N, M))
        mask, diag = vm.masks.EgoMask(L, N, M, rep=rep, diag=False), False
    spec = {"kind": "ego", "rep": rep, "diag": diag}
    eng, o, P = _engine_and_oracle(net, mask, spec, K, mutuality=mutuality, tile_h=32)
    assert eng.simple_mode and int(P.t["u_simple"].sum()) > 0 and P.n_cx < P.U
    assert bool(P.t["u_single"].any()) == mutuality
    ref, _, P2 = _engine_and_oracle(net, mask, None, K, mutuality=mutuality, tile_h=32, simple=False)
    assert not ref.simple_mode and P2.n_cx == P2.U

    def check(tag, slab):
        p, q = eng.params(), ref.params()
        for k in ("gamma_shp", "gamma_rte", "phi_shp", "phi_rte"):
            np.testing.assert_allclose(p[k], getattr(o, k), rtol=1e-5, err_msg=f"{k} vs oracle {tag}")
            np.testing.assert_allclose(p[k], q[k], rtol=5e-6, err_msg=f"{k} vs fp64 path {tag}")
        if mutuality:
            np.testing.assert_allclose(p["nu_shp"], o.nu_shp, rtol=1e-5, err_msg=tag)
        if slab:
            a = eng.rho_slab().cpu().numpy().astype(np.float64)
            np.testing.assert_allclose(a, o.rho, rtol=2e-5, atol=1e-30, err_msg=tag)
            np.testing.assert_allclose(a, ref.rho_slab().cpu().numpy(), rtol=1e-5, atol=1e-30, err_msg=tag)

    # the layers do take the shortcut (flag written by k_phi_finish), and the special-tie kernel skips the simple ties
    for e in (eng, ref):
        e.iterate(2)  # two iterations without ELBO
    o.iterate()
    o.iterate()
    lc = eng.layer_consts.cpu().numpy().reshape(L, 3 * K + 5)
    assert (lc[:, 2 * K + 4] == 1.0).all()
    check("after 2 fast iterations", slab=True)
    for e in (eng, ref):
        e.iterate(4, elbo_last=True)  # three more without, then one with the ELBO (every special tie in fp64)
    for _ in range(4):
        o.iterate()
    np.testing.assert_allclose(eng.elbo(), o.elbo(), rtol=1e-6)
    np.testing.assert_allclose(eng.elbo(), ref.elbo(), rtol=1e-7)
    check("after an ELBO iteration", slab=True)
    for e in (eng, ref):
        e.iterate(3)
    for _ in range(3):
        o.iterate()
    check("fast iterations after an ELBO iteration", slab=True)
    torch.cuda.synchronize()


def test_shortcut_ties_vs_fp64_path_at_config3_size():
    """N = 20 000 (config 3): 10 iterations in which the shortcut kernel evaluates the SIMPLE and SINGLE special ties in
    fp32 against the same 10 iterations with every special tie in fp64 (simple=False).  The fp32 table rounding is common
    to all ties of a node, so its effect does not average down with N: this is the size at which it has to be checked."""
    torch = _cuda()
    import vimure_b200.synthetic as syn

    N, K = 20000, 2
    net = syn.StandardSBM(N=N, L=1, K=K, C=2, avg_degree=10, seed=10).build_X(mutuality=0.5, seed=20)
    res = {}
    for mode in ("shortcut", "fp64"):
        eng, _, P = _engine_and_oracle(net, net.R, None, K, tile_h=128, simple=(mode == "shortcut"))
        assert eng.simple_mode == (mode == "shortcut")
        if mode == "shortcut":
            frac = 1.0 - P.n_cx / P.U
            assert frac > 0.9, frac  # almost every special tie takes the shortcut at this density
        eng.iterate(9)
        p9 = eng.params()
        eng.iterate(1, elbo_last=True)
        res[mode] = (p9, eng.params(), eng.elbo())
        del eng, P
        torch.cuda.empty_cache()
    for which in (0, 1):
        a, b = res["shortcut"][which], res["fp64"][which]
        for k in ("gamma_shp", "gamma_rte", "phi_shp", "phi_rte", "nu_shp"):
            np.testing.assert_allclose(a[k], b[k], rtol=5e-6, err_msg=f"{k} after {9 + which} iterations")
    np.testing.assert_allclose(res["shortcut"][2], res["fp64"][2], rtol=1e-7)


@pytest.mark.parametrize("cfg", ["c3", "c5"])
def test_oracle_parity_at_n4096(cfg):
    """Configs 3 and 5 at N = 4096 (8 column tiles, 32 row tiles) against the CPU oracle, on the production cadence:
    iteration 1 with ELBO, three without (shortcut ties in fp32), one with."""
    import vimure_b200.synthetic as syn

    if cfg == "c3":
        L, N, K = 1, 4096, 2
        net = syn.StandardSBM(N=N, L=L, K=K, C=2, avg_degree=10, seed=10).build_X(mutuality=0.5, seed=20)
    else:
        L, N, K = 2, 4096, 3
        net = syn.Multitensor(N=N, L=L, K=K, C=2, avg_degree=10, eta=0.5, seed=10).build_X(mutuality=0.5, seed=20)
    spec = {"kind": "ego", "rep": np.ones((L, N), dtype=np.uint8), "diag": True}
    eng, o, P = _engine_and_oracle(net, net.R, spec, K, tile_h=128)
    assert eng.simple_mode

    def check(tag, elbo):
        p = eng.params()
        for k in ("gamma_shp", "gamma_rte", "phi_shp", "phi_rte", "nu_shp"):
            np.testing.assert_allclose(p[k], getattr(o, k), rtol=1e-5, err_msg=f"{k} {tag}")
        if elbo:
            np.testing.assert_allclose(eng.elbo(), o.elbo(), rtol=1e-6, err_msg=tag)

    eng.iterate(1, elbo_last=True)
    o.iterate()
    check("it1", True)
    for it in range(3):
        eng.iterate(1)
        o.iterate()
        check(f"it{it + 2}", False)
    eng.iterate(1, elbo_last=True)
    o.iterate()
    check("it5", True)
    rho = eng.rho_slab().cpu().numpy().astype(np.float64)
    np.testing.assert_allclose(rho, o.rho, rtol=2e-5, atol=1e-30)
    top = np.sort(o.rho, axis=-1)
    clear = (top[..., -1] - top[..., -2]) >= 1e-6
    assert np.array_equal(np.argmax(rho, -1)[clear], np.argmax(o.rho, -1)[clear])


def test_simple_special_ties_sharded_rows():
    """The shortcut with row-block sharding (row0 > 0): three shards of the N=1100 problem, statistics vectors summed by
    hand between the phases (what the NCCL all-reduce does), iterations without ELBO -- against the single-rank engine."""
    torch = _cuda()
    import vimure_b200.synthetic as syn
    from vimure_b200.model import shard_rows

    L, N, K, W = 1, 1100, 2, 3
    net = syn.StandardSBM(N=N, L=L, K=K, C=2, avg_degree=10, seed=10).build_X(mutuality=0.5, seed=20)
    one, _, _ = _engine_and_oracle(net, net.R, None, K, tile_h=32)
    engs = [_engine_and_oracle(net, net.R, None, K, tile_h=32, row0=r0, nloc=nl)[0]
            for r0, nl in (shard_rows(N, W, r) for r in range(W))]
    assert all(e.simple_mode for e in engs) and sum(e.P.U - e.P.n_cx for e in engs) == one.P.U - one.P.n_cx
    F = one.C
    # the helper draws the priors of a shard's ties from one stream: key them by the GLOBAL tie instead, so that every
    # decomposition starts from the same state
    rs = np.random.RandomState(3).random_sample
    st = dict(gamma_shp=0.1 * rs((L, N)) + 0.1, phi_shp=10.0 * rs((L, K)) + 10.0, gamma_rte=0.1 * rs((L, N)) + 0.1,
              phi_rte=10.0 * rs((L, K)) + 10.0, nu_shp=0.5 * rs(1)[0] + 0.5)
    table = 1 + 0.01 * np.random.RandomState(4).random_sample((1 << 16, K))
    for e in [one] + engs:
        P = e.P
        keep = (P.t["u_has_x"] & P.t["u_reported"]).cpu().numpy()
        flat = P.t["u_gflat"].cpu().numpy()
        pr_u = np.zeros((P.U, K))
        pr_u[:, 0] = 1.0
        pr = table[(flat[keep] * 2654435761) % (1 << 16)]
        pr_u[keep] = pr / pr.sum(axis=1)[:, None]
        e.set_state(st["gamma_shp"], st["gamma_rte"], st["phi_shp"], st["phi_rte"], st["nu_shp"],
                    PRIORS["beta_eta"] + float(np.sum(net.X.vals)), pr_u, 1e-12)

    def allreduce(attr):
        tot = sum(getattr(e, attr) for e in engs)
        for e in engs:
            getattr(e, attr).copy_(tot)

    allreduce("red3")  # the initial statistics were computed per shard
    for it in range(5):
        fl = F["VM_F_ELBO"] if it == 3 else 0
        for e in engs:
            e.phase("gamma")
        allreduce("red1")
        for e in engs:
            e.phase("phi")
        allreduce("red2")
        for e in engs:
            e.phase("rho", fl)
        allreduce("red3")
        for e in engs:
            e.phase("finish", fl)
        one.iterate(1, elbo_last=bool(fl))
        p = one.params()
        for e in engs:
            q = e.params()
            for k in ("gamma_shp", "gamma_rte", "phi_shp", "phi_rte", "nu_shp"):
                np.testing.assert_allclose(q[k], p[k], rtol=1e-6, err_msg=f"{k} it{it}")
            if fl:
                np.testing.assert_allclose(e.elbo(), one.elbo(), rtol=1e-8)
    slab = torch.cat([e.rho_slab() for e in engs], dim=1)
    # (the shards' parameters differ from the single rank's by reduction order, ~1e-8; a shortcut tie's fp32 posterior then
    # differs by a few ulp)
    np.testing.assert_allclose(slab.cpu().numpy(), one.rho_slab().cpu().numpy(), rtol=5e-6, atol=1e-30)
