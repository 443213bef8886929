"""Fits without the dense posterior slab (`CaviEngine(slab=False)`, `fit(store_rho="never")`): the posterior stays implicit
in the row/column tables and the special ties' rho_u32 and is evaluated on demand (`vm_materialize_rows`).  Everything
must be bit-identical to a fit that stores the slab: statistics, parameters, ELBO, the evaluated posterior and every
consumer."""
import os
import socket
import sys
import warnings

import numpy as np
import pytest

from tests.test_gpu_scaled import PRIORS, _cuda

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _pair(subs, vals, L, N, M, K, mask, mutuality=True, tile_h=64, may_dead=False, seed=3, slabs=(True, False)):
    """Engines over the same packed data and initial state, with the slab or without it as `slabs` says (default: one
    with, one without), then the packed data."""
    torch = _cuda()
    from vimure_b200 import _packing
    from vimure_b200._engine import CaviEngine

    P = _packing.pack(np.asarray(subs), np.asarray(vals), L, N, M, K, mask, "cuda", tile_h=tile_h, mutuality=mutuality)
    rs = np.random.RandomState(seed).random_sample
    st = dict(gamma_shp=0.1 * rs((L, M)) + 0.1, phi_shp=10.0 * rs((L, K)) + 10.0, gamma_rte=0.1 * rs((L, M)) + 0.1,
              phi_rte=10.0 * rs((L, K)) + 10.0, nu_shp=0.5 * rs(1)[0] + 0.5)
    keep = (P.t["u_has_x"] & P.t["u_reported"]).cpu().numpy()
    pr_u = np.zeros((P.U, K))
    pr_u[:, 0] = 1.0
    pr = 1 + 0.01 * rs((int(keep.sum()), K))
    pr_u[keep] = pr / pr.sum(axis=1)[:, None]
    nu_rte = PRIORS["beta_eta"] + float(np.asarray(vals).sum()) if mutuality else 1.0
    engs = []
    for slab in slabs:
        e = CaviEngine(P, PRIORS, mutuality=mutuality, eps=1e-12, may_dead=may_dead, slab=slab)
        e.set_state(st["gamma_shp"], st["gamma_rte"], st["phi_shp"], st["phi_rte"], st["nu_shp"] if mutuality else 1e-6,
                    nu_rte, pr_u, 1e-12)
        engs.append(e)
    torch.cuda.synchronize()
    return (*engs, P)


def _sbm(N, K=2, mutuality=0.5, L=1):
    import vimure_b200.synthetic as syn

    net = syn.StandardSBM(N=N, L=L, K=K, C=2, avg_degree=10, seed=10).build_X(mutuality=mutuality, seed=20)
    return np.stack(net.X.subs), np.asarray(net.X.vals), net.R


def _case(name):
    import vimure_b200 as vm

    if name == "ego_k2_partial_tile":  # N = 1100: two full column tiles and a partial one
        s, v, R = _sbm(1100)
        return dict(subs=s, vals=v, L=1, N=1100, M=1100, K=2, mask=R)
    if name == "hub_tile_h32":  # row segments with > 64 and 33..64 shortcut ties (tests/test_gpu_dense_sc.py)
        from tests.test_gpu_dense_sc import _hub_network

        net = _hub_network(1100, 2)
        return dict(subs=np.stack(net.X.subs), vals=np.asarray(net.X.vals), L=1, N=1100, M=1100, K=2, mask=net.R,
                    tile_h=32)
    if name == "gm_n640_l2_k3":
        from tests.golden_util import Golden
        from tests.test_gpu_parity import build_inputs

        g = Golden(name)
        X, R = build_inputs(g, structured=True)
        return dict(subs=g.X_subs, vals=g.X_vals, L=g.L, N=g.N, M=g.M, K=g.K, mask=vm.masks.from_input(R, g.L, g.N, g.M),
                    mutuality=g.mutuality)
    if name == "all_reporters_k_all32":  # N >= 512: fast dense kernel next to k_all32
        import vimure_b200.synthetic as syn

        y = syn.StandardSBM(N=600, M=16, L=2, K=2, C=2, avg_degree=8, seed=5)
        X, _ = syn.dense_reporting_X(y, M=16, mutuality=0.4, seed=6)
        return dict(subs=np.stack(X.subs), vals=np.asarray(X.vals), L=2, N=600, M=16, K=2,
                    mask=vm.masks.AllMask(2, 600, 16))
    if name == "may_dead":
        s, v, R = _sbm(1100)
        return dict(subs=s, vals=v, L=1, N=1100, M=1100, K=2, mask=R, may_dead=True)
    if name == "no_mutuality":
        s, v, R = _sbm(1024, mutuality=0.0)
        return dict(subs=s, vals=v, L=1, N=1024, M=1024, K=2, mask=R, mutuality=False)
    raise KeyError(name)


CASES = ["ego_k2_partial_tile", "hub_tile_h32", "gm_n640_l2_k3", "all_reporters_k_all32", "may_dead", "no_mutuality"]

# every buffer an iteration leaves behind besides the posterior
STATE = ("gamma_shp", "gamma_rte", "phi_shp", "phi_rte", "nu", "red3", "elbo_out", "rho_u32", "fixA", "fixP")


@pytest.mark.parametrize("name", CASES)
def test_engine_without_slab_is_bit_identical(name):
    """Without a slab (imp), and with one that only the last iteration of each step stores (nst)."""
    torch = _cuda()
    kw = _case(name)
    ref, imp, nst, P = _pair(**kw, slabs=(True, False, True))
    L, N, K, nloc = P.L, P.N, P.K, P.nloc
    assert ref.rho is not None and imp.rho is None and imp.ctx.rho is None
    if name == "all_reporters_k_all32":
        assert imp.all32_mode
    elif name in ("ego_k2_partial_tile", "hub_tile_h32"):
        assert imp.simple_mode
    with pytest.raises(RuntimeError, match="no posterior yet"):
        imp.infer(0)
    imp.block_rows = 37  # several consumer blocks per layer, the last one partial
    for step, (n, elbo) in enumerate(((1, False), (2, False), (1, True), (3, False), (1, True))):
        for e in (ref, imp):
            e.iterate(n, elbo_last=elbo)
        nst.iterate(n, elbo_last=elbo, store=False, store_last=True)
        tag = f"{name} step {step}"
        for k in STATE:
            assert torch.equal(getattr(ref, k), getattr(imp, k)), f"{k}: {tag}"
            assert torch.equal(getattr(ref, k), getattr(nst, k)), f"{k}: {tag}, store=False"
        slab = ref.rho_slab().view(L * nloc, N, K)
        for blk in (7, 64, L * nloc):
            for a in range(0, L * nloc, blk):
                b = min(a + blk, L * nloc)
                assert torch.equal(imp.materialize_rows(a, b - a), slab[a:b]), f"rows {a}:{b}, {tag}"
        assert torch.equal(ref.materialize_rows(0, L * nloc), slab), tag
        assert torch.equal(imp.rho_slab(), ref.rho_slab()), tag
        assert torch.equal(imp.infer(0), ref.infer(0)), tag
        assert torch.equal(imp.infer(1, 0.3), ref.infer(1, 0.3)), tag
        assert torch.equal(imp.infer_mean(), ref.infer_mean()), tag
        assert torch.equal(imp.sample(5, seed=11 + step), ref.sample(5, seed=11 + step)), tag
        assert torch.equal(nst.rho_slab(), ref.rho_slab()), tag
    # an iteration that stores nothing leaves the slab stale and the posterior implicit
    for e in (ref, imp):
        e.iterate(1)
    nst.iterate(1, store=False, store_last=False)
    for k in STATE:
        assert torch.equal(getattr(ref, k), getattr(nst, k)), f"{k}: {name}, store_last=False"
    with pytest.raises(RuntimeError, match="not stored"):
        nst.rho_slab()
    assert torch.equal(nst.materialize_rows(0, L * nloc), ref.rho_slab().view(L * nloc, N, K)), name
    # a copy of the implicit posterior (what a fit keeps of an earlier restart) still reads as it did
    snap, before = imp.snapshot(), ref.rho_slab().clone()
    for e in (ref, imp):
        e.iterate(2, elbo_last=True)
    assert torch.equal(imp.rho_slab(snap), before)
    assert torch.equal(imp.infer(0, slab=snap), ref.infer(0, slab=before))
    assert torch.equal(imp.sample(3, seed=5, slab=snap), ref.sample(3, seed=5, slab=before))


def test_entry_points_that_need_a_slab_refuse_without_one():
    torch = _cuda()
    import ctypes

    from vimure_b200 import _capi

    kw = _case("ego_k2_partial_tile")
    ref, imp, P = _pair(**kw)
    for e in (ref, imp):
        e.iterate(1, elbo_last=True)
    lib, st, F = imp.lib, imp._stream(), imp.C
    out = torch.empty(P.L * P.nloc * P.N, dtype=torch.uint8, device="cuda")
    assert lib.vm_infer(imp._cref, 0, 0.5, ctypes.c_void_p(out.data_ptr()), st) == F["VM_EINVAL"]
    assert lib.vm_materialize_prior(imp._cref, st) == F["VM_EINVAL"]
    assert lib.vm_dense_only(imp._cref, 0, st) == F["VM_EINVAL"]
    assert lib.vm_iteration(imp._cref, 0, st) == F["VM_EINVAL"]
    assert lib.vm_run(imp._cref, 2, F["VM_F_NO_STORE"], 0, st) == F["VM_EINVAL"]
    assert lib.vm_phase_rho(imp._cref, F["VM_F_ELBO"], st) == F["VM_EINVAL"]
    assert lib.vm_materialize_rows(imp._cref, 0, P.L * P.nloc + 1, ctypes.c_void_p(out.data_ptr()), st) == F["VM_EINVAL"]
    torch.cuda.synchronize()
    # nothing ran: the state is that of one iteration on both engines
    ref.iterate(1, elbo_last=True)
    imp.iterate(1, elbo_last=True)
    assert torch.equal(ref.gamma_shp, imp.gamma_shp) and torch.equal(ref.red3, imp.red3)
    assert _capi.consts()["VM_ABI_VERSION"] == 17


def _fit(g, X, R, **kw):
    import vimure_b200 as vm

    mk = dict(g.model_kwargs)
    model = vm.VimureModel(**mk)
    fk = dict(g.fit_kwargs)
    fk.update(kw)
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        model.fit(X, R=R, **fk)
    return model


def _assert_fits_identical(a, b):
    cols = ["realisation", "seed", "iter", "elbo", "reached_convergence"]
    assert a.trace[cols].equals(b.trace[cols])
    assert a.maxL == b.maxL and a.n_iter_ == b.n_iter_
    for k in ("gamma_shp", "gamma_rte", "phi_shp", "phi_rte", "nu_shp", "nu_rte", "G_exp_theta", "G_exp_lambda",
              "G_exp_nu"):
        assert np.array_equal(getattr(a, k + "_f"), getattr(b, k + "_f")), k + "_f"
        assert np.array_equal(getattr(a, k), getattr(b, k)), k
    for args in (("rho_max",), ("rho_mean",), ("fixed_threshold", 0.3), ("heuristic_threshold",)):
        with warnings.catch_warnings():
            warnings.simplefilter("ignore")
            assert np.array_equal(a.get_inferred_model(*args), b.get_inferred_model(*args)), args
    for rng in ("numpy", "device"):
        ya, yb = a.sample_inferred_model(N=3, seed=5, rng=rng), b.sample_inferred_model(N=3, seed=5, rng=rng)
        assert all(np.array_equal(p, q) for p, q in zip(ya, yb)), rng
    assert np.array_equal(a.rho, b.rho) and np.array_equal(a.rho_f, b.rho_f)
    pa, pb = a.get_posterior_estimates(), b.get_posterior_estimates()
    assert all(np.array_equal(pa[k], pb[k]) for k in pa)


def test_fit_without_slab_is_bit_identical():
    _cuda()
    from tests.golden_util import Golden
    from tests.test_gpu_parity import build_inputs

    g = Golden("f1_over")
    X, R = build_inputs(g)
    # a seed whose best restart is not the last one (rho_f is then kept from an earlier restart)
    for seed in range(3, 20):
        ref = _fit(g, X, R, num_realisations=2, max_iter=40, seed=seed, concurrent_realisations=False)
        last = ref.trace.groupby("realisation")["elbo"].last()
        if last[0] > last[1]:
            break
    else:
        pytest.fail("no seed with an earlier best restart")
    assert ref._rho_f_dev is not None
    for conc in (False, True):
        imp = _fit(g, X, R, num_realisations=2, max_iter=40, seed=seed, concurrent_realisations=conc, store_rho="never")
        assert imp._engine.rho is None and imp._engine_of_rho_f().rho is None
        if not conc:
            assert isinstance(imp._rho_f_dev, dict)  # the restart's tables, not a slab
        _assert_fits_identical(ref, imp)
        _assert_fits_identical(ref, _fit(g, X, R, num_realisations=2, max_iter=40, seed=seed,
                                         concurrent_realisations=conc, store_rho=False))

    g = Golden("karnataka_vil1")
    X, R = build_inputs(g)
    a = _fit(g, X, R, init_state=g.init_state())
    b = _fit(g, X, R, init_state=g.init_state(), store_rho="never")
    assert b._engine.rho is None
    _assert_fits_identical(a, b)
    _assert_fits_identical(a, _fit(g, X, R, init_state=g.init_state(), store_rho=False))


def test_general_mask_without_slab_raises():
    torch = _cuda()
    from tests.golden_util import Golden
    from tests.test_gpu_parity import build_inputs, make_engine

    g = Golden("custom_mask")
    assert g.R_spec["kind"] == "coo"
    X, R = build_inputs(g)
    for store in ("never", False, "sometimes"):
        with pytest.raises(ValueError, match="store_rho"):
            _fit(g, X, R, store_rho=store, max_iter=3)
    # the C ABI refuses an iteration without the slab write before any phase has changed the state
    csr, _ = make_engine(g, structured=False)
    assert csr.P.r_mode == 2 and csr.rho is not None
    csr.iterate(1, elbo_last=True)
    before = {k: getattr(csr, k).clone() for k in ("gamma_shp", "red3", "rho_u32")}
    lib, st, F = csr.lib, csr._stream(), csr.C
    assert lib.vm_iteration(csr._cref, F["VM_F_NO_STORE"], st) == F["VM_ENOTSUP"]
    assert lib.vm_phase_rho(csr._cref, F["VM_F_NO_STORE"], st) == F["VM_ENOTSUP"]
    torch.cuda.synchronize()
    for k, v in before.items():
        assert torch.equal(getattr(csr, k), v), k


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _dist_worker(rank, world, port, out):
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    sys.path.insert(0, ROOT)
    import torch
    import torch.distributed as dist

    torch.cuda.set_device(0)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    res = {}
    try:
        from tests.golden_util import Golden
        from tests.test_gpu_parity import build_inputs

        g = Golden("sbm_n520")  # N >= 512: the fast dense kernels and a partial column tile on every rank
        X, R = build_inputs(g)
        fits = [_fit(g, X, R, init_state=g.init_state(), max_iter=12, convergence_tol=0.0, **kw)
                for kw in ({}, {"store_rho": "never"}, {"store_rho": False})]
        a = fits[0]
        res["world"] = fits[1]._world
        res["no_slab"] = fits[1]._engine.rho is None
        for b, tag in zip(fits[1:], ("never", "no_store")):
            res[tag] = dict(
                params=all(np.array_equal(getattr(a, k), getattr(b, k)) for k in
                           ("gamma_shp", "gamma_rte", "phi_shp", "phi_rte", "nu_shp")) and a.maxL == b.maxL,
                rho_max=bool(np.array_equal(a.get_inferred_model("rho_max"), b.get_inferred_model("rho_max"))),
                sample=bool(np.array_equal(a.sample_inferred_model(N=2, seed=4, rng="device")[1],
                                           b.sample_inferred_model(N=2, seed=4, rng="device")[1])),
                rho=bool(np.array_equal(a.rho, b.rho)))
        res["ok"] = True
    except Exception:  # noqa: BLE001
        import traceback

        res["ok"] = False
        res["error"] = traceback.format_exc()[-1500:]
    out.put((rank, res))
    dist.destroy_process_group()


def test_two_rank_fit_without_slab_is_bit_identical():
    torch = _cuda()
    import torch.multiprocessing as mp

    world = 2
    ctx = mp.get_context("spawn")
    out = ctx.Queue()
    port = _free_port()
    ps = [ctx.Process(target=_dist_worker, args=(r, world, port, out)) for r in range(world)]
    for p in ps:
        p.start()
    results = dict(out.get(timeout=900) for _ in ps)
    for p in ps:
        p.join(timeout=120)
    for rank in range(world):
        res = results[rank]
        assert res["ok"], res.get("error")
        assert res["world"] == world and res["no_slab"], res
        for tag in ("never", "no_store"):
            assert set(res[tag]) == {"params", "rho_max", "sample", "rho"} and all(res[tag].values()), (tag, res)
    del torch


@pytest.mark.slow
def test_sparse_network_beyond_the_slab():
    """N = 160 000 nodes, K = 2, a sparse report law: the slab (205 GB) exceeds the device's memory, the fit without it
    runs.  The argmax of the posterior (the consumer behind get_inferred_model("rho_max"), on the device: the public
    method returns an int64 host array of N^2 entries) is checked on sampled rows against a host argmax of the rows
    evaluated on their own, and the evaluated rows hold the special ties' posteriors."""
    torch = _cuda()
    import vimure_b200 as vm
    from vimure_b200 import synthetic as syn

    L, N, K = 1, 160_000, 2
    assert float(L) * N * N * K * 4 > torch.cuda.mem_get_info()[1]
    rng = np.random.RandomState(7)
    nY = 2 * N
    ys = np.stack([np.zeros(nY, np.int64), rng.randint(0, N, nY), rng.randint(0, N, nY)])
    ys = ys[:, ys[1] != ys[2]]
    ys = ys[:, np.unique(ys[1] * N + ys[2], return_index=True)[1]]
    theta = 0.5 + rng.random_sample((L, N))
    subs, vals = syn.device_reports(L, N, N, K, ys, np.ones(ys.shape[1], np.int32), theta, 0.5, seed=11,
                                    lam=np.array([[1e-4, 1.0]]))
    X = vm.sptensor.sptensor(tuple(subs.cpu().numpy()), vals.cpu().numpy(), shape=(L, N, N, N))
    del subs, vals
    model = vm.VimureModel(mutuality=True)
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        model.fit(X, R=vm.masks.EgoMask(L, N, N), K=K, seed=3, max_iter=20, store_rho="never")
    assert np.isfinite(model.maxL) and model.n_iter_ == 20
    eng = model._engine_of_rho_f()
    assert eng.rho is None
    Y = eng.infer(0)
    u_row, u_col = eng.P.t["u_lrow"].long(), eng.P.t["u_col"].long()
    # rows where the posterior favours a tie somewhere (an all-zero argmax row would prove nothing), and random rows
    tied = u_row[eng.rho_u32[:, 1] > eng.rho_u32[:, 0]].cpu().numpy()
    assert len(tied) > 0
    rows = np.concatenate([rng.choice(tied, 3, replace=False), rng.choice(N, 3, replace=False)])
    assert int(Y[0, rows[:3]].sum()) > 0
    for i in rows:
        r = eng.materialize_rows(int(i), 1)[0]
        assert np.array_equal(Y[0, i].cpu().numpy(), np.argmax(r.cpu().numpy(), axis=-1)), i
        sel = u_row == int(i)
        assert torch.equal(r[u_col[sel]], eng.rho_u32[sel]), i
    del Y
    torch.cuda.synchronize()
