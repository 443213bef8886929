"""Sparse consumers (`vm_edges_count` / `vm_edges_emit`, `CaviEngine.infer_edges` / `sample_edges`,
`get_inferred_model(..., sparse=True)`, `sample_inferred_model(..., sparse=True)`): the ties whose label is nonzero, as an
edge list evaluated on the device.  Every result must equal the nonzero entries of the dense consumer exactly: keys,
labels and dtypes."""
import ctypes
import os
import sys
import warnings

import numpy as np
import pytest

from tests.test_gpu_implicit import CASES, ROOT, _case, _fit, _free_port, _pair
from tests.test_gpu_scaled import _cuda

pytestmark = pytest.mark.gpu


def _nonzero(eng, y):
    """Dense labels (L, nloc, N) of `eng` -> (global keys (l*N+i)*N+j int64, labels uint8), as the sparse consumers."""
    torch = _cuda()
    L, nloc, N = y.shape
    idx = torch.nonzero(y.reshape(-1)).reshape(-1)
    lrow, j = idx // N, idx % N
    l, i = lrow // nloc, lrow % nloc + eng.P.row0
    return (l * N + i) * N + j, y.reshape(-1)[idx]


def _assert_edges(got, want, tag):
    torch = _cuda()
    assert got[0].dtype == torch.int64 and got[1].dtype == torch.uint8, tag
    assert torch.equal(got[0], want[0]), "keys: " + tag
    assert torch.equal(got[1], want[1]), "labels: " + tag


def _heuristic(eng):
    return 0.54 * float(eng.nu[eng.C["VM_NU_G_STALE"]]) - 0.01


def _check_engine(eng, tag, slab=None):
    thr = _heuristic(eng)
    for mode, t in ((0, 0.5), (1, 0.3), (1, thr)):
        _assert_edges(eng.infer_edges(mode, t, slab=slab), _nonzero(eng, eng.infer(mode, t, slab=slab)),
                      f"infer({mode}, {t}) {tag}")
    _assert_edges(eng.sample_edges(5, seed=17, slab=slab), _nonzero(eng, eng.sample(5, seed=17, slab=slab)),
                  f"sample {tag}")


@pytest.mark.parametrize("name", CASES)
def test_engine_edges_equal_dense(name):
    torch = _cuda()
    ref, imp, P = _pair(**_case(name))
    with pytest.raises(RuntimeError, match="no posterior yet"):
        imp.infer_edges(0)
    # the prior of a storing engine: slab source
    _check_engine(ref, f"{name} prior")
    imp.block_rows = 37
    for step, (n, elbo) in enumerate(((1, False), (2, False), (1, True), (3, False))):
        for e in (ref, imp):
            e.iterate(n, elbo_last=elbo)
        tag = f"{name} step {step}"
        _check_engine(ref, "storing, implicit source " + tag)
        _check_engine(ref, "storing, slab source " + tag, slab=ref.rho_slab().clone())
        _check_engine(imp, "slab-free " + tag)
        # the implicit source on the storing engine reads the same posterior as its slab
        _assert_edges(ref.infer_edges(0), imp.infer_edges(0), tag)
    # an earlier restart's posterior: a snapshot (implicit source) and a cloned slab (slab source)
    snap, before = imp.snapshot(), ref.rho_slab().clone()
    for e in (ref, imp):
        e.iterate(2, elbo_last=True)
    _check_engine(imp, f"{name} snapshot", slab=snap)
    _check_engine(ref, f"{name} cloned slab", slab=before)
    _assert_edges(imp.infer_edges(0, slab=snap), ref.infer_edges(0, slab=before), name)
    _assert_edges(imp.sample_edges(3, seed=5, slab=snap), ref.sample_edges(3, seed=5, slab=before), name)
    torch.cuda.synchronize()


def _skip_bounds(eng, rows, rng):
    """Rewrite tab_q of a few columns (ties without reports that become edges) and tab_p of `rows` so that fl(p_k + qmax_k)
    sits at each bound of the row skip and 2^-10 log2 units either side of it, or well above it."""
    torch = _cuda()
    P, K = eng.P, eng.P.K
    q = eng.tab_q.view(P.L, P.N, K)
    cols = torch.as_tensor(rng.choice(P.N, 8, replace=False), device="cuda")
    q[:, cols, 1:] += 40.0
    qmax = q.max(dim=1)[0]  # (L, K)
    p = eng.tab_p.view(P.L, P.nloc, K)
    bounds = [-1.0, float(np.log2(np.float32(0.3))) - 1.0, -30.0, 0.5, 3.0]
    targets = [b + d for b in bounds for d in (-2.0 ** -10, 0.0, 2.0 ** -10)]
    for n, i in enumerate(rows):
        t = torch.tensor(targets[n % len(targets)], dtype=torch.float32, device="cuda")
        for k in range(1, K):
            p[:, i, k] = t - qmax[:, k]
    return len(targets)


@pytest.mark.parametrize("name", ["ego_k2_partial_tile", "gm_n640_l2_k3", "all_reporters_k_all32", "may_dead"])
def test_closed_form_edges_and_skip_bounds(name):
    torch = _cuda()
    _, imp, P = _pair(**_case(name))
    imp.iterate(2, elbo_last=True)
    rng = np.random.RandomState(1)
    rows = rng.choice(P.nloc, 40, replace=False)
    _skip_bounds(imp, rows, rng)
    _check_engine(imp, name)
    y = imp.infer(0)
    assert int((y != 0).sum()) > 0, "no edges: the test would prove nothing"
    if name == "may_dead":
        # a row whose closed form underflows completely: its ties without reports are dead (all zero), which the device
        # sampler sends to the last category and argmax / threshold leave at 0
        i = int(rows[0])
        imp.tab_p.view(P.L, P.nloc, P.K)[:, i, 0] = -4000.0
        keys, lab = imp.sample_edges(3, seed=2)
        _assert_edges((keys, lab), _nonzero(imp, imp.sample(3, seed=2)), "dead row")
        u_col = P.t["u_col"][P.t["u_lrow"] == i].long()
        plain = torch.ones(P.N, dtype=torch.bool, device="cuda")
        plain[u_col] = False
        row_keys = keys[(keys // P.N) == i]
        row_lab = lab[(keys // P.N) == i]
        assert torch.equal(plain.nonzero().reshape(-1), row_keys[plain[row_keys % P.N]] % P.N)
        assert bool((row_lab[plain[row_keys % P.N]] == P.K - 1).all())
        for mode, t in ((0, 0.5), (1, 0.3)):
            k2, _ = imp.infer_edges(mode, t)
            assert not bool(plain[k2[(k2 // P.N) == i] % P.N].any()), mode


def test_whole_range_thresholds():
    torch = _cuda()
    ref, imp, P = _pair(**_case("gm_n640_l2_k3"))
    for e in (ref, imp):
        e.iterate(3, elbo_last=True)
    n_all = P.L * P.nloc * P.N
    for e in (ref, imp):
        keys, lab = e.infer_edges(1, 0.0)
        assert keys.numel() == n_all and bool((lab == 1).all())
        assert torch.equal(keys, torch.arange(n_all, device="cuda"))
        for t in (0.0, 1.0):
            _assert_edges(e.infer_edges(1, t), _nonzero(e, e.infer(1, t)), f"threshold {t}")
        rho1 = e.rho_slab()[..., 1]
        assert e.infer_edges(1, 1.0)[0].numel() == int((rho1 >= 1.0).sum())


METHODS = (("rho_max",), ("rho_mean",), ("fixed_threshold", 0.3), ("heuristic_threshold",))


def _assert_sparse_model(m):
    import vimure_b200 as vm

    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        for args in METHODS:
            if args[0] == "rho_mean" and m.mutuality:
                with pytest.raises(ValueError, match="rho_mean"):
                    m.get_inferred_model(*args, sparse=True)
                continue
            got, want = m.get_inferred_model(*args, sparse=True), vm.sptensor.sptensor.fromarray(m.get_inferred_model(*args))
            assert got.shape == want.shape and got.vals.dtype == want.vals.dtype, args
            assert all(a.dtype == b.dtype and np.array_equal(a, b) for a, b in zip(got.subs, want.subs)), args
            assert np.array_equal(got.vals, want.vals), args
    ys = m.sample_inferred_model(N=3, seed=5, sparse=True)
    yd = m.sample_inferred_model(N=3, seed=5, rng="device")
    assert len(ys) == 3
    for a, b in zip(ys, yd):
        b = vm.sptensor.sptensor.fromarray(b)
        assert a.vals.dtype == b.vals.dtype and np.array_equal(a.vals, b.vals)
        assert all(np.array_equal(p, q) for p, q in zip(a.subs, b.subs))
    with pytest.raises(ValueError, match="numpy"):
        m.sample_inferred_model(N=1, seed=5, rng="numpy", sparse=True)


def test_fits_sparse_equal_dense():
    _cuda()
    from tests.golden_util import Golden
    from tests.test_gpu_parity import build_inputs

    g = Golden("f1_over")
    X, R = build_inputs(g)
    for seed in range(3, 20):  # a seed whose best restart is not the last one (rho_f kept from an earlier restart)
        ref = _fit(g, X, R, num_realisations=2, max_iter=40, seed=seed, concurrent_realisations=False)
        last = ref.trace.groupby("realisation")["elbo"].last()
        if last[0] > last[1]:
            break
    else:
        pytest.fail("no seed with an earlier best restart")
    assert ref._rho_f_dev is not None
    _assert_sparse_model(ref)
    for conc in (False, True):
        for store in (True, "never"):
            _assert_sparse_model(_fit(g, X, R, num_realisations=2, max_iter=40, seed=seed, concurrent_realisations=conc,
                                      store_rho=store))
    for name in ("karnataka_vil1", "custom_mask"):
        g = Golden(name)
        X, R = build_inputs(g)
        for store in ((True, "never") if name == "karnataka_vil1" else (True,)):
            _assert_sparse_model(_fit(g, X, R, init_state=g.init_state(), store_rho=store))


def test_edges_c_abi_rejects_bad_arguments():
    torch = _cuda()
    from tests.golden_util import Golden
    from tests.test_gpu_parity import make_engine
    from vimure_b200 import _capi

    ref, imp, P = _pair(**_case("ego_k2_partial_tile"))
    for e in (ref, imp):
        e.iterate(1, elbo_last=True)
    C, A = imp.C, _capi.edges_class()
    assert imp.lib.vm_edges_size() == ctypes.sizeof(A)
    rows = P.L * P.nloc
    bufs = dict(row_count=torch.full((rows,), -7, dtype=torch.int64, device="cuda"),
                row_off=torch.zeros(rows, dtype=torch.int64, device="cuda"),
                o_key=torch.full((16,), -7, dtype=torch.int64, device="cuda"),
                o_val=torch.full((16,), 9, dtype=torch.uint8, device="cuda"),
                workspace=torch.full((P.L * P.K,), -7.0, device="cuda"))
    before = {k: v.clone() for k, v in bufs.items()}

    def args(**kw):
        d = dict(what=C["VM_EDGES_ARGMAX"], source=C["VM_EDGES_IMPLICIT"], threshold=0.5, n_trials=1, seed=0)
        d.update({k: v.data_ptr() for k, v in bufs.items()})
        d.update(kw)
        return A(**d)

    st = imp._stream()
    count, emit = imp.lib.vm_edges_count, imp.lib.vm_edges_emit
    E = C["VM_EINVAL"]
    for fn in (count, emit):
        assert fn(imp._cref, None, st) == E
        assert fn(imp._cref, ctypes.byref(args(what=3)), st) == E
        assert fn(imp._cref, ctypes.byref(args(what=-1)), st) == E
        assert fn(imp._cref, ctypes.byref(args(source=2)), st) == E
        assert fn(imp._cref, ctypes.byref(args(what=C["VM_EDGES_SAMPLE"], n_trials=0)), st) == E
        assert fn(imp._cref, ctypes.byref(args(workspace=None)), st) == E
        assert fn(imp._cref, ctypes.byref(args(source=C["VM_EDGES_SLAB"])), st) == E  # no slab
    assert count(imp._cref, ctypes.byref(args(row_count=None)), st) == E
    for k in ("row_off", "o_key", "o_val"):
        assert emit(imp._cref, ctypes.byref(args(**{k: None})), st) == E
    # the general mask has no tables: the implicit source is not supported, the slab source is
    csr, _ = make_engine(Golden("custom_mask"), structured=False)
    assert csr.P.r_mode == 2
    csr.iterate(1, elbo_last=True)
    for fn in (count, emit):
        assert fn(csr._cref, ctypes.byref(args()), st) == C["VM_ENOTSUP"]
    torch.cuda.synchronize()
    for k, v in bufs.items():
        assert torch.equal(v, before[k]), k  # nothing was written
    _assert_edges(csr.infer_edges(0), _nonzero(csr, csr.infer(0)), "custom_mask")


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
        import vimure_b200 as vm
        from tests.golden_util import Golden
        from tests.test_gpu_parity import build_inputs

        g = Golden("gm_n640_l2_k3")  # L = 2: the gathered edge lists must be merged by layer
        X, R = build_inputs(g, structured=True)
        for store in (True, "never"):
            m = _fit(g, X, R, init_state=g.init_state(), max_iter=12, convergence_tol=0.0, store_rho=store)
            res["world"] = m._world
            with warnings.catch_warnings():
                warnings.simplefilter("ignore")
                sp = m.get_inferred_model("rho_max", sparse=True)
                dense = vm.sptensor.sptensor.fromarray(m.get_inferred_model("rho_max"))
            ys = m.sample_inferred_model(N=2, seed=4, sparse=True)[1]
            yd = vm.sptensor.sptensor.fromarray(m.sample_inferred_model(N=2, seed=4, rng="device")[1])
            res[store] = dict(sp=(sp.subs, sp.vals), dense=(dense.subs, dense.vals), ys=(ys.subs, ys.vals),
                              yd=(yd.subs, yd.vals))
        res["ok"] = True
    except Exception:  # noqa: BLE001
        import traceback

        res["ok"] = False
        res["error"] = traceback.format_exc()[-1500:]
    out.put((rank, res))
    dist.destroy_process_group()


def _same(a, b):
    return all(np.array_equal(p, q) and p.dtype == q.dtype for p, q in zip(a[0], b[0])) and \
        np.array_equal(a[1], b[1]) and a[1].dtype == b[1].dtype


def test_two_rank_sparse_equals_dense():
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
        assert res["world"] == world
        for store in (True, "never"):
            r, r0 = res[store], results[0][store]
            assert len(r["sp"][1]) > 0
            assert _same(r["sp"], r["dense"]) and _same(r["ys"], r["yd"]), (rank, store)
            assert all(_same(r[k], r0[k]) for k in r), (rank, store)  # every rank holds the whole result
            assert all(_same(r[k], results[0][True][k]) for k in r), (rank, store)  # with or without the slab
    del torch


@pytest.mark.slow
def test_sparse_inferred_network_beyond_the_slab():
    """N = 160 000 nodes without the slab (205 GB): `get_inferred_model("rho_max", sparse=True)` and a sparse sample
    through the public API, checked on sampled rows against a host evaluation of the rows on their own; the call adds
    far less device memory than the dense result alone (25.6 GB)."""
    torch = _cuda()
    import vimure_b200 as vm
    from vimure_b200 import synthetic as syn

    L, N, K = 1, 160_000, 2
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
    eng = model._engine_of_rho_f()
    assert eng.rho is None
    torch.cuda.synchronize()
    base = torch.cuda.memory_allocated()
    torch.cuda.reset_peak_memory_stats()
    Y = model.get_inferred_model("rho_max", sparse=True)
    added = torch.cuda.max_memory_allocated() - base
    assert added < 1e9, added
    assert Y.shape == (L, N, N) and Y.vals.dtype == np.int64 and len(Y.vals) > 0
    S = model.sample_inferred_model(N=2, seed=9, sparse=True)
    u_row, u_col = eng.P.t["u_lrow"].long(), eng.P.t["u_col"].long()
    tied = u_row[eng.rho_u32[:, 1] > eng.rho_u32[:, 0]].cpu().numpy()
    rows = np.concatenate([rng.choice(tied, 3, replace=False), rng.choice(N, 3, replace=False)])
    from vimure_b200 import _capi

    view = _capi.ctx_class()()  # a one-row ctx over an evaluated row, for the dense sampler (as CaviEngine._consume)
    ctypes.memmove(ctypes.byref(view), eng._cref, ctypes.sizeof(view))
    view.L, view.nloc, view.nrt = 1, 1, 1
    out = torch.empty(N, dtype=torch.uint8, device="cuda")

    def row_of(sp, i):
        y = np.zeros(N, np.int64)
        sel = sp.subs[1] == i
        y[sp.subs[2][sel]] = sp.vals[sel]
        return y

    for i in rows:
        r = eng.materialize_rows(int(i), 1)
        assert np.array_equal(row_of(Y, i), np.argmax(r[0].cpu().numpy(), axis=-1)), i
        view.row0, view.rho = int(i), r.data_ptr()
        for n, s in enumerate(S):
            _capi.check(eng.lib.vm_sample(ctypes.byref(view), 2, ctypes.c_uint64(9 + n), ctypes.c_void_p(out.data_ptr()),
                                          eng._stream()), "vm_sample")
            assert np.array_equal(row_of(s, i), out.cpu().numpy().astype(np.int64)), (i, n)
    assert int(np.isin(Y.subs[1], rows[:3]).sum()) > 0
    for s in S:
        assert s.shape == (L, N, N) and len(s.vals) > 0
    torch.cuda.synchronize()
