"""The posterior at given ties (`vm_rho_at`, `CaviEngine.rho_at`, `VimureModel.rho_f_at`): evaluated tie by tie on the
device, without the dense slab or an (L, N, N, K) array.  Every value must equal the slab's (or `vm_materialize_rows`'s)
for that tie exactly, and the ties a rank does not own must be left alone."""
import ctypes
import os
import sys
import warnings

import numpy as np
import pytest

from tests.test_gpu_implicit import CASES, ROOT, _case, _fit, _free_port, _pair
from tests.test_gpu_scaled import _cuda

pytestmark = pytest.mark.gpu


def _kw(name):
    if name == "random_k5":  # K = 5: the general kernels (two layers, an ego mask with a subset of reporters, no diagonal)
        from tests.test_gpu_random import _random_problem

        p = _random_problem(37)
        assert p["K"] == 5 and p["kind"] == "ego_subset"
        return {k: p[k] for k in ("subs", "vals", "L", "N", "M", "K", "mask", "mutuality", "tile_h")}
    return _case(name)


def _local(P, keys):
    """Global keys (l*N+i)*N+j of this engine's rows -> local ties lrow*N + j (the slab's flat index)."""
    li, j = keys // P.N, keys % P.N
    l, i = li // P.N, li % P.N
    return (l * P.nloc + i - P.row0) * P.N + j


def _queries(P, seed=0, n_rand=4000):
    """Random ties of every layer, every special tie (diagonal ones included), ties in the last (partial) column tile, the
    first and last column of every tile, and a quarter of them again: shuffled."""
    torch = _cuda()
    rng = np.random.RandomState(seed)
    L, N, nloc, row0, tw = P.L, P.N, P.nloc, P.row0, P.tile_w

    def key(l, i, j):
        return (np.asarray(l, np.int64) * N + np.asarray(i, np.int64)) * N + np.asarray(j, np.int64)

    ur, uc = P.t["u_lrow"].long().cpu().numpy(), P.t["u_col"].long().cpu().numpy()
    parts = [key(rng.randint(0, L, n_rand), rng.randint(row0, row0 + nloc, n_rand), rng.randint(0, N, n_rand)),
             key(ur // nloc, ur % nloc + row0, uc)]
    last0 = (P.nct - 1) * tw
    n = 500
    parts.append(key(rng.randint(0, L, n), rng.randint(row0, row0 + nloc, n), rng.randint(last0, N, n)))
    edges = np.unique(np.concatenate([np.arange(0, N, tw), np.minimum(np.arange(tw, N + tw, tw), N) - 1]))
    rows = rng.randint(row0, row0 + nloc, 8)
    ll, ii, jj = np.meshgrid(np.arange(L), rows, edges, indexing="ij")
    parts.append(key(ll.ravel(), ii.ravel(), jj.ravel()))
    keys = np.concatenate(parts)
    keys = np.concatenate([keys, keys[rng.choice(len(keys), len(keys) // 4)]])
    rng.shuffle(keys)
    return torch.as_tensor(keys, device="cuda")


def _assert_at(eng, keys, slab, tag, src=None):
    """eng.rho_at(keys, slab=src) equals `slab` (L, nloc, N, K) at those ties."""
    torch = _cuda()
    got = eng.rho_at(keys, slab=src)
    want = slab.reshape(-1, eng.P.K)[_local(eng.P, keys)]
    assert got.dtype == torch.float32 and got.shape == want.shape, tag
    assert torch.equal(got, want), tag


@pytest.mark.parametrize("name", CASES + ["random_k5"])
def test_engine_rho_at_equals_slab(name):
    torch = _cuda()
    ref, imp, P = _pair(**_kw(name))
    L, N, K, nloc = P.L, P.N, P.K, P.nloc
    keys = _queries(P)
    with pytest.raises(RuntimeError, match="no posterior yet"):
        imp.rho_at(keys)
    # the prior of a storing engine: slab source
    _assert_at(ref, keys, ref.rho_slab(), f"{name} prior")
    for step, (n, elbo) in enumerate(((1, False), (2, False), (1, True), (3, False))):
        for e in (ref, imp):
            e.iterate(n, elbo_last=elbo)
        tag = f"{name} step {step}"
        slab = ref.rho_slab()
        _assert_at(ref, keys, slab, "storing, implicit source " + tag)
        _assert_at(ref, keys, slab, "storing, slab source " + tag, src=slab.clone())
        _assert_at(imp, keys, imp.materialize_rows(0, L * nloc), "slab-free " + tag)
        assert torch.equal(imp.rho_at(keys), ref.rho_at(keys)), tag
    # an earlier restart's posterior: a snapshot (implicit source) and a cloned slab (slab source)
    snap, before = imp.snapshot(), ref.rho_slab().clone()
    for e in (ref, imp):
        e.iterate(2, elbo_last=True)
    _assert_at(imp, keys, before, f"{name} snapshot", src=snap)
    _assert_at(ref, keys, before, f"{name} cloned slab", src=before)
    assert torch.equal(imp.rho_at(keys[:0]), torch.zeros(0, K, device="cuda"))
    if name == "may_dead":
        # a row whose closed form underflows completely: its ties without reports are dead (all zero), as the slab holds them
        i = int(np.random.RandomState(1).randint(nloc))
        imp.tab_p.view(L, nloc, K)[:, i, 0] = -4000.0
        row = torch.arange(N, device="cuda", dtype=torch.int64) + i * N
        got = imp.rho_at(row)
        assert torch.equal(got, imp.materialize_rows(i, 1)[0]), "dead row"
        plain = torch.ones(N, dtype=torch.bool, device="cuda")
        plain[P.t["u_col"][P.t["u_lrow"] == i].long()] = False
        assert bool(plain.any()) and bool((got[plain] == 0).all()), "dead row"
    torch.cuda.synchronize()


def _call(eng, source, keys, out, n=None, view=None):
    """vm_rho_at on `eng`'s ctx, or on `view` (a copy of it) if given."""
    return eng.lib.vm_rho_at(eng._cref if view is None else ctypes.byref(view), source,
                             keys.numel() if n is None else n, ctypes.c_void_p(keys.data_ptr() if keys is not None else 0),
                             ctypes.c_void_p(out.data_ptr() if out is not None else 0), eng._stream())


def test_keys_outside_the_rows_are_not_written():
    torch = _cuda()
    from vimure_b200 import _capi

    ref, imp, P = _pair(**_case("ego_k2_partial_tile"))
    for e in (ref, imp):
        e.iterate(2, elbo_last=True)
    L, N, K, C = P.L, P.N, P.K, ref.C
    SLAB, IMPL = C["VM_EDGES_SLAB"], C["VM_EDGES_IMPLICIT"]
    bad = torch.tensor([-1, -N * N, -(2 ** 62), L * N * N, L * N * N + 5, 2 ** 62], dtype=torch.int64, device="cuda")
    for e, src in ((ref, SLAB), (ref, IMPL), (imp, IMPL)):
        out = torch.full((bad.numel(), K), 7.0, device="cuda")
        assert _call(e, src, bad, out) == 0
        torch.cuda.synchronize()
        assert bool((out == 7.0).all()), src
    # a ctx view over the rows [r0, r0+nv) only (L = 1, as CaviEngine._consume narrows it), its row arrays offset to them
    r0, nv = 300, 250
    slab = ref.rho_slab()
    view = _capi.ctx_class()()
    ctypes.memmove(ctypes.byref(view), ref._cref, ctypes.sizeof(view))
    view.row0, view.nloc, view.nrt = r0, nv, -(-nv // P.tile_h)
    view.rho = slab.data_ptr() + r0 * N * K * 4
    view.tab_p = ref.tab_p.data_ptr() + r0 * K * 4
    view.utile_ptr = P.t["utile_ptr"].data_ptr() + r0 * P.nct * P.t["utile_ptr"].element_size()
    keys = _queries(P, seed=4)
    i = keys // N
    mine = (i >= r0) & (i < r0 + nv)
    assert bool(mine.any()) and not bool(mine.all())
    for src in (SLAB, IMPL):
        out = torch.full((keys.numel(), K), 7.0, device="cuda")
        assert _call(ref, src, keys, out, view=view) == 0
        torch.cuda.synchronize()
        assert torch.equal(out[mine], slab.reshape(-1, K)[keys[mine]]), src
        assert bool((out[~mine] == 7.0).all()), src
    # keys the engine cannot hand to the kernel: another dtype, or not on its device
    for k in (keys.to(torch.int32), keys.cpu()):
        with pytest.raises(ValueError, match="int64 tensor"):
            ref.rho_at(k)


def test_special_tie_search_at_indices_beyond_2_30():
    """The special-tie search of the implicit source on indices where lo + hi no longer fits an int32 (a rank with more
    than 2^30 special ties): a ctx view whose utile_ptr is shifted up by 2^30 and whose u_col / rho_u32 start 2^30 ties
    earlier addresses the very same ties, so the values must still equal the slab."""
    torch = _cuda()
    from vimure_b200 import _capi

    ref, P = _pair(**_case("ego_k2_partial_tile"), slabs=(True,))
    ref.iterate(2, elbo_last=True)
    K, S = P.K, 2 ** 30
    assert P.U + S < 2 ** 31 - 1
    uptr = (P.t["utile_ptr"].to(torch.int64) + S).to(torch.int32)
    view = _capi.ctx_class()()
    ctypes.memmove(ctypes.byref(view), ref._cref, ctypes.sizeof(view))
    view.utile_ptr = uptr.data_ptr()
    view.u_col = P.t["u_col"].data_ptr() - S * P.t["u_col"].element_size()
    view.rho_u32 = ref.rho_u32.data_ptr() - S * K * ref.rho_u32.element_size()
    keys = _queries(P, seed=6)
    out = torch.full((keys.numel(), K), 7.0, device="cuda")
    assert _call(ref, ref.C["VM_EDGES_IMPLICIT"], keys, out, view=view) == 0
    torch.cuda.synchronize()
    assert torch.equal(out, ref.rho_slab().reshape(-1, K)[keys])


def test_rho_at_c_abi_rejects_bad_arguments():
    torch = _cuda()
    from tests.golden_util import Golden
    from tests.test_gpu_parity import make_engine

    ref, imp, P = _pair(**_case("ego_k2_partial_tile"))
    for e in (ref, imp):
        e.iterate(1, elbo_last=True)
    C = imp.C
    E, SLAB, IMPL = C["VM_EINVAL"], C["VM_EDGES_SLAB"], C["VM_EDGES_IMPLICIT"]
    keys = _queries(P)
    out = torch.full((keys.numel(), P.K), 7.0, device="cuda")
    assert _call(imp, IMPL, None, out, n=keys.numel()) == E
    assert _call(imp, IMPL, keys, None) == E
    assert _call(imp, IMPL, keys, out, n=-1) == E
    for src in (2, -1):
        assert _call(ref, src, keys, out) == E
    assert _call(imp, SLAB, keys, out) == E  # no slab
    assert _call(imp, IMPL, None, None, n=0) == 0
    csr, _ = make_engine(Golden("custom_mask"), structured=False)
    assert csr.P.r_mode == 2
    csr.iterate(1, elbo_last=True)
    ckeys = _queries(csr.P)
    cout = torch.full((ckeys.numel(), csr.P.K), 7.0, device="cuda")
    assert _call(csr, IMPL, ckeys, cout) == C["VM_ENOTSUP"]
    torch.cuda.synchronize()
    assert bool((out == 7.0).all()) and bool((cout == 7.0).all())  # nothing was written
    # the general mask: the slab source (which the engine picks there) reads its slab
    _assert_at(csr, ckeys, csr.rho_slab(), "custom_mask")
    assert _call(csr, SLAB, ckeys, cout) == 0
    assert torch.equal(cout, csr.rho_slab().reshape(-1, csr.P.K)[ckeys])


def _assert_rho_f_at(m):
    rho_f = m.rho_f
    rng = np.random.RandomState(2)
    n = 3000
    subs = (rng.randint(0, m.L, n), rng.randint(0, m.N, n), rng.randint(0, m.N, n))
    got = m.rho_f_at(subs)
    assert got.dtype == np.float64 and got.shape == (n, m.K)
    assert np.array_equal(got, rho_f[subs])
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        Y = m.get_inferred_model("rho_max", sparse=True)
    assert len(Y.vals) > 0
    assert np.array_equal(m.rho_f_at(Y.subs), rho_f[Y.subs])
    assert m.rho_f_at(tuple(np.zeros(0, np.int64) for _ in range(3))).shape == (0, m.K)
    for bad in ((subs[0], subs[1], subs[2][:-1]), (subs[0], subs[1], subs[2].astype(float)),
                (subs[0], subs[1] + m.N, subs[2]), (subs[0], -1 - subs[1], subs[2]), (subs[0] + m.L, subs[1], subs[2]),
                subs[:2], tuple(np.zeros(0) for _ in range(3))):
        with pytest.raises(ValueError):
            m.rho_f_at(bad)


def test_fits_rho_f_at_equals_rho_f():
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
    _assert_rho_f_at(ref)
    for conc in (False, True):
        for store in (True, False, "never"):
            _assert_rho_f_at(_fit(g, X, R, num_realisations=2, max_iter=40, seed=seed, concurrent_realisations=conc,
                                  store_rho=store))
    for name in ("karnataka_vil1", "custom_mask"):
        g = Golden(name)
        X, R = build_inputs(g)
        for store in ((True, "never") if name == "karnataka_vil1" else (True,)):
            _assert_rho_f_at(_fit(g, X, R, init_state=g.init_state(), store_rho=store))


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

        g = Golden("gm_n640_l2_k3")  # L = 2, K = 3
        X, R = build_inputs(g, structured=True)
        rng = np.random.RandomState(8)  # the same queries on every rank
        n = 5000
        subs = (rng.randint(0, g.L, n), rng.randint(0, g.N, n), rng.randint(0, g.N, n))
        for store in (True, "never"):
            m = _fit(g, X, R, init_state=g.init_state(), max_iter=12, convergence_tol=0.0, store_rho=store)
            res["world"] = m._world
            with warnings.catch_warnings():
                warnings.simplefilter("ignore")
                Y = m.get_inferred_model("rho_max", sparse=True)
            q = tuple(np.concatenate([a, b]) for a, b in zip(subs, Y.subs))
            res[store] = dict(got=m.rho_f_at(q), want=m.rho_f[q], n_edges=len(Y.vals))
        res["ok"] = True
    except Exception:  # noqa: BLE001
        import traceback

        res["ok"] = False
        res["error"] = traceback.format_exc()[-1500:]
    out.put((rank, res))
    dist.destroy_process_group()


def test_two_rank_rho_f_at():
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
            r = res[store]
            assert r["n_edges"] > 0 and r["got"].shape == (5000 + r["n_edges"], 3)
            assert np.array_equal(r["got"], r["want"]), (rank, store)
            assert np.array_equal(r["got"], results[0][store]["got"]), (rank, store)  # every rank holds the whole result
        assert np.array_equal(res[True]["got"], res["never"]["got"]), rank  # with or without the slab
    del torch


@pytest.mark.slow
def test_rho_f_at_beyond_the_slab():
    """N = 160 000 nodes without the slab (205 GB): `rho_f_at` on the rho_max edge list and on random ties adds far less
    than 1 GB of device memory, equals `materialize_rows` on sampled rows, and its argmax gives the sparse labels."""
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
    Y = model.get_inferred_model("rho_max", sparse=True)
    assert len(Y.vals) > 0
    n = 100_000
    rows = rng.choice(N, 4, replace=False)
    q = tuple(np.concatenate([a, b, c]) for a, b, c in
              zip(Y.subs, (np.zeros(n, np.int64), rng.randint(0, N, n), rng.randint(0, N, n)),
                  (np.zeros(2 * N, np.int64), np.repeat(rows, N // 2), rng.randint(0, N, 2 * N))))
    torch.cuda.synchronize()
    base = torch.cuda.memory_allocated()
    torch.cuda.reset_peak_memory_stats()
    got = model.rho_f_at(q)
    added = torch.cuda.max_memory_allocated() - base
    assert added < 0.25e9, added
    ne = len(Y.vals)
    assert np.array_equal(np.argmax(got[:ne], axis=-1), Y.vals)
    tail = got[ne + n:]
    for i in rows:
        r = eng.materialize_rows(int(i), 1)[0].cpu().numpy().astype(np.float64)
        sel = q[1][ne + n:] == i
        assert sel.sum() > 0 and np.array_equal(tail[sel], r[q[2][ne + n:][sel]]), i
    torch.cuda.synchronize()
