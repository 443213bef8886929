"""CPU-only checks: the C-ABI library loads and exports every declared symbol; packing logic; masks."""
import ctypes
import os

import numpy as np
import pytest
import torch

from tests.golden_util import Golden


def test_library_exports_every_declared_symbol():
    from vimure_b200 import _capi, build

    build.build()
    lib = _capi.load()
    names = _capi.header_symbols()
    assert len(names) >= 12
    for n in names:
        assert hasattr(lib, n), n
    assert lib.vm_ctx_size() == ctypes.sizeof(_capi.ctx_class())
    assert lib.vm_abi_version() == _capi.consts()["VM_ABI_VERSION"]


def test_no_cpu_fallback():
    import vimure_b200 as vm

    if torch.cuda.is_available():
        pytest.skip("GPU present")
    g = Golden("sbm_k3")
    X = vm.sptensor.sptensor(tuple(g.X_subs), g.X_vals, shape=(g.L, g.N, g.N, g.M))
    with pytest.raises(RuntimeError, match="CUDA"):
        vm.VimureModel().fit(X, K=3, R=vm.masks.EgoMask(g.L, g.N, g.M))


@pytest.mark.parametrize("name", ["f1_over", "karnataka_vil1", "custom_mask", "dense_reporting"])
def test_mask_detection(name):
    import vimure_b200 as vm

    g = Golden(name)
    spec = g.R_spec
    if spec["kind"] == "all":
        m = vm.masks.from_input(np.ones((g.L, g.N, g.N, g.M)), g.L, g.N, g.M)
        assert m.kind == "all"
        return
    subs, vals = g.R_coo()
    R = vm.sptensor.sptensor(tuple(subs), vals, shape=(g.L, g.N, g.N, g.M))
    m = vm.masks.from_input(R, g.L, g.N, g.M)
    assert m.kind == spec["kind"]
    if m.kind == "ego":
        assert m.diag == spec["diag"]
        assert np.array_equal(m.rep, spec["rep"])
        # round trip through the explicit form
        R2 = m.to_sptensor()
        k1 = np.sort(np.ravel_multi_index(tuple(subs), R.shape))
        k2 = np.sort(np.ravel_multi_index(R2.subs, R.shape))
        assert np.array_equal(k1, k2)
    # membership queries agree with the explicit mask
    rng = np.random.RandomState(0)
    q = np.stack([rng.randint(0, g.L, 500), rng.randint(0, g.N, 500), rng.randint(0, g.N, 500), rng.randint(0, g.M, 500)])
    q[:, :250] = subs[:, rng.randint(0, subs.shape[1], 250)]
    dense = R.toarray()
    mult = m.entry_multiplicity(*[torch.as_tensor(a) for a in q]).numpy()
    assert np.array_equal(mult > 0, dense[tuple(q)] > 0)
    rep_any = dense.sum(axis=-1) > 0
    tr = m.tie_reported(*[torch.as_tensor(a) for a in q[:3]]).numpy()
    assert np.array_equal(tr, rep_any[tuple(q[:3])])


def test_ego_detection_rejects_duplicates_and_near_misses():
    """An explicit mask is only recognised as an ego mask if it is EXACTLY one (same entries, each once)."""
    import vimure_b200 as vm

    L, N, M = 2, 30, 20
    ego = vm.masks.EgoMask(L, N, M, rep=np.arange(0, M, 2), diag=True)
    R = ego.to_sptensor()
    subs, vals = [np.asarray(s) for s in R.subs], np.asarray(R.vals)
    m = vm.masks.from_input(R, L, N, M)
    assert m.kind == "ego" and m.diag and np.array_equal(m.rep, ego.rep)
    # one entry replaced by a copy of another entry of the same reporter and side: same counts, not distinct
    l, i, j, r = (a.copy() for a in subs)
    idx = np.nonzero((l == l[0]) & (r == r[0]) & (i == r) & (j != r))[0][:2]
    for a in (l, i, j, r):
        a[idx[1]] = a[idx[0]]
    assert vm.masks._detect_ego((l, i, j, r), vals, L, N, M) is None
    assert vm.masks.from_input(vm.sptensor.sptensor((l, i, j, r), vals, shape=R.shape), L, N, M).kind == "coo"
    # a reporter that reports a tie it is not part of / a non-unit value / a missing entry
    l, i, j, r = (a.copy() for a in subs)
    i[5], j[5] = (r[5] + 1) % N, (r[5] + 2) % N
    assert vm.masks._detect_ego((l, i, j, r), vals, L, N, M) is None
    v2 = vals.copy()
    v2[3] = 2
    assert vm.masks._detect_ego(subs, v2, L, N, M) is None
    assert vm.masks._detect_ego([a[1:] for a in subs], vals[1:], L, N, M) is None
    # without the diagonal entries it is the diag=False ego mask
    keep = ~((subs[1] == subs[3]) & (subs[2] == subs[3]))
    m2 = vm.masks._detect_ego([a[keep] for a in subs], vals[keep], L, N, M)
    assert m2 is not None and not m2.diag
    # the sort-based path (far fewer entries than slots) gives the same verdicts
    assert vm.masks._ego_entries_distinct(*[a[:7] for a in subs], L=L, N=10**6, M=M)
    dup = [np.concatenate([a[:7], a[:1]]) for a in subs]
    assert not vm.masks._ego_entries_distinct(*dup, L=L, N=10**6, M=M)


@pytest.mark.parametrize("name,world", [("f1_over", 1), ("karnataka_vil1", 1), ("gm_l2_k3", 3), ("custom_mask", 2), ("nomut", 2),
                                        ("dense_reporting", 3), ("f1_over", 8)])
def test_packing_invariants(name, world):
    import vimure_b200 as vm
    from vimure_b200 import _packing
    from vimure_b200.model import shard_rows

    g = Golden(name)
    spec = g.R_spec
    if spec["kind"] == "ego":
        mask = vm.masks.EgoMask(g.L, g.N, g.M, rep=spec["rep"], diag=spec["diag"])
    elif spec["kind"] == "all":
        mask = vm.masks.AllMask(g.L, g.N, g.M)
    else:
        mask = vm.masks.CooMask(spec["subs"], spec["vals"], (g.L, g.N, g.N, g.M))
    Xd = np.zeros((g.L, g.N, g.N, g.M))
    Xd[tuple(g.X_subs)] = g.X_vals
    tot_I, tot_IT = 0, 0
    for r in range(world):
        row0, nloc = shard_rows(g.N, world, r)
        P = _packing.pack(g.X_subs, g.X_vals, g.L, g.N, g.M, g.K, mask, "cpu", row0=row0, nloc=nloc, tile_h=16,
                          mutuality=g.mutuality)
        t = {k: v.numpy() for k, v in P.t.items()}
        tot_I += P.I
        tot_IT += P.IT
        # every entry: tie, reporter, value and reciprocal are right
        eu = t["e_u"]
        lrow, col = t["u_lrow"][eu], t["u_col"][eu]
        l, i = lrow // nloc, lrow % nloc + row0
        assert np.array_equal(Xd[l, i, col, t["e_m"]], t["e_x"])
        assert np.array_equal(Xd[l, col, i, t["e_m"]], t["e_xT"])
        # CSR by tie is consistent
        assert t["u_ptr"][0] == 0 and t["u_ptr"][-1] == P.I
        assert np.all(np.diff(t["u_ptr"]) >= 0)
        assert np.array_equal(np.repeat(np.arange(P.U), np.diff(t["u_ptr"])), eu)
        # special ties sorted, tile pointers monotone and complete
        key = t["u_lrow"].astype(np.int64) * g.N + t["u_col"]
        assert np.all(np.diff(key) > 0)
        tp = t["utile_ptr"]
        assert tp[0] == 0 and tp[-1] == P.U and np.all(np.diff(tp) >= 0)
        # E1 = entries with a reciprocal report (the only ones the gamma / phi passes visit); E0 = the rest
        e1 = t["e1_idx"]
        is1 = np.zeros(P.I, dtype=bool)
        is1[e1] = True
        assert np.array_equal(is1, (t["e_xT"] != 0) if g.mutuality else np.zeros(P.I, dtype=bool))
        assert P.I1 == int(is1.sum())
        assert np.array_equal(t["f_u"], eu[e1]) and np.array_equal(t["f_x"], t["e_x"][e1])
        lm_of_entry = l * g.M + t["e_m"]
        g0_ref = np.zeros(g.L * g.M)
        np.add.at(g0_ref, lm_of_entry[~is1], t["e_x"][~is1].astype(np.float64))
        np.testing.assert_allclose(t["g0"], g0_ref, rtol=0, atol=1e-9)
        x0_ref = np.zeros(P.U)
        np.add.at(x0_ref, eu[~is1], t["e_x"][~is1].astype(np.float64))
        np.testing.assert_allclose(t["u_x0sum"], x0_ref, rtol=0, atol=1e-6)
        # layer ranges of the E1 entries
        lp = t["lay_eptr"]
        assert lp[0] == 0 and lp[-1] == P.I1 and np.all(np.diff(lp) >= 0)
        assert np.array_equal(np.repeat(np.arange(g.L), np.diff(lp)), l[e1])
        # reporter chunks partition the E1 entries by reporter
        gp, cp, clm = t["g_perm"], t["g_chunk_ptr"], t["g_chunk_lm"]
        assert sorted(gp.tolist()) == list(range(P.I1))
        lm1 = lm_of_entry[e1]
        for c in range(P.n_gchunk):
            assert np.all(lm1[gp[cp[c]:cp[c + 1]]] == clm[c])
            assert 0 < cp[c + 1] - cp[c] <= _packing.GAMMA_CHUNK
        assert np.array_equal(t["g_u"], t["f_u"][gp])
    assert tot_I == len(g.X_vals)
    if g.mutuality:
        l, i, j, m = g.X_subs
        mult = mask.entry_multiplicity(*[torch.as_tensor(a) for a in (l, j, i, m)]).numpy()
        assert tot_IT == int((mult > 0).sum())


def test_reference_prior_stream():
    """`reference_prior_draws` reproduces `prng.rand(L,N,N,K)` (model.py:470) at the requested ties."""
    from vimure_b200._packing import reference_prior_draws

    L, N, K = 2, 37, 3
    full = np.random.RandomState(5).rand(L, N, N, K).reshape(-1, K)
    ties = np.sort(np.random.RandomState(1).choice(L * N * N, 200, replace=False))
    prng = np.random.RandomState(5)
    got = reference_prior_draws(prng, L, N, K, ties, chunk=1000)
    assert np.array_equal(got, full[ties])
    # the stream continues exactly where the reference's would
    ref = np.random.RandomState(5)
    ref.rand(L, N, N, K)
    assert prng.random_sample() == ref.random_sample()


@pytest.mark.parametrize("mutuality", [True, False])
def test_simple_special_tie_classification(mutuality):
    """vm_ctx.simple_mode contract: a special tie is SIMPLE iff it has X entries, none of them with a reciprocal report
    (all of them when mutuality is off), it is off the diagonal and lies in a full column tile; it is SINGLE iff it has
    exactly one X entry, that entry has a reciprocal report and was reported by the row or the column node (same position
    constraints); `cx_idx` lists the other special ties in ascending order with per-layer ranges `cx_ptr`, and `cx_*` are
    their compacted per-tie arrays."""
    import vimure_b200.synthetic as syn
    from vimure_b200 import _packing
    from vimure_b200.model import shard_rows

    L, N, K = 2, 1100, 2
    net = syn.Multitensor(N=N, L=L, K=K, C=2, avg_degree=6, eta=0.5, seed=2).build_X(mutuality=0.5, seed=3)
    tw = _packing.dense_tile_w(K)
    n_simple = n_single = 0
    for r in range(2):
        row0, nloc = shard_rows(N, 2, r)
        P = _packing.pack(net.X.subs, net.X.vals, L, N, N, K, net.R, "cpu", row0=row0, nloc=nloc, tile_h=32,
                          mutuality=mutuality)
        assert P.simple_ok
        t = {k: v.numpy() for k, v in P.t.items()}
        s = t["u_simple"]
        n_simple += int(s.sum())
        has_e1 = np.zeros(P.U, dtype=bool)
        has_e1[t["e_u"][t["e1_idx"]]] = True
        l = t["u_lrow"] // nloc
        i = t["u_lrow"] % nloc + row0
        expect = (t["u_cnt"] >= 1) & ~has_e1 & (i != t["u_col"]) & (t["u_col"] < (N // tw) * tw)
        assert np.array_equal(s, expect)
        g = t["u_single"]
        inside = (i != t["u_col"]) & (t["u_col"] < (N // tw) * tw)
        expect_g = (t["u_cnt"] == 1) & (t["u_xT0"] != 0) & inside & ((t["u_m0"] == i) | (t["u_m0"] == t["u_col"]))
        if not mutuality:
            assert P.I1 == 0 and np.array_equal(s, (t["u_cnt"] >= 1) & inside) and not g.any()
        else:
            assert np.array_equal(g, expect_g) and g.any() and not (g & s).any()
            n_single += int(g.sum())
            # patch constants: X = the entry's x; +x^T when the row node reported, -x^T when the column node did
            assert np.array_equal(t["u_px"][g], t["u_x0"][g])
            assert np.array_equal(t["u_pxt"][g], np.where(t["u_m0"][g] == i[g], t["u_xT0"][g], -t["u_xT0"][g]))
            assert (t["u_pxt"][~g] == 0).all() and (t["u_pxt"][g] != 0).all()
        assert np.array_equal(t["u_px"][s], t["u_x0sum"][s]) and (t["u_px"][~(s | g)] == 0).all()
        cx = t["cx_idx"]
        assert P.n_cx == len(cx) and np.array_equal(cx, np.nonzero(~(s | g))[0])
        cp = t["cx_ptr"]
        assert cp[0] == 0 and cp[-1] == P.n_cx
        assert np.array_equal(np.repeat(np.arange(L), np.diff(cp)), l[cx])
        for name in ("lrow", "col", "cnt", "m0", "x0", "xT0", "x0sum"):
            assert np.array_equal(t["cx_" + name], t["u_" + name][cx]), name
        # X of a simple tie = the sum of its entries
        x = np.zeros(P.U)
        np.add.at(x, t["e_u"], t["e_x"].astype(np.float64))
        np.testing.assert_allclose(t["u_x0sum"][s], x[s], rtol=0, atol=1e-6)
    assert n_simple > 0 and (n_single > 0) == mutuality
    # the A/B switches
    P0 = _packing.pack(net.X.subs, net.X.vals, L, N, N, K, net.R, "cpu", tile_h=32, mutuality=mutuality, simple=False)
    assert not P0.simple_ok and P0.n_cx == P0.U and not P0.t["u_simple"].any() and not P0.t["u_single"].any()
    P1 = _packing.pack(net.X.subs, net.X.vals, L, N, N, K, net.R, "cpu", tile_h=32, mutuality=mutuality, single=False)
    assert P1.simple_ok and not P1.t["u_single"].any() and P1.n_cx == P1.U - int(P1.t["u_simple"].sum())
    # no fast dense kernel (N*K % 4 != 0 or N below one column tile) -> no shortcut
    small = syn.StandardSBM(N=300, L=1, K=2, C=2, avg_degree=4, seed=1).build_X(mutuality=0.3, seed=2)
    Ps = _packing.pack(small.X.subs, small.X.vals, 1, 300, 300, 2, small.R, "cpu", mutuality=mutuality)
    assert not Ps.simple_ok and Ps.n_cx == Ps.U
    # the packer itself records whether the E0 / E1 split holds (what the engine's fp32 paths require)
    Pt = _packing.pack_torch(small.X.subs, small.X.vals, 1, 300, 300, 2, small.R, "cpu", mutuality=mutuality,
                             split_e0=False)
    assert Pt.split_e0 == (not mutuality)
