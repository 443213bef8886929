"""The device report generators under every reporter mask: `vm_synth_all` (all-reporter mask), `vm_synth_masked`
(explicit mask) and the routing of `device_reports`, against `vm_synth_ego` and against each other.

Every generator draws reporter m's counts on a pair with the same function of (seed, layer, m, pair), so the reports of
one mask restricted to the entries of a smaller mask are exactly the smaller mask's reports.  The law of the new
counter space (a reporter that is not an endpoint of the pair) is checked by per-class moments against the host
all-reporter generator `dense_reporting_X`, and the self ties against their analytic mean.  Then
`PosteriorSyntheticNetwork` from ego, all-reporter and explicit-mask fits."""
import ctypes
import resource
import warnings

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

L, N, K = 2, 150, 3


def _cuda():
    torch = pytest.importorskip("torch")
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")
    return torch


def _net(n=N, seed=4):
    import vimure_b200.synthetic as syn

    return syn.Multitensor(N=n, L=L, K=K, C=2, avg_degree=8, eta=0.5, seed=seed)


def _lam(with_table):
    return np.array([[0.02, 1.5, 2.5], [0.005, 0.8, 3.0]]) if with_table else None


def _run(entry, net, M, theta, lam=None, seed=9, row0=0, nloc=None, tr=False, mask=None, eta=0.4):
    import vimure_b200.synthetic as syn

    return syn._generate(entry, net.L, net.N, M, K, net.Y_subs, net.Y_vals, theta, eta, seed, lam, "cuda", row0, nloc, tr,
                         mask=mask)


def _masked(net, M, theta, entries, lam=None, seed=9, row0=0, nloc=None, tr=False):
    import vimure_b200.synthetic as syn

    return syn.masked_reports(net.L, net.N, M, K, net.Y_subs, net.Y_vals, theta, 0.4, seed, entries, lam=lam,
                              row0=row0, nloc=nloc, emit_transposed=tr)


def _sorted(out, n, M):
    """(keys, vals) of a generator's output, sorted by key ((l*N+i)*N+j)*M+m; the keys are distinct and the vals > 0"""
    s = out[0].cpu().numpy().astype(np.int64)
    v = out[1].cpu().numpy().astype(np.int64)
    k = ((s[0] * n + s[1]) * n + s[2]) * M + s[3]
    o = np.argsort(k)
    k, v = k[o], v[o]
    assert len(np.unique(k)) == len(k) and (v > 0).all()
    return k, v


def _same(a, b):
    return np.array_equal(a[0], b[0]) and np.array_equal(a[1], b[1])


def _restrict(a, keys):
    sel = np.isin(a[0], keys)
    return a[0][sel], a[1][sel]


def _decode(k, n, M):
    m = k % M
    r = k // M
    return r // (n * n), (r // n) % n, r % n, m


@pytest.mark.parametrize("with_table", [False, True])
def test_every_mask_draws_the_same_counts(with_table):
    _cuda()
    import vimure_b200.masks as masks
    import vimure_b200.synthetic as syn

    net = _net()
    lam = _lam(with_table)
    theta = np.random.RandomState(3).gamma(2.0, 0.5, size=(L, N))
    ego = _sorted(_run("vm_synth_ego", net, N, theta, lam), N, N)
    assert len(ego[0]) > 1000
    # the full ego mask as explicit entries
    full = np.stack(masks.EgoMask(L, N, N, diag=True).to_sptensor().subs)
    assert _same(_sorted(_masked(net, N, theta, full, lam), N, N), ego)
    # a subset of the reporters, without the self ties: explicit entries == device_reports' filtered ego output
    rep = np.zeros((L, N), np.uint8)
    rep[0, ::3] = 1
    rep[1, 1::2] = 1
    sub = masks.EgoMask(L, N, N, rep=rep, diag=False)
    want = _sorted(syn.device_reports(L, N, N, K, net.Y_subs, net.Y_vals, theta, 0.4, 9, lam=lam, mask=sub), N, N)
    assert _same(_sorted(_masked(net, N, theta, np.stack(sub.to_sptensor().subs), lam), N, N), want)
    l, i, j, m = _decode(want[0], N, N)
    assert rep[l, m].all() and (i != j).all() and ((m == i) | (m == j)).all()
    # the all-reporter mask restricted to the ego entries (M = N)
    al = _sorted(_run("vm_synth_all", net, N, theta, lam), N, N)
    l, i, j, m = _decode(al[0], N, N)
    on = (m == i) | (m == j)
    assert _same((al[0][on], al[1][on]), ego)
    assert (~on).sum() > 10 * on.sum()  # most reports come from reporters off the pair
    assert ((i == j) & (m != i)).sum() > 0  # self ties of every reporter
    # a random explicit mask == the all-reporter reports restricted to it: reporters off the pair, self ties, true ties,
    # duplicates
    rng = np.random.RandomState(5)
    n = 200_000
    rnd = np.stack([rng.randint(0, L, n), rng.randint(0, N, n), rng.randint(0, N, n), rng.randint(0, N, n)])
    pos = rng.choice(len(al[0]), 20_000, replace=False)
    hit = np.stack(_decode(al[0][pos], N, N))  # entries known to be positive
    ys = net.Y_subs[:, rng.choice(net.Y_subs.shape[1], 5000)]
    tie = np.stack([ys[0], ys[1], ys[2], rng.randint(0, N, 5000)])  # true ties, any reporter
    selfs = rng.randint(0, N, (2, 3000))
    slf = np.stack([rng.randint(0, L, 3000), selfs[0], selfs[0], selfs[1]])
    entries = np.concatenate([rnd, hit, tie, slf, hit[:, :4000], tie[:, :1000]], axis=1)
    entries = entries[:, rng.permutation(entries.shape[1])]
    got = _sorted(_masked(net, N, theta, entries, lam), N, N)
    ek = np.unique(((entries[0] * N + entries[1]) * N + entries[2]) * N + entries[3])
    want = _restrict(al, ek)
    assert _same(got, want)
    l, i, j, m = _decode(got[0], N, N)
    assert ((m != i) & (m != j) & (i != j)).sum() > 1000 and ((i == j) & (m != i)).sum() > 0
    # the same mask through device_reports (CooMask route) and through an sptensor
    from vimure_b200.sptensor import sptensor

    sp = sptensor(tuple(entries), np.ones(entries.shape[1]), shape=(L, N, N, N))
    dr = syn.device_reports(L, N, N, K, net.Y_subs, net.Y_vals, theta, 0.4, 9, lam=lam, mask=sp)
    assert _same(_sorted(dr, N, N), want)


@pytest.mark.parametrize("with_table", [False, True])
def test_explicit_all_ones_mask_is_the_all_reporter_mask(with_table):
    _cuda()
    n, M = 40, 10
    net = _net(n, seed=6)
    lam = _lam(with_table)
    theta = np.random.RandomState(2).gamma(2.0, 0.5, size=(L, M))
    al = _sorted(_run("vm_synth_all", net, M, theta, lam), n, M)
    everything = np.indices((L, n, n, M)).reshape(4, -1)
    assert _same(_sorted(_masked(net, M, theta, everything, lam), n, M), al)
    assert len(al[0]) > 100


@pytest.mark.parametrize("entry", ["vm_synth_all", "vm_synth_masked"])
def test_shards_agree_with_the_whole(entry):
    """As the ego generator: a row block's entries are the whole's entries of its rows, plus with emit_transposed the
    whole's entries of its columns whose rows it does not own; two identical calls give identical sets."""
    _cuda()
    from vimure_b200.model import shard_rows

    n, M = 300, 40
    net = _net(n, seed=8)
    theta = np.random.RandomState(1).gamma(2.0, 0.5, size=(L, M))
    if entry == "vm_synth_masked":
        rng = np.random.RandomState(3)
        ent = np.stack([rng.randint(0, L, 400_000), rng.randint(0, n, 400_000), rng.randint(0, n, 400_000),
                        rng.randint(0, M, 400_000)])
        ys = net.Y_subs
        ent = np.concatenate([ent, np.stack([ys[0], ys[1], ys[2], rng.randint(0, M, ys.shape[1])])], axis=1)

        def gen(**kw):
            return _masked(net, M, theta, ent, **kw)
    else:
        def gen(**kw):
            tr = kw.pop("tr", False)
            return _run(entry, net, M, theta, tr=tr, **kw)
    whole = _sorted(gen(), n, M)
    assert len(whole[0]) > 500
    assert _same(_sorted(gen(), n, M), whole)
    _, i_all, j_all, _ = _decode(whole[0], n, M)
    for r in range(3):
        row0, nloc = shard_rows(n, 3, r)
        own = (i_all >= row0) & (i_all < row0 + nloc)
        tr = ~own & (j_all >= row0) & (j_all < row0 + nloc)
        assert _same(_sorted(gen(row0=row0, nloc=nloc, tr=True), n, M), (whole[0][own | tr], whole[1][own | tr]))
        assert _same(_sorted(gen(row0=row0, nloc=nloc, tr=False), n, M), (whole[0][own], whole[1][own]))


def _class_stats(X, Yd):
    """per class (Y_lij > 0, Y_lji > 0, reporter is an endpoint) of the off-diagonal entries: count, sum X, #X>0, sum X^2,
    sum X X^T"""
    Ln, n, _, M = X.shape
    yij = (Yd > 0)[:, :, :, None]
    yji = np.transpose(Yd > 0, (0, 2, 1))[:, :, :, None]
    idx = np.arange(n)
    m = np.arange(M)
    endp = (idx[:, None, None] == m[None, None, :]) | (idx[None, :, None] == m[None, None, :])
    off = (idx[:, None] != idx[None, :])[None, :, :, None]
    XT = np.transpose(X, (0, 2, 1, 3))
    cls = (yij * 4 + yji * 2 + endp[None]).astype(np.int64)
    out = np.zeros((8, 5))
    for c in range(8):
        sel = (cls == c) & off
        x = X[np.broadcast_to(sel, X.shape)]
        xt = XT[np.broadcast_to(sel, X.shape)]
        out[c] = (x.size, x.sum(), (x > 0).sum(), (x * x).sum(), (x * xt).sum())
    return out


def test_all_reporter_law_against_the_host_generator():
    """Off the diagonal, `vm_synth_all` and `dense_reporting_X` per class over 40 seeds each, within 5 standard errors;
    the self ties against their analytic mean theta lam_0 (1 + eta/(1-eta))."""
    torch = _cuda()
    import vimure_b200.synthetic as syn

    n, M, eta = 60, 60, 0.5
    net = syn.Multitensor(N=n, L=L, K=K, C=2, avg_degree=10, eta=0.5, seed=12)
    Yd = net.Y.toarray()
    assert ((Yd > 0) & (np.transpose(Yd, (0, 2, 1)) > 0)).any() and ((Yd > 0) & (np.transpose(Yd, (0, 2, 1)) == 0)).any()
    host, dev = [], []
    self_sum, self_mean, self_var = 0.0, 0.0, 0.0
    for sd in range(40):
        X, theta = syn.dense_reporting_X(net, M=M, mutuality=eta, seed=100 + sd)
        host.append(_class_stats(X.toarray(), Yd))
        s, v = _run("vm_synth_all", net, M, theta, seed=5000 + sd, eta=eta)
        Xd = np.zeros((L, n, n, M), np.int64)
        s = s.cpu().numpy().astype(np.int64)
        Xd[tuple(s)] = v.cpu().numpy()
        dev.append(_class_stats(Xd, Yd))
        d = np.arange(n)
        self_sum += Xd[:, d, d, :].sum()
        mu = theta * syn.LAMBDA_0  # (L, M): every self tie of reporter m
        mm = mu / (1 - eta)
        self_mean += n * (mu * (1 + eta / (1 - eta))).sum()
        self_var += n * (mu + eta * mm + eta * eta * mm).sum()
    a, b = np.stack(dev), np.stack(host)
    assert np.array_equal(a[:, :, 0], b[:, :, 0])
    for c in range(8):
        for q, name in ((1, "sum X"), (2, "#X>0"), (3, "sum X^2"), (4, "sum X X^T")):
            x, y = a[:, c, q], b[:, c, q]
            se = np.sqrt(x.var(ddof=1) / len(x) + y.var(ddof=1) / len(y))
            assert abs(x.mean() - y.mean()) <= 5 * se + 1e-9, (c, name, x.mean(), y.mean(), se)
    assert abs(self_sum - self_mean) <= 5 * np.sqrt(self_var), (self_sum, self_mean, np.sqrt(self_var))
    del torch


def test_c_abi_refusals_and_capacity():
    torch = _cuda()
    import vimure_b200.synthetic as syn
    from vimure_b200 import _capi

    lib = _capi.load()
    C = _capi.consts()
    n, M = 50, 8
    net = _net(n, seed=2)
    theta = np.random.RandomState(1).gamma(2.0, 0.5, size=(L, M))
    ykey = (net.Y_subs[0] * n + net.Y_subs[1]) * n + net.Y_subs[2]
    o = np.argsort(ykey)
    yk = torch.as_tensor(ykey[o], device="cuda")
    yv = torch.as_tensor(net.Y_vals[o].astype(np.int32), device="cuda")
    th = torch.as_tensor(theta, device="cuda")
    counter = torch.full((1,), 12345, dtype=torch.int64, device="cuda")
    ent = torch.zeros((4, 10), dtype=torch.int32, device="cuda")
    stream = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)

    def args(**kw):
        S = _capi.synth_class()()
        S.L, S.N, S.M, S.K, S.row0, S.nloc, S.emit_transposed, S.seed, S.eta = L, n, M, K, 0, n, 0, 9, 0.4
        S.theta, S.y_key, S.y_val, S.nY = th.data_ptr(), yk.data_ptr(), yv.data_ptr(), int(yk.numel())
        S.cap, S.counter = 0, counter.data_ptr()
        for k, v in kw.items():
            setattr(S, k, v)
        return S

    def mask(**kw):
        Mk = _capi.synth_mask_class()()
        Mk.l, Mk.i, Mk.j, Mk.m = (ent[d].data_ptr() for d in range(4))
        Mk.n = 10
        for k, v in kw.items():
            setattr(Mk, k, v)
        return Mk

    bad = [dict(L=0), dict(N=0), dict(M=0), dict(nloc=-1), dict(row0=-1), dict(row0=10, nloc=n), dict(eta=1.0),
           dict(eta=-0.1), dict(cap=-1), dict(counter=None), dict(theta=None), dict(y_key=None), dict(nY=-1),
           dict(N=2 ** 31), dict(cap=5)]  # cap > 0 without output arrays
    for kw in bad:
        S = args(**kw)
        assert lib.vm_synth_all(ctypes.byref(S), stream) == C["VM_EINVAL"], kw
        Mk = mask()
        assert lib.vm_synth_masked(ctypes.byref(S), ctypes.byref(Mk), stream) == C["VM_EINVAL"], kw
    S = args()
    assert lib.vm_synth_masked(ctypes.byref(S), None, stream) == C["VM_EINVAL"]
    for kw in (dict(n=-1), dict(l=None), dict(m=None)):
        Mk = mask(**kw)
        assert lib.vm_synth_masked(ctypes.byref(S), ctypes.byref(Mk), stream) == C["VM_EINVAL"], kw
    torch.cuda.synchronize()
    assert int(counter.item()) == 12345  # nothing was launched, the counter untouched
    # a capacity below the output: the full count, only `cap` entries stored, the rest untouched
    full = _sorted(_run("vm_synth_all", net, M, theta, seed=9), n, M)
    nfull = len(full[0])
    cap = nfull // 3
    out = torch.full((5, nfull), -7, dtype=torch.int32, device="cuda")
    S = args(cap=cap)
    S.o_l, S.o_i, S.o_j, S.o_m, S.o_x = (out[d].data_ptr() for d in range(5))
    _capi.check(lib.vm_synth_all(ctypes.byref(S), stream), "vm_synth_all")
    assert int(counter.item()) == nfull
    h = out.cpu().numpy().astype(np.int64)
    assert (h[:, cap:] == -7).all() and (h[:, :cap] >= 0).all()
    k = ((h[0, :cap] * n + h[1, :cap]) * n + h[2, :cap]) * M + h[3, :cap]
    pos = np.searchsorted(full[0], k)
    assert np.array_equal(full[0][pos], k) and np.array_equal(full[1][pos], h[4, :cap])
    # the same for the explicit mask (every entry of the shape)
    everything = torch.as_tensor(np.indices((L, n, n, M)).reshape(4, -1).astype(np.int32), device="cuda")
    Mk = mask(n=int(everything.shape[1]))
    Mk.l, Mk.i, Mk.j, Mk.m = (everything[d].data_ptr() for d in range(4))
    out.fill_(-7)
    _capi.check(lib.vm_synth_masked(ctypes.byref(S), ctypes.byref(Mk), stream), "vm_synth_masked")
    assert int(counter.item()) == nfull
    h = out.cpu().numpy().astype(np.int64)
    assert (h[:, cap:] == -7).all()
    k = ((h[0, :cap] * n + h[1, :cap]) * n + h[2, :cap]) * M + h[3, :cap]
    pos = np.searchsorted(full[0], k)
    assert np.array_equal(full[0][pos], k) and np.array_equal(full[1][pos], h[4, :cap])
    # host validation of explicit masks
    with pytest.raises(ValueError):
        _masked(net, M, theta, np.array([[0], [0], [n], [0]]))
    with pytest.raises(ValueError):
        _masked(net, M, theta, np.array([[0], [0], [1], [M]]))
    with pytest.raises(ValueError):
        _masked(net, M, theta, np.array([[-1], [0], [1], [0]]))
    del syn


def _fit(X, R, K_, seed=5, **kw):
    import vimure_b200 as vm

    model = vm.VimureModel(mutuality=True)
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        model.fit(X, R=R, K=K_, seed=seed, max_iter=21, **kw)
    return model


def _check_posterior_network(model, ps, kind, M, seed_X=7):
    Lm, n, Km = model.L, model.N, model.K
    assert ps.R.kind == kind and tuple(ps.R.shape) == (Lm, n, n, M)
    prng = np.random.RandomState(seed_X)
    np.testing.assert_array_equal(ps.theta, prng.gamma(shape=model.gamma_shp_f, scale=1.0 / model.gamma_rte_f, size=(Lm, M)))
    np.testing.assert_array_equal(ps.lambda_k, prng.gamma(shape=model.phi_shp_f, scale=1.0 / model.phi_rte_f, size=(Lm, Km)))
    assert ps.mutuality == prng.gamma(shape=model.nu_shp_f, scale=1.0 / model.nu_rte_f, size=1)[0]
    assert ps.X.shape == (Lm, n, n, M) and len(ps.X.vals) > 0 and ps.X.vals.min() >= 1
    # baselines
    tk = (ps.X.subs[0] * n + ps.X.subs[1]) * n + ps.X.subs[2]
    u, c = np.unique(tk, return_counts=True)
    uk = (ps.X_union.subs[0] * n + ps.X_union.subs[1]) * n + ps.X_union.subs[2]
    ik = (ps.X_intersection.subs[0] * n + ps.X_intersection.subs[1]) * n + ps.X_intersection.subs[2]
    assert np.array_equal(uk, u) and np.array_equal(ik, u[c == 2])
    # a refit on what was generated takes (X, R) as they are
    refit = _fit(ps.X, ps.R, Km, seed=3)
    assert np.isfinite(refit.maxL)
    # the device draw of Y, without the (L, N, N) array, is the dense device draw
    psd = type(ps)(model, seed_Y=11).build_Y(rng="device")
    want = np.minimum(model.sample_inferred_model(N=1, seed=11, rng="device")[0], Km - 1)
    assert np.array_equal(psd.Y.toarray(), want)
    assert psd.Y_vals.dtype == np.int64 and psd.Y_subs.dtype == np.int64


def test_posterior_network_all_reporter_fit():
    _cuda()
    import vimure_b200 as vm
    import vimure_b200.synthetic as syn

    n, M = 120, 12
    net = syn.Multitensor(N=n, L=2, K=2, C=2, avg_degree=8, eta=0.3, seed=3)
    X, _ = syn.dense_reporting_X(net, M=M, mutuality=0.3, seed=4)
    model = _fit(X, vm.masks.AllMask(2, n, M), 2)
    ps = syn.PosteriorSyntheticNetwork(model, seed_Y=11).build_Y()
    ps.build_X(flag_self_reporter=False, seed_X=7)
    assert isinstance(ps.R, vm.masks.AllMask)
    assert ps.X.subs[3].max() < M
    l, i, j, m = ps.X.subs
    assert ((m != i) & (m != j)).sum() > 0 and (i == j).sum() > 0
    _check_posterior_network(model, ps, "all", M)


def test_posterior_network_explicit_mask_fit():
    _cuda()
    import vimure_b200 as vm
    import vimure_b200.synthetic as syn
    from vimure_b200.sptensor import sptensor

    n, M = 120, 30
    net = syn.Multitensor(N=n, M=M, L=2, K=2, C=2, avg_degree=8, eta=0.3, seed=3)
    rng = np.random.RandomState(2)
    # each reporter reports her own row and column, and a random set of other ties
    ego = np.stack(vm.masks.EgoMask(2, n, M, diag=False).to_sptensor().subs)
    extra = np.stack([rng.randint(0, 2, 20_000), rng.randint(0, n, 20_000), rng.randint(0, n, 20_000),
                      rng.randint(0, M, 20_000)])
    ent = np.concatenate([ego, extra], axis=1)
    ent = ent[:, np.unique(((ent[0] * n + ent[1]) * n + ent[2]) * M + ent[3], return_index=True)[1]]
    Rsp = sptensor(tuple(ent), np.ones(ent.shape[1], np.int64), shape=(2, n, n, M))
    s, v = net.build_X_device(mutuality=0.3, seed=4, Rinput=Rsp)
    assert isinstance(net.R, vm.masks.CooMask)
    X = sptensor(tuple(s.cpu().numpy().astype(np.int64)), v.cpu().numpy().astype(np.int64), shape=(2, n, n, M))
    model = _fit(X, Rsp, 2)
    ps = syn.PosteriorSyntheticNetwork(model, seed_Y=11).build_Y()
    ps.build_X(Rinput=Rsp, seed_X=7)
    assert isinstance(ps.R, vm.masks.CooMask)
    ek = ((ent[0] * n + ent[1]) * n + ent[2]) * M + ent[3]
    xs = ps.X.subs
    assert np.isin(((xs[0] * n + xs[1]) * n + xs[2]) * M + xs[3], ek).all()  # X within the mask
    _check_posterior_network(model, ps, "coo", M)


def test_posterior_network_ego_fit():
    _cuda()
    import vimure_b200 as vm
    import vimure_b200.synthetic as syn

    net = syn.Multitensor(N=120, L=2, K=3, C=2, avg_degree=8, eta=0.3, seed=3).build_X(mutuality=0.3, seed=4)
    model = _fit(net.X, net.R, 3)
    ps = syn.PosteriorSyntheticNetwork(model, seed_Y=11).build_Y()
    ps.build_X(seed_X=7)
    assert isinstance(ps.R, vm.masks.EgoMask) and ps.R.diag
    l, i, j, m = ps.X.subs
    assert np.all((m == i) | (m == j))
    _check_posterior_network(model, ps, "ego", 120)
    # an ego mask passed explicitly is the same generator
    ps2 = syn.PosteriorSyntheticNetwork(model, seed_Y=11).build_Y()
    ps2.build_X(Rinput=vm.masks.EgoMask(2, 120, 120).to_sptensor(), seed_X=7)
    a = np.lexsort(ps.X.subs[::-1])
    b = np.lexsort(ps2.X.subs[::-1])
    assert all(np.array_equal(p[a], q[b]) for p, q in zip(ps.X.subs, ps2.X.subs))
    assert np.array_equal(ps.X.vals[a], ps2.X.vals[b])


@pytest.mark.slow
def test_posterior_network_beyond_the_slab():
    """N = 160 000 without the slab: build_Y and build_X never build an (L, N, N) array."""
    torch = _cuda()
    import vimure_b200 as vm
    from vimure_b200 import synthetic as syn

    Ln, n, Kn = 1, 160_000, 2
    rng = np.random.RandomState(7)
    nY = 2 * n
    ys = np.stack([np.zeros(nY, np.int64), rng.randint(0, n, nY), rng.randint(0, n, nY)])
    ys = ys[:, ys[1] != ys[2]]
    ys = ys[:, np.unique(ys[1] * n + ys[2], return_index=True)[1]]
    theta = 0.5 + rng.random_sample((Ln, n))
    subs, vals = syn.device_reports(Ln, n, n, Kn, ys, np.ones(ys.shape[1], np.int32), theta, 0.5, seed=11,
                                    lam=np.array([[1e-4, 1.0]]))
    X = vm.sptensor.sptensor(tuple(subs.cpu().numpy()), vals.cpu().numpy(), shape=(Ln, n, n, n))
    del subs, vals
    model = vm.VimureModel(mutuality=True)
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        model.fit(X, R=vm.masks.EgoMask(Ln, n, n), K=Kn, seed=3, max_iter=20, store_rho="never")
    assert model._engine_of_rho_f().rho is None
    del X
    torch.cuda.synchronize()
    base = torch.cuda.memory_allocated()
    torch.cuda.reset_peak_memory_stats()
    rss0 = resource.getrusage(resource.RUSAGE_SELF).ru_maxrss * 1024
    ps = syn.PosteriorSyntheticNetwork(model, seed_Y=5).build_Y()
    ps.build_X(seed_X=7)
    grew = resource.getrusage(resource.RUSAGE_SELF).ru_maxrss * 1024 - rss0
    added = torch.cuda.max_memory_allocated() - base
    want = model.sample_inferred_model(N=1, seed=5, sparse=True)[0]
    assert all(np.array_equal(p, q) for p, q in zip(ps.Y.subs, want.subs))
    assert np.array_equal(ps.Y.vals, np.minimum(want.vals, Kn - 1)) and len(ps.Y.vals) > 0
    assert ps.X.shape == (Ln, n, n, n) and len(ps.X.vals) > 0 and isinstance(ps.R, vm.masks.EgoMask)
    assert grew < 4e9, grew  # one (N, N) uint8 array is 25.6 GB
    assert added < 8e9, added
    print("posterior network N=%d: %d ties, %d reports, host peak RSS +%.2f GB, device +%.2f GB"
          % (n, len(ps.Y.vals), len(ps.X.vals), grew / 1e9, added / 1e9))
