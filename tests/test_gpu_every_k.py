"""Every K the library is built for (2..32 = VM_MAX_K), each against references that do not share its code.

The kernels are templates on K, instantiated once per K; the dense column tile, the gather depth of the gamma / phi passes,
the dense kernel's staging layout and the tie-sorted gamma pass all change with K.  For each K: an ego-mask problem with
two full column tiles and a partial one, counts 1..K-1 all present, against the fp64 oracle over the production cadence;
the slab-free, store-last and graph-replaying engines bit for bit against the storing one; and every consumer (argmax,
`rho_at`, edge lists, the sampler) against a reference that is not the kernel under test -- for the sampler, a numpy
restatement of Philox4x32-10 and of `vm_sample_label`.  Then the all-reporter and general masks at the K where their
kernels switch, and the count guard of the tie-sorted gamma pass."""
import copy
import ctypes
from types import SimpleNamespace

import numpy as np
import pytest

from tests.test_gpu_rho_at import _call, _queries
from tests.test_gpu_scaled import PRIORS, _cuda
from tests.test_gpu_sparse_infer import _assert_edges, _check_engine, _nonzero, _skip_bounds

KS = list(range(2, 33))
STATE = ("gamma_shp", "gamma_rte", "phi_shp", "phi_rte", "nu", "red3", "elbo_out", "rho_u32", "fixA", "fixP")
# the production cadence: (iterations, ELBO on the last one)
CADENCE = ((1, True), (1, False), (1, False), (1, False), (1, True))
RTOL_P, RTOL_E, RTOL_RHO = 1e-5, 1e-6, 3e-5

M32 = np.uint64(0xFFFFFFFF)


# ------------------------------------------------------------------ host reference of the device sampler
def _philox4x32_10(ctr, key):
    """Philox4x32-10 (Salmon et al. 2011) as `vm_philox4x32`: `ctr` four uint32 words (arrays broadcast), `key` two.
    The 32x32 -> 64 bit products in uint64.  Returns the four output words as uint32 arrays."""
    c = [np.asarray(x, dtype=np.uint64) & M32 for x in ctr]
    k0, k1 = (np.asarray(x, dtype=np.uint64) & M32 for x in key)
    for _ in range(10):
        p0 = np.uint64(0xD2511F53) * c[0]
        p1 = np.uint64(0xCD9E8D57) * c[2]
        c = [(p1 >> np.uint64(32)) ^ c[1] ^ k0, p1 & M32, (p0 >> np.uint64(32)) ^ c[3] ^ k1, p0 & M32]
        k0 = (k0 + np.uint64(0x9E3779B9)) & M32
        k1 = (k1 + np.uint64(0xBB67AE85)) & M32
    return [x.astype(np.uint32) for x in c]


def _sample_labels_host(r32, gt, n_trials, seed):
    """`vm_sample_label` for every row of `r32` (n, K) float32, tie ids `gt` (n,): the category drawn most often in
    `n_trials` draws, operation by operation in float32 (none of them can be contracted into an FMA, so numpy gives the
    device's bits).  Counter (gt_lo, gt_hi, blk_lo, blk_hi), key (seed_lo, seed_hi), four draws per block."""
    r = np.ascontiguousarray(r32, dtype=np.float32)
    n, K = r.shape
    gt = np.asarray(gt, dtype=np.int64).astype(np.uint64)
    s = np.zeros(n, np.float32)
    for k in range(K):
        s = s + r[:, k]
    out = np.zeros(n, np.uint8)
    # early return: every draw lands in category 0 when the sum is p[0] > 0
    live = np.nonzero(~((s == r[:, 0]) & (s > 0)))[0]
    p, s, g = r[live], s[live], gt[live]
    cnt = np.zeros((len(live), K), np.int64)
    rows = np.arange(len(live))
    seed = int(seed) & (2 ** 64 - 1)
    key = (seed & 0xFFFFFFFF, seed >> 32)
    for d0 in range(0, n_trials, 4):
        blk = d0 >> 2
        x = _philox4x32_10((g & M32, g >> np.uint64(32), blk & 0xFFFFFFFF, blk >> 32), key)
        for q in range(min(4, n_trials - d0)):
            u = ((x[q] >> np.uint32(9)).astype(np.float32) + np.float32(0.5)) * np.float32(2.0 ** -23) * s
            cum = np.zeros(len(live), np.float32)
            lab = np.full(len(live), K - 1)  # the remainder goes to the last category
            open_ = np.ones(len(live), bool)
            for k in range(K - 1):
                cum = cum + p[:, k]
                hit = open_ & (u < cum)
                lab[hit] = k
                open_ &= ~hit
            cnt[rows, lab] += 1
    out[live] = np.argmax(cnt, axis=1)  # the first category with the largest count
    return out


def test_philox_known_answers():
    """The Random123 known-answer vectors of philox4x32-10."""
    for ctr, key, want in (
            ((0, 0, 0, 0), (0, 0), (0x6627e8d5, 0xe169c58d, 0xbc57ac4c, 0x9b00dbd8)),
            ((0xffffffff,) * 4, (0xffffffff,) * 2, (0x408f276d, 0x41c83b0e, 0xa20bc7c6, 0x6d5451fd)),
            ((0x243f6a88, 0x85a308d3, 0x13198a2e, 0x03707344), (0xa4093822, 0x299f31d0),
             (0xd16cfe09, 0x94fdcceb, 0x5001e420, 0x24126ea1))):
        got = _philox4x32_10(ctr, key)
        assert [int(w) for w in got] == list(want), [hex(int(w)) for w in got]
    # vectorised over counters: each lane equals its scalar evaluation
    ctr = (np.array([0, 0xffffffff, 0x243f6a88], np.uint64), np.array([0, 0xffffffff, 0x85a308d3], np.uint64),
           np.array([0, 0xffffffff, 0x13198a2e], np.uint64), np.array([0, 0xffffffff, 0x03707344], np.uint64))
    got = _philox4x32_10(ctr, (0, 0))
    for i in range(3):
        one = _philox4x32_10(tuple(c[i] for c in ctr), (0, 0))
        assert all(int(a[i]) == int(b) for a, b in zip(got, one))


def test_host_sampler_rules():
    """The rules of `vm_sample_label` the host reference restates, on rows where the answer is known."""
    K = 4
    r = np.array([[1.0, 0.0, 0.0, 0.0],      # sum == p[0] > 0: always 0
                  [0.0, 0.0, 0.0, 0.0],      # dead tie: every draw goes to the last category
                  [0.0, 0.0, 1.0, 0.0],      # all mass on category 2
                  [0.0, 0.0, 0.0, 1.0]], np.float32)
    gt = np.arange(K, dtype=np.int64) + 2 ** 33
    for n in (1, 2, 5, 8):
        assert list(_sample_labels_host(r, gt, n, 2 ** 64 - 1)) == [0, K - 1, 2, 3]
    # two equally likely categories and two draws: the draws of a tie that split 1 / 1 give the first category
    r2 = np.tile(np.array([[0.5, 0.5]], np.float32), (4000, 1))
    g2 = np.arange(4000, dtype=np.int64)
    x = _philox4x32_10((g2, 0, 0, 0), (7, 0))
    u = [((w >> np.uint32(9)).astype(np.float32) + np.float32(0.5)) * np.float32(2.0 ** -23) for w in x[:2]]
    split = (u[0] < 0.5) != (u[1] < 0.5)
    lab = _sample_labels_host(r2, g2, 2, 7)
    assert split.any() and (lab[split] == 0).all()
    assert np.array_equal(lab[~split], np.where(u[0][~split] < 0.5, 0, 1))


# ------------------------------------------------------------------ problems
def _tile_n(K):
    """N with two full column tiles of the dense kernels and a partial one (DenseCfg<K>::TW = 512 / 256 / 128)."""
    return 1100 if K <= 3 else 600 if K <= 5 else 300


def _cover_counts(vals, K, rng):
    """Counts clipped to K-1, and K-1 random entries set to 1..K-1: every count occurs and max(X) = K-1."""
    vals = np.minimum(np.asarray(vals).astype(np.int64), K - 1)
    pick = rng.choice(len(vals), K - 1, replace=False)
    vals[pick] = np.arange(1, K)
    return vals


def _problem(K):
    """Ego-mask problem at K: L, tile_h and mutuality vary with K (two layers for odd K; row tiles of 32 or 128, partial
    either way; mutuality off for K = 5, 10, .., 30)."""
    import vimure_b200.synthetic as syn

    N, L = _tile_n(K), 1 + K % 2
    tile_h, mutuality = (32 if K % 3 else 128), K % 5 != 0
    net = syn.StandardSBM(N=N, L=L, K=K, C=2, avg_degree=6, seed=K).build_X(mutuality=0.4, seed=K + 100)
    vals = _cover_counts(net.X.vals, K, np.random.RandomState(K))
    return dict(subs=np.stack(net.X.subs).astype(np.int64), vals=vals, L=L, N=N, M=N, K=K, mask=net.R,
                spec={"kind": "ego", "rep": np.ones((L, N), dtype=np.uint8), "diag": True}, mutuality=mutuality,
                tile_h=tile_h)


def _engines(subs, vals, L, N, M, K, mask, spec=None, mutuality=True, tile_h=64, slabs=(True,), seed=3):
    """Engines over the same packed data and initial state (`slabs`: with or without a slab), the packed data, and the
    fp64 oracle from that state if `spec` is given."""
    torch = _cuda()
    from oracle.cavi_numpy import OracleCAVI
    from vimure_b200 import _packing
    from vimure_b200._engine import CaviEngine

    P = _packing.pack(subs, vals, L, N, M, K, mask, "cuda", tile_h=tile_h, mutuality=mutuality)
    rs = np.random.RandomState(seed).random_sample
    st = dict(gamma_shp=0.1 * rs((L, M)) + 0.1, phi_shp=10.0 * rs((L, K)) + 10.0, gamma_rte=0.1 * rs((L, M)) + 0.1,
              phi_rte=10.0 * rs((L, K)) + 10.0, nu_shp=0.5 * rs(1)[0] + 0.5)
    keep = (P.t["u_has_x"] & P.t["u_reported"]).cpu().numpy()
    pr_u = np.zeros((P.U, K))
    pr_u[:, 0] = 1.0
    pr = 1 + 0.01 * rs((int(keep.sum()), K))
    pr_u[keep] = pr / pr.sum(axis=1)[:, None]
    nu_rte = PRIORS["beta_eta"] + float(np.sum(vals)) if mutuality else 1.0
    engs = []
    for slab in slabs:
        e = CaviEngine(P, PRIORS, mutuality=mutuality, eps=1e-12, slab=slab)
        e.set_state(st["gamma_shp"], st["gamma_rte"], st["phi_shp"], st["phi_rte"], st["nu_shp"] if mutuality else 1e-6,
                    nu_rte, pr_u, 1e-12)
        engs.append(e)
    o = None
    if spec is not None:
        o = OracleCAVI(L, N, M, K, subs, vals, spec, mutuality=mutuality, EPS=1e-12, **PRIORS)
        flat = P.t["u_gflat"].cpu().numpy()[keep]
        ties = np.stack([flat // (N * N), (flat // N) % N, flat % N], axis=1)
        o.set_state(st["gamma_shp"], st["gamma_rte"], st["phi_shp"], st["phi_rte"], st["nu_shp"],
                    o.default_pr_rho(ties, pr_u[keep]))
    torch.cuda.synchronize()
    return engs, P, o


def _oracle_step(eng, o, P, elbo, mutuality, tag):
    """After one iteration of `eng` and `o`: gamma, phi, nu, the ELBO (if evaluated) and rho_u32 against the oracle."""
    p = eng.params()
    for k in ("gamma_shp", "gamma_rte", "phi_shp", "phi_rte"):
        np.testing.assert_allclose(p[k], getattr(o, k), rtol=RTOL_P, err_msg=f"{k} {tag}")
    if mutuality:
        np.testing.assert_allclose(p["nu_shp"], o.nu_shp, rtol=RTOL_P, err_msg=f"nu {tag}")
    if elbo:
        np.testing.assert_allclose(eng.elbo(), o.elbo(), rtol=RTOL_E, err_msg=f"elbo {tag}")
    flat = P.t["u_gflat"].cpu().numpy()
    np.testing.assert_allclose(eng.rho_u32[:P.U].cpu().numpy().astype(np.float64), o.rho.reshape(-1, P.K)[flat],
                               rtol=RTOL_RHO, atol=1e-30, err_msg=f"rho_u32 {tag}")


def _oracle_parity(eng, o, P, mutuality, tag):
    for step, (n, elbo) in enumerate(CADENCE):
        eng.iterate(n, elbo_last=elbo)
        for _ in range(n):
            o.iterate()
        _oracle_step(eng, o, P, elbo, mutuality, f"{tag} step {step}")
    np.testing.assert_allclose(eng.rho_slab().cpu().numpy().astype(np.float64), o.rho, rtol=RTOL_RHO, atol=1e-30,
                               err_msg=f"slab {tag}")


# ------------------------------------------------------------------ parts 2-4: the ego problem at every K
@pytest.fixture(scope="module", params=KS, ids=lambda K: f"K{K}")
def every_k(request):
    """The ego problem of one K run over the cadence on the storing engine (`ref`) and the fp64 oracle, side by side with
    a slab-free engine (`imp`), one that stores only the last iteration of a call (`nst`: the three iterations without
    the ELBO in one call) and one that replays captured graphs (`gr`).  Records the oracle comparison and the
    bit-identity mismatches per step; the tests assert them, so a failure names the part of the check that failed."""
    torch = _cuda()
    K = request.param
    pb = _problem(K)
    spec, mut = pb.pop("spec"), pb["mutuality"]
    (ref, imp, nst, gr), P, o = _engines(**pb, spec=spec, slabs=(True, False, True, True))
    assert ref.rho is not None and imp.rho is None
    assert gr.enable_graphs()
    parity, mismatch = [], []
    for step, (n, elbo) in enumerate(CADENCE):
        for e in (ref, imp, gr):
            e.iterate(n, elbo_last=elbo)
        if step != 2 and step != 3:  # nst: steps 1..3 as one call iterate(3, store=False, store_last=True)
            nst.iterate(3 if step == 1 else n, elbo_last=elbo, store=False, store_last=True)
        o.iterate()
        try:
            _oracle_step(ref, o, P, elbo, mut, f"K={K} step {step}")
        except AssertionError as ex:
            parity.append(str(ex))
        others = (("slab-free", imp), ("graphs", gr)) + ((("store-last", nst),) if step not in (1, 2) else ())
        for what, e in others:
            for k in STATE:
                if not torch.equal(getattr(ref, k), getattr(e, k)):
                    mismatch.append(f"{k}: {what}, step {step}")
        slab = ref.rho_slab()
        if not torch.equal(gr.rho_slab(), slab):
            mismatch.append(f"slab: graphs, step {step}")
        if step not in (1, 2) and not torch.equal(nst.rho_slab(), slab):
            mismatch.append(f"slab: store-last, step {step}")
        if not torch.equal(imp.materialize_rows(0, P.L * P.nloc), slab.view(P.L * P.nloc, P.N, K)):
            mismatch.append(f"slab: slab-free, step {step}")
    try:
        np.testing.assert_allclose(ref.rho_slab().cpu().numpy().astype(np.float64), o.rho, rtol=RTOL_RHO, atol=1e-30,
                                   err_msg=f"slab K={K}")
    except AssertionError as ex:
        parity.append(str(ex))
    yield SimpleNamespace(K=K, P=P, o=o, ref=ref, imp=imp, nst=nst, gr=gr, parity=parity, mismatch=mismatch,
                          vals=pb["vals"])
    del ref, imp, nst, gr, o
    torch.cuda.synchronize()


@pytest.mark.gpu
def test_problem_covers_every_count(every_k):
    K, P, vals = every_k.K, every_k.P, every_k.vals
    assert set(np.unique(vals).tolist()) == set(range(1, K)) and int(vals.max()) == K - 1
    assert P.nct == 3 and P.N % P.tile_w != 0 and P.N > 2 * P.tile_w, (P.N, P.tile_w)
    assert P.nloc % P.tile_h != 0 and (P.N * K) % 4 == 0


@pytest.mark.gpu
def test_iteration_matches_oracle(every_k):
    assert not every_k.parity, "\n".join(every_k.parity)


@pytest.mark.gpu
def test_engine_paths_bit_identical(every_k):
    torch = _cuda()
    assert not every_k.mismatch, every_k.mismatch
    ref, imp, P = every_k.ref, every_k.imp, every_k.P
    rows = P.L * P.nloc
    slab = ref.rho_slab().view(rows, P.N, P.K)
    for blk in (7, 37):  # neither divides the row count
        assert rows % blk
        for a in range(0, rows, blk):
            b = min(a + blk, rows)
            assert torch.equal(imp.materialize_rows(a, b - a), slab[a:b]), (blk, a)


def _host_sample_check(eng, slab, cases, tag):
    """eng.sample(n, seed) (dense) and eng.sample_edges(n, seed) against the host reference on `slab` (L, nloc, N, K)."""
    torch = _cuda()
    P = eng.P
    r32 = slab.reshape(-1, P.K).cpu().numpy()
    gt = np.arange(P.L * P.N * P.N, dtype=np.int64)  # one rank: local tie t = global id
    for n, seed in cases:
        want = _sample_labels_host(r32, gt, n, seed)
        got = eng.sample(n, seed=seed).reshape(-1).cpu().numpy()
        bad = np.nonzero(got != want)[0]
        assert len(bad) == 0, f"sample({n}, {seed}) {tag}: {len(bad)} ties differ, first {bad[:5]}"
        wt = torch.as_tensor(want.reshape(P.L, P.nloc, P.N), device="cuda")
        _assert_edges(eng.sample_edges(n, seed=seed), _nonzero(eng, wt), f"sample_edges({n}, {seed}) {tag}")


SAMPLE_CASES = ((1, 0), (2, 7), (3, 2 ** 40 + 7), (4, 2 ** 64 - 1), (5, 12345), (8, 2 ** 32))


@pytest.mark.gpu
def test_consumers_against_references(every_k):
    torch = _cuda()
    K, P, o, ref, imp = every_k.K, every_k.P, every_k.o, every_k.ref, every_k.imp
    L, N, nloc = P.L, P.N, P.nloc
    slab = ref.rho_slab()
    s_np = slab.cpu().numpy()
    # argmax: the first maximum of the device slab, exactly; the oracle's wherever its top two are apart
    y = ref.infer(0)
    y_np = y.cpu().numpy()
    assert np.array_equal(y_np, np.argmax(s_np, axis=-1))
    assert torch.equal(imp.infer(0), y)
    top = np.sort(o.rho, axis=-1)
    clear = (top[..., -1] - top[..., -2]) >= 1e-6
    assert clear.mean() > 0.5
    assert np.array_equal(y_np[clear], np.argmax(o.rho, axis=-1)[clear])
    # rho_at: random ties, every special tie, the tile edges -- the slab gather
    keys = _queries(P, seed=K)
    want = slab.reshape(-1, K)[keys]
    for e in (ref, imp):
        assert torch.equal(e.rho_at(keys), want)
    assert torch.equal(ref.rho_at(keys, slab=slab.clone()), want)
    C = ref.C
    bad = torch.tensor([-1, -N * N, -(2 ** 62), L * N * N, L * N * N + 5, 2 ** 62], dtype=torch.int64, device="cuda")
    mixed = torch.cat([keys[:500], bad, keys[500:1000]])
    good = torch.ones(mixed.numel(), dtype=torch.bool, device="cuda")
    good[500:500 + bad.numel()] = False
    for e, src in ((ref, C["VM_EDGES_SLAB"]), (ref, C["VM_EDGES_IMPLICIT"]), (imp, C["VM_EDGES_IMPLICIT"])):
        out = torch.full((mixed.numel(), K), 7.0, device="cuda")
        assert _call(e, src, mixed, out) == 0
        torch.cuda.synchronize()
        assert torch.equal(out[good], slab.reshape(-1, K)[mixed[good]]), src
        assert bool((out[~good] == 7.0).all()), src
    if L == 1:
        # a ctx view over rows [r0, r0+nv) only: the keys of the other rows are left alone (row offsets scale with K)
        from vimure_b200 import _capi

        r0, nv = nloc // 3, nloc // 3
        view = _capi.ctx_class()()
        ctypes.memmove(ctypes.byref(view), ref._cref, ctypes.sizeof(view))
        view.row0, view.nloc, view.nrt = r0, nv, -(-nv // P.tile_h)
        view.rho = slab.data_ptr() + r0 * N * K * 4
        view.tab_p = ref.tab_p.data_ptr() + r0 * K * 4
        view.utile_ptr = P.t["utile_ptr"].data_ptr() + r0 * P.nct * P.t["utile_ptr"].element_size()
        mine = (keys // N >= r0) & (keys // N < r0 + nv)
        assert bool(mine.any()) and not bool(mine.all())
        for src in (C["VM_EDGES_SLAB"], C["VM_EDGES_IMPLICIT"]):
            out = torch.full((keys.numel(), K), 7.0, device="cuda")
            assert _call(ref, src, keys, out, view=view) == 0
            torch.cuda.synchronize()
            assert torch.equal(out[mine], want[mine]), src
            assert bool((out[~mine] == 7.0).all()), src
    # edge lists: the nonzero entries of the dense consumers, implicit source and a cloned slab
    _check_engine(ref, f"K={K} implicit")
    _check_engine(ref, f"K={K} cloned slab", slab=slab.clone())
    _check_engine(imp, f"K={K} slab-free")
    # the sampler against the host reference, bit for bit, on the device's own slab
    _host_sample_check(ref, slab, SAMPLE_CASES, f"K={K}")
    assert torch.equal(imp.sample(3, seed=2 ** 40 + 7), ref.sample(3, seed=2 ** 40 + 7))
    rng = np.random.RandomState(K)
    u = P.t["u_gflat"].cpu().numpy()
    ties = np.concatenate([rng.choice(L * N * N, 2000, replace=False), u[rng.choice(len(u), min(len(u), 1000))]])
    got = ref.sample(2001, seed=2 ** 64 - 1).reshape(-1).cpu().numpy()[ties]
    want_s = _sample_labels_host(s_np.reshape(-1, K)[ties], ties, 2001, 2 ** 64 - 1)
    assert np.array_equal(got, want_s), np.nonzero(got != want_s)[0][:5]
    assert (got != 0).any(), "no tie drew a nonzero label: the comparison would prove little"
    if K in (9, 17, 32):
        # the row skip of the sparse consumers at each of its bounds (K = 32: K-1 = 31 terms, where the SAMPLE bound's
        # half-ulp argument is tight), then the edge lists and the sampler again
        # (on the fixture's slab-free engine: its tables are put back afterwards, whatever runs after this test)
        saved = {k: getattr(imp, k).clone() for k in ("tab_p", "tab_q")}
        try:
            rows = rng.choice(nloc, 40, replace=False)
            _skip_bounds(imp, rows, rng)
            _check_engine(imp, f"K={K} skip bounds")
            assert int((imp.infer(0) != 0).sum()) > 0
            m = imp.materialize_rows(0, L * nloc).view(L, nloc, N, K)
            _host_sample_check(imp, m, ((1, 3), (4, 2 ** 64 - 1), (5, 2 ** 40 + 7)), f"K={K} skip bounds")
        finally:
            for k, v in saved.items():
                getattr(imp, k).copy_(v)


# ------------------------------------------------------------------ part 5: the other masks at the boundary K
def _rel(a, b):
    """Largest relative difference of `a` from `b` over the entries where |b| > 1e-30 (the tolerances' atol)."""
    a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
    m = np.abs(b) > 1e-30
    return float(np.max(np.abs(a[m] - b[m]) / np.abs(b[m]))) if m.any() else 0.0


def _sensitivity(o, o32, flat, K):
    """How far the oracle `o32`, whose posterior is rounded to fp32 after every update, has moved from `o`: per quantity
    of the part-2 check, relative to its tolerance."""
    d = [_rel(getattr(o32, k), getattr(o, k)) / RTOL_P for k in ("gamma_shp", "gamma_rte", "phi_shp", "phi_rte")]
    d.append(_rel(o32.nu_shp, o.nu_shp) / RTOL_P)
    d.append(_rel(o32.rho.reshape(-1, K)[flat], o.rho.reshape(-1, K)[flat]) / RTOL_RHO)
    return max(d)


@pytest.mark.gpu
@pytest.mark.parametrize("K", [4, 5, 8, 9, 32])
def test_all_mask_boundary_k(K):
    """All-reporter mask, M = 16 <= 256, N = 300: k_all32 only at K <= 4, the tie-sorted gamma pass only at K <= 8.

    Every iteration of the cadence is checked at the part-2 tolerances against one fp64 oracle iteration started from the
    engine's own state (its parameters, nu and slab): that isolates the error of the engine's passes from the conditioning
    of the problem.  The conditioning is what limits the check against the free-running oracle here.  The fp64 oracle whose
    posterior is only rounded to fp32 after each update (the precision the gamma / phi passes read rho_u32 in) leaves the
    unrounded oracle by about x10 per iteration at K >= 4 on this problem, whose posteriors swing between categories in the
    first iterations: up to 1e-4 relative on rho and 7e-6 on phi_shp by the fifth iteration.  No fp32 posterior can follow
    the fp64 trajectory closer than that.  So the free-running comparison holds the part-2 tolerances for as long as that
    measured sensitivity stays below a thirtieth of them (at least the first two iterations)."""
    import vimure_b200 as vm
    import vimure_b200.synthetic as syn

    L, N, M = 2, 300, 16
    y = syn.StandardSBM(N=N, M=M, L=L, K=K, C=2, avg_degree=8, seed=K)
    X, _ = syn.dense_reporting_X(y, M=M, mutuality=0.4, seed=K + 1)
    (eng,), P, o = _engines(np.stack(X.subs).astype(np.int64), np.asarray(X.vals), L, N, M, K, vm.masks.AllMask(L, N, M),
                            spec={"kind": "all", "dense_input": True}, tile_h=32)
    assert eng.all32_mode == (K <= 4) and eng.gamma_ts == (K <= 8), (eng.all32_mode, eng.gamma_ts)
    flat = P.t["u_gflat"].cpu().numpy()
    o32 = copy.deepcopy(o)
    free = 0
    for step, (n, elbo) in enumerate(CADENCE):
        one = copy.deepcopy(o)
        if step:  # the engine's state after the previous iteration (the slab holds the rho_u32 the next passes read)
            p = eng.params()
            one.gamma_shp, one.gamma_rte, one.phi_shp, one.phi_rte = (p[k] for k in ("gamma_shp", "gamma_rte", "phi_shp",
                                                                                     "phi_rte"))
            one.nu_shp = float(p["nu_shp"])
            one.rho = eng.rho_slab().cpu().numpy().astype(np.float64)
        eng.iterate(n, elbo_last=elbo)
        for x in (one, o, o32):
            x.iterate()
        o32.rho = o32.rho.astype(np.float32).astype(np.float64)
        _oracle_step(eng, one, P, elbo, True, f"all K={K} step {step}, one oracle iteration from the engine's state")
        if free == step and _sensitivity(o, o32, flat, K) < 1 / 30:
            _oracle_step(eng, o, P, elbo, True, f"all K={K} step {step}, free-running oracle")
            free += 1
    np.testing.assert_allclose(eng.rho_slab().cpu().numpy().astype(np.float64), one.rho, rtol=RTOL_RHO, atol=1e-30,
                               err_msg=f"slab all K={K}")
    assert free >= 2, free


def _coo_problem(K, seed):
    """General COO mask (as tests/test_gpu_random.py builds it): most of the ego entries, some weights of 2, extra
    reporters on random ties, X entries outside R, second reports on existing ties and self-loops."""
    import vimure_b200 as vm
    import vimure_b200.synthetic as syn

    rng = np.random.RandomState(2000 + seed)
    L, N, M = 2, 128, 30
    net = syn.StandardSBM(N=N, M=M, L=L, K=K, C=2, avg_degree=8, seed=seed).build_X(mutuality=0.3, seed=seed + 1)
    subs, vals = np.stack(net.X.subs).astype(np.int64), np.asarray(net.X.vals)
    rep = (rng.rand(L, M) < 0.7).astype(np.uint8)
    rep[:, 0] = 1
    keep = rep[subs[0], np.minimum(subs[3], M - 1)] == 1
    subs, vals = subs[:, keep], vals[keep]
    R = vm.masks.EgoMask(L, N, M, rep=rep, diag=False).to_sptensor()
    rs, rv = np.stack(R.subs).astype(np.int64), np.asarray(R.vals).astype(np.float64)
    k2 = rng.rand(rs.shape[1]) < 0.9
    rs, rv = rs[:, k2], rv[k2]
    rv[rng.rand(rv.size) < 0.05] = 2.0
    n_extra = 3 * N
    ex = np.stack([rng.randint(0, L, n_extra), rng.randint(0, N, n_extra), rng.randint(0, N, n_extra),
                   rng.randint(0, M, n_extra)])
    allk = np.concatenate([rs, ex], axis=1)
    _, first = np.unique(np.ravel_multi_index(tuple(allk), (L, N, N, M)), return_index=True)
    first.sort()
    rs, rv = allk[:, first], np.concatenate([rv, np.ones(n_extra)])[first]
    mask = vm.masks.CooMask(tuple(rs), rv, (L, N, N, M), dense_input=False)
    spec = {"kind": "coo", "subs": rs, "vals": rv, "dense_input": False}
    take = rng.choice(subs.shape[1], size=min(20, subs.shape[1]), replace=False)
    extra = subs[:, take].copy()
    extra[3] = (extra[3] + 1 + rng.randint(0, M - 1, extra.shape[1])) % M
    loops = subs[:, take[:5]].copy()
    loops[2] = loops[1]
    allk = np.concatenate([subs, extra, loops], axis=1)
    allv = np.concatenate([vals, rng.randint(1, 4, extra.shape[1]), rng.randint(1, 3, loops.shape[1])])
    _, first = np.unique(np.ravel_multi_index(tuple(allk), (L, N, N, M)), return_index=True)
    first.sort()
    subs, vals = allk[:, first], allv[first]
    return dict(subs=subs, vals=vals, L=L, N=N, M=M, K=K, mask=mask, spec=spec)


@pytest.mark.parametrize("K", [6, 9, 17, 32])
@pytest.mark.gpu
def test_general_mask_boundary_k(K):
    pb = _coo_problem(K, seed=K)
    (eng,), P, o = _engines(**pb, tile_h=32)
    assert P.r_mode == 2
    _oracle_parity(eng, o, P, True, f"coo K={K}")


@pytest.mark.gpu
@pytest.mark.parametrize("xmax", [2 ** 19 - 1, 2 ** 19])
def test_gamma_ts_count_guard(xmax, monkeypatch):
    """The tie-sorted gamma pass accumulates x * rho in fixed point (2^-30, three 20-bit limbs) and runs only while every
    count is below 2^19; at 2^19 the reporter-sorted pass takes over.  At such a count the fp64 oracle itself overflows
    (its exp of the tie's log-posterior is not shifted by the maximum), so the reference here is the same engine with the
    tie-sorted pass switched off (VM_NO_GAMMA_TS=1).  Only at 2^19 - 1 does that compare two different kernels: there the
    passes must agree at the part-2 tolerances over the cadence.  At 2^19 both engines run the reporter-sorted pass, so
    that case pins the guard itself (which pass runs) and that the fit stays finite.  The count is put on every entry of
    one reporter that has a reciprocal report, so that a warp's shared limbs sum many terms of ~2^19 (the 512-term
    headroom argument of k_gamma_partial_ts), not a single one."""
    import vimure_b200 as vm
    import vimure_b200.synthetic as syn

    L, N, M, K = 1, 300, 12, 2
    y = syn.StandardSBM(N=N, M=M, L=L, K=K, C=2, avg_degree=8, seed=5)
    X, _ = syn.dense_reporting_X(y, M=M, mutuality=0.5, seed=6)
    subs, vals = np.stack(X.subs).astype(np.int64), np.asarray(X.vals).astype(np.int64).copy()
    # the entries of one reporter that have a reciprocal report (only those visit the gamma pass, f_x)
    key = ((subs[0] * N + subs[1]) * N + subs[2]) * M + subs[3]
    rkey = ((subs[0] * N + subs[2]) * N + subs[1]) * M + subs[3]
    recip = np.nonzero(np.isin(rkey, key) & (subs[1] != subs[2]))[0]
    recip = recip[subs[3, recip] == subs[3, recip[0]]]
    assert len(recip) >= 64, len(recip)
    vals[recip] = xmax
    mask = vm.masks.AllMask(L, N, M)
    (eng,), P, _ = _engines(subs, vals, L, N, M, K, mask)
    monkeypatch.setenv("VM_NO_GAMMA_TS", "1")
    (ref,), _, _ = _engines(subs, vals, L, N, M, K, mask)
    assert float(P.t["f_x"].max()) == xmax
    assert eng.gamma_ts == (xmax < 2 ** 19) and not ref.gamma_ts
    for step, (n, elbo) in enumerate(CADENCE):
        for e in (eng, ref):
            e.iterate(n, elbo_last=elbo)
        p, q = eng.params(), ref.params()
        for k in ("gamma_shp", "gamma_rte", "phi_shp", "phi_rte", "nu_shp"):
            assert np.all(np.isfinite(p[k])), k
            np.testing.assert_allclose(p[k], q[k], rtol=RTOL_P, err_msg=f"{k} xmax={xmax} step {step}")
        if elbo:
            assert np.isfinite(eng.elbo())
            np.testing.assert_allclose(eng.elbo(), ref.elbo(), rtol=RTOL_E, err_msg=f"elbo xmax={xmax} step {step}")
    np.testing.assert_allclose(eng.rho_slab().cpu().numpy(), ref.rho_slab().cpu().numpy(), rtol=RTOL_RHO, atol=1e-30)


# ------------------------------------------------------------------ part 6: tie ids >= 2^32
@pytest.mark.gpu
@pytest.mark.slow
def test_sampler_at_tie_ids_beyond_2_32():
    """N = 70 000 without the slab: rows with (l*N+i)*N >= 2^32 key the sampler's Philox counter with a nonzero high word.
    The row's materialised posterior, the sparse sampler restricted to the row, and the host reference agree exactly."""
    torch = _cuda()
    import vimure_b200 as vm
    from vimure_b200 import synthetic as syn

    L, N, K = 1, 70_000, 2
    rng = np.random.RandomState(7)
    nY = 2 * N
    ys = np.stack([np.zeros(nY, np.int64), rng.randint(0, N, nY), rng.randint(0, N, nY)])
    ys = ys[:, ys[1] != ys[2]]
    ys = ys[:, np.unique(ys[1] * N + ys[2], return_index=True)[1]]
    theta = 0.5 + rng.random_sample((L, N))
    subs, vals = syn.device_reports(L, N, N, K, ys, np.ones(ys.shape[1], np.int32), theta, 0.5, seed=11,
                                    lam=np.array([[1e-4, 1.0]]))
    subs, vals = subs.cpu().numpy().astype(np.int64), vals.cpu().numpy()
    (imp,), P, _ = _engines(subs, vals, L, N, N, K, vm.masks.EgoMask(L, N, N), slabs=(False,))
    imp.iterate(2, elbo_last=True)
    lo = -(-(2 ** 32) // N)
    u_row = P.t["u_lrow"].long()
    hi_u = u_row[(u_row >= lo) & (imp.rho_u32[:P.U, 1] > 1e-3)].cpu().numpy()
    assert len(hi_u) > 0
    rows = np.unique(np.concatenate([[lo, N - 1], rng.choice(hi_u, min(3, len(hi_u)), replace=False),
                                     rng.randint(lo, N, 2)]))
    post = {int(i): imp.materialize_rows(int(i), 1)[0].cpu().numpy() for i in rows}
    n_edges = 0
    for n, seed in ((3, 5), (4, 2 ** 64 - 1), (2001, 2 ** 40 + 7)):
        keys, lab = imp.sample_edges(n, seed=seed)
        for i, r in post.items():
            gt = i * N + np.arange(N, dtype=np.int64)
            assert gt[0] >= 2 ** 32
            want = _sample_labels_host(r, gt, n, seed)
            sel = (keys // N) == i
            nz = np.nonzero(want)[0]
            assert np.array_equal(keys[sel].cpu().numpy(), gt[nz]), (i, n, seed)
            assert np.array_equal(lab[sel].cpu().numpy(), want[nz]), (i, n, seed)
            n_edges += len(nz)
    assert n_edges > 0, "no sampled edge in the rows: the comparison would prove little"
    torch.cuda.synchronize()

