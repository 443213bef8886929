"""`vm_pack` (the device-side packer behind the C ABI, csrc/vm_pack.cu) against the torch restatement of the packed
layout (`_packing.pack_torch`), array by array; and a fit driven WITHOUT the torch packer."""
import os
import subprocess
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _cuda():
    import torch

    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")
    return torch


def _sorted_coo(X):
    """Entries in (l,i,j,m) order: the two packers then also agree on the order of the entries WITHIN a tie."""
    s = np.stack(X.subs).astype(np.int64)
    o = np.lexsort((s[3], s[2], s[1], s[0]))
    return s[:, o], np.asarray(X.vals)[o]


CASES = ["ego_k2", "ego_l2_k3_shard", "ego_nomut", "ego_subset_nodiag", "all_mask", "ego_no_shortcut", "all_mask_shard",
         "ego_subset_nodiag_k4_shard", "ego_empty_shard"]


@pytest.mark.parametrize("case", CASES)
def test_vm_pack_matches_the_torch_packer(case):
    torch = _cuda()
    import vimure_b200 as vm
    import vimure_b200.synthetic as syn
    from vimure_b200 import _packing
    from vimure_b200.model import shard_rows

    kw = dict(mutuality=True, split_e0=True)
    row0, nloc = 0, None
    if case == "ego_k2":
        L, N, K = 1, 1100, 2
        net = syn.StandardSBM(N=N, L=L, K=K, C=2, avg_degree=10, seed=10).build_X(mutuality=0.5, seed=20)
        mask, M = net.R, N
    elif case == "ego_l2_k3_shard":
        L, N, K = 2, 640, 3
        net = syn.Multitensor(N=N, L=L, K=K, C=2, avg_degree=8, eta=0.5, seed=3).build_X(mutuality=0.5, seed=4)
        mask, M = net.R, N
        row0, nloc = shard_rows(N, 3, 1)
    elif case == "ego_nomut":
        L, N, K = 1, 600, 2
        net = syn.StandardSBM(N=N, L=L, K=K, C=2, avg_degree=6, seed=5).build_X(mutuality=0.3, seed=6)
        mask, M = net.R, N
        kw = dict(mutuality=False, split_e0=True)
    elif case in ("ego_subset_nodiag", "ego_subset_nodiag_k4_shard"):
        L, N, K, M = 2, 520, 4, 60
        net = syn.StandardSBM(N=N, M=M, L=L, K=K, C=2, avg_degree=6, seed=7).build_X(mutuality=0.4, seed=8)
        rep = np.zeros((L, M), dtype=np.uint8)
        rep[:, ::2] = 1
        mask = vm.masks.EgoMask(L, N, M, rep=rep, diag=False)  # X keeps entries of inactive reporters: outside R
        if case == "ego_subset_nodiag_k4_shard":  # rows >= M: no row node of the shard reports
            row0, nloc = shard_rows(N, 3, 2)
    elif case == "ego_empty_shard":  # every report that touches the shard's rows dropped: only its diagonal ties remain
        L, N, K = 1, 1100, 2
        net = syn.StandardSBM(N=N, L=L, K=K, C=2, avg_degree=10, seed=10).build_X(mutuality=0.5, seed=20)
        mask, M = net.R, N
        row0, nloc = shard_rows(N, 3, 1)
        s = np.stack(net.X.subs)
        inside = lambda a: (a >= row0) & (a < row0 + nloc)  # noqa: E731
        keep = ~(inside(s[1]) | inside(s[2]))
        net.X = vm.sptensor.sptensor(tuple(s[:, keep]), np.asarray(net.X.vals)[keep], shape=net.X.shape)
    elif case in ("all_mask", "all_mask_shard"):
        L, N, K, M = 2, 300, 2, 16
        y = syn.StandardSBM(N=N, M=M, L=L, K=K, C=2, avg_degree=8, seed=5)
        X, _ = syn.dense_reporting_X(y, M=M, mutuality=0.4, seed=6)

        class Net:
            pass

        net = Net()
        net.X = X
        mask = vm.masks.AllMask(L, N, M)
        if case == "all_mask_shard":
            row0, nloc = shard_rows(N, 3, 1)
    else:  # no fast dense kernel (N below a column tile): no shortcut ties; every entry visited (split_e0 off)
        L, N, K = 1, 300, 2
        net = syn.StandardSBM(N=N, L=L, K=K, C=2, avg_degree=4, seed=1).build_X(mutuality=0.3, seed=2)
        mask, M = net.R, N
        kw = dict(mutuality=True, split_e0=False)
    subs, vals = _sorted_coo(net.X)
    a = _packing.pack_device(subs, vals, L, N, M, K, mask, "cuda", row0=row0, nloc=nloc, tile_h=32, **kw)
    b = _packing.pack_torch(subs, vals, L, N, M, K, mask, "cuda", row0=row0, nloc=nloc, tile_h=32, **kw)
    for f in ("L", "N", "M", "K", "row0", "nloc", "tile_w", "tile_h", "nct", "nrt", "U", "I", "I1", "IT", "n_cx", "n_gchunk",
              "n_ublk", "phi_chunk", "n_phichunk", "n_cxblk", "r_mode", "ego_diag", "simple_ok", "split_e0"):
        assert getattr(a, f) == getattr(b, f), f
    assert a.b_all == b.b_all
    assert a.sumX_owned == (b.sumX_owned if b.sumX_owned is not None else b.sumX)
    skip = {"u_key", "e1_idx", "g_perm", "e_src"}
    for name in sorted(set(b.t) - skip):
        assert name in a.t, name
        x, y = a.t[name].cpu().numpy(), b.t[name].cpu().numpy()
        assert x.shape == y.shape, (name, x.shape, y.shape)
        assert np.array_equal(x, y), name
    assert np.array_equal(a.entry_src.cpu().numpy(), b.entry_src.cpu().numpy())
    assert int(a.t["u_single"].sum()) > 0 or case in ("ego_nomut", "all_mask", "ego_no_shortcut", "all_mask_shard",
                                                      "ego_empty_shard")
    if case == "ego_empty_shard":
        assert a.I == 0 and a.U == nloc and a.n_cx == a.U
    if case == "ego_subset_nodiag_k4_shard":
        assert a.row0 >= M and a.I > 0


def _assert_same_packing(a, b, src_a, src_b, tag):
    """Two packings of one shard from different inputs: every array equal; the packed entries come from the same entries
    of the whole list (`src_*` maps a position in each input to the whole list)."""
    for f in ("U", "I", "I1", "IT", "n_cx", "n_gchunk", "n_ublk", "n_phichunk", "n_cxblk", "simple_ok"):
        assert getattr(a, f) == getattr(b, f), (f, tag)
    assert a.b_all == b.b_all and a.sumX_owned == b.sumX_owned, tag
    assert set(a.t) == set(b.t), tag
    for name in sorted(set(a.t) - {"e_src"}):
        x, y = a.t[name].cpu().numpy(), b.t[name].cpu().numpy()
        assert x.shape == y.shape and np.array_equal(x, y), (name, tag)
    assert np.array_equal(src_a[a.entry_src.cpu().numpy()], src_b[b.entry_src.cpu().numpy()]), tag


@pytest.mark.parametrize("kind", ["ego", "all"])
def test_vm_pack_of_a_shard_from_its_own_rows_and_reciprocals(kind):
    """A shard packed from the entries of its own rows plus the reciprocal entries of other rows (in the order
    `_exchange_reciprocals` delivers them: own entries, then the received ones by sending rank; and as
    `device_reports(..., emit_transposed=True)` generates them) is the shard packed from the whole list."""
    torch = _cuda()
    import vimure_b200 as vm
    import vimure_b200.synthetic as syn
    from vimure_b200._pack_native import pack_device
    from vimure_b200.model import shard_rows

    W, r = 3, 1
    if kind == "ego":
        L, N, M, K = 2, 1100, 1100, 3
        net = syn.Multitensor(N=N, L=L, K=K, C=2, avg_degree=8, eta=0.5, seed=3).build_X(mutuality=0.5, seed=4)
        mask = net.R
    else:
        L, N, M, K = 2, 600, 16, 2
        net = syn.StandardSBM(N=N, M=M, L=L, K=K, C=2, avg_degree=8, seed=5)
        net.X, _ = syn.dense_reporting_X(net, M=M, mutuality=0.4, seed=6)
        mask = vm.masks.AllMask(L, N, M)
    row0, nloc = shard_rows(N, W, r)
    kw = dict(row0=row0, nloc=nloc, tile_h=128)
    # 1. a host list: the whole of it, and the shard's own entries followed by the reciprocals it receives
    s, v = np.stack(net.X.subs).astype(np.int64), np.asarray(net.X.vals).astype(np.int64)
    owner = np.searchsorted(np.array([shard_rows(N, W, q)[0] for q in range(1, W)]), s[1], side="right")
    col_owner = np.searchsorted(np.array([shard_rows(N, W, q)[0] for q in range(1, W)]), s[2], side="right")
    own = np.nonzero(owner == r)[0]
    recv = np.nonzero((col_owner == r) & (owner != r))[0]
    recv = recv[np.argsort(owner[recv], kind="stable")]
    sel = np.concatenate([own, recv])
    assert len(recv) and len(own)
    a = pack_device(s, v, L, N, M, K, mask, "cuda", **kw)
    b = pack_device(s[:, sel], v[sel], L, N, M, K, mask, "cuda", **kw)
    _assert_same_packing(a, b, np.arange(len(v)), sel, f"{kind}: own rows + received reciprocals")
    # 2. the device generator: the shard's rows with their transposed entries, against the whole generated list
    theta = np.random.RandomState(7).gamma(2.0, 0.5, size=(L, M))
    gen = dict(mask=mask) if kind == "all" else {}
    fs, fv = syn.device_reports(L, N, M, K, net.Y_subs, net.Y_vals, theta, 0.4, 17, **gen)
    ps, pv = syn.device_reports(L, N, M, K, net.Y_subs, net.Y_vals, theta, 0.4, 17, row0=row0, nloc=nloc,
                                emit_transposed=True, **gen)
    fk = (((fs[0].long() * N + fs[1]) * N + fs[2]) * M + fs[3]).cpu().numpy()
    pk = (((ps[0].long() * N + ps[1]) * N + ps[2]) * M + ps[3]).cpu().numpy()
    o = np.argsort(fk)
    pos = o[np.searchsorted(fk[o], pk)]
    assert np.array_equal(fk[pos], pk) and np.array_equal(fv.cpu().numpy()[pos], pv.cpu().numpy())
    a = pack_device(fs, fv, L, N, M, K, mask, "cuda", **kw)
    b = pack_device(ps, pv, L, N, M, K, mask, "cuda", **kw)
    _assert_same_packing(a, b, np.arange(fk.size), pos, f"{kind}: device_reports(emit_transposed=True)")
    torch.cuda.synchronize()


def test_vm_pack_reports_bad_input():
    _cuda()
    import vimure_b200 as vm
    from vimure_b200 import _packing

    mask = vm.masks.EgoMask(1, 50, 50)
    subs = np.array([[0, 0], [1, 1], [2, 2], [1, 1]])
    with pytest.raises(ValueError, match="Duplicate entries"):
        _packing.pack_device(subs, np.array([1, 2]), 1, 50, 50, 2, mask, "cuda")
    subs = np.array([[0], [1], [50], [1]])
    with pytest.raises(ValueError, match="outside its shape"):
        _packing.pack_device(subs, np.array([1]), 1, 50, 50, 2, mask, "cuda")
    # an empty network packs (only the diagonal ties of the ego mask are special)
    P = _packing.pack_device(np.zeros((4, 0), dtype=np.int64), np.zeros(0, dtype=np.int64), 1, 50, 50, 2, mask, "cuda")
    assert P.U == 50 and P.I == 0 and P.I1 == 0 and P.IT == 0


def test_pack_and_iterate_without_the_torch_packer():
    """A host that never runs the torch packer (it is made to raise): vm_pack + the engine, against a golden of the
    reference."""
    _cuda()
    code = r'''
import sys
sys.path.insert(0, %r)
import numpy as np
from tests.golden_util import Golden
import vimure_b200._pack_native as pn
import vimure_b200._packing as pk
def boom(*a, **k):
    raise AssertionError("the torch packer was used")
pk.pack_torch = pk.pack = boom
from vimure_b200._engine import CaviEngine
from vimure_b200 import masks
g = Golden("sbm_n520")
mask = masks.EgoMask(g.L, g.N, g.M, rep=g.R_spec["rep"], diag=g.R_spec["diag"])
P = pn.pack_device(g.X_subs, g.X_vals, g.L, g.N, g.M, g.K, mask, "cuda", tile_h=128)
eng = CaviEngine(P, g.priors(), mutuality=True, eps=1e-12)
st = g.init_state()
flat = P.t["u_gflat"].cpu().numpy()
pr_u = np.zeros((P.U, g.K)); pr_u[:, 0] = 1.0
ties = st["pr_ties"]
tf = (ties[:, 0] * g.N + ties[:, 1]) * g.N + ties[:, 2]
o = np.argsort(tf)
pos = np.minimum(np.searchsorted(tf[o], flat), len(tf) - 1)
hit = tf[o][pos] == flat
pr_u[hit] = st["pr_vals"][o][pos[hit]]
eng.set_state(st["gamma_shp"], st["gamma_rte"], st["phi_shp"], st["phi_rte"], st["nu_shp"],
              g.priors()["beta_eta"] + g.X_vals.sum(), pr_u, 1e-12)
for it in range(g.n_iter):
    eng.iterate(1, elbo_last=(it == g.n_iter - 1))
p = eng.params()
np.testing.assert_allclose(p["gamma_shp"], g.z["it_gamma_shp"][-1], rtol=1e-5)
np.testing.assert_allclose(p["phi_rte"], g.z["it_phi_rte"][-1], rtol=1e-5)
np.testing.assert_allclose(eng.elbo(), g.z["it_elbo"][-1], rtol=1e-6)
print("OK")
''' % ROOT
    r = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0 and "OK" in r.stdout, r.stdout + r.stderr
