"""The dense kernel that evaluates the shortcut ties itself (k_dense_sc) on row segments with many of them: a hub whose
segments of one column tile carry more than 32 and more than 64 shortcut ties (the kernel's per-lane loop over a
segment's ties), next to segments without special ties.  Against the CPU oracle and the fp64 path (VM_NO_SIMPLE=1);
the slab must equal rho_u32 at every special tie."""
import os

import numpy as np
import pytest

from tests.test_gpu_scaled import _cuda, _engine_and_oracle

pytestmark = pytest.mark.gpu


def _hub_network(N=1100, K=2):
    import vimure_b200 as vm
    import vimure_b200.synthetic as syn

    net = syn.StandardSBM(N=N, L=1, K=K, C=2, avg_degree=4, seed=11).build_X(mutuality=0.5, seed=21)
    s = np.stack(net.X.subs)
    vals = np.asarray(net.X.vals)
    # hubs: node 5 reports its ties to 100 nodes of the first column tile, node 9 to 40 nodes of the second (no
    # reciprocal reports: SIMPLE shortcut ties); rows 13 and 17 (the same warps' next rows) carry no entries, so
    # their only special tie is the diagonal
    hub = [(5, j) for j in range(20, 420, 4)] + [(9, j) for j in range(600, 1000, 10)]
    quiet = np.isin(s[1], [13, 17]) | np.isin(s[2], [13, 17])
    s, vals = s[:, ~quiet], vals[~quiet]
    extra = np.array([[0, i, j, i] for i, j in hub], dtype=s.dtype).T
    s = np.concatenate([s, extra], axis=1)
    vals = np.concatenate([vals, np.full(extra.shape[1], 2, dtype=vals.dtype)])
    key = ((s[0] * N + s[1]) * N + s[2]) * N + s[3]
    _, first = np.unique(key, return_index=True)
    s, vals = s[:, np.sort(first)], vals[np.sort(first)]
    net.X = vm.sptensor.sptensor(tuple(s), vals, shape=(1, N, N, N))
    return net


def test_crowded_row_segments_in_the_fused_dense_kernel(monkeypatch):
    torch = _cuda()
    N, K = 1100, 2
    net = _hub_network(N, K)
    spec = {"kind": "ego", "rep": np.ones((1, N), dtype=np.uint8), "diag": True}
    eng, o, P = _engine_and_oracle(net, net.R, spec, K, tile_h=32)
    assert eng.simple_mode
    # the hub segments are as crowded as intended
    sc = (P.t["u_simple"] | P.t["u_single"]).cpu().numpy()
    row = P.t["u_lrow"].cpu().numpy()
    ct = P.t["u_col"].cpu().numpy() // 512
    per_seg = np.bincount((row * 3 + ct)[sc], minlength=N * 3)
    assert per_seg[5 * 3 + 0] > 64 and 32 < per_seg[9 * 3 + 1] <= 64
    quiet = np.isin(row, [13, 17])
    assert (P.t["u_col"].cpu().numpy()[quiet] == row[quiet]).all()  # their only special tie is the diagonal
    monkeypatch.setenv("VM_NO_SIMPLE", "1")
    ref, _, _ = _engine_and_oracle(net, net.R, None, K, tile_h=32)
    monkeypatch.delenv("VM_NO_SIMPLE")
    assert not ref.simple_mode

    u_row, u_col = P.t["u_lrow"].long(), P.t["u_col"].long()
    for step, (n, elbo) in enumerate(((1, False), (2, False), (2, True), (1, False))):
        for e in (eng, ref):
            e.iterate(n, elbo_last=elbo)
        for _ in range(n):
            o.iterate()
        lc = eng.layer_consts.cpu().numpy().reshape(1, 3 * K + 5)
        assert lc[0, 2 * K + 4] == 1.0  # the layer takes the shortcut
        p, q = eng.params(), ref.params()
        for k in ("gamma_shp", "gamma_rte", "phi_shp", "phi_rte", "nu_shp"):
            np.testing.assert_allclose(p[k], getattr(o, k), rtol=1e-5, err_msg=f"{k} vs oracle, step {step}")
            np.testing.assert_allclose(p[k], q[k], rtol=5e-6, err_msg=f"{k} vs fp64 path, step {step}")
        slab = eng.rho_slab()
        assert torch.equal(slab[0, u_row, u_col], eng.rho_u32), f"slab != rho_u32 at the special ties, step {step}"
        a = slab.cpu().numpy().astype(np.float64)
        np.testing.assert_allclose(a, o.rho, rtol=2e-5, atol=1e-30, err_msg=f"step {step}")
        np.testing.assert_allclose(a, ref.rho_slab().cpu().numpy(), rtol=1e-5, atol=1e-30, err_msg=f"step {step}")
    torch.cuda.synchronize()
