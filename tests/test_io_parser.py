"""Edgelist parser (vimure_b200.io) -- CPU only."""
import warnings

import numpy as np
import pandas as pd
import pytest

from tests.golden_util import Golden


def _coo_set(subs, vals):
    return set(zip(*[np.asarray(s).tolist() for s in subs], np.asarray(vals).tolist()))


def test_round_trip_from_fixture():
    import vimure_b200 as vm
    from vimure_b200.io import read_from_edgelist

    g = Golden("gm_l2_k3")
    l, i, j, m = g.X_subs
    df = pd.DataFrame({"ego": [f"n{a:03d}" for a in i], "alter": [f"n{a:03d}" for a in j],
                       "reporter": [f"n{a:03d}" for a in m], "layer": [f"L{a}" for a in l], "weight": g.X_vals})
    nodes = [f"n{a:03d}" for a in range(g.N)]
    with warnings.catch_warnings(record=True) as w:
        warnings.simplefilter("always")
        net = read_from_edgelist(df, nodes=nodes, reporters=nodes, is_weighted=True)
    assert any("Reporters Mask was not informed" in str(x.message) for x in w)
    assert any("Parameter K was None" in str(x.message) for x in w)
    assert net.X.shape == (g.L, g.N, g.N, g.N) and net.K == int(g.X_vals.max()) + 1
    assert _coo_set(net.X.subs, net.X.vals) == _coo_set(g.X_subs, g.X_vals)
    assert isinstance(net.R, vm.masks.EgoMask) and not net.R.diag and net.R.rep.all()
    # unweighted: counts collapse to 1
    net2 = read_from_edgelist(df, nodes=nodes, reporters=nodes, K=2)
    assert set(np.unique(net2.X.vals)) == {1}


def test_errors_and_warnings():
    from vimure_b200.io import read_from_edgelist

    df = pd.DataFrame({"ego": ["a", "b"], "alter": ["b", "c"], "reporter": ["a", "b"]})
    with pytest.raises(ValueError, match="Required columns not found"):
        read_from_edgelist(df.rename(columns={"ego": "from"}))
    with pytest.raises(ValueError, match="'nodes' should be a list"):
        read_from_edgelist(df, nodes={"a", "b", "c"})
    with pytest.raises(ValueError, match="does not contain all nodes"):
        read_from_edgelist(df, nodes=["a", "b"])
    with pytest.raises(ValueError, match="do not appear in the list of reporters"):
        read_from_edgelist(df, nodes=["a", "b", "c"], reporters=["a"])
    with pytest.warns(UserWarning):
        net = read_from_edgelist(df)
    assert (net.L, net.N, net.M) == (1, 3, 3)
    # undirected: symmetrised per reporter
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        net = read_from_edgelist(df, is_undirected=True, K=2)
    s = _coo_set(net.X.subs, net.X.vals)
    assert (0, 0, 1, 0, 1) in s and (0, 1, 0, 0, 1) in s and (0, 1, 2, 1, 1) in s and (0, 2, 1, 1, 1) in s


def test_matches_reference_parser_on_karnataka():
    """The golden fixture karnataka_vil1 holds the reference parser's output on Karnataka village 1 (X and the reporter
    mask, oracle/gen_golden.py).  The same reports as an edgelist -- node ids that do not sort like their indices,
    rows in random order -- must parse to exactly that X and mask."""
    from vimure_b200.io import read_from_edgelist

    g = Golden("karnataka_vil1")
    rng = np.random.RandomState(1)
    names = [str(v) for v in 1000 + rng.permutation(10 * g.N)[: g.N]]
    l, i, j, m = g.X_subs
    df = pd.DataFrame({"ego": [names[a] for a in i], "alter": [names[a] for a in j],
                       "reporter": [names[a] for a in m], "layer": ["layer%d" % a for a in l]})
    df = df.iloc[rng.permutation(len(df))].reset_index(drop=True)
    rep = g.R_spec["rep"].astype(bool)
    assert (rep == rep[0]).all()  # every layer has the same reporters
    nodes, reporters = names, [names[a] for a in rng.permutation(np.nonzero(rep[0])[0])]
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        got = read_from_edgelist(df, nodes=nodes, reporters=reporters, K=2)
    # the fixture's M is X.shape[3]; the parser's M counts the reporters
    assert got.X.shape == (g.L, g.N, g.N, g.M) and (got.L, got.N, got.M, got.K) == (g.L, g.N, len(reporters), g.K)
    assert _coo_set(got.X.subs, got.X.vals) == _coo_set(g.X_subs, g.X_vals)
    subs, _ = g.R_coo()
    k_ref = np.sort(np.ravel_multi_index(tuple(subs), (g.L, g.N, g.N, g.M)))
    R2 = got.R.to_sptensor()
    k_got = np.sort(np.ravel_multi_index(R2.subs, R2.shape))
    assert np.array_equal(k_ref, k_got)
