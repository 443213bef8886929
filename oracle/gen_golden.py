"""Generates the golden vectors under `tests/golden/` by running the UNMODIFIED reference
(`/root/reference`, through `oracle/ref_runner.py`).  TEST INFRASTRUCTURE ONLY.

Run in the build container (the only place `/root/reference` exists):

    python oracle/gen_golden.py [scenario ...]

Each fixture `tests/golden/<name>.npz` holds the inputs (X in COO form, the reporter mask R as a
structure spec or COO, priors / fit kwargs), the initial state the reference drew (so that it can be
injected), and the state after every CAVI iteration (gamma/phi/nu and the ELBO evaluated every
iteration) plus the final rho.  The reference has no per-iteration golden vectors of its own
(SURVEY.md section 8c); its only known answers (the F1 assertions of `test_model.py:188,261,334`)
are reproduced in the `f1_*` scenarios and stored alongside.
"""
import json
import os
import sys
import warnings

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
sys.path.insert(0, ROOT)

from oracle.ref_runner import import_reference, run_reference_trace  # noqa: E402

GOLDEN_DIR = os.path.join(ROOT, "tests", "golden")


def describe_R(R, L, N, M):
    """Return a compact spec of the reporter mask: ego / all / coo."""
    if isinstance(R, np.ndarray):
        Rd = np.asarray(R)
        if np.all(Rd == 1):
            return {"kind": "all"}
        subs = np.nonzero(Rd)
        vals = Rd[subs]
    else:
        subs = tuple(np.asarray(s) for s in R.subs)
        vals = np.asarray(R.vals)
    l, i, j, m = subs
    if np.all(vals == 1) and np.all((i == m) | (j == m)):
        # candidate ego mask: per (l, m) either a full cross (with or without the (m,m) tie) or nothing
        diag_cnt = np.count_nonzero((i == m) & (j == m))
        cnt = np.zeros((L, M), dtype=np.int64)
        np.add.at(cnt, (l, m), 1)
        rep = cnt > 0
        for diag in (True, False):
            full = 2 * N - 1 if diag else 2 * N - 2
            if np.all(cnt[rep] == full) and diag_cnt == (rep.sum() if diag else 0):
                key = np.unique(np.stack([l, i, j, m]), axis=1)
                if key.shape[1] == len(l):
                    return {"kind": "ego", "diag": bool(diag), "rep": rep.astype(np.uint8)}
    return {"kind": "coo", "subs": np.stack(subs).astype(np.int32), "vals": vals.astype(np.float64)}


def save_fixture(name, X, R, L, N, M, K, model_kwargs, fit_kwargs, rec, extra=None, keep_rho="final"):
    os.makedirs(GOLDEN_DIR, exist_ok=True)
    out = {}
    out["dims"] = np.array([L, N, M, K], dtype=np.int64)
    out["X_subs"] = np.stack([np.asarray(s) for s in X.subs]).astype(np.int32)
    out["X_vals"] = np.asarray(X.vals).astype(np.int64)
    spec = describe_R(R, L, N, M)
    out["R_kind"] = np.array(spec["kind"])
    if spec["kind"] == "ego":
        out["R_diag"] = np.array(spec["diag"])
        out["R_rep"] = spec["rep"]
    elif spec["kind"] == "coo":
        out["R_subs"] = spec["subs"]
        out["R_vals"] = spec["vals"]
    out["R_dense_input"] = np.array(isinstance(R, np.ndarray))

    meta = {"model_kwargs": model_kwargs, "fit_kwargs": {}}
    for k, v in fit_kwargs.items():
        if k == "R":
            continue
        if isinstance(v, np.ndarray):
            out["fitarr_" + k] = v
        else:
            meta["fit_kwargs"][k] = v
    out["meta_json"] = np.array(json.dumps(meta))

    init = rec["init"]
    for k in ("gamma_shp", "gamma_rte", "phi_shp", "phi_rte"):
        out["init_" + k] = init[k]
    out["init_nu_shp"] = np.array(init["nu_shp"])
    out["init_nu_rte"] = np.array(init["nu_rte"])
    # the prior differs from the one-hot [1,0,..] only on ties that carry an X entry and an R entry
    pr = init["pr_rho"]
    onehot = np.zeros(K)
    onehot[0] = 1.0
    special = np.argwhere(np.any(pr != onehot, axis=-1))
    out["init_pr_ties"] = special.astype(np.int32)  # (n,3) l,i,j
    out["init_pr_vals"] = pr[special[:, 0], special[:, 1], special[:, 2], :]

    its = rec["iters"]
    for k in ("gamma_shp", "gamma_rte", "phi_shp", "phi_rte"):
        out["it_" + k] = np.stack([it[k] for it in its])
    out["it_nu_shp"] = np.array([it["nu_shp"] for it in its])
    out["it_elbo"] = np.array([it["elbo"] for it in its])
    rho_final = its[-1]["rho"]
    if keep_rho == "final":
        out["rho_final"] = rho_final
    else:  # large: keep the union ties only + summary statistics
        l, i, j = (np.asarray(s) for s in X.subs[:3])
        ties = np.unique(np.stack([l, i, j]), axis=1).T
        out["rho_final_ties"] = ties.astype(np.int32)
        out["rho_final_vals"] = rho_final[ties[:, 0], ties[:, 1], ties[:, 2], :]
        out["rho_final_colsum"] = rho_final.sum(axis=1)
        out["rho_final_rowsum"] = rho_final.sum(axis=2)
    out["rho_argmax_sum"] = np.array(int(np.argmax(rho_final, axis=-1).sum()))
    model = rec["model"]
    out["trace"] = model.trace[["realisation", "iter", "elbo", "reached_convergence"]].to_numpy(dtype=float)
    out["maxL"] = np.array(float(model.maxL))
    if extra:
        out.update(extra)
    path = os.path.join(GOLDEN_DIR, name + ".npz")
    np.savez_compressed(path, **out)
    print("wrote", path, os.path.getsize(path) // 1024, "KiB", "iters", len(its), "elbo[-1]", its[-1]["elbo"])


def reference_prior(seed, L, N, K, ties):
    """The reference's random prior of `ties` ((n, 3) l,i,j): `1 + 0.01 * RandomState(seed).rand(L, N, N, K)` normalised
    per tie (model.py:470-472, bias0 = 0), the first draw of the fit's stream."""
    d = np.random.RandomState(int(seed)).rand(L, N, N, K)
    pr = 1.0 + 0.01 * d[ties[:, 0], ties[:, 1], ties[:, 2]]
    return pr / pr.sum(axis=-1)[:, None]


def shrink_fixture(name, rho_fraction=0.5, check_rows=64):
    """Keep a fixture under 1 MB: the random prior is replaced by its seed (redrawn by tests/golden_util.py and checked
    against its first `check_rows` rows, which stay stored), and the final rho is kept on a seeded sample of
    `rho_fraction` of the ties (the column/row sums and the argmax sum still cover all of them)."""
    path = os.path.join(GOLDEN_DIR, name + ".npz")
    z = np.load(path)
    out = {k: z[k] for k in z.files}
    L, N, M, K = (int(v) for v in z["dims"])
    seed = json.loads(str(z["meta_json"]))["fit_kwargs"]["seed"]
    pr = reference_prior(seed, L, N, K, z["init_pr_ties"].astype(np.int64))
    assert np.array_equal(pr, z["init_pr_vals"]), "the stored prior is not the seed's first draw"
    del out["init_pr_vals"]
    out["init_pr_seed"] = np.array(seed, dtype=np.int64)
    out["init_pr_vals_head"] = z["init_pr_vals"][:check_rows]
    n = len(z["rho_final_ties"])
    keep = np.sort(np.random.RandomState(0).choice(n, int(rho_fraction * n), replace=False))
    out["rho_final_ties"] = z["rho_final_ties"][keep]
    out["rho_final_vals"] = z["rho_final_vals"][keep]
    np.savez_compressed(path, **out)
    print("shrunk", path, os.path.getsize(path) // 1024, "KiB")


def scenario_f1(vm, exaggeration):
    """`test_model.py:117-188` (over) / `:263-334` (under): the reference's only known answers."""
    from sklearn.metrics import f1_score

    seed, eta, K = 25, 0.2, 2
    gt = vm.synthetic.Multitensor(N=100, M=100, L=1, C=2, K=K, avg_degree=5, sparsify=True, seed=seed,
                                  ExpM=None, eta=eta)
    theta = vm.synthetic.build_custom_theta(gt_network=gt, theta_ratio=0.1, exaggeration_type=exaggeration,
                                            seed=seed)
    gt._build_X(mutuality=eta, theta=theta, cutoff_X=False, lambda_diff=0.99, flag_self_reporter=True, seed=seed)
    lam = np.array([[0.01, 1.0]])
    beta_lambda = 10000 * np.ones(lam.shape)
    alpha_lambda = lam * beta_lambda
    fit_kwargs = dict(K=K, seed=seed, theta_prior=(0.1, 0.1), eta_prior=(0.5, 1.0), alpha_lambda=alpha_lambda,
                      beta_lambda=beta_lambda, max_iter=21, R=gt.R)
    model_kwargs = dict(mutuality=True)
    rec = run_reference_trace(gt.X, fit_kwargs, model_kwargs)
    # the full 2-realisation fit of the reference test, for the F1 known answer
    m = vm.model.VimureModel(mutuality=True)
    fk = dict(fit_kwargs)
    fk["num_realisations"] = 2
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        m.fit(gt.X, **fk)
    Y_true = gt.Y.toarray()[0].flatten()
    Y_rec = vm.utils.apply_rho_threshold(m, threshold=0.5)[0].flatten()
    f1 = f1_score(Y_true, Y_rec)
    extra = {
        "Y_true": (gt.Y.toarray()[0] > 0).astype(np.uint8),
        "ref_f1": np.array(f1),
        "ref2_trace": m.trace[["realisation", "seed", "iter", "elbo", "reached_convergence"]].to_numpy(dtype=float),
        "ref2_maxL": np.array(float(m.maxL)),
        "ref2_nu_shp_f": np.array(float(m.nu_shp_f)),
        "ref2_gamma_shp_f": m.gamma_shp_f,
        "ref2_phi_shp_f": m.phi_shp_f,
    }
    print("F1", exaggeration, f1, "maxL", m.maxL)
    save_fixture("f1_" + exaggeration, gt.X, gt.R, 1, 100, 100, K, model_kwargs, fit_kwargs, rec, extra)


def scenario_sbm_k3(vm):
    """`test_model.py:59-84`: StandardSBM N=20 M=20 K=3, default priors (default convergence rule)."""
    gt = vm.synthetic.StandardSBM(N=20, M=20, L=1, K=3, C=2, avg_degree=2, sparsify=False)
    gt._build_X(flag_self_reporter=True)
    fit_kwargs = dict(K=3, seed=3, max_iter=60, R=gt.R)
    rec = run_reference_trace(gt.X, fit_kwargs, {})
    save_fixture("sbm_k3", gt.X, gt.R, 1, 20, 20, 3, {}, fit_kwargs, rec)


def scenario_gm_l2_k3(vm):
    gt = vm.synthetic.Multitensor(N=60, M=60, L=2, C=2, K=3, avg_degree=6, sparsify=True, seed=7, eta=0.5)
    gt._build_X(mutuality=0.5, flag_self_reporter=True, seed=11)
    fit_kwargs = dict(K=3, seed=5, max_iter=25, R=gt.R)
    model_kwargs = dict(mutuality=True, convergence_tol=0.0)
    rec = run_reference_trace(gt.X, fit_kwargs, model_kwargs)
    save_fixture("gm_l2_k3", gt.X, gt.R, 2, 60, 60, 3, model_kwargs, fit_kwargs, rec)


def scenario_nomut(vm):
    gt = vm.synthetic.StandardSBM(N=50, M=50, L=1, K=2, C=2, avg_degree=4, sparsify=True, seed=4)
    gt._build_X(mutuality=0.0, flag_self_reporter=True, seed=4)
    fit_kwargs = dict(K=2, seed=9, max_iter=15, R=gt.R)
    model_kwargs = dict(mutuality=False, convergence_tol=0.0)
    rec = run_reference_trace(gt.X, fit_kwargs, model_kwargs)
    save_fixture("nomut", gt.X, gt.R, 1, 50, 50, 2, model_kwargs, fit_kwargs, rec)


def scenario_dense_reporting(vm):
    """All reporters report all ties: R is a dense all-ones array (the `dtensor` branches,
    `model.py:706-709, 737-738, 766-769, 1251-1252`)."""
    gt = vm.synthetic.StandardSBM(N=30, M=8, L=2, K=2, C=2, avg_degree=4, sparsify=True, seed=2)
    gt._build_X(mutuality=0.3, flag_self_reporter=False, seed=2)
    R = np.ones((2, 30, 30, 8))
    fit_kwargs = dict(K=2, seed=8, max_iter=15, R=R)
    model_kwargs = dict(mutuality=True, convergence_tol=0.0)
    rec = run_reference_trace(gt.X, fit_kwargs, model_kwargs)
    save_fixture("dense_reporting", gt.X, R, 2, 30, 8, 2, model_kwargs, fit_kwargs, rec)


def scenario_custom_mask(vm):
    """A general sparse mask (random subset of reporters per tie), with some X entries outside R
    and a few ties reported by nobody (`model.py:536-545`)."""
    import sktensor as skt

    gt = vm.synthetic.StandardSBM(N=40, M=10, L=2, K=2, C=2, avg_degree=4, sparsify=True, seed=6)
    gt._build_X(mutuality=0.4, flag_self_reporter=False, seed=6)
    prng = np.random.RandomState(123)
    Rd = (prng.rand(2, 40, 40, 10) < 0.3).astype(int)
    subs = np.nonzero(Rd)
    R = skt.sptensor(subs, Rd[subs], shape=Rd.shape, dtype=int)
    fit_kwargs = dict(K=2, seed=12, max_iter=15, R=R)
    model_kwargs = dict(mutuality=True, convergence_tol=0.0)
    rec = run_reference_trace(gt.X, fit_kwargs, model_kwargs)
    save_fixture("custom_mask", gt.X, R, 2, 40, 10, 2, model_kwargs, fit_kwargs, rec)


def scenario_karnataka(vm):
    """BASELINE config 2: Karnataka vil1, all 4 layers, via the reference edgelist parser
    (`test/__init__.py:18-28`, `_io.py:132`)."""
    sys.path.insert(0, "/root/reference/notebooks/python/experiments/")
    from karnataka import read_village_data  # type: ignore

    df, nodes, reporters = read_village_data(
        "vil1", data_folder="/root/reference/data/input/india_microfinance/formatted/", print_details=False)
    df.rename(columns={"Ego": "ego", "Alter": "alter"}, inplace=True)
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        net = vm._io.read_from_edgelist(df, nodes=list(nodes), reporters=list(reporters), K=2)
    L, N, M = net.L, net.N, net.X.shape[3]
    fit_kwargs = dict(K=2, seed=1, max_iter=12, R=net.R)
    model_kwargs = dict(mutuality=True, convergence_tol=0.0)
    rec = run_reference_trace(net.X, fit_kwargs, model_kwargs)
    save_fixture("karnataka_vil1", net.X, net.R, L, N, M, 2, model_kwargs, fit_kwargs, rec, keep_rho="summary")


def scenario_rho_prior(vm):
    """User-supplied rho_prior (`model.py:485-500`)."""
    gt = vm.synthetic.StandardSBM(N=30, M=30, L=1, K=3, C=2, avg_degree=3, sparsify=True, seed=13)
    gt._build_X(mutuality=0.2, flag_self_reporter=True, seed=13)
    Xd = gt.X.toarray()
    rho_prior = Xd.sum(axis=-1).astype(float) / 2.0
    fit_kwargs = dict(K=3, seed=21, max_iter=12, R=gt.R, rho_prior=rho_prior)
    model_kwargs = dict(mutuality=True, convergence_tol=0.0)
    rec = run_reference_trace(gt.X, fit_kwargs, model_kwargs)
    save_fixture("rho_prior", gt.X, gt.R, 1, 30, 30, 3, model_kwargs, fit_kwargs, rec)


def scenario_undirected(vm):
    """undirected=True (model.py:58-65, 127-132, 477-478): symmetric dense X, mutuality forced off, symmetrised prior."""
    gt = vm.synthetic.StandardSBM(N=30, M=30, L=1, K=2, C=2, avg_degree=4, sparsify=True, seed=17)
    gt._build_X(mutuality=0.0, flag_self_reporter=True, seed=17)
    Xd = gt.X.toarray()
    Xs = np.maximum(Xd, np.transpose(Xd, axes=(0, 2, 1, 3)))
    fit_kwargs = dict(K=2, seed=31, max_iter=12, R=gt.R)
    model_kwargs = dict(undirected=True, convergence_tol=0.0)
    rec = run_reference_trace(Xs, fit_kwargs, model_kwargs)
    X = rec["model"].X
    save_fixture("undirected", X, gt.R, 1, 30, 30, 2, model_kwargs, fit_kwargs, rec)


def scenario_sbm_n520(vm):
    """N >= the dense kernel's column tile (512 at K=2): the fast dense kernel, the simple-tie shortcut and the partial
    last tile are compared with the REFERENCE itself, not only with the oracle (VERDICT r1, item 5a)."""
    gt = vm.synthetic.StandardSBM(N=520, M=520, L=1, K=2, C=2, avg_degree=8, sparsify=True, seed=10)
    gt._build_X(mutuality=0.5, flag_self_reporter=True, seed=20)
    fit_kwargs = dict(K=2, seed=1, max_iter=12, R=gt.R)
    model_kwargs = dict(mutuality=True, convergence_tol=0.0)
    rec = run_reference_trace(gt.X, fit_kwargs, model_kwargs)
    save_fixture("sbm_n520", gt.X, gt.R, 1, 520, 520, 2, model_kwargs, fit_kwargs, rec, keep_rho="summary")


def scenario_gm_n640_l2_k3(vm):
    """Config 5's law (Multitensor / GMReciprocity, L > 1, K = 3) at a size that reaches the K = 3 fast dense kernel
    (column tile 512) with a partial last tile."""
    gt = vm.synthetic.Multitensor(N=640, M=640, L=2, C=2, K=3, avg_degree=8, sparsify=True, seed=7, eta=0.5)
    gt._build_X(mutuality=0.5, flag_self_reporter=True, seed=11)
    fit_kwargs = dict(K=3, seed=5, max_iter=11, R=gt.R)
    model_kwargs = dict(mutuality=True, convergence_tol=0.0)
    rec = run_reference_trace(gt.X, fit_kwargs, model_kwargs)
    save_fixture("gm_n640_l2_k3", gt.X, gt.R, 2, 640, 640, 3, model_kwargs, fit_kwargs, rec, keep_rho="summary")
    shrink_fixture("gm_n640_l2_k3")


SCENARIOS = {
    "f1_over": lambda vm: scenario_f1(vm, "over"),
    "f1_under": lambda vm: scenario_f1(vm, "under"),
    "sbm_k3": scenario_sbm_k3,
    "gm_l2_k3": scenario_gm_l2_k3,
    "nomut": scenario_nomut,
    "dense_reporting": scenario_dense_reporting,
    "custom_mask": scenario_custom_mask,
    "karnataka_vil1": scenario_karnataka,
    "rho_prior": scenario_rho_prior,
    "undirected": scenario_undirected,
    "sbm_n520": scenario_sbm_n520,
    "gm_n640_l2_k3": scenario_gm_n640_l2_k3,
}

if __name__ == "__main__":
    vm = import_reference()
    names = sys.argv[1:] or list(SCENARIOS)
    for n in names:
        print("== scenario", n)
        SCENARIOS[n](vm)
