"""Loading of the golden fixtures in tests/golden (made by oracle/gen_golden.py from the reference)."""
import json
import os

import numpy as np

GOLDEN_DIR = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
ALL_FIXTURES = ["f1_over", "f1_under", "sbm_k3", "gm_l2_k3", "nomut", "dense_reporting", "custom_mask",
                "karnataka_vil1", "rho_prior", "undirected", "sbm_n520", "gm_n640_l2_k3"]
# fixtures large enough (N >= the dense kernel's column tile of 512) to reach the fast dense kernel and its shortcut ties
LARGE_FIXTURES = ["sbm_n520", "gm_n640_l2_k3"]


class Golden:
    def __init__(self, name):
        z = np.load(os.path.join(GOLDEN_DIR, name + ".npz"), allow_pickle=False)
        self.name = name
        self.z = z
        self.L, self.N, self.M, self.K = (int(v) for v in z["dims"])
        self.X_subs = z["X_subs"].astype(np.int64)
        self.X_vals = z["X_vals"]
        meta = json.loads(str(z["meta_json"]))
        self.model_kwargs = meta["model_kwargs"]
        self.fit_kwargs = meta["fit_kwargs"]
        for k in z.files:
            if k.startswith("fitarr_"):
                self.fit_kwargs[k[len("fitarr_"):]] = z[k]
        for k in ("theta_prior", "lambda_prior", "eta_prior"):
            if k in self.fit_kwargs:
                self.fit_kwargs[k] = tuple(self.fit_kwargs[k])
        kind = str(z["R_kind"])
        self.R_spec = {"kind": kind, "dense_input": bool(z["R_dense_input"])}
        if kind == "ego":
            self.R_spec["diag"] = bool(z["R_diag"])
            self.R_spec["rep"] = z["R_rep"]
        elif kind == "coo":
            self.R_spec["subs"] = z["R_subs"].astype(np.int64)
            self.R_spec["vals"] = z["R_vals"]
        self.mutuality = bool(self.model_kwargs.get("mutuality", True)) and not self.model_kwargs.get("undirected", False)
        self.n_iter = len(z["it_elbo"])

    # priors as the reference resolves them (model.py:238-317)
    def priors(self):
        fk = self.fit_kwargs
        tp = fk.get("theta_prior", (0.1, 0.1))
        lp = fk.get("lambda_prior", (10.0, 10.0))
        ep = fk.get("eta_prior", (0.5, 1.0))
        return dict(
            alpha_theta=fk.get("alpha_theta", tp[0]), beta_theta=fk.get("beta_theta", tp[1]),
            alpha_lambda=fk.get("alpha_lambda", lp[0]), beta_lambda=fk.get("beta_lambda", lp[1]),
            alpha_eta=ep[0], beta_eta=ep[1],
        )

    def init_state(self):
        z = self.z
        return dict(
            gamma_shp=z["init_gamma_shp"], gamma_rte=z["init_gamma_rte"], phi_shp=z["init_phi_shp"],
            phi_rte=z["init_phi_rte"], nu_shp=float(z["init_nu_shp"]),
            pr_ties=z["init_pr_ties"].astype(np.int64), pr_vals=self.init_pr_vals(),
        )

    def init_pr_vals(self):
        """Prior of the ties `init_pr_ties`.  Large fixtures store the reference's seed instead of the values
        (oracle/gen_golden.py, shrink_fixture): the draw is redone and checked against the rows kept."""
        from oracle.gen_golden import reference_prior

        z = self.z
        if "init_pr_vals" in z.files:
            return z["init_pr_vals"]
        pr = reference_prior(int(z["init_pr_seed"]), self.L, self.N, self.K, z["init_pr_ties"].astype(np.int64))
        head = z["init_pr_vals_head"]
        assert np.array_equal(pr[: len(head)], head), "redrawn prior differs from the stored rows"
        return pr

    def R_coo(self):
        """Explicit COO (subs (4,nnz), vals) of the mask -- for feeding the public API."""
        L, N, M = self.L, self.N, self.M
        spec = self.R_spec
        if spec["kind"] == "coo":
            return spec["subs"], spec["vals"]
        if spec["kind"] == "all":
            l, i, j, m = np.meshgrid(np.arange(L), np.arange(N), np.arange(N), np.arange(M), indexing="ij")
            subs = np.stack([l.ravel(), i.ravel(), j.ravel(), m.ravel()])
            return subs, np.ones(subs.shape[1])
        rep = spec["rep"].astype(bool)
        out = []
        for l in range(L):
            for m in np.nonzero(rep[l])[0]:
                others = np.array([n for n in range(N) if n != m])
                rows = np.stack([np.full(N - 1, l), np.full(N - 1, m), others, np.full(N - 1, m)])
                cols = np.stack([np.full(N - 1, l), others, np.full(N - 1, m), np.full(N - 1, m)])
                out += [rows, cols]
                if spec["diag"]:
                    out.append(np.array([[l], [m], [m], [m]]))
        subs = np.concatenate(out, axis=1)
        return subs, np.ones(subs.shape[1])
