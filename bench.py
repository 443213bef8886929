#!/usr/bin/env python
"""Benchmark of the CAVI hot path (BASELINE.json metric: CAVI iter/s and ties/s at N=20k, % of HBM roofline; 1/2/4/8 B200).

    python bench.py --gpus N --steps K --warmup W            # this repo's CUDA path
    python bench.py --impl reference --gpus N --steps K ...  # the reference's CPU algorithm (numpy oracle port)
    python bench.py ... --dump-outputs DIR                   # also save what the last timed step computed, as .npy

A "step" is ONE CAVI iteration (reference `_update_CAVI`, model.py:623-660) over the whole synthetic network, with the
ELBO evaluated on the reference's cadence (iteration 1, every 10th, the last; model.py:1036) inside the timed region.

Headline workload (config 3 of BASELINE.json): StandardSBM law, N = 20 000 nodes, M = N ego-only reporters, L = 1,
K = 2, mutuality.  With G > 1 GPUs the ties are sharded by node-row blocks and the network is grown so that every GPU
keeps 4e8 ties ("weak" scaling): N = 20 000 * sqrt(G).  `value` = ties processed per second by the whole job
= steps * L * N^2 / time (max over ranks, CUDA events).

Second workload, reported under `configs.c5` of the same JSON line (config 5 of BASELINE.json): Multitensor /
"GMReciprocity" law, ego-only, L = 4, K = 3, weak-scaled so that 8 GPUs run N = 64 000 (N = 64 000 * sqrt(G/8):
22 628 on one GPU, 24.6 GB of posterior slab per GPU).

`parity`: before anything is timed, reference golden scenarios are fitted through `VimureModel.fit` on the very path
being benchmarked (NCCL row-block sharding when G > 1) and compared with the unmodified reference's trajectories.

Inputs come from the device-side generator (`vm_synth_ego`: counter-based RNG, every rank generates its own row block
and the reciprocal entries it needs, nothing is exchanged); the e2e figure feeds the SAME entries back in as pinned
host buffers through the public API.  Prints ONE JSON line on rank 0.
"""
import argparse
import json
import math
import os
import subprocess
import sys
import time
import warnings

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

BASE_N = 20000
C5_N8 = 64000
PRIORS = dict(alpha_theta=0.1, beta_theta=0.1, alpha_lambda=10.0, beta_lambda=10.0, alpha_eta=0.5, beta_eta=1.0)


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--nodes", type=int, default=0, help="override the number of nodes of the headline workload")
    ap.add_argument("--cpu-nodes", type=int, default=2048, help="nodes of the bounded CPU-baseline sample")
    ap.add_argument("--cpu-procs", type=int, default=0,
                    help="concurrent replicas of the CPU sample (0 = one per host core, at most 64)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-parity", action="store_true")
    ap.add_argument("--no-c5", action="store_true", help="skip the config-5 workload (configs.c5)")
    ap.add_argument("--c5-steps", type=int, default=None, help="timed steps of the config-5 workload (default: --steps)")
    ap.add_argument("--c5-nodes", type=int, default=0)
    ap.add_argument("--tile-h", type=int, default=128)
    ap.add_argument("--trace", action="store_true", help="print per-batch device times (rank 0, stderr)")
    ap.add_argument("--no-graphs", action="store_true",
                    help="launch the kernels of an iteration one by one instead of replaying a captured CUDA graph")
    ap.add_argument("--host-generator", action="store_true", help="generate the inputs with the numpy generator (1 GPU)")
    ap.add_argument("--config", default="c3", choices=["c3", "c4", "c5", "c5s"],
                    help="headline workload: c3 (default, BASELINE's metric); builder runs: c4 = dense reporting N=8k "
                         "M=64 L=2 K=2, c5 = config 5 weak-scaled, c5s = config 5 at N=16k")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last one computed as DIR/<name>.npy: posterior "
                         "parameters, ELBO and a fixed sample of the rho slab (rank 0's rows); the config-5 "
                         "workload's as DIR/c5_<name>.npy")
    return ap.parse_args()


def _round4(n):
    return (int(round(n)) + 3) // 4 * 4


def config_dims(config, world, nodes=0):
    """(law, L, K, N) of a workload at `world` GPUs."""
    if config == "c3":
        return "sbm", 1, 2, nodes or _round4(BASE_N * math.sqrt(world))
    if config == "c4":
        return "sbm", 2, 2, nodes or 8000
    if config == "c5s":
        return "gm", 4, 3, nodes or 16000
    return "gm", 4, 3, nodes or _round4(C5_N8 * math.sqrt(world / 8.0))


def workload_name(config, N, L, K, world):
    return {"c3": "StandardSBM ego-only N=%d M=N L=%d K=%d mutuality (config 3 of BASELINE.json%s)"
                  % (N, L, K, "" if world == 1 else ", grown to keep 4e8 ties per GPU"),
            "c4": "dense reporting N=%d M=64 all-report-all L=%d K=%d (config 4 of BASELINE.json)" % (N, L, K),
            "c5": "GMReciprocity ego-only N=%d L=%d K=%d (config 5 of BASELINE.json, weak-scaled: N=64000 on 8 GPUs)" % (N, L, K),
            "c5s": "GMReciprocity ego-only N=%d L=%d K=%d (config 5 of BASELINE.json scaled to one GPU)" % (N, L, K)}[config]


def make_network(N, L, K, seed_y=10, seed_x=20, config="c3"):
    """Host (numpy) generator: the CPU baseline's sample, config 4, and --host-generator."""
    from vimure_b200 import masks
    from vimure_b200 import synthetic as syn

    if config == "c4":  # every one of M=64 reporters reports every tie
        net = syn.StandardSBM(N=N, M=64, L=L, K=K, C=2, avg_degree=10, seed=seed_y)
        net.X, net.theta = syn.dense_reporting_X(net, M=64, mutuality=0.5, seed=seed_x)
        net.R = masks.AllMask(L, N, 64)
        net.M = 64
        return net
    if config in ("c5", "c5s"):
        net = syn.Multitensor(N=N, L=L, K=K, C=2, avg_degree=10, eta=0.5, seed=seed_y)
    else:
        net = syn.StandardSBM(N=N, L=L, K=K, C=2, avg_degree=10, seed=seed_y)
    net.build_X(mutuality=0.5, seed=seed_x)
    return net


class Shard:
    """This rank's part of a synthetic network: COO on the device (own rows + the reciprocal entries it needs)."""


def make_shard(config, N, L, K, rank, world, dev, host_generator=False, seed_y=10, seed_x=20):
    import torch

    from vimure_b200 import masks
    from vimure_b200 import synthetic as syn
    from vimure_b200.model import shard_rows

    sh = Shard()
    sh.L, sh.N, sh.K = L, N, K
    sh.row0, sh.nloc = shard_rows(N, world, rank)
    t0 = time.time()
    if config == "c4" or host_generator:
        if world > 1:
            raise SystemExit("config c4 / --host-generator run on one GPU")
        net = make_network(N, L, K, seed_y, seed_x, config)
        sh.M, sh.R = net.M, net.R
        sh.subs = torch.from_numpy(np.stack(net.X.subs).astype(np.int32)).to(dev)
        sh.vals = torch.from_numpy(np.asarray(net.X.vals).astype(np.int32)).to(dev)
        sh.generator = "host numpy (vimure_b200.synthetic)"
    else:
        # the ground truth Y is small (avg_degree ties per node): every rank draws the same one on the host
        net = (syn.Multitensor(N=N, L=L, K=K, C=2, avg_degree=10, eta=0.5, seed=seed_y) if config in ("c5", "c5s")
               else syn.StandardSBM(N=N, L=L, K=K, C=2, avg_degree=10, seed=seed_y))
        sh.subs, sh.vals = net.build_X_device(mutuality=0.5, seed=seed_x, device=dev, row0=sh.row0, nloc=sh.nloc,
                                              emit_transposed=world > 1)
        sh.M, sh.R = N, masks.EgoMask(L, N, N, diag=True)
        sh.generator = "device (vm_synth_ego)"
    own = (sh.subs[1] >= sh.row0) & (sh.subs[1] < sh.row0 + sh.nloc)
    sh.nnz_owned = int(own.sum())
    sh.sumX_owned = float(sh.vals[own].sum())
    torch.cuda.synchronize(dev)
    sh.gen_s = time.time() - t0
    return sh


def draw_state(L, M, K, seed=1):
    """Initial variational state as `_initialize_priors` draws it (model.py:570-595), default priors."""
    prng = np.random.RandomState(seed)
    rs = prng.random_sample
    st = dict(gamma_shp=0.1 * rs((L, M)) + 0.1, phi_shp=10.0 * rs((L, K)) + 10.0,
              gamma_rte=0.1 * rs((L, M)) + 0.1, phi_rte=10.0 * rs((L, K)) + 10.0,
              nu_shp=0.5 * rs(1)[0] + 0.5)
    return st, prng


# ----------------------------------------------------------------------------------------- CPU arm
def _cpu_worker(idx, n_nodes, L, K, iters, barrier, out):
    """One replica of the bounded CPU sample (spawned process, one numpy thread)."""
    try:
        from oracle.cavi_numpy import OracleCAVI

        net = make_network(n_nodes, L, K)
        spec = {"kind": "ego", "rep": np.ones((L, net.M), dtype=np.uint8), "diag": True}
        o = OracleCAVI(L, n_nodes, net.M, K, np.stack(net.X.subs), net.X.vals, spec, mutuality=True, **PRIORS)
        st, prng = draw_state(L, net.M, K, seed=1 + idx)
        s = np.stack(net.X.subs[:3])
        ties = np.unique(s, axis=1).T
        pr = 1 + 0.01 * prng.random_sample((len(ties), K))
        pr /= pr.sum(axis=1)[:, None]
        o.set_state(st["gamma_shp"], st["gamma_rte"], st["phi_shp"], st["phi_rte"], st["nu_shp"],
                    o.default_pr_rho(ties, pr))
        o.iterate()  # warm-up
        if barrier is not None:
            barrier.wait(timeout=300)  # all replicas start their timed iterations together
        t0 = time.time()
        for it in range(iters):
            o.iterate()
            if it == 0 or it == iters - 1:
                o.elbo()
        res = (idx, time.time() - t0, len(net.X.vals), None)
    except Exception as e:  # noqa: BLE001
        try:
            barrier.abort()
        except Exception:
            pass
        res = (idx, 0.0, 0, repr(e))
    if out is None:
        return res
    out.put(res)


def cpu_oracle_throughput_all_cores(n_nodes, L, K, iters=3, procs=0):
    """The path shards by node-row blocks with no exchange but the statistics vector, so a CPU implementation that uses
    every host core is, to a good approximation, one replica of the single-threaded implementation per core: `procs`
    replicas of the bounded sample run CONCURRENTLY (so that they compete for memory bandwidth as a parallel
    implementation would); throughput = procs * iters * ties / slowest replica.  Returns (ties/s, s/iter, nnz, procs)."""
    import multiprocessing as mp
    import queue as _queue

    if not procs:
        # the cores this process may run on (a cgroup / cpuset can be narrower than os.cpu_count()), at most 64, and no
        # more replicas than the host memory holds (a replica of the N=2048 sample peaks at 1.5 GB; scaled by N^2)
        try:
            ncpu = len(os.sched_getaffinity(0))
        except Exception:  # noqa: BLE001
            ncpu = os.cpu_count() or 1
        per_replica = 1.6e9 * (n_nodes / 2048.0) ** 2 * L
        try:
            import psutil

            avail = float(psutil.virtual_memory().available)
        except Exception:  # noqa: BLE001
            avail = 32e9
        procs = max(1, min(ncpu, 64, int(0.6 * avail / per_replica)))
    ties = float(L) * n_nodes * n_nodes

    def attempt(procs):
        if procs == 1:
            r = _cpu_worker(0, n_nodes, L, K, iters, None, None)
            if r[3] is not None:
                raise RuntimeError("CPU sample failed: %s" % r[3])
            return iters * ties / r[1], r[1] / iters, r[2], 1
        ctx = mp.get_context("spawn")  # never fork a process that may hold a CUDA context
        barrier, out = ctx.Barrier(procs), ctx.Queue()
        saved = {k: os.environ.get(k) for k in ("OMP_NUM_THREADS", "MKL_NUM_THREADS", "OPENBLAS_NUM_THREADS")}
        for k in saved:
            os.environ[k] = "1"
        try:
            ps = [ctx.Process(target=_cpu_worker, args=(i, n_nodes, L, K, iters, barrier, out), daemon=True)
                  for i in range(procs)]
            for p_ in ps:
                p_.start()
        finally:
            for k, v in saved.items():
                if v is None:
                    os.environ.pop(k, None)
                else:
                    os.environ[k] = v
        # collect the results; a replica that died without reporting (e.g. killed for memory) would leave the others at
        # their barrier: notice it, release them and fail this attempt instead of waiting
        res, deadline = [], time.time() + 600
        try:
            while len(res) < procs:
                try:
                    res.append(out.get(timeout=1.0))
                    continue
                except _queue.Empty:
                    pass
                dead = [p_ for p_ in ps if p_.exitcode not in (None, 0)]
                if dead or time.time() > deadline:
                    try:
                        barrier.abort()
                    except Exception:  # noqa: BLE001
                        pass
                    raise RuntimeError("CPU replica died (exit code %s) or timed out" % (dead[0].exitcode if dead else "-"))
        finally:
            for p_ in ps:
                p_.join(timeout=5)
                if p_.is_alive():
                    p_.terminate()  # (exact processes this function started)
        bad = [r for r in res if r[3] is not None]
        if bad:
            raise RuntimeError("CPU replica failed: %s" % bad[0][3])
        slowest = max(r[1] for r in res)
        return procs * iters * ties / slowest, slowest / iters, res[0][2], procs

    while True:
        try:
            return attempt(procs)
        except RuntimeError:
            if procs == 1:
                raise
            procs = max(1, procs // 4)  # fewer replicas (memory), finally one in-process


def cpu_baseline_record(n_nodes, L, K, iters, procs):
    v, s_it, nnz, procs = cpu_oracle_throughput_all_cores(n_nodes, L, K, iters=iters, procs=procs)
    return {"value": v, "unit": "ties/s", "cores": procs, "kind": "port", "sample_nodes": n_nodes,
            "sample_ms_per_iteration": s_it * 1e3,
            "sample": "numpy oracle port of model.py:623-1019 (pinned to the reference's goldens), SAME LAW as the workload "
                      "but at N=%d (nnz(X)=%d), %d iterations incl. 2 ELBO evaluations, %d concurrent single-threaded "
                      "replicas (one per host core, at most 64) started together; ties/s = replicas * iterations * N^2 / "
                      "slowest replica (%.2f s/iteration).  The reference itself cannot run N=20000 (dense (L,N,N,M) arrays)"
                      % (n_nodes, nnz, iters, procs, s_it)}


def reference_small_configs():
    """BASELINE configs 1 and 2 (the ones the reference CAN run): the UNMODIFIED reference (`oracle/_ref/vimure`, put
    there by `__graft_entry__.build()` in the build container; it travels to the GPU box as a built artefact) timed on
    this box's host CPU, on the golden fixtures' inputs.  Returns None when oracle/_ref is absent."""
    ref_dir = os.path.join(ROOT, "oracle", "_ref")
    if not os.path.isdir(os.path.join(ref_dir, "vimure")):
        return None
    for p_ in (os.path.join(ROOT, "oracle", "shims"), ref_dir):
        if p_ not in sys.path:
            sys.path.insert(0, p_)
    out = {}
    try:
        with warnings.catch_warnings():
            warnings.simplefilter("ignore")
            import sktensor as skt  # the COO container stand-in (oracle/shims)
            import vimure as ref  # noqa: F401
            from vimure.model import VimureModel as RefModel

            from tests.golden_util import Golden

            for tag, name, iters in (("c1", "f1_over", 21), ("c2", "karnataka_vil1", 11)):
                g = Golden(name)
                X = skt.sptensor(tuple(g.X_subs), g.X_vals, shape=(g.L, g.N, g.N, g.M), dtype=int)
                rs, rv = g.R_coo()
                R = skt.sptensor(tuple(rs.astype(np.int64)), rv.astype(int), shape=(g.L, g.N, g.N, g.M), dtype=int)
                fk = {k: v for k, v in g.fit_kwargs.items() if k not in ("max_iter", "num_realisations")}
                m = RefModel(mutuality=True, convergence_tol=0.0)
                t0 = time.time()
                m.fit(X, R=R, max_iter=iters, num_realisations=1, **fk)
                wall = time.time() - t0
                rt = float(np.mean(m.trace["runtime"])) if len(m.trace) else 0.0
                out[tag] = {"fixture": name, "N": g.N, "L": g.L, "K": g.K, "iterations": iters, "fit_wall_s": wall,
                            "cavi_s_per_iteration": rt if rt > 0 else None, "iter_per_s": (1.0 / rt) if rt > 0 else None,
                            "ties_per_s": (g.L * g.N * g.N / rt) if rt > 0 else None, "cores": 1,
                            "what": "unmodified reference VimureModel.fit; trace['runtime'] = CAVI only (model.py:406-410)"}
    except Exception as e:  # noqa: BLE001
        out["error"] = repr(e)[:300]
    return out


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    try:
        import torch

        torch.set_num_threads(os.cpu_count() or 1)
    except Exception:
        pass
    law, L, K, N_full = config_dims(args.config, args.gpus, args.nodes)
    n = args.cpu_nodes
    iters = max(1, min(args.steps, 3))
    t_all = time.time()
    rec = cpu_baseline_record(n, L, K, iters, args.cpu_procs)
    line = {
        "impl": "reference", "metric": "cavi_ties_per_s", "value": rec["value"], "unit": "ties/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": rec["sample_ms_per_iteration"],
        "ms_per_step_is": "one iteration of the N=%d SAMPLE (not of the N=%d workload)" % (n, N_full),
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": workload_name(args.config, N_full, L, K, args.gpus),
                   "ran": "bounded sample of that workload: same law at N=%d, per-tie normalised" % n},
        "cpu_baseline": rec,
        "e2e": {"value": rec["value"], "unit": "ties/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "reference_small_configs": reference_small_configs(),
        "wall_s": time.time() - t_all,
    }
    print(json.dumps(line))


# ----------------------------------------------------------------------------------------- clocks
class ClockSampler:
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.samples, self.proc = index, [], None

    def __enter__(self):
        # ONE long-lived nvidia-smi sampling every 20 ms (spawning one per sample is too slow for a ~0.1 s region)
        if self.index is None:
            return self
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "20"], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            time.sleep(0.3)  # let it finish its NVML initialisation
        except Exception:
            self.proc = None
        return self

    def __exit__(self, *a):
        if self.proc is None:
            return
        time.sleep(0.05)
        self.proc.terminate()
        try:
            out, _ = self.proc.communicate(timeout=5)
        except Exception:
            self.proc.kill()
            out = ""
        for line in out.strip().splitlines():
            self.samples.append([x.strip() for x in line.split(",")])

    def summary(self):
        rows, reasons = [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for s in self.samples:
            try:
                rows.append((float(s[0]), float(s[1]), float(s[2])))
                for nm, v in zip(names, s[4:8]):
                    if v.lower().startswith("active"):
                        reasons.add(nm)
            except Exception:
                pass
        if not rows:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        pmax = max(r[2] for r in rows)
        load = [r for r in rows if r[2] >= 0.6 * pmax] or rows  # samples taken under load
        return {"sm_mhz": float(np.median([r[0] for r in load])), "sm_max_mhz": max(r[1] for r in rows),
                "power_w_max": pmax, "reasons": sorted(reasons), "samples": len(rows), "samples_under_load": len(load)}


# ----------------------------------------------------------------------------------------- parity on the benched path
def run_parity(world, rank, dev):
    """Reference golden scenarios through `VimureModel.fit` on the path being benchmarked (NCCL row-block sharding when
    world > 1; same code as tests/run_dist_gpu.py): final gamma/phi after the fixture's iterations within rtol 1e-5 of
    the unmodified reference's, ELBO within 1e-6."""
    import torch

    import vimure_b200 as vm
    from tests.golden_util import Golden
    from tests.test_gpu_parity import build_inputs

    res, ok = {}, True
    for name in ("f1_over", "gm_l2_k3", "karnataka_vil1", "sbm_n520"):
        g = Golden(name)
        X, R = build_inputs(g, structured=(name == "sbm_n520"))
        mk = dict(g.model_kwargs)
        mk["convergence_tol"] = 0.0
        model = vm.VimureModel(**mk)
        fk = dict(g.fit_kwargs)
        n_it = min(g.n_iter, 20)
        fk["max_iter"] = n_it
        with warnings.catch_warnings():
            warnings.simplefilter("ignore")
            model.fit(X, R=R, init_state=g.init_state(), **fk)
        z, it = g.z, n_it - 1
        err = 0.0
        for k in ("gamma_shp", "gamma_rte", "phi_shp", "phi_rte"):
            a, b = getattr(model, k), z["it_" + k][it]
            err = max(err, float(np.max(np.abs(a - b) / np.abs(b))))
        err = max(err, abs(float(model.nu_shp) - float(z["it_nu_shp"][it])) / abs(float(z["it_nu_shp"][it])))
        e_elbo = abs(model.maxL - float(z["it_elbo"][it])) / abs(float(z["it_elbo"][it]))
        good = bool(err <= 1e-5 and e_elbo <= 1e-6)
        ok = ok and good
        res[name] = {"max_rel_err_params": err, "rel_err_elbo": e_elbo, "iterations": n_it, "pass": good}
    if world > 1:
        import torch.distributed as dist

        t = torch.tensor([1 if ok else 0], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MIN)
        ok = bool(int(t.item()) == 1)
    return {"path": "VimureModel.fit, %s" % ("row-block sharded over %d ranks, NCCL all-reduce of the statistics" % world
                                              if world > 1 else "single rank"),
            "against": "golden trajectories of the unmodified reference (tests/golden/*.npz, oracle/gen_golden.py)",
            "tolerance": {"params_rtol": 1e-5, "elbo_rtol": 1e-6}, "scenarios": res, "pass": ok, "rank": rank}


# ----------------------------------------------------------------------------------------- GPU arm
def hbm_peak():
    try:
        mp = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        return float(mp["hbm_gbs"]), "MEASURED_PEAKS.json hbm_gbs (of measured)"
    except Exception:
        return 6650.0, "fallback of B200_PROFILING.md (of fallback)"


def dump_outputs(eng, row0, out_dir, prefix, n_sample=1 << 18):
    """What the timed iterations hand their caller: posterior parameters and ELBO (float64) and the dense rho slab
    (float32), the slab as a fixed sample of at most `n_sample` ties with their global flat ids (l*N + i)*N + j."""
    import torch

    os.makedirs(out_dir, exist_ok=True)
    p = eng.params()
    rho = eng.rho_slab()
    L, nloc, N, K = rho.shape
    total = L * nloc * N
    idx = np.unique(np.random.RandomState(0).randint(0, total, size=min(n_sample, total), dtype=np.int64))
    sample = rho.view(-1, K)[torch.from_numpy(idx).to(rho.device)].cpu().numpy()
    l, rest = np.divmod(idx, nloc * N)
    i, j = np.divmod(rest, N)
    out = {k: p[k] for k in ("gamma_shp", "gamma_rte", "phi_shp", "phi_rte", "nu_shp", "nu_rte")}
    out.update(elbo=np.float64(eng.elbo()), rho_sample=sample,
               rho_sample_tie=((l * N + row0 + i) * N + j).astype(np.float64))
    for name, a in out.items():
        np.save(os.path.join(out_dir, prefix + name + ".npy"), np.asarray(a))


def run_workload(args, config, N, L, K, steps, warmup, dist, world, rank, dev, do_e2e, clock_index, dump_prefix=""):
    """Generate this rank's shard, pack it, run warm-up + `steps` timed iterations, the dense kernel in isolation, and
    (optionally) the end-to-end fit from pinned host buffers.  Returns the result dict (rank 0 uses it)."""
    import torch

    from vimure_b200 import _packing
    from vimure_b200._engine import CaviEngine
    from vimure_b200.model import VimureModel

    sh = make_shard(config, N, L, K, rank, world, dev, host_generator=args.host_generator)
    M = sh.M
    T = float(L) * N * N

    def allsum(v):
        if dist is None:
            return float(v)
        t = torch.tensor([float(v)], device=dev, dtype=torch.float64)
        dist.all_reduce(t)
        return float(t.item())

    def allmax(v):
        if dist is None:
            return float(v)
        t = torch.tensor([float(v)], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    nnzX = allsum(sh.nnz_owned)
    sumX = allsum(sh.sumX_owned)
    t0 = time.time()
    P = _packing.pack(sh.subs, sh.vals, L, N, M, K, sh.R, dev, row0=sh.row0, nloc=sh.nloc, tile_h=args.tile_h)
    eng = CaviEngine(P, PRIORS, mutuality=True, eps=1e-12, group=True if world > 1 else None)
    torch.cuda.synchronize(dev)
    pack_s = time.time() - t0
    if not args.no_graphs:
        eng.enable_graphs()  # what VimureModel.fit does
    st, prng = draw_state(L, M, K)
    # prior of the ties that carry a report: a device draw (what fit(init="fast") does), keyed per rank
    keep = P.t["u_has_x"] & P.t["u_reported"]
    gen = torch.Generator(device=dev)
    gen.manual_seed(1234 + rank)
    pr_u = torch.rand((P.U, K), generator=gen, dtype=torch.float64, device=dev).mul_(0.01).add_(1.0)
    pr_u /= pr_u.sum(dim=-1, keepdim=True)
    pr_u.masked_fill_(~keep[:, None], 0.0)
    pr_u[:, 0].masked_fill_(~keep, 1.0)
    nu_rte = PRIORS["beta_eta"] + sumX
    eng.set_state(st["gamma_shp"], st["gamma_rte"], st["phi_shp"], st["phi_rte"], st["nu_shp"], nu_rte, pr_u, 1e-12)
    del pr_u

    def run_iters(first, count, total):
        """iterations first..first+count-1 of a `total`-iteration fit, ELBO on the reference cadence"""
        it = first
        end = first + count - 1
        while it <= end:
            nxt = it
            while not (nxt == 1 or nxt % 10 == 0 or nxt == total) and nxt < end:
                nxt += 1
            is_elbo = (nxt == 1 or nxt % 10 == 0 or nxt == total)
            if args.trace:
                torch.cuda.synchronize(dev)
                t_b = time.time()
            eng.iterate(nxt - it + 1, elbo_last=is_elbo)
            if args.trace:
                torch.cuda.synchronize(dev)
                t_i = time.time()
            if is_elbo:
                e = eng.elbo()  # the one D2H scalar of `_check_for_convergence`
                if not np.isfinite(e):
                    raise RuntimeError("ELBO is not finite")
            if args.trace and rank == 0:
                print("trace: iters %d..%d elbo=%s  %.3f ms (+%.3f ms elbo readback)" %
                      (it, nxt, is_elbo, (t_i - t_b) * 1e3, (time.time() - t_i) * 1e3), file=sys.stderr)
            it = nxt + 1

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize(dev)

    total = warmup + steps
    # the clock sampler (one nvidia-smi process, rank 0 only) is started BEFORE the warm-up: its NVML initialisation
    # takes driver locks for a few hundred ms and must not fall into the timed region
    clk = ClockSampler(clock_index)
    with clk:
        run_iters(1, warmup, total)
        barrier()
        n0 = eng.n_launch
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ev0.record()
        run_iters(warmup + 1, steps, total)
        ev1.record()
        barrier()
    ms = allmax(ev0.elapsed_time(ev1))
    launches = eng.n_launch - n0
    value = steps * T / (ms * 1e-3)
    elbo_final = eng.elbo()
    if args.dump_outputs and rank == 0:
        dump_outputs(eng, sh.row0, args.dump_outputs, dump_prefix)

    # ---- dominant kernel in isolation: the per-tie dense kernel (writes 4*K bytes per owned tie)
    reps = 20
    eng.dense_only(0)
    torch.cuda.synchronize(dev)
    d0, d1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    d0.record()
    for _ in range(reps):
        eng.dense_only(0)
    d1.record()
    torch.cuda.synchronize(dev)
    dense_ms = allmax(d0.elapsed_time(d1) / reps)
    # the same iteration without the slab write (fit(store_rho=False): rho materialised at ELBO iterations only)
    eng.iterate(2, store=False, store_last=False)
    n0e, n1e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    n0e.record()
    eng.iterate(10, store=False, store_last=True)
    n1e.record()
    torch.cuda.synchronize(dev)
    ms_nostore = n0e.elapsed_time(n1e) / 10
    ties_local = float(L) * sh.nloc * N
    alg_bytes = 4.0 * K * ties_local
    achieved = alg_bytes / (dense_ms * 1e-3) / 1e9
    peak, peak_src = hbm_peak()
    traffic = None
    try:
        tr = json.load(open(os.path.join(ROOT, "profiles", "dense_traffic.json")))
        if tr.get("N") == N and tr.get("K") == K and tr.get("nloc") == sh.nloc:
            traffic = tr["dram_bytes_per_launch"]
    except Exception:
        pass
    shortcut = bool(eng.simple_mode)
    lcs = eng.layer_consts.cpu().numpy().reshape(L, 3 * K + 5)
    all32 = bool(getattr(eng, "all32_mode", False))
    fp32_layers = int((lcs[:, 2 * K + 4] == 1.0).sum()) if (eng.simple_mode or all32) else 0
    fast = P.N >= P.tile_w and K <= 4 and P.r_mode != 2 and (P.N * K) % 4 == 0
    tma = os.environ.get("VM_X_NOTMA") != "1"
    kname = (("k_dense_tma<K=%d,ELBO=false>" if tma else "k_dense_fast<K=%d,ELBO=false>") % K) if fast else "k_dense<K=%d>" % K
    roofline = {"bound": "hbm", "kernel": kname + (" (+ k_dense on the aux stream for the partial last column tile)" if fast else ""),
                "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "traffic": traffic,
                "traffic_source": "ncu --set full dram__bytes_read.sum + dram__bytes_write.sum per launch "
                                  "(profiles/dense_traffic.json)" if traffic else None,
                "peak_source": peak_src, "algorithmic_bytes_per_launch": alg_bytes,
                "algorithmic_bytes_rule": "4*K bytes per owned tie: the fp32 posterior written once (SURVEY.md 8d)",
                "kernel_ms": dense_ms, "share_of_step": dense_ms / (ms / steps),
                "timing": "CUDA events around %d back-to-back launches on the launching stream (max over ranks)" % reps}
    # whole iteration against the SURVEY 8(d) algorithmic bytes: 4*K*T + 3*16*nnz(X) + 3*4*K*U
    U_all = allsum(P.U)
    b_iter = 4.0 * K * T + 48.0 * nnzX + 12.0 * K * U_all
    step_gbs = b_iter / world / (ms / steps * 1e-3) / 1e9
    roofline_step = {"achieved": step_gbs, "peak": peak, "unit": "GB/s per GPU", "frac": step_gbs / peak,
                     "algorithmic_bytes_per_iteration": b_iter,
                     "rule": "4*K*T [rho written once] + 3*16*nnz(X) [three sparse passes] + 3*4*K*U [special ties] "
                             "(SURVEY.md 8d), divided by the measured ms_per_step (ELBO iterations included)",
                     "frac_of_8TBs_spec": step_gbs / 8000.0}

    # ---- end to end through the public API, host buffers in, posterior parameters + ELBO out
    e2e = None
    if do_e2e:
        from vimure_b200.sptensor import sptensor

        barrier()
        # this rank's entries as PINNED host buffers (int32 indices / counts), as the contract asks
        # (several ranks: only the entries of the rank's OWN rows travel over PCIe; fit(presharded="rows") fetches the
        # reciprocal entries it needs from their owners, device to device)
        own_e = (sh.subs[1] >= sh.row0) & (sh.subs[1] < sh.row0 + sh.nloc)
        e_subs, e_vals = (sh.subs[:, own_e], sh.vals[own_e]) if world > 1 else (sh.subs, sh.vals)
        host = torch.empty((5, e_subs.shape[1]), dtype=torch.int32, pin_memory=True)
        host[:4].copy_(e_subs)
        host[4].copy_(e_vals)
        del e_subs, e_vals, own_e
        torch.cuda.synchronize(dev)
        hn = host.numpy()
        Xh = sptensor(tuple(hn[d] for d in range(4)), hn[4], shape=(L, N, N, M))
        h2d = hn.nbytes
        # free the engine of the device-timed part: the fits below allocate their own
        del eng, P
        torch.cuda.empty_cache()
        runs = []
        for rep_i in range(3):
            model = VimureModel(mutuality=True, convergence_tol=0.0)  # tol 0: never stops early -> exactly `steps` iterations
            barrier()
            t0 = time.time()
            model.fit(Xh, R=sh.R, K=K, seed=1, max_iter=steps, init="fast", graphs=not args.no_graphs,
                      presharded="rows" if world > 1 else False)
            d2h = model.gamma_shp.nbytes * 4 + model.phi_shp.nbytes * 4 + 8 * (2 + len(model.trace))
            torch.cuda.synchronize(dev)
            wall = allmax(time.time() - t0)
            tm = {k: round(v, 4) for k, v in model.timings.items()}
            tm["batch_ms_per_iteration"] = [round(float(v) * 1e3, 3) for v in model.trace["runtime"]]
            runs.append((wall, model.pack_time, tm, d2h))
            del model
        wall, pack_t, timings, d2h = sorted(runs, key=lambda r_: r_[0])[1]
        warm = sorted(r_[0] for r_ in runs[1:])[0]
        e2e = {"value": steps * T / wall, "unit": "ties/s", "h2d_bytes_per_step": h2d / steps,
               "d2h_bytes_per_step": d2h / steps, "wall_s": wall, "wall_s_all_runs": [round(r_[0], 4) for r_ in runs],
               "e2e_first_fit": {"wall_s": runs[0][0], "value": steps * T / runs[0][0],
                                 "note": "first complete fit of the process after the device-timed part (allocator and "
                                         "lazily loaded kernels not yet warm)"},
               "e2e_warm": {"wall_s": warm, "value": steps * T / warm, "note": "faster of fits 2 and 3"},
               "pack_s": pack_t, "timings_s": timings,
               "what": "VimureModel.fit(X = this rank's entries as pinned host COO, R=EgoMask, max_iter=steps%s): H2D + "
                       "pack + CAVI + ELBO + D2H of gamma/phi/nu posteriors; rho stays on the device; `value` = median "
                       "of 3 consecutive complete fits, wall clock, max over ranks"
                       % (', presharded="rows"' if world > 1 else "")}
    return {"N": N, "L": L, "K": K, "ties": T, "nnz_X": nnzX, "special_ties": U_all, "ms": ms, "steps": steps, "value": value,
            "elbo_final": elbo_final, "launches": launches, "dense_ms": dense_ms, "ms_nostore": ms_nostore,
            "roofline": roofline, "roofline_step": roofline_step, "e2e": e2e, "clocks": clk.summary(), "pack_s": pack_s,
            "generate_s": sh.gen_s, "generator": sh.generator, "M": M, "slab_gb_per_gpu": alg_bytes / 1e9,
            "shortcut_ties": shortcut, "nloc": sh.nloc, "fp32_layers": fp32_layers,
            "all32": all32}


def run_ours(args):
    import torch

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    dist = None
    if world > 1:
        import torch.distributed as dist

        dist.init_process_group("nccl", device_id=dev)
    assert world == args.gpus or world == 1, "launch with torchrun --nproc-per-node == --gpus"
    t_all = time.time()

    parity = None
    if not args.no_parity:
        parity = run_parity(world, rank, dev)

    law, L, K, N = config_dims(args.config, world, args.nodes)
    main = run_workload(args, args.config, N, L, K, args.steps, args.warmup, dist, world, rank, dev,
                        do_e2e=not args.no_e2e, clock_index=local if rank == 0 else None)
    torch.cuda.empty_cache()

    c5 = None
    if not args.no_c5 and args.config == "c3":
        _, L5, K5, N5 = config_dims("c5", world, args.c5_nodes)
        c5_steps = args.steps if args.c5_steps is None else args.c5_steps
        r5 = run_workload(args, "c5", N5, L5, K5, c5_steps, min(args.warmup, 5), dist, world, rank, dev,
                          do_e2e=False, clock_index=None, dump_prefix="c5_")
        c5 = {"workload": workload_name("c5", N5, L5, K5, world), "n_gpus": world, "steps": c5_steps,
              "ms_per_step": r5["ms"] / r5["steps"], "value": r5["value"], "unit": "ties/s",
              "iter_per_s": r5["steps"] / (r5["ms"] * 1e-3), "ties": r5["ties"], "nnz_X": r5["nnz_X"],
              "special_ties": r5["special_ties"], "slab_gb_per_gpu": r5["slab_gb_per_gpu"],
              "roofline": r5["roofline"], "roofline_step": r5["roofline_step"], "elbo_final": r5["elbo_final"],
              "generate_s": r5["generate_s"], "pack_s": r5["pack_s"], "scaling": "weak (N = 64000*sqrt(G/8))"}
        torch.cuda.empty_cache()

    cpu = None
    small = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        cpu = cpu_baseline_record(args.cpu_nodes, L, K, 3, args.cpu_procs)
        small = reference_small_configs()

    if rank == 0:
        ms, steps = main["ms"], main["steps"]
        line = {
            "metric": "cavi_ties_per_s", "value": main["value"], "unit": "ties/s", "n_gpus": world, "steps": steps,
            "warmup": args.warmup, "ms_per_step": ms / steps, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32 storage / f64 accumulate", "data": "synthetic",
            "config": {"workload": workload_name(args.config, N, L, K, world), "nnz_X": main["nnz_X"],
                       "special_ties": main["special_ties"], "ties": main["ties"], "row_block_sharding": world,
                       "generator": main["generator"],
                       "l2": "per-iteration output (%.1f GB slab per GPU) exceeds L2" % main["slab_gb_per_gpu"],
                       "elbo_cadence": "iter 1, every 10th, last (inside the timed region)",
                       "shortcut_ties_kernel": main["shortcut_ties"], "fp32_special_tie_kernel_all_mask": main["all32"],
                       "layers_on_the_fp32_special_tie_path": main["fp32_layers"]},
            "iter_per_s": steps / (ms * 1e-3),
            "reports_per_s": steps * ((2.0 * N - 1) * main["M"] * L if args.config != "c4" else float(N) * N * main["M"] * L) / (ms * 1e-3),
            "elbo_final": main["elbo_final"], "ms_per_step_store_rho_false": main["ms_nostore"],
            "roofline": main["roofline"], "roofline_step": main["roofline_step"], "cpu_baseline": cpu, "e2e": main["e2e"],
            "gpu_launches": main["launches"], "clocks": main["clocks"], "parity": parity, "configs": {"c5": c5},
            "reference_small_configs": small, "generate_s": main["generate_s"], "pack_s": main["pack_s"],
            "bench_wall_s": time.time() - t_all,
        }
        print(json.dumps(line))
    if dist is not None:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    a = parse()
    if a.impl == "reference":
        run_reference(a)
    else:
        run_ours(a)
