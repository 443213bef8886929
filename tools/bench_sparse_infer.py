"""The sparse consumers (`infer_edges` / `sample_edges`, `get_inferred_model(..., sparse=True)`) against the dense device
consumers they replace, on one GPU, in one process.

Config 3 (StandardSBM ego, N = 20 000, L = 1, K = 2) with and without the slab, after a few iterations: the sparse
rho_max, fixed threshold (0.3) and 5-trial sample against the dense consumer + torch.nonzero.  Then the sparse network of
tools/bench_implicit.py beyond the slab's reach (N = 160 000, L = 1, K = 2, store_rho="never", 20 iterations through
`VimureModel.fit`): the sparse rho_max and sample (the device part and the whole public call) against the dense device
argmax `infer(0)`.  Each pair alternates, warm, `--reps` times (CUDA events around the device part, a host clock around
the public call, which ends in a device-to-host copy); per call the device memory it adds (torch.cuda.max_memory_allocated
over what was allocated before) and the number of edges.  One JSON object per line on stdout (and in --out); the card's
name and power limit first.

    python tools/bench_sparse_infer.py --out profiles/bench_sparse_infer.jsonl
"""
import argparse
import os
import subprocess
import sys
import time
import warnings

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

from bench_implicit import emit, make_engine, run_iters, sparse_reports  # noqa: E402


def measure(fn):
    """(ms by CUDA events, device memory added in GB, result) of one call of fn()"""
    import torch

    torch.cuda.synchronize()
    base = torch.cuda.memory_allocated()
    torch.cuda.reset_peak_memory_stats()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    r = fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1), (torch.cuda.max_memory_allocated() - base) / 1e9, r


def host_timed(fn):
    import torch

    torch.cuda.synchronize()
    base = torch.cuda.memory_allocated()
    torch.cuda.reset_peak_memory_stats()
    t0 = time.perf_counter()
    r = fn()
    torch.cuda.synchronize()
    return (time.perf_counter() - t0) * 1e3, (torch.cuda.max_memory_allocated() - base) / 1e9, r


def dense_nonzero(y):
    import torch

    return torch.nonzero(y.reshape(-1)).reshape(-1)


def config3(reps, out):
    import torch

    from bench import make_shard

    sh = make_shard("c3", 20000, 1, 2, 0, 1, torch.device("cuda"))
    name = "c3 N=20000 L=1 K=2"
    for slab in (True, False):
        eng, P = make_engine(sh, slab)
        run_iters(eng, 1, 10, 10)
        pairs = {
            "rho_max": (lambda: eng.infer_edges(0), lambda: dense_nonzero(eng.infer(0))),
            "fixed_threshold_0.3": (lambda: eng.infer_edges(1, 0.3), lambda: dense_nonzero(eng.infer(1, 0.3))),
            "sample_5": (lambda: eng.sample_edges(5, seed=3), lambda: dense_nonzero(eng.sample(5, seed=3))),
        }
        for what, (sparse, dense) in pairs.items():
            sparse(), dense()  # warm
            for rep in range(reps):
                ms_s, gb_s, (keys, _) = measure(sparse)
                ms_d, gb_d, nz = measure(dense)
                assert keys.numel() == nz.numel()
                emit(dict(workload=name, mode="store" if slab else "never", what=what, rep=rep, edges=int(keys.numel()),
                          sparse_ms=ms_s, sparse_added_GB=gb_s, dense_plus_nonzero_ms=ms_d, dense_added_GB=gb_d), out)
                del keys, nz
        del eng, P, pairs
        torch.cuda.empty_cache()


def sparse160k(N, reps, out):
    import torch

    import vimure_b200 as vm

    L, K, subs, vals = sparse_reports(N)
    X = vm.sptensor.sptensor(tuple(subs.cpu().numpy()), vals.cpu().numpy(), shape=(L, N, N, N))
    del subs, vals
    model = vm.VimureModel(mutuality=True)
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        model.fit(X, R=vm.masks.EgoMask(L, N, N), K=K, seed=3, max_iter=20, store_rho="never")
    eng = model._engine_of_rho_f()
    assert eng.rho is None
    name = "sparse ego N=%d L=%d K=%d lam=(1e-4,1), store_rho=never, %d special ties" % (N, L, K, eng.P.U)
    calls = {
        "rho_max device": lambda: eng.infer_edges(0),
        "rho_max public": lambda: model.get_inferred_model("rho_max", sparse=True),
        "sample_1 device": lambda: eng.sample_edges(1, seed=3),
        "sample_1 public": lambda: model.sample_inferred_model(N=1, seed=3, sparse=True)[0],
        "dense argmax infer(0)": lambda: eng.infer(0),
    }
    for fn in calls.values():  # warm
        r = fn()
        del r
        torch.cuda.empty_cache()
    for rep in range(reps):
        for what, fn in calls.items():
            if "public" in what:
                ms, gb, r = host_timed(fn)
                n = len(r.vals)
            else:
                ms, gb, r = measure(fn)
                n = int(r[0].numel()) if isinstance(r, tuple) else \
                    sum(int(torch.count_nonzero(r[:, a:a + 4096])) for a in range(0, N, 4096))
            emit(dict(workload=name, what=what, rep=rep, ms=ms, added_GB=gb, edges=n,
                      clock="host" if "public" in what else "cuda events"), out)
            del r
            torch.cuda.empty_cache()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=2)
    ap.add_argument("--sparse-n", type=int, default=160_000)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch

    if not torch.cuda.is_available():
        raise SystemExit("bench_sparse_infer.py measures on a GPU; none found")
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                       text=True).stdout.strip().splitlines()
    emit(dict(gpu=q[0] if q else "unknown", torch=torch.__version__, time=time.strftime("%Y-%m-%d %H:%M:%S")), args.out)
    config3(args.reps, args.out)
    if args.sparse_n:
        sparse160k(args.sparse_n, args.reps, args.out)


if __name__ == "__main__":
    main()
