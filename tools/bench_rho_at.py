"""The posterior at given ties (`vm_rho_at`, `VimureModel.rho_f_at`) on one GPU, in one process.

Config 3 (StandardSBM ego, N = 20 000, L = 1, K = 2) with and without the slab, after 10 iterations: device time of
`vm_rho_at` (CUDA events around `--launches` back-to-back launches into a preallocated output, after a warm-up) for 1e6 and
1e7 uniformly random keys and for the keys of the rho_max edge list (sorted), with every source the engine has (a storing
engine: implicit and slab; a slab-free one: implicit).  Baseline on the same queries: the obvious alternative,
`vm_materialize_rows` of the rows the queries touch (one range, from the first to the last touched row: every row for the
random keys) and a gather.  Then the sparse network of tools/bench_implicit.py beyond the slab's reach (N = 160 000,
L = 1, K = 2, store_rho="never", 20 iterations through `VimureModel.fit`): `rho_f_at` on the rho_max edge list -- the
device part (`CaviEngine.rho_at`, CUDA events), the whole public call (host clock, ends in the device-to-host copy) and the
device memory each adds (torch.cuda.max_memory_allocated over what was allocated before).  One JSON object per line on
stdout (and in --out); the card's name and power limit first.

    python tools/bench_rho_at.py --out profiles/bench_rho_at.jsonl
"""
import argparse
import ctypes
import os
import subprocess
import sys
import time
import warnings

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

from bench_implicit import emit, make_engine, run_iters, sparse_reports  # noqa: E402
from bench_sparse_infer import host_timed, measure  # noqa: E402


def events_ms(fn, launches):
    """mean ms per call of `launches` back-to-back calls of fn(), by CUDA events (one warm call first)"""
    import torch

    fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(launches):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / launches


def config3(launches, reps, out):
    import torch

    from bench import make_shard
    from vimure_b200 import _capi

    sh = make_shard("c3", 20000, 1, 2, 0, 1, torch.device("cuda"))
    name = "c3 N=20000 L=1 K=2"
    for slab in (True, False):
        eng, P = make_engine(sh, slab)
        run_iters(eng, 1, 10, 10)
        N, K, C = P.N, P.K, eng.C
        gen = torch.Generator(device="cuda")
        gen.manual_seed(5)
        queries = {"random_1e6": torch.randint(0, P.L * N * N, (10 ** 6,), generator=gen, device="cuda"),
                   "random_1e7": torch.randint(0, P.L * N * N, (10 ** 7,), generator=gen, device="cuda"),
                   "rho_max_edges": eng.infer_edges(0)[0]}
        sources = {"implicit": C["VM_EDGES_IMPLICIT"]}
        if slab:
            sources["slab"] = C["VM_EDGES_SLAB"]
        for what, keys in queries.items():
            n = keys.numel()
            out_buf = torch.empty(n, K, dtype=torch.float32, device="cuda")
            want = None
            lrow = keys // N
            r0, r1 = int(lrow.min()), int(lrow.max()) + 1
            rows_buf = torch.empty(r1 - r0, N, K, dtype=torch.float32, device="cuda")
            local = (lrow - r0) * N + keys % N

            def baseline():
                eng.materialize_rows(r0, r1 - r0, rows_buf)
                return rows_buf.view(-1, K)[local]

            for sname, src in sources.items():
                def call(src=src):  # the C ABI directly, into the preallocated output: the kernel alone
                    _capi.check(eng.lib.vm_rho_at(eng._cref, src, n, ctypes.c_void_p(keys.data_ptr()),
                                                  ctypes.c_void_p(out_buf.data_ptr()), eng._stream()), "vm_rho_at")

                call()
                got = out_buf.clone()
                want = baseline() if want is None else want
                assert torch.equal(got, want), (what, sname)
                for rep in range(reps):
                    ms = events_ms(call, launches)
                    ms_b = events_ms(baseline, max(2, launches // 10))
                    emit(dict(workload=name, mode="store" if slab else "never", queries=what, n=n, source=sname, rep=rep,
                              rho_at_ms=ms, rho_at_launches=launches, baseline_rows=r1 - r0, baseline_ms=ms_b,
                              clock="cuda events"), out)
            del out_buf, rows_buf, local, lrow, want
        del eng, P, queries
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
    Y = model.get_inferred_model("rho_max", sparse=True)
    keys = torch.as_tensor((Y.subs[0] * np.int64(N) + Y.subs[1]) * N + Y.subs[2], device="cuda")
    calls = {"rho_at device": lambda: eng.rho_at(keys), "rho_f_at public": lambda: model.rho_f_at(Y.subs)}
    for fn in calls.values():  # warm
        r = fn()
        del r
        torch.cuda.empty_cache()
    got = model.rho_f_at(Y.subs)
    assert np.array_equal(np.argmax(got, axis=-1), Y.vals)
    for rep in range(reps):
        for what, fn in calls.items():
            ms, gb, r = host_timed(fn) if "public" in what else measure(fn)
            emit(dict(workload=name, what=what, rep=rep, ms=ms, added_GB=gb, n=len(Y.vals),
                      clock="host" if "public" in what else "cuda events"), out)
            del r
            torch.cuda.empty_cache()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--launches", type=int, default=50)
    ap.add_argument("--reps", type=int, default=2)
    ap.add_argument("--sparse-n", type=int, default=160_000)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch

    if not torch.cuda.is_available():
        raise SystemExit("bench_rho_at.py measures on a GPU; none found")
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                       text=True).stdout.strip().splitlines()
    emit(dict(gpu=q[0] if q else "unknown", torch=torch.__version__, time=time.strftime("%Y-%m-%d %H:%M:%S")), args.out)
    config3(args.launches, args.reps, args.out)
    if args.sparse_n:
        sparse160k(args.sparse_n, args.reps, args.out)


if __name__ == "__main__":
    main()
