"""Fits with and without the dense posterior slab (`store_rho="never"`, engine `slab=False`) on one GPU, in one process.

For config 3 (StandardSBM ego, N = 20 000, L = 1, K = 2) and config 5 weak-scaled to one GPU (GMReciprocity ego,
N = 22 628, L = 4, K = 3) the two modes alternate `--reps` times, each over `--steps` iterations on the reference's
ELBO cadence after `--warmup` (CUDA events).  Per mode: ms per step, torch.cuda.max_memory_allocated after pack + engine
and after the iterations, and (torch.profiler, a run of its own) the dense kernels' device time per iteration.  Then a
sparse network beyond the slab's reach (N = 160 000, L = 1, K = 2, report law lam = (1e-4, 1)) without the slab: ms per
iteration and peak memory.  One JSON object per line on stdout (and in --out); the card's name and power limit first.

    python tools/bench_implicit.py --out profiles/bench_implicit.jsonl
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def emit(rec, out):
    line = json.dumps(rec)
    print(line, flush=True)
    if out:
        with open(out, "a") as f:
            f.write(line + "\n")


def make_engine(sh, slab, tile_h=128):
    import torch

    from bench import PRIORS, draw_state
    from vimure_b200 import _packing
    from vimure_b200._engine import CaviEngine

    dev = torch.device("cuda")
    P = _packing.pack(sh.subs, sh.vals, sh.L, sh.N, sh.M, sh.K, sh.R, dev, row0=0, nloc=sh.N, tile_h=tile_h)
    eng = CaviEngine(P, PRIORS, mutuality=True, eps=1e-12, slab=slab)
    eng.enable_graphs()
    st, _ = draw_state(sh.L, sh.M, sh.K)
    keep = P.t["u_has_x"] & P.t["u_reported"]
    gen = torch.Generator(device=dev)
    gen.manual_seed(1234)
    pr_u = torch.rand((P.U, sh.K), generator=gen, dtype=torch.float64, device=dev).mul_(0.01).add_(1.0)
    pr_u /= pr_u.sum(dim=-1, keepdim=True)
    pr_u.masked_fill_(~keep[:, None], 0.0)
    pr_u[:, 0].masked_fill_(~keep, 1.0)
    nu_rte = PRIORS["beta_eta"] + float(sh.vals.sum())
    eng.set_state(st["gamma_shp"], st["gamma_rte"], st["phi_shp"], st["phi_rte"], st["nu_shp"], nu_rte, pr_u, 1e-12)
    del pr_u
    torch.cuda.synchronize()
    return eng, P


def run_iters(eng, first, count, total):
    """iterations first..first+count-1 of a `total`-iteration fit, ELBO on the reference cadence (as bench.py)"""
    it, end = first, first + count - 1
    while it <= end:
        nxt = it
        while not (nxt == 1 or nxt % 10 == 0 or nxt == total) and nxt < end:
            nxt += 1
        is_elbo = nxt == 1 or nxt % 10 == 0 or nxt == total
        eng.iterate(nxt - it + 1, elbo_last=is_elbo)
        if is_elbo and not np.isfinite(eng.elbo()):
            raise RuntimeError("ELBO is not finite")
        it = nxt + 1


def timed(sh, slab, steps, warmup):
    import torch

    torch.cuda.empty_cache()
    torch.cuda.reset_peak_memory_stats()
    base = torch.cuda.memory_allocated()
    eng, P = make_engine(sh, slab)
    mem_pack = torch.cuda.max_memory_allocated() - base
    total = warmup + steps
    run_iters(eng, 1, warmup, total)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    run_iters(eng, warmup + 1, steps, total)
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / steps
    mem_fit = torch.cuda.max_memory_allocated() - base
    elbo = eng.elbo()
    del eng, P
    return dict(ms_per_step=ms, mem_after_pack_GB=mem_pack / 1e9, mem_after_fit_GB=mem_fit / 1e9, elbo=elbo)


def profiled(sh, slab, iters, prof_dir, tag):
    """device time of the dense kernels per iteration, from a torch.profiler run of its own"""
    import torch
    from torch.profiler import ProfilerActivity, profile

    eng, P = make_engine(sh, slab)
    eng._graphs = None  # eager launches: one trace event per kernel
    run_iters(eng, 1, 3, 3 + iters)
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        run_iters(eng, 4, iters, 3 + iters)
        torch.cuda.synchronize()
    per = {}
    for ev in prof.key_averages():
        if "k_dense" in ev.key or "k_patch_rest" in ev.key:
            name = ev.key.split("(")[0].replace("void ", "")
            per[name] = dict(us_per_launch=ev.device_time_total / ev.count, launches=ev.count)
    if prof_dir:
        with open(os.path.join(prof_dir, "prof_implicit_%s_%s.txt" % (tag, "slab" if slab else "never")), "w") as f:
            f.write(prof.key_averages().table(sort_by="device_time_total", row_limit=25))
    del eng, P
    return per


def sparse_reports(N):
    """The sparse ego network of `sparse_run`: L = 1, K = 2, two true ties per node, report law lam = (1e-4, 1).
    Returns (L, K, subs, vals) on the device."""
    from vimure_b200 import synthetic as syn

    L, K = 1, 2
    rng = np.random.RandomState(7)
    ys = np.stack([np.zeros(2 * N, np.int64), rng.randint(0, N, 2 * N), rng.randint(0, N, 2 * N)])
    ys = ys[:, ys[1] != ys[2]]
    ys = ys[:, np.unique(ys[1] * N + ys[2], return_index=True)[1]]
    theta = 0.5 + rng.random_sample((L, N))
    subs, vals = syn.device_reports(L, N, N, K, ys, np.ones(ys.shape[1], np.int32), theta, 0.5, seed=11,
                                    lam=np.array([[1e-4, 1.0]]))
    return L, K, subs, vals


def sparse_run(N, iters):
    import torch

    import vimure_b200 as vm
    from bench import PRIORS
    from vimure_b200 import _packing
    from vimure_b200._engine import CaviEngine

    torch.cuda.empty_cache()
    torch.cuda.reset_peak_memory_stats()
    L, K, subs, vals = sparse_reports(N)
    P = _packing.pack(subs, vals, L, N, N, K, vm.masks.EgoMask(L, N, N), torch.device("cuda"), tile_h=128)
    eng = CaviEngine(P, PRIORS, mutuality=True, eps=1e-12, slab=False)
    eng.enable_graphs()
    rs = np.random.RandomState(1).random_sample
    pr_u = np.zeros((P.U, K))
    pr_u[:, 0] = 1.0
    keep = (P.t["u_has_x"] & P.t["u_reported"]).cpu().numpy()
    pr = 1 + 0.01 * rs((int(keep.sum()), K))
    pr_u[keep] = pr / pr.sum(axis=1)[:, None]
    eng.set_state(0.1 * rs((L, N)) + 0.1, 0.1 * rs((L, N)) + 0.1, 10.0 * rs((L, K)) + 10.0, 10.0 * rs((L, K)) + 10.0,
                  0.5 * rs(1)[0] + 0.5, PRIORS["beta_eta"] + float(vals.sum()), pr_u, 1e-12)
    torch.cuda.synchronize()
    mem_pack = torch.cuda.max_memory_allocated()
    run_iters(eng, 1, 2, iters)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    run_iters(eng, 3, iters - 2, iters)
    e1.record()
    torch.cuda.synchronize()
    ms_iter = e0.elapsed_time(e1) / (iters - 2)
    # the argmax of the whole posterior (get_inferred_model("rho_max")'s device part), block by block
    torch.cuda.synchronize()
    e0.record()
    Y = eng.infer(0)
    e1.record()
    torch.cuda.synchronize()
    ms_argmax = e0.elapsed_time(e1)
    ones = sum(int(torch.count_nonzero(Y[:, a:a + 4096])) for a in range(0, N, 4096))
    del Y
    rec = dict(workload="sparse ego N=%d L=%d K=%d lam=(1e-4,1), %d reports, %d special ties" % (N, L, K, int(vals.numel()), P.U),
               mode="never", ms_per_iter=ms_iter, iters=iters, elbo=eng.elbo(), ms_rho_max_all_rows=ms_argmax,
               rho_max_ones=ones,
               slab_GB_if_stored=4.0 * L * N * N * K / 1e9, mem_after_pack_GB=mem_pack / 1e9,
               mem_peak_GB=torch.cuda.max_memory_allocated() / 1e9,
               device_total_GB=torch.cuda.mem_get_info()[1] / 1e9)
    del eng, P
    return rec


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--reps", type=int, default=2)
    ap.add_argument("--prof-iters", type=int, default=10)
    ap.add_argument("--sparse-n", type=int, default=160_000)
    ap.add_argument("--sparse-iters", type=int, default=20)
    ap.add_argument("--out", default=None)
    ap.add_argument("--prof-dir", default=None)
    args = ap.parse_args()
    import torch

    if not torch.cuda.is_available():
        raise SystemExit("bench_implicit.py measures on a GPU; none found")
    from bench import make_shard

    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                       text=True).stdout.strip().splitlines()
    emit(dict(gpu=q[0] if q else "unknown", torch=torch.__version__, time=time.strftime("%Y-%m-%d %H:%M:%S")), args.out)
    dev = torch.device("cuda")
    for config, N, L, K in (("c3", 20000, 1, 2), ("c5", 22628, 4, 3)):
        sh = make_shard(config, N, L, K, 0, 1, dev)
        name = "%s N=%d L=%d K=%d" % (config, N, L, K)
        for rep in range(args.reps):
            for slab in (True, False):
                r = timed(sh, slab, args.steps, args.warmup)
                emit(dict(workload=name, mode="store" if slab else "never", rep=rep, steps=args.steps, **r), args.out)
        for slab in (True, False):
            per = profiled(sh, slab, args.prof_iters, args.prof_dir, config)
            emit(dict(workload=name, mode="store" if slab else "never", profiler_iters=args.prof_iters, profiler=per),
                 args.out)
        del sh
    if args.sparse_n:
        emit(sparse_run(args.sparse_n, args.sparse_iters), args.out)


if __name__ == "__main__":
    main()
