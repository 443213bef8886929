"""The device report generators on one GPU, in one process.

- `vm_synth_all` at config 4's shape (StandardSBM Y, L = 2, N = 8000, M = 64 reporters, mutuality 0.5) against the host
  all-reporter generator `dense_reporting_X` on the same Y and theta (host clock, one call);
- `vm_synth_masked` on a uniformly random explicit mask of `--mask-entries` entries of that shape;
- `vm_synth_ego` at config 3 (StandardSBM, N = 20 000, L = 1, K = 2), in this build and, with `--parent-lib`, in another
  build of the library (for instance the parent commit's), alternately, on the same inputs; the two outputs are
  compared entry by entry.

Device times are CUDA events around the C entry point (counter reset + kernels): the counting pass (cap = 0, nothing
stored) and the filling pass, after one warm call of each, `--reps` times.  One JSON object per line on stdout (and in
--out); the card's name and power limit first.

    python tools/bench_synth.py --out profiles/bench_synth.jsonl [--parent-lib path/to/libvimure_b200.so]
"""
import argparse
import ctypes
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


class Call:
    """The arguments of one `vm_synth_*` call on the device (counting pass; `fill()` switches to a filling pass)."""

    def __init__(self, net, M, K, theta, eta, seed, mask=None):
        import torch

        from vimure_b200 import _capi

        N, L = net.N, net.L
        ykey = (net.Y_subs[0] * N + net.Y_subs[1]) * N + net.Y_subs[2]
        o = np.argsort(ykey)
        self.yk = torch.as_tensor(ykey[o], device="cuda")
        self.yv = torch.as_tensor(np.asarray(net.Y_vals)[o].astype(np.int32), device="cuda")
        self.th = torch.as_tensor(np.ascontiguousarray(theta, dtype=np.float64), device="cuda")
        self.counter = torch.zeros(1, dtype=torch.int64, device="cuda")
        S = _capi.synth_class()()
        S.L, S.N, S.M, S.K, S.row0, S.nloc, S.emit_transposed = L, N, M, K, 0, N, 0
        S.seed, S.eta = seed, eta
        S.theta, S.y_key, S.y_val, S.nY = self.th.data_ptr(), self.yk.data_ptr(), self.yv.data_ptr(), int(self.yk.numel())
        S.cap, S.counter = 0, self.counter.data_ptr()
        self.S, self.out, self.mask = S, None, None
        if mask is not None:
            Mk = _capi.synth_mask_class()()
            Mk.l, Mk.i, Mk.j, Mk.m = (int(t.data_ptr()) for t in mask)
            Mk.n = int(mask[0].numel())
            self.mask, self._keep = Mk, mask
        self.stream = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)

    def args(self):
        a = (ctypes.byref(self.S),)
        return a + ((ctypes.byref(self.mask),) if self.mask is not None else ()) + (self.stream,)

    def count(self, fn):
        self.S.cap = 0
        rc = fn(*self.args())
        assert rc == 0, rc
        return int(self.counter.item())

    def fill(self, n):
        import torch

        self.out = torch.empty((5, max(n, 1)), dtype=torch.int32, device="cuda")
        self.S.cap = n
        self.S.o_l, self.S.o_i, self.S.o_j, self.S.o_m, self.S.o_x = (self.out[d].data_ptr() for d in range(5))

    def sorted_output(self, n, M):
        h = self.out[:, :n].cpu().numpy().astype(np.int64)
        k = ((h[0] * self.S.N + h[1]) * self.S.N + h[2]) * M + h[3]
        o = np.argsort(k)
        return k[o], h[4][o]


def events_ms(fn, args, launches=1):
    import torch

    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(launches):
        rc = fn(*args)
    e1.record()
    torch.cuda.synchronize()
    assert rc == 0, rc
    return e0.elapsed_time(e1) / launches


def timed_passes(fn, call, n, reps):
    """(count ms, fill ms) per rep, each after one warm call"""
    cap = call.S.cap
    res = []
    for phase, c in (("count", 0), ("fill", n)):
        call.S.cap = c
        events_ms(fn, call.args())
        res.append([events_ms(fn, call.args()) for _ in range(reps)])
    call.S.cap = cap
    return res


def config4(lib, reps, mask_entries, out):
    import torch

    from vimure_b200 import synthetic as syn

    L, N, M, K, eta = 2, 8000, 64, 2, 0.5
    net = syn.StandardSBM(N=N, M=64, L=L, K=K, C=2, avg_degree=10, seed=10)
    t0 = time.time()
    X, theta = syn.dense_reporting_X(net, M=M, mutuality=eta, seed=20)
    host_s = time.time() - t0
    call = Call(net, M, K, theta, eta, seed=20)
    n = call.count(lib.vm_synth_all)
    call.fill(n)
    cnt, fill = timed_passes(lib.vm_synth_all, call, n, reps)
    assert int(call.counter.item()) == n
    k, v = call.sorted_output(n, M)
    l_, r = np.divmod(k // M, N * N)
    i_, j_ = np.divmod(r, N)
    off = i_ != j_
    hv = np.asarray(X.vals)
    name = "config 4 shape: StandardSBM N=%d L=%d, M=%d reporters, mutuality %.1f" % (N, L, M, eta)
    emit(dict(workload=name, generator="vm_synth_all", entries=n, entries_off_diagonal=int(off.sum()),
              sum_x_off_diagonal=int(v[off].sum()), count_ms=cnt, fill_ms=fill, clock="cuda events",
              philox_draws_per_pass=L * N * N * M + 2 * int(call.S.nY) * M), out)
    emit(dict(workload=name, generator="dense_reporting_X (host numpy, no self ties)", entries=int(len(hv)),
              sum_x=int(hv.sum()), seconds=host_s, clock="host", calls=1), out)
    del call
    torch.cuda.empty_cache()
    # an explicit mask of `mask_entries` uniformly random entries of the same shape
    g = torch.Generator(device="cuda")
    g.manual_seed(3)
    ent = [torch.randint(0, d, (mask_entries,), generator=g, device="cuda", dtype=torch.int32) for d in (L, N, N, M)]
    call = Call(net, M, K, theta, eta, seed=20, mask=ent)
    n = call.count(lib.vm_synth_masked)
    call.fill(n)
    cnt, fill = timed_passes(lib.vm_synth_masked, call, n, reps)
    emit(dict(workload=name + ", uniformly random explicit mask", generator="vm_synth_masked", mask_entries=mask_entries,
              entries=n, count_ms=cnt, fill_ms=fill, clock="cuda events"), out)
    del call, ent
    torch.cuda.empty_cache()


def config3_ego(lib, parent, reps, out):
    import torch

    from vimure_b200 import synthetic as syn

    L, N, K, eta = 1, 20000, 2, 0.5
    net = syn.StandardSBM(N=N, L=L, K=K, C=2, avg_degree=10, seed=10)
    theta = np.random.RandomState(20).gamma(shape=2.0, scale=0.5, size=(L, N))  # as build_X_device draws it
    libs = {"this build": lib}
    if parent is not None:
        libs["parent build"] = parent
    calls, outs, n = {}, {}, None
    for nm, lb in libs.items():
        c = Call(net, N, K, theta, eta, seed=20)
        nn = c.count(lb.vm_synth_ego)
        assert n is None or nn == n, (nm, nn, n)
        n = nn
        c.fill(n)
        assert lb.vm_synth_ego(*c.args()) == 0
        outs[nm] = c.sorted_output(n, N)
        calls[nm] = c
    same = all(np.array_equal(outs[k][0], outs["this build"][0]) and np.array_equal(outs[k][1], outs["this build"][1])
               for k in outs)
    times = {nm: ([], []) for nm in libs}
    for _ in range(reps):  # alternate the builds
        for nm, lb in libs.items():
            c, f = timed_passes(lb.vm_synth_ego, calls[nm], n, 1)
            times[nm][0].extend(c)
            times[nm][1].extend(f)
    name = "config 3: StandardSBM ego N=%d L=%d K=%d, mutuality %.1f, seed 20" % (N, L, K, eta)
    for nm in libs:
        emit(dict(workload=name, generator="vm_synth_ego", library=nm, entries=n, count_ms=times[nm][0],
                  fill_ms=times[nm][1], clock="cuda events", outputs_identical_across_builds=same), out)
    del calls
    torch.cuda.empty_cache()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--mask-entries", type=int, default=100_000_000)
    ap.add_argument("--parent-lib", default=None, help="another build of libvimure_b200.so to time vm_synth_ego against")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch

    from vimure_b200 import _capi

    if not torch.cuda.is_available():
        raise SystemExit("bench_synth.py measures on a GPU; none found")
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                       text=True).stdout.strip().splitlines()
    emit(dict(gpu=q[0] if q else "unknown", torch=torch.__version__, time=time.strftime("%Y-%m-%d %H:%M:%S")), args.out)
    lib = _capi.load()
    parent = None
    if args.parent_lib:
        parent = ctypes.CDLL(os.path.abspath(args.parent_lib))
        parent.vm_synth_ego.restype = ctypes.c_int
        parent.vm_synth_ego.argtypes = [ctypes.POINTER(_capi.synth_class()), ctypes.c_void_p]
        assert parent.vm_synth_size() == ctypes.sizeof(_capi.synth_class())
    config3_ego(lib, parent, args.reps, args.out)
    config4(lib, args.reps, args.mask_entries, args.out)


if __name__ == "__main__":
    main()
