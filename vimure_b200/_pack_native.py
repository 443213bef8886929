"""Packing through the library's own packer: `vm_pack` behind the C ABI (include/vimure_b200.h, csrc/vm_pack.cu).

The Python here only allocates the output buffers by their upper bounds, fills `vm_pack_args`, makes the one call and reads
the counts back; nothing of the layout is computed on the host.  (`_packing.pack_torch` is the torch restatement of the
same layout: the executable specification the tests compare this against, and the path for CPU tests / general masks.)
"""
import numpy as np
import torch


def dense_tile_w(K):
    """Column-tile width of the dense kernel (a K-dependent constant of the CUDA library)."""
    from . import _capi

    w = int(_capi.load().vm_dense_tile_w(int(K)))
    if w <= 0:
        raise ValueError("vimure_b200 supports 2 <= K <= 32 = VM_MAX_K (got K=%d)" % K)
    return w

GAMMA_CHUNK = 256
PHI_CHUNK = 4096
SPECIAL_TIES_PER_BLOCK = 1024  # == VM_SPECIAL_TIES_PER_BLOCK of include/vimure_b200.h


def dense_fast_eligible(K, r_mode, N, tile_w, tile_h):
    """Does a rho update run the fast (TMA) dense kernel?  A copy of `dense_fast_eligible` in csrc/vm_kernels.cu, which
    decides it: an ego or all-reporter mask (not the general COO mask, r_mode 2), K <= 4, N*K % 4 == 0, at least one
    full column tile, and row tiles of at most 128 = VM_FAST_MAX_TILE_H rows."""
    return K <= 4 and r_mode != 2 and (N * K) % 4 == 0 and N >= tile_w and tile_h <= 128


def shortcut_ties_eligible(K, r_mode, N, tile_w, tile_h, split_e0, U):
    """Can the fast dense kernel evaluate special ties itself (shortcut ties, include/vimure_b200.h: vm_ctx.simple_mode)?
    An ego mask (r_mode 0) on the fast dense kernel, the E0 / E1 split of the packed layout (`Packed.split_e0`), some
    special ties, and column ids exact in fp32 (N < 2^24: the per-tie record stores them as floats)."""
    return (r_mode == 0 and dense_fast_eligible(K, r_mode, N, tile_w, tile_h) and split_e0 and U > 0
            and N < (1 << 24))


def _i32(t):
    return t.to(torch.int32).contiguous()


class _Trace:
    """VM_PACK_TRACE=1: print the wall time of the packer's stages (each closed by a device synchronisation)."""

    def __init__(self, dev):
        import os
        import time

        self.on = os.environ.get("VM_PACK_TRACE") == "1"
        self.dev, self.time = dev, time
        if self.on:
            self._sync()
            self.t = time.time()

    def _sync(self):
        if self.dev.type == "cuda":
            torch.cuda.synchronize(self.dev)

    def __call__(self, label):
        if self.on:
            self._sync()
            now = self.time.time()
            print("pack: %-24s %7.2f ms" % (label, (now - self.t) * 1e3), flush=True)
            self.t = now


class Packed:
    """Plain container of the packed tensors + dimensions."""

    def __init__(self):
        self.t = {}

    def __getattr__(self, k):
        t = self.__dict__.get("t", {})
        if k in t:
            return t[k]
        raise AttributeError(k)


def pack_device(X_subs, X_vals, L, N, M, K, mask, device, row0=0, nloc=None, tile_h=64, mutuality=True, split_e0=True,
                simple=True, single=True):
    """The packed layout through `vm_pack` (include/vimure_b200.h) for an ego or all-reporter mask on a CUDA device: one
    call, one host synchronisation (to read the counts).  Same contract as `pack_torch`, `simple` and `single` included;
    within a tie the entries are ordered by reporter (the sort key is (l,i,j,m)) instead of by their position in the
    caller's list."""
    import ctypes

    from . import _capi

    dev = torch.device(device)
    nloc = N - row0 if nloc is None else int(nloc)
    _mark = _Trace(dev)
    lib = _capi.load()
    P = Packed()
    P.L, P.N, P.M, P.K, P.row0, P.nloc = int(L), int(N), int(M), int(K), int(row0), nloc
    TILE_W = dense_tile_w(K)
    P.tile_w, P.tile_h = TILE_W, int(tile_h)
    P.nct = (N + TILE_W - 1) // TILE_W
    P.nrt = (nloc + P.tile_h - 1) // P.tile_h
    P.mask = mask
    P.mutuality = bool(mutuality)
    # (the fp32 paths need the E0 / E1 split's precondition: no prior so small that exp(E[log theta/lambda]) can be 0)
    P.split_e0 = bool(split_e0 or not mutuality)

    def up32(a):
        if torch.is_tensor(a):
            return a.to(device=dev, dtype=torch.int32).contiguous()
        a = np.asarray(a)
        if a.dtype.kind not in "iu":
            if a.dtype.kind == "f" and a.size and not np.all(a == np.floor(a)):
                raise ValueError("X must hold integer counts")
            a = a.astype(np.int64)
        # (a host scan of a 1.5e7-entry column costs ~4 ms: only where the narrowing cast could wrap)
        if a.dtype.itemsize > 4 or (a.dtype.itemsize == 4 and a.dtype.kind == "u"):
            if a.size and (a.max() >= 2**31 or a.min() < -2**31):
                raise ValueError("X has subscripts outside its shape")
        return torch.from_numpy(np.ascontiguousarray(a.astype(np.int32, copy=False))).to(dev)

    xs = [up32(X_subs[d]) for d in range(4)]
    xv = up32(X_vals)
    n_in = int(xv.numel())
    _mark("h2d")
    ego = mask.kind == "ego"
    cap_e = max(n_in, 1)
    cap_u = n_in + (L * nloc if ego else 0) + 1
    cap_g = n_in // GAMMA_CHUNK + L * M + 2
    i32 = dict(dtype=torch.int32, device=dev)
    f32 = dict(dtype=torch.float32, device=dev)
    i64 = dict(dtype=torch.int64, device=dev)
    u8 = dict(dtype=torch.uint8, device=dev)
    out = {}
    for name in ("e_u", "e_m", "e_src", "f_u", "f_m", "g_u", "t_u", "t_lrow", "t_col"):
        out[name] = torch.empty(cap_e, **i32)
    for name in ("e_x", "e_xT", "f_x", "f_xT", "g_x", "g_xT", "t_x"):
        out[name] = torch.empty(cap_e, **f32)
    out["e_flags"] = torch.empty(cap_e, **u8)
    for name in ("u_lrow", "u_col", "u_cnt", "u_m0", "cx_idx", "cx_lrow", "cx_col", "cx_cnt", "cx_m0"):
        out[name] = torch.empty(cap_u, **i32)
    for name in ("u_x0", "u_xT0", "u_x0sum", "u_px", "u_pxt", "cx_x0", "cx_xT0", "cx_x0sum"):
        out[name] = torch.empty(cap_u, **f32)
    out["u_ptr"] = torch.empty(cap_u + 1, **i64)
    out["u_gflat"] = torch.empty(cap_u, **i64)
    out["u_has_x"] = torch.empty(cap_u, **u8)
    out["u_reported"] = torch.empty(cap_u, **u8)
    out["utile_ptr"] = torch.empty(L * nloc * P.nct + 1, **i32)
    out["cx_ptr"] = torch.empty(L + 1, **i64)
    out["lay_eptr"] = torch.empty(L + 1, **i64)
    out["g0"] = torch.empty(L * M, dtype=torch.float64, device=dev)
    out["g_chunk_ptr"] = torch.empty(cap_g + 1, **i64)
    out["g_chunk_lm"] = torch.empty(cap_g, **i32)
    out["g_lm_cptr"] = torch.empty(L * M + 1, **i64)
    counts = torch.zeros(16, **i64)
    rep = torch.as_tensor(mask.rep, device=dev).to(torch.uint8).flatten().contiguous() if ego else None

    # vm_pack classifies the shortcut ties, so the rule is decided before U is known: only an ego mask can have them,
    # and it makes every owned diagonal tie special, so there U > 0 exactly when L * nloc > 0
    P.r_mode = 0 if ego else 1
    P.simple_ok = bool(simple) and shortcut_ties_eligible(P.K, P.r_mode, P.N, TILE_W, P.tile_h, P.split_e0, L * nloc)
    A = _capi.pack_class()()
    A.L, A.N, A.M, A.K, A.row0, A.nloc, A.tile_h = P.L, P.N, P.M, P.K, P.row0, nloc, P.tile_h
    A.r_mode, A.ego_diag = P.r_mode, int(getattr(mask, "diag", False))
    A.mutuality, A.split_e0 = int(bool(mutuality)), int(bool(split_e0))
    A.simple, A.single = int(P.simple_ok), int(bool(single))
    A.n_in = n_in
    A.x_l, A.x_i, A.x_j, A.x_m = (t.data_ptr() for t in xs)
    A.x_v = xv.data_ptr()
    A.rep = rep.data_ptr() if rep is not None else None
    A.cap_e, A.cap_u, A.cap_g = cap_e, cap_u, cap_g
    for name, t in out.items():
        setattr(A, name, t.data_ptr())
    A.counts = counts.data_ptr()
    wsb = int(lib.vm_pack_workspace_bytes(ctypes.byref(A)))
    if wsb < 0:
        raise ValueError("vm_pack: unsupported problem size (more than 2^31 entries on one rank?)")
    ws = torch.empty(wsb, dtype=torch.uint8, device=dev)
    A.workspace, A.workspace_bytes = ws.data_ptr(), wsb
    stream = ctypes.c_void_p(torch.cuda.current_stream(dev).cuda_stream)
    _capi.check(lib.vm_pack(ctypes.byref(A), stream), "vm_pack")
    cn = counts.cpu().numpy()  # the one synchronisation
    del ws
    _mark("vm_pack")
    if cn[10]:
        raise ValueError("X has subscripts outside its shape")
    if cn[9]:
        raise ValueError("Duplicate entries without specified accumulation function")
    U, I, I1, IT, n_cx, n_gchunk = (int(v) for v in cn[:6])
    if U >= 2**31 or I >= 2**31:
        raise ValueError("too many special ties / entries for one rank (int32 indices)")
    P.U, P.I, P.I1, P.IT, P.n_cx, P.n_gchunk = U, I, I1, IT, n_cx, n_gchunk
    P.n_ublk = max(1, (int(cn[6]) + SPECIAL_TIES_PER_BLOCK - 1) // SPECIAL_TIES_PER_BLOCK)
    P.phi_chunk = PHI_CHUNK
    P.n_phichunk = max(1, (int(cn[7]) + PHI_CHUNK - 1) // PHI_CHUNK)
    P.n_cxblk = max(1, (int(cn[8]) + SPECIAL_TIES_PER_BLOCK - 1) // SPECIAL_TIES_PER_BLOCK)
    P.sumX_owned = float(cn[11])
    P.sumX = float(cn[11])
    P.b_all = float(cn[12])
    size = dict(e_u=I, e_m=I, e_src=I, e_x=I, e_xT=I, e_flags=I, f_u=I1, f_m=I1, f_x=I1, f_xT=I1, g_u=I1, g_x=I1, g_xT=I1,
                t_u=IT, t_lrow=IT, t_col=IT, t_x=IT, u_lrow=U, u_col=U, u_cnt=U, u_m0=U, u_x0=U, u_xT0=U, u_x0sum=U, u_px=U,
                u_pxt=U, u_ptr=U + 1, u_gflat=U, u_has_x=U, u_reported=U, cx_idx=n_cx, cx_lrow=n_cx, cx_col=n_cx, cx_cnt=n_cx,
                cx_m0=n_cx, cx_x0=n_cx, cx_xT0=n_cx, cx_x0sum=n_cx, g_chunk_ptr=n_gchunk + 1, g_chunk_lm=n_gchunk)
    for name, t in out.items():
        P.t[name] = t[: size[name]] if name in size else t
    P.t["u_has_x"] = P.t["u_has_x"].to(torch.bool)
    P.t["u_reported"] = P.t["u_reported"].to(torch.bool)
    P.t["u_single"] = P.t["u_pxt"] != 0
    P.t["u_simple"] = (P.t["u_px"] > 0) & ~P.t["u_single"]
    P.entry_src = P.t["e_src"].to(torch.int64)
    P.ego_diag = int(getattr(mask, "diag", False))
    if ego:
        P.t["rep"] = rep
    _mark("finish")
    return P


