"""Data packing: the sptensor X and the reporter mask R -> the tie-sorted device layout the kernels read.

Replaces, for the hot path, the reference's `__check_fit_params` data preparation (`model.py:147-176`):
`data_T` / `data_T_vals` (an O(nnz^2) python lookup, `utils.py:73-84`) become one sort + searchsorted that
pre-pairs every report X[l,i,j,m] with its reciprocal X[l,j,i,m]; the union-of-ties DataFrame merges of
`_set_rho_prior` (`model.py:509-556`) become a `unique` over the tie keys.

Everything here is index plumbing done with torch ops on whatever device it is given (the GPU in
production, the CPU in the `-m "not gpu"` tests); the arithmetic of the model lives in `csrc/`.

Layout (see include/vimure_b200.h): this rank owns node rows [row0, row0+nloc) of every layer;
`special ties` = owned ties that carry at least one X entry, plus (ego mask) every owned diagonal tie.
"""
import numpy as np
import torch


from ._pack_native import (GAMMA_CHUNK, PHI_CHUNK, SPECIAL_TIES_PER_BLOCK, Packed, _Trace, _i32,  # noqa: F401
                           dense_tile_w, pack_device)


def pack(X_subs, X_vals, L, N, M, K, mask, device, row0=0, nloc=None, tile_h=64, mutuality=True, split_e0=True,
         simple=None, single=None):
    """Build the packed layout: on a CUDA device and for a structured mask through the library's own packer (`vm_pack`
    behind the C ABI, csrc/vm_pack.cu); otherwise (CPU tests, general COO masks, VM_PY_PACKER=1) with the torch index
    ops of `pack_torch`, which doubles as the executable specification of the layout."""
    import os

    dev = torch.device(device)
    if dev.type == "cuda" and mask.kind in ("ego", "all") and os.environ.get("VM_PY_PACKER") != "1":
        P = pack_device(X_subs, X_vals, L, N, M, K, mask, dev, row0=row0, nloc=nloc, tile_h=tile_h, mutuality=mutuality,
                        split_e0=split_e0, simple=simple, single=single)
    else:
        P = pack_torch(X_subs, X_vals, L, N, M, K, mask, device, row0=row0, nloc=nloc, tile_h=tile_h, mutuality=mutuality,
                       split_e0=split_e0, simple=simple, single=single)
    # (the fp32 paths need the E0 / E1 split's precondition: no prior so small that exp(E[log theta/lambda]) can be 0)
    P.split_e0 = bool(split_e0 or not mutuality)
    return P


def pack_torch(X_subs, X_vals, L, N, M, K, mask, device, row0=0, nloc=None, tile_h=64, mutuality=True, split_e0=True,
               simple=None, single=None):
    """Build the packed layout with torch index ops (any device).

    X_subs : (4, I) integer array-like (l, i, j, m);  X_vals : (I,) counts;  mask : masks.ReporterMask.
    mutuality / split_e0 : the gamma and phi passes only visit the entries with a reciprocal report (x^T > 0); for the
        others dz1_k = x, a constant (reference model.py:679-681, 693 with z2 = 0).  `split_e0=False` makes every entry
        visited (needed when a prior is so small that exp(E[log theta]) can underflow to 0, where model.py:692 gives 0).
    simple : classify the special ties whose posterior the fast dense kernel can evaluate itself (default: yes, unless the
        environment says VM_NO_SIMPLE=1 -- the A/B switch of the tests and tools).
    single : ... including the ties with exactly one report that has a reciprocal report (default: yes, unless
        VM_NO_SINGLE=1).
    """
    import os

    if simple is None:
        simple = os.environ.get("VM_NO_SIMPLE") != "1"
    if single is None:
        single = os.environ.get("VM_NO_SINGLE") != "1"
    dev = torch.device(device)
    nloc = N - row0 if nloc is None else int(nloc)
    _mark = _Trace(dev)
    P = Packed()
    P.L, P.N, P.M, P.K, P.row0, P.nloc = int(L), int(N), int(M), int(K), int(row0), nloc
    TILE_W = dense_tile_w(K)
    P.tile_w, P.tile_h = TILE_W, int(tile_h)
    P.nct = (N + TILE_W - 1) // TILE_W
    P.nrt = (nloc + P.tile_h - 1) // P.tile_h
    P.mask = mask
    P.mutuality = bool(mutuality)

    def _up(a, small):
        """host array -> device int64/float64 tensor, moving as few bytes as possible over PCIe"""
        if torch.is_tensor(a):
            return a.to(dev)
        a = np.asarray(a)
        if small and a.dtype.kind in "iu" and a.dtype.itemsize > 4:
            a = a.astype(np.int32)
        return torch.from_numpy(np.ascontiguousarray(a)).to(dev)

    small = max(L, N, M) < 2**31
    xl, xi, xj, xm = (_up(X_subs[d], small) for d in range(4))
    xv = _up(X_vals, small and (torch.is_tensor(X_vals) or np.asarray(X_vals).dtype.kind in "iu"))
    if xv.numel():
        mx = torch.stack([xl.max(), xi.max(), xj.max(), xm.max(), -torch.stack([xl.min(), xi.min(), xj.min(), xm.min()]).min()])
        mx = mx.cpu().numpy()
        if mx[0] >= L or mx[1] >= N or mx[2] >= N or mx[3] >= M or mx[4] > 0:
            raise ValueError("X has subscripts outside its shape")
    P.sumX_owned = None
    keep_idx = None
    if nloc < N and xv.numel():
        # a row-block shard only needs the entries of its own rows (i in the block) and their reciprocals (j in the block):
        # everything else is dropped BEFORE the 64-bit keys, the sorts and the pairing (sharded ingestion; with G ranks
        # about 2/G of the list survives)
        own_i = (xi >= row0) & (xi < row0 + nloc)
        need = own_i | ((xj >= row0) & (xj < row0 + nloc))
        P.sumX_owned = float(xv[own_i].sum())
        keep_idx = torch.nonzero(need).flatten()
        xl, xi, xj, xm, xv = xl[keep_idx], xi[keep_idx], xj[keep_idx], xm[keep_idx], xv[keep_idx]
        del own_i, need
    xl, xi, xj, xm = (t.to(torch.int64) for t in (xl, xi, xj, xm))
    xv = xv.to(torch.float64)
    I_all = xv.numel()

    _mark("h2d+check")
    # ---- reciprocal pairing: xT[I] = X[l, j, i, m]   (model.py:152-161)
    key = ((xl * N + xi) * N + xj) * M + xm
    skey, order = torch.sort(key)
    if I_all > 1 and bool((skey[1:] == skey[:-1]).any()):
        raise ValueError("Duplicate entries without specified accumulation function")
    keyT = ((xl * N + xj) * N + xi) * M + xm
    if I_all:
        pos = torch.searchsorted(skey, keyT).clamp(max=I_all - 1)
        found = skey[pos] == keyT
        xT = torch.where(found, xv[order][pos], torch.zeros_like(xv))
    else:
        xT = xv.clone()
    P.sumX = float(xv.sum()) if I_all else 0.0
    # named temporaries live until the function returns: release the big ones so that the allocator can reuse their blocks
    # (in a cold process every tensor of this size is a fresh cudaMalloc, a few ms each)
    if I_all:
        del pos, found
    del key, skey, order, keyT

    _mark("pairing")
    in_R = mask.entry_multiplicity(xl, xi, xj, xm) if I_all else xv.clone()
    in_RT = mask.entry_multiplicity(xl, xj, xi, xm) if I_all else xv.clone()

    # ---- ownership and tie-sorted order of the owned entries
    own = (xi >= row0) & (xi < row0 + nloc)
    sel = torch.nonzero(own).flatten()
    tk = (xl[sel] * nloc + (xi[sel] - row0)) * N + xj[sel]  # local tie id
    tk_sorted, o2 = torch.sort(tk, stable=True)
    sel = sel[o2]
    I = sel.numel()
    P.I = int(I)
    P.entry_src = sel if keep_idx is None else keep_idx[sel]  # position of each packed entry in the caller's COO order
    del own, tk, o2

    _mark("mask+tie sort")
    # ---- special ties
    ukeys = torch.unique_consecutive(tk_sorted)
    if mask.kind == "ego":
        ii = torch.arange(row0, row0 + nloc, device=dev, dtype=torch.int64)
        ll = torch.arange(L, device=dev, dtype=torch.int64)
        dk = ((ll[:, None] * nloc + (ii[None, :] - row0)) * N + ii[None, :]).flatten()
        ukeys = torch.unique(torch.cat([ukeys, dk]))
    U = ukeys.numel()
    P.U = int(U)
    if U >= 2**31 or I >= 2**31:
        raise ValueError("too many special ties / entries for one rank (int32 indices)")
    u_lrow = ukeys // N
    u_col = ukeys - u_lrow * N
    P.t["u_lrow"] = _i32(u_lrow)
    P.t["u_col"] = _i32(u_col)
    P.t["u_key"] = ukeys
    e_u = torch.searchsorted(ukeys, tk_sorted)
    P.t["e_u"] = _i32(e_u)
    u_ptr = torch.searchsorted(tk_sorted, torch.cat([ukeys, ukeys.new_tensor([L * nloc * N])]))
    P.t["u_ptr"] = u_ptr.to(torch.int64).contiguous()
    P.t["e_m"] = _i32(xm[sel])
    P.t["e_x"] = xv[sel].to(torch.float32).contiguous()
    P.t["e_xT"] = xT[sel].to(torch.float32).contiguous()
    P.t["e_flags"] = (in_R[sel] > 0).to(torch.uint8).contiguous()
    # first entry of every special tie, inline
    cnt = u_ptr[1:] - u_ptr[:-1]
    first = u_ptr[:-1].clamp(max=max(I - 1, 0))
    has = cnt > 0
    P.t["u_cnt"] = _i32(cnt)
    if I:
        P.t["u_m0"] = torch.where(has, P.t["e_m"][first], torch.zeros_like(P.t["e_m"][first])).contiguous()
        P.t["u_x0"] = torch.where(has, P.t["e_x"][first], torch.zeros_like(P.t["e_x"][first])).contiguous()
        P.t["u_xT0"] = torch.where(has, P.t["e_xT"][first], torch.zeros_like(P.t["e_xT"][first])).contiguous()
    else:
        P.t["u_m0"] = torch.zeros(U, dtype=torch.int32, device=dev)
        P.t["u_x0"] = torch.zeros(U, dtype=torch.float32, device=dev)
        P.t["u_xT0"] = torch.zeros(U, dtype=torch.float32, device=dev)
    # has this special tie any X entry / is it reported by anybody (model.py:536-556)
    u_l = u_lrow // nloc
    u_i = u_lrow - u_l * nloc + row0
    P.t["u_has_x"] = (u_ptr[1:] > u_ptr[:-1])
    P.t["u_reported"] = mask.tie_reported(u_l, u_i, u_col) if U else torch.zeros(0, dtype=torch.bool, device=dev)
    P.t["u_gflat"] = (u_l * N + u_i) * N + u_col  # global flat tie id (l,i,j) -> position in the reference's arrays

    _mark("special ties")
    # dense-tile pointers: first special tie of every (local row, column tile)
    rows = torch.arange(L * nloc, device=dev, dtype=torch.int64)
    bounds = (rows[:, None] * N + torch.arange(P.nct, device=dev, dtype=torch.int64)[None, :] * TILE_W).flatten()
    bounds = torch.cat([bounds, bounds.new_tensor([L * nloc * N])])
    P.t["utile_ptr"] = _i32(torch.searchsorted(ukeys, bounds))
    n_ul = (P.t["utile_ptr"][:: nloc * P.nct][1:] - P.t["utile_ptr"][:: nloc * P.nct][:-1]) if U else None
    max_ul = int(n_ul.max()) if U else 0
    P.n_ublk = max(1, (max_ul + SPECIAL_TIES_PER_BLOCK - 1) // SPECIAL_TIES_PER_BLOCK)

    _mark("tile/col pointers")
    # ---- layer ranges and reporter chunks of the entries
    P.phi_chunk = PHI_CHUNK
    e_l = tk_sorted // (nloc * N)
    lm_all = e_l * M + xm[sel]
    # E1 = entries the gamma / phi passes visit; E0 = the rest (constant Poisson allocation dz1 = x)
    if not split_e0:
        is1 = torch.ones(I, dtype=torch.bool, device=dev)
    elif mutuality:
        is1 = P.t["e_xT"] != 0
    else:
        is1 = torch.zeros(I, dtype=torch.bool, device=dev)
    e1 = torch.nonzero(is1).flatten()
    P.I1 = int(e1.numel())
    P.t["e1_idx"] = e1
    P.t["f_u"] = P.t["e_u"][e1].contiguous()
    P.t["f_m"] = P.t["e_m"][e1].contiguous()
    P.t["f_x"] = P.t["e_x"][e1].contiguous()
    P.t["f_xT"] = P.t["e_xT"][e1].contiguous()
    x64 = P.t["e_x"].to(torch.float64)
    x0 = torch.where(is1, torch.zeros_like(x64), x64)
    # per-reporter / per-tie sums of x over E0 (deterministic: sorted segments, no atomics)
    g0 = torch.zeros(L * M, dtype=torch.float64, device=dev)
    if I:
        o_lm = torch.sort(lm_all, stable=True)[1]
        cs = torch.cat([x0.new_zeros(1), torch.cumsum(x0[o_lm], 0)])
        bnd = torch.searchsorted(lm_all[o_lm], torch.arange(L * M + 1, device=dev, dtype=torch.int64))
        g0 = cs[bnd[1:]] - cs[bnd[:-1]]
        cs_t = torch.cat([x0.new_zeros(1), torch.cumsum(x0, 0)])
        x0sum = (cs_t[u_ptr[1:]] - cs_t[u_ptr[:-1]])
    else:
        x0sum = torch.zeros(U, dtype=torch.float64, device=dev)
    P.t["g0"] = g0.contiguous()
    P.t["u_x0sum"] = x0sum.to(torch.float32).contiguous()
    # ---- shortcut ties (include/vimure_b200.h, vm_ctx.simple_mode): off the diagonal, in a full column tile, and either
    # SIMPLE (no entry with a reciprocal report) or SINGLE (exactly one entry, with a reciprocal report, reported by the row
    # or the column node).  On iterations without ELBO the dense kernel (k_dense_sc) evaluates them and the special-tie kernel walks
    # `cx_idx`, the others, through compacted copies of their per-tie arrays.
    P.simple_ok = bool(simple and mask.kind == "ego" and K <= 4 and (N * K) % 4 == 0 and N >= TILE_W and P.tile_h <= 128
                       and (split_e0 or not mutuality) and U > 0 and N < (1 << 24))
    u_simple = torch.zeros(U, dtype=torch.bool, device=dev)
    u_single = torch.zeros(U, dtype=torch.bool, device=dev)
    if P.simple_ok:
        has_e1 = torch.zeros(U, dtype=torch.bool, device=dev)
        if P.I1:
            has_e1[P.t["e_u"][e1].to(torch.int64)] = True
        inside = (u_i != u_col) & (u_col < (N // TILE_W) * TILE_W)
        u_simple = P.t["u_has_x"] & ~has_e1 & inside
        if mutuality and split_e0 and single:
            m0 = P.t["u_m0"].to(torch.int64)
            u_single = (P.t["u_cnt"] == 1) & has_e1 & inside & ((m0 == u_i) | (m0 == u_col))
    P.t["u_simple"] = u_simple
    P.t["u_single"] = u_single
    # patch constants of the shortcut ties: X (= x of a SINGLE tie's entry) and +-x^T (sign: reported by the row / column node)
    zf = torch.zeros(U, dtype=torch.float32, device=dev)
    P.t["u_px"] = torch.where(u_simple, P.t["u_x0sum"], torch.where(u_single, P.t["u_x0"], zf)).contiguous()
    P.t["u_pxt"] = torch.where(u_single, torch.where(P.t["u_m0"].to(torch.int64) == u_i, P.t["u_xT0"], -P.t["u_xT0"]),
                               zf).contiguous()
    cx = torch.nonzero(~(u_simple | u_single)).flatten()
    P.n_cx = int(cx.numel())
    P.t["cx_idx"] = _i32(cx)
    P.t["cx_ptr"] = torch.searchsorted(u_l[cx].contiguous(), torch.arange(L + 1, device=dev, dtype=torch.int64)).contiguous()
    n_cxl = int((P.t["cx_ptr"][1:] - P.t["cx_ptr"][:-1]).max()) if L else 0
    P.n_cxblk = max(1, (n_cxl + SPECIAL_TIES_PER_BLOCK - 1) // SPECIAL_TIES_PER_BLOCK)
    if P.simple_ok:  # compacted copies of the per-tie arrays: the list mode of the special-tie kernel reads them coalesced
        for name in ("lrow", "col", "cnt", "m0", "x0", "xT0", "x0sum"):
            P.t["cx_" + name] = P.t["u_" + name][cx].contiguous()
    # layer ranges of the E1 entries (phi pass)
    lay_eptr = torch.searchsorted(e_l[e1].contiguous(), torch.arange(L + 1, device=dev, dtype=torch.int64))
    P.t["lay_eptr"] = lay_eptr.contiguous()
    n_lay = lay_eptr[1:] - lay_eptr[:-1]
    P.n_phichunk = max(1, int((int(n_lay.max()) + PHI_CHUNK - 1) // PHI_CHUNK)) if L else 1
    # reporter-sorted E1 entries (gamma pass)
    lm = lm_all[e1]
    I1 = P.I1
    lm_sorted, gperm = torch.sort(lm, stable=True)
    P.t["g_perm"] = _i32(gperm)
    P.t["g_u"] = P.t["f_u"][gperm].contiguous()
    P.t["g_x"] = P.t["f_x"][gperm].contiguous()
    P.t["g_xT"] = P.t["f_xT"][gperm].contiguous()
    cnt = torch.bincount(lm, minlength=L * M) if I1 else torch.zeros(L * M, dtype=torch.int64, device=dev)
    nch = (cnt + GAMMA_CHUNK - 1) // GAMMA_CHUNK
    cptr = torch.cat([nch.new_zeros(1), torch.cumsum(nch, 0)])
    P.t["g_lm_cptr"] = cptr.contiguous()
    n_gchunk = int(cptr[-1])
    P.n_gchunk = n_gchunk
    chunk_lm = torch.repeat_interleave(torch.arange(L * M, device=dev, dtype=torch.int64), nch)
    estart = torch.cat([cnt.new_zeros(1), torch.cumsum(cnt, 0)])
    within = torch.arange(n_gchunk, device=dev, dtype=torch.int64) - cptr[chunk_lm]
    cstart = estart[chunk_lm] + within * GAMMA_CHUNK
    P.t["g_chunk_lm"] = _i32(chunk_lm)
    P.t["g_chunk_ptr"] = torch.cat([cstart, cstart.new_tensor([I1])]).contiguous()

    _mark("E0/E1 + reporter order")
    # ---- transposed-position list for the eta part of the ELBO (model.py:1269-1290): the X entry (l,i,j,m)
    # is the "X_T" value of the mask entry (l,j,i,m); it belongs to the rank that owns row j
    ownT = (xj >= row0) & (xj < row0 + nloc) & (in_RT > 0)
    st = torch.nonzero(ownT).flatten()
    t_lrow = xl[st] * nloc + (xj[st] - row0)
    t_col = xi[st]
    tkey = t_lrow * N + t_col
    if U and st.numel():
        pos = torch.searchsorted(ukeys, tkey).clamp(max=U - 1)
        t_u = torch.where(ukeys[pos] == tkey, pos, torch.full_like(pos, -1))
    else:
        t_u = torch.full_like(tkey, -1)
    P.IT = int(st.numel())
    P.t["t_u"] = _i32(t_u)
    P.t["t_lrow"] = _i32(t_lrow)
    P.t["t_col"] = _i32(t_col)
    P.t["t_x"] = (xv[st] * in_RT[st]).to(torch.float32).contiguous()
    P.b_all = float(P.t["t_x"].to(torch.float64).sum()) if P.IT else 0.0

    _mark("transposed list")
    # ---- reporter mask
    P.r_mode = {"ego": 0, "all": 1, "coo": 2}[mask.kind]
    P.ego_diag = int(getattr(mask, "diag", False))
    if mask.kind == "ego":
        P.t["rep"] = torch.as_tensor(mask.rep, device=dev).to(torch.uint8).flatten().contiguous()
    elif mask.kind == "coo":
        rs = torch.as_tensor(mask.subs, device=dev)
        rv = torch.as_tensor(mask.vals, device=dev)
        rown = (rs[1] >= row0) & (rs[1] < row0 + nloc)
        rsel = torch.nonzero(rown).flatten()
        rtie = (rs[0][rsel] * nloc + (rs[1][rsel] - row0)) * N + rs[2][rsel]
        rtie_s, ro = torch.sort(rtie, stable=True)
        rsel = rsel[ro]
        T = L * nloc * N
        P.t["r_ptr"] = torch.searchsorted(rtie_s, torch.arange(T + 1, device=dev, dtype=torch.int64)).contiguous()
        P.t["r_m"] = _i32(rs[3][rsel])
        P.t["r_val"] = rv[rsel].to(torch.float32).contiguous()
        rlm = rs[0][rsel] * M + rs[3][rsel]
        rlm_s, co = torch.sort(rlm, stable=True)
        P.t["c_ptr"] = torch.searchsorted(rlm_s, torch.arange(L * M + 1, device=dev, dtype=torch.int64)).contiguous()
        P.t["c_tie"] = rtie_s[co].contiguous()
    _mark("mask arrays")
    return P


def reference_prior_draws(prng, L, N, K, flat_ties_sorted, chunk=1 << 22):
    """The reference draws `prng.rand(L, N, N, K)` (model.py:470) and then keeps the result only on the ties
    that carry an X and an R entry.  Reproduce the stream: consume L*N*N*K doubles in chunks, keeping the K
    values of the requested ties (`flat_ties_sorted` = sorted flat (l,i,j) ids).  Returns (n, K) float64."""
    flat = np.asarray(flat_ties_sorted, dtype=np.int64)
    out = np.empty((flat.size, K), dtype=np.float64)
    T = L * N * N
    per = max(1, chunk // K)
    t0 = 0
    while t0 < T:
        t1 = min(T, t0 + per)
        block = prng.random_sample((t1 - t0) * K)
        a, b = np.searchsorted(flat, t0), np.searchsorted(flat, t1)
        if b > a:
            idx = (flat[a:b] - t0)[:, None] * K + np.arange(K)[None, :]
            out[a:b] = block[idx]
        t0 = t1
    return out
