"""ctypes binding of the C ABI declared in include/vimure_b200.h.

There is NO CPU fallback: if the CUDA library is missing this module raises, loudly.
The `vm_ctx` mirror is generated from the header itself (single source of truth) and its size is checked
against `vm_ctx_size()` at load time.
"""
import ctypes
import os
import re

HERE = os.path.dirname(os.path.abspath(__file__))
HEADER = os.path.join(os.path.dirname(HERE), "include", "vimure_b200.h")
LIB_PATH = os.environ.get("VIMURE_B200_LIB") or os.path.join(HERE, "_lib", "libvimure_b200.so")

_lib = None
_ctx_cls = None
_consts = None


def _parse_struct(src, name):
    body = re.search(r"typedef struct %s \{(.*?)\}\s*%s;" % (name, name), src, re.S).group(1)
    body = re.sub(r"/\*.*?\*/", "", body, flags=re.S)
    fields = []
    for decl in body.split(";"):
        decl = " ".join(decl.split())
        if not decl:
            continue
        m = re.match(r"(const\s+)?(\w+)\s*(.*)$", decl)
        base, rest = m.group(2), m.group(3)
        for name in rest.split(","):
            name = name.strip()
            ptr = name.startswith("*") or base.endswith("*")
            name = name.lstrip("* ")
            if ptr:
                ctype = ctypes.c_void_p
            elif base == "int64_t":
                ctype = ctypes.c_int64
            elif base == "uint64_t":
                ctype = ctypes.c_uint64
            elif base == "double":
                ctype = ctypes.c_double
            else:
                raise RuntimeError("%s may only hold int64_t/double/pointers, got %r" % (name, decl))
            fields.append((name, ctype))
    return fields


def _parse_header():
    src = open(HEADER).read()
    consts = {m.group(1): int(m.group(2), 0) for m in re.finditer(r"#define\s+(VM_\w+)\s+\(?(-?\d+)\)?\s", src)}
    return _parse_struct(src, "vm_ctx"), consts


_synth_cls = None
_synth_mask_cls = None
_pack_cls = None
_edges_cls = None


def pack_class():
    """ctypes mirror of `vm_pack_args` (device-side packer), generated from the header."""
    global _pack_cls
    if _pack_cls is None:
        fields = _parse_struct(open(HEADER).read(), "vm_pack_args")

        class VmPackArgs(ctypes.Structure):
            _fields_ = fields

        _pack_cls = VmPackArgs
    return _pack_cls


def synth_class():
    """ctypes mirror of `vm_synth` (device-side synthetic reports), generated from the header."""
    global _synth_cls
    if _synth_cls is None:
        fields = _parse_struct(open(HEADER).read(), "vm_synth")

        class VmSynth(ctypes.Structure):
            _fields_ = fields

        _synth_cls = VmSynth
    return _synth_cls


def synth_mask_class():
    """ctypes mirror of `vm_synth_mask` (explicit mask of `vm_synth_masked`), generated from the header."""
    global _synth_mask_cls
    if _synth_mask_cls is None:
        fields = _parse_struct(open(HEADER).read(), "vm_synth_mask")

        class VmSynthMask(ctypes.Structure):
            _fields_ = fields

        _synth_mask_cls = VmSynthMask
    return _synth_mask_cls


def edges_class():
    """ctypes mirror of `vm_edges_args` (sparse consumers), generated from the header."""
    global _edges_cls
    if _edges_cls is None:
        fields = _parse_struct(open(HEADER).read(), "vm_edges_args")

        class VmEdgesArgs(ctypes.Structure):
            _fields_ = fields

        _edges_cls = VmEdgesArgs
    return _edges_cls


def header_symbols():
    """Names of every function the header declares."""
    src = open(HEADER).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(?:int|int64_t)\s+(vm_\w+)\s*\(", src)))


def ctx_class():
    global _ctx_cls, _consts
    if _ctx_cls is None:
        fields, _consts = _parse_header()

        class VmCtx(ctypes.Structure):
            _fields_ = fields

        _ctx_cls = VmCtx
    return _ctx_cls


def consts():
    ctx_class()
    return _consts


def load():
    """Load the CUDA library (building is `__graft_entry__.build()` / `python -m vimure_b200.build`)."""
    global _lib
    if _lib is None:
        _lib = open_library(LIB_PATH)
    return _lib


def open_library(path):
    """dlopen `path`, declare the prototypes of the header's entry points and verify the ABI (not cached: the A/B timing
    tool opens several builds of the library in one process)."""
    if not os.path.exists(path):
        raise RuntimeError(
            "vimure_b200: CUDA library %s is missing -- run `python -m vimure_b200.build` (needs nvcc). "
            "There is no CPU fallback." % path)
    lib = ctypes.CDLL(path)
    Ctx = ctx_class()
    P = ctypes.POINTER(Ctx)
    vp, i, i64, d = ctypes.c_void_p, ctypes.c_int, ctypes.c_int64, ctypes.c_double
    protos = {
        "vm_ctx_size": (i64, []),
        "vm_abi_version": (i64, []),
        "vm_dense_tile_w": (i64, [i64]),
        "vm_refresh_cache": (i, [P, vp]),
        "vm_init_stats": (i, [P, vp]),
        "vm_phase_gamma": (i, [P, vp]),
        "vm_phase_phi": (i, [P, vp]),
        "vm_phase_rho": (i, [P, i, vp]),
        "vm_phase_finish": (i, [P, i, vp]),
        "vm_dense_only": (i, [P, i, vp]),
        "vm_iteration": (i, [P, i, vp]),
        "vm_run": (i, [P, i, i, i, vp]),
        "vm_materialize_prior": (i, [P, vp]),
        "vm_materialize_rows": (i, [P, i64, i64, vp, vp]),
        "vm_infer": (i, [P, i, d, vp, vp]),
        "vm_sample": (i, [P, i64, ctypes.c_uint64, vp, vp]),
        "vm_infer_mean": (i, [P, vp, vp]),
        "vm_edges_size": (i64, []),
        "vm_edges_count": (i, [P, ctypes.POINTER(edges_class()), vp]),
        "vm_edges_emit": (i, [P, ctypes.POINTER(edges_class()), vp]),
        "vm_rho_at": (i, [P, i64, i64, vp, vp, vp]),
        "vm_test_special": (i, [vp, vp, vp, i64, vp]),
        "vm_pack_size": (i64, []),
        "vm_pack_workspace_bytes": (i64, [ctypes.POINTER(pack_class())]),
        "vm_pack": (i, [ctypes.POINTER(pack_class()), vp]),
        "vm_synth_size": (i64, []),
        "vm_synth_ego": (i, [ctypes.POINTER(synth_class()), vp]),
        "vm_synth_all": (i, [ctypes.POINTER(synth_class()), vp]),
        "vm_synth_mask_size": (i64, []),
        "vm_synth_masked": (i, [ctypes.POINTER(synth_class()), ctypes.POINTER(synth_mask_class()), vp]),
    }
    for name, (res, args) in protos.items():
        fn = getattr(lib, name)
        fn.restype = res
        fn.argtypes = args
    if lib.vm_ctx_size() != ctypes.sizeof(Ctx):
        raise RuntimeError("vm_ctx layout mismatch: library %d bytes, python mirror %d bytes (stale build?)"
                           % (lib.vm_ctx_size(), ctypes.sizeof(Ctx)))
    if lib.vm_pack_size() != ctypes.sizeof(pack_class()):
        raise RuntimeError("vm_pack_args layout mismatch between header and library (stale build?)")
    if lib.vm_synth_size() != ctypes.sizeof(synth_class()):
        raise RuntimeError("vm_synth layout mismatch between header and library (stale build?)")
    if lib.vm_synth_mask_size() != ctypes.sizeof(synth_mask_class()):
        raise RuntimeError("vm_synth_mask layout mismatch between header and library (stale build?)")
    if lib.vm_edges_size() != ctypes.sizeof(edges_class()):
        raise RuntimeError("vm_edges_args layout mismatch between header and library (stale build?)")
    if lib.vm_abi_version() != consts()["VM_ABI_VERSION"]:
        raise RuntimeError("vimure_b200: ABI version mismatch between header and library (stale build?)")
    return lib


def check(rc, what):
    if rc != 0:
        if rc > 0:
            raise RuntimeError("vimure_b200: %s failed with cudaError %d" % (what, rc))
        raise RuntimeError("vimure_b200: %s failed with error code %d (see include/vimure_b200.h)" % (what, rc))
