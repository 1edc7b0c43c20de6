"""ctypes binding of tests/sim/libjpsim.so — the CPU simulation of the kernels' algorithm
(test infrastructure; see tests/sim/jpsim.cpp)."""
import ctypes as C
import os
import subprocess
import sys

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(_HERE)
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
from jpeg_rust_b200 import _ffi  # noqa: E402

_lib = None


def lib():
    global _lib
    if _lib is None:
        path = os.environ.get("JPSIM_LIB") or os.path.join(_HERE, "sim", "libjpsim.so")   # JPSIM_LIB: e.g. an ASAN build
        if not os.path.exists(path):
            subprocess.check_call(["make", "-s", "-C", ROOT, "tests/sim/libjpsim.so"])
        L = C.CDLL(path)
        L.jpgpu_parse.argtypes = [C.c_void_p, C.c_size_t, C.c_uint32, C.c_uint32, C.POINTER(_ffi.ImageDesc)]
        L.jpsim_decode_batch.argtypes = [C.POINTER(_ffi.ImageDesc), C.c_size_t, C.POINTER(C.c_void_p),
                                         C.POINTER(C.c_void_p), C.POINTER(C.c_size_t), C.POINTER(C.c_uint32),
                                         C.POINTER(C.c_int32), C.POINTER(C.c_uint64), C.POINTER(C.c_uint64), C.c_uint32]
        L.jpsim_idct_8x8.argtypes = [C.c_void_p, C.c_void_p]
        _lib = L
    return _lib


class SimResult:
    pass


def decode_scans(files, layout=_ffi.LAYOUT_SPEC, ext=_ffi.EXT_NONE, sub_bits=0):
    """Files that may hold one non-interleaved scan per component (jpgpu_parse_scans): every scan a descriptor of the
    one simulated batch.  Returns (list of HxWx3 arrays, statuses, per file the list of per-scan SimResult)."""
    from jpeg_rust_b200.jpeg import parse_scans
    descs, owners, first, count = [], [], [], []
    for f in files:
        st, ds, buf = parse_scans(f, ext, layout)
        assert st == 0, st
        first.append(len(descs)); count.append(len(ds))
        descs += ds; owners.append(buf)
    rs, _ = decode_batch(None, layout=layout, ext=ext, sub_bits=sub_bits, descs=descs)
    outs = [rs[first[i]].rgb for i in range(len(files))]
    return outs, [rs[first[i]].status for i in range(len(files))], [rs[first[i]:first[i] + count[i]] for i in range(len(files))]


def decode_batch(files, layout=_ffi.LAYOUT_SPEC, ext=_ffi.EXT_NONE, sub_bits=0, descs=None):
    """files: list of bytes (or descs: a list of ready descriptors). Returns (list of SimResult, diag)."""
    L = lib()
    if descs is not None:
        n = len(descs)
        arr = (_ffi.ImageDesc * n)(*descs)
        descs = arr
        parse_status = [0] * n
    else:
        n = len(files)
        descs = (_ffi.ImageDesc * n)()
        bufs = [np.frombuffer(f, np.uint8).copy() for f in files]
        parse_status = []
        for i, b in enumerate(bufs):
            parse_status.append(L.jpgpu_parse(b.ctypes.data, len(b), ext, layout, C.byref(descs[i])))

    def out_shape(d):   # a frame's first scan owns the frame's pixels, further scans none
        if d.frame_part == 1:
            return (d.frame_height, d.frame_width, 3)
        if d.frame_part == 2:
            return (1, 1, 3)
        return (max(1, d.height), max(1, d.width), 3)
    rgb = [np.zeros(out_shape(descs[i]), np.uint8) for i in range(n)]
    cap = [(((descs[i].width + 15) // 16 + 1) * ((descs[i].height + 15) // 16 + 1) * 12 * 64) for i in range(n)]
    coefs = [np.zeros(cap[i], np.int16) for i in range(n)]
    rgb_p = (C.c_void_p * n)(*[a.ctypes.data for a in rgb])
    coef_p = (C.c_void_p * n)(*[a.ctypes.data for a in coefs])
    caps = (C.c_size_t * n)(*cap)
    nblocks = (C.c_uint32 * (4 * n))()
    statuses = (C.c_int32 * n)()
    bytes_read = (C.c_uint64 * n)()
    diag = (C.c_uint64 * 8)()
    st = L.jpsim_decode_batch(descs, n, rgb_p, coef_p, caps, nblocks, statuses, bytes_read, diag, sub_bits)
    assert st == 0, st
    out = []
    for i in range(n):
        r = SimResult()
        r.parse_status = parse_status[i]
        r.status = statuses[i] if parse_status[i] == 0 else parse_status[i]
        r.width, r.height, r.ncomp = descs[i].width, descs[i].height, descs[i].ncomp
        r.rgb = rgb[i]
        r.bytes_read = bytes_read[i]
        nb = [nblocks[4 * i + c] for c in range(4)]
        r.coefs = []
        off = 0
        for c in range(r.ncomp):
            r.coefs.append(coefs[i][off:off + nb[c] * 64].reshape(-1, 64))
            off += nb[c] * 64
        out.append(r)
    return out, {"repair_iters": diag[0], "repairs": diag[1], "sync_decodes": diag[2], "flush_phases": diag[3],
                 "sync_digest": diag[4], "max_broken": diag[5],
                 "crowded_rounds": diag[6]}


def set_sync_multi(on):
    """The simulated synchronisation pass through the multi-symbol tables (default, as the product) or symbol by symbol."""
    lib().jpsim_set_sync_multi(1 if on else 0)


def idct_8x8(block_natural):
    a = np.ascontiguousarray(block_natural, np.float32).reshape(64)
    out = np.empty(64, np.float32)
    lib().jpsim_idct_8x8(a.ctypes.data, out.ctypes.data)
    return out.reshape(8, 8)
