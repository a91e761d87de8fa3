"""Linear check of bwtparse's outputs (.ilist, .bwlast, .bwsai) against its inputs (.parse, .last, .sai).

TEST INFRASTRUCTURE ONLY: used by tests/ and tools/ as the checker of parses too large for the oracle's
suffix sort; nothing under big-bwt_b200/ may import this.  The check is plain C (oracle/lf_check.c, which
states what it checks), compiled on first use into a temporary directory and called through ctypes.
"""
from __future__ import annotations

import atexit
import ctypes as C
import os
import shutil
import subprocess
import tempfile

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
_lib = None


def _load():
    global _lib
    if _lib is None:
        d = tempfile.mkdtemp(prefix="lf_check_")
        atexit.register(shutil.rmtree, d, True)
        so = os.path.join(d, "liblf_check.so")
        subprocess.check_call([os.environ.get("CC", "cc"), "-O2", "-std=c99", "-shared", "-fPIC", "-o", so,
                               os.path.join(HERE, "lf_check.c")])
        L = C.CDLL(so)
        vp = C.c_void_p
        L.lf_check.argtypes = [vp, C.c_uint64, vp, vp, vp, vp, vp, C.c_uint64, C.c_char_p, C.c_int]
        L.lf_check.restype = C.c_int
        _lib = L
    return _lib


def _arr(x, dtype):
    if x is None:
        return None
    if isinstance(x, (bytes, bytearray, memoryview)):
        return np.frombuffer(x, dtype=dtype)
    return np.ascontiguousarray(x).view(dtype)


def check(parse, last, sai, ilist, bwlast, bwsai) -> str:
    """parse (u32 symbols), last, sai (5 bytes per phrase, or None) and the three outputs, as bytes or
    numpy arrays.  Returns "" when the outputs are bwtparse's for these inputs, else what is wrong."""
    t, la, sv = _arr(parse, np.uint32), _arr(last, np.uint8), _arr(sai, np.uint8)
    il, bl, bs = _arr(ilist, np.uint32), _arr(bwlast, np.uint8), _arr(bwsai, np.uint8)
    n = t.size
    if la.size != n or (sv is not None and sv.size != 5 * n):
        return f"inputs: {n} phrases, {la.size} .last bytes, {None if sv is None else sv.size} .sai bytes"
    if bl.size != il.size or (sv is not None and (bs is None or bs.size != 5 * il.size)):
        return f"outputs: {il.size} .ilist entries, {bl.size} .bwlast bytes, {None if bs is None else bs.size} .bwsai bytes"
    msg = C.create_string_buffer(512)
    ptr = lambda a: None if a is None or a.size == 0 else a.ctypes.data
    rc = _load().lf_check(ptr(t), n, ptr(la), ptr(sv), ptr(il), ptr(bl), ptr(bs) if sv is not None else None,
                          il.size, msg, len(msg))
    return "" if rc == 0 else msg.value.decode()


def check_files(base, sai=True) -> str:
    """check() on <base>.parse .last [.sai] .ilist .bwlast [.bwsai], memory-mapped"""
    m = lambda ext, dt: np.memmap(f"{base}.{ext}", dtype=dt, mode="r")
    return check(m("parse", np.uint32), m("last", np.uint8), m("sai", np.uint8) if sai else None,
                 m("ilist", np.uint32), m("bwlast", np.uint8), m("bwsai", np.uint8) if sai else None)
