"""ctypes binding of libpfpb200.so -- the host-side mirror of the reference scanner.

The reference's interface for this stage is the `newscan.x` command line and its five output
files (bigbwt:71-86).  `Scanner` exposes the same knobs (w, p, -s, -f, -c, -t) over the C ABI
declared in include/pfpb200.h.  There is no CPU path here: if the CUDA library is missing or no
GPU is usable, construction raises.
"""
from __future__ import annotations

import ctypes as C
import os
from dataclasses import dataclass, field

import numpy as np

PKG_DIR = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(PKG_DIR, "libpfpb200.so")
CLI_PATH = os.path.join(PKG_DIR, "gpuscan.x")
BWTPARSE_CLI_PATH = os.path.join(PKG_DIR, "gpubwtparse.x")
UNPARSE_CLI_PATH = os.path.join(PKG_DIR, "gpuunparse.x")
PFBWT_CLI_PATH = os.path.join(PKG_DIR, "gpupfbwt.x")
BIGBWT_CLI_PATH = os.path.join(PKG_DIR, "gpubigbwt.x")
PFBWT_SA, PFBWT_SSA, PFBWT_ESA = 1, 2, 4

F_SAI, F_FASTA, F_COMPRESS, F_VERBOSE, F_VERIFY = 1, 2, 4, 8, 16

ERRORS = {0: "OK", -1: "E_ARG", -2: "E_IO", -3: "E_CUDA", -4: "E_NOMEM", -5: "E_LIMIT",
          -6: "E_COLLISION", -7: "E_INTERNAL"}


class PfpError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__(f"pfpb200 {ERRORS.get(code, code)}: {msg}")
        self.code = code


class Opts(C.Structure):
    _fields_ = [("w", C.c_uint32), ("p", C.c_uint32), ("flags", C.c_uint32), ("nseg", C.c_int32)]


class Stats(C.Structure):
    _fields_ = [("n_text", C.c_uint64), ("n_phrases", C.c_uint64), ("n_distinct", C.c_uint64),
                ("sum_word_len", C.c_uint64), ("dict_bytes", C.c_uint64), ("alg_bytes", C.c_uint64),
                ("rank_rounds", C.c_uint32), ("launches", C.c_uint32),
                ("ms_total", C.c_float), ("ms_scan", C.c_float), ("ms_emit", C.c_float),
                ("ms_hash", C.c_float), ("ms_dedup", C.c_float), ("ms_rank", C.c_float),
                ("ms_dict", C.c_float), ("ms_remap", C.c_float), ("ms_h2d", C.c_float),
                ("ms_d2h", C.c_float), ("sec_read", C.c_float), ("sec_write", C.c_float)]

    def as_dict(self):
        return {k: getattr(self, k) for k, _ in self._fields_}


class Outputs(C.Structure):
    _fields_ = [("dict", C.c_void_p), ("dict_bytes", C.c_uint64),
                ("occ", C.c_void_p), ("n_distinct", C.c_uint64),
                ("parse", C.c_void_p), ("n_phrases", C.c_uint64),
                ("last", C.c_void_p), ("sai", C.c_void_p)]


class BwtParseResult(C.Structure):
    """include/pfpb200.h: pfpb200_bwtparse_result."""
    _fields_ = [("ilist", C.c_void_p), ("bwlast", C.c_void_p), ("bwsai", C.c_void_p), ("n_out", C.c_uint64),
                ("alphabet", C.c_uint64), ("rounds", C.c_uint32), ("launches", C.c_uint32),
                ("ms_sa", C.c_float), ("ms_lists", C.c_float), ("ms_total", C.c_float)]

    def as_dict(self):
        return {k: getattr(self, k) for k, _ in self._fields_ if k not in ("ilist", "bwlast", "bwsai")}


class PfbwtResult(C.Structure):
    """include/pfpb200.h: pfpb200_pfbwt_result."""
    _fields_ = [("bwt", C.c_void_p), ("n_bwt", C.c_uint64), ("sa", C.c_void_p), ("n_sa", C.c_uint64),
                ("ssa", C.c_void_p), ("n_ssa", C.c_uint64), ("esa", C.c_void_p), ("n_esa", C.c_uint64),
                ("dict_bytes", C.c_uint64), ("dict_words", C.c_uint64), ("parse_size", C.c_uint64),
                ("easy", C.c_uint64), ("hard", C.c_uint64), ("rounds", C.c_uint32), ("launches", C.c_uint32),
                ("ms_sa", C.c_float), ("ms_fill", C.c_float), ("ms_total", C.c_float)]

    def as_dict(self):
        return {k: getattr(self, k) for k, _ in self._fields_ if k not in ("bwt", "sa", "ssa", "esa")}


class PfbwtRank(C.Structure):
    """include/pfpb200.h: pfpb200_pfbwt_rank (one rank of a sharded pfbwt call)."""
    _fields_ = [("suffixes", C.c_uint64), ("chars", C.c_uint64), ("hard", C.c_uint64), ("peak_bytes", C.c_uint64),
                ("ms_read", C.c_float), ("ms_sort", C.c_float), ("ms_emit", C.c_float), ("ms_write", C.c_float)]

    def as_dict(self):
        return {k: getattr(self, k) for k, _ in self._fields_}


@dataclass
class BwtParseFiles:
    """.ilist / .bwlast / .bwsai as bytes (host copies)."""
    ilist: bytes
    bwlast: bytes
    bwsai: bytes
    stats: dict = field(default_factory=dict)


@dataclass
class PfpFiles:
    """The five output streams as bytes (host copies)."""
    dict: bytes
    occ: bytes
    parse: bytes
    last: bytes
    sai: bytes
    stats: dict = field(default_factory=dict)

    @property
    def n_phrases(self):
        return len(self.parse) // 4

    @property
    def n_distinct(self):
        return len(self.occ) // 4


_lib = None

SYMBOLS = ["pfpb200_create", "pfpb200_destroy", "pfpb200_set_stream", "pfpb200_parse_device",
           "pfpb200_parse_host", "pfpb200_parse_file", "pfpb200_fasta_extract", "pfpb200_fasta_extract_device",
           "pfpb200_read_input",
           "pfpb200_free_host",
           "pfpb200_scan_triggers", "pfpb200_memcpy_d2h", "pfpb200_strerror",
           "pfpb200_shard_scan", "pfpb200_shard_words", "pfpb200_dict_merge", "pfpb200_shard_remap",
           "pfpb200_shard_first_keys", "pfpb200_shard_sample_keys", "pfpb200_shard_route", "pfpb200_shard_route_plan",
           "pfpb200_shard_route_push", "pfpb200_dict_merge_words", "pfpb200_dict_merge_begin",
           "pfpb200_dict_merge_finish",
           "pfpb200_shard_ranks_back", "pfpb200_multi_create", "pfpb200_multi_destroy", "pfpb200_multi_n_gpus",
           "pfpb200_multi_parse_host", "pfpb200_multi_parse_file", "pfpb200_multi_last_error",
           "pfpb200_multi_phase_ms", "pfpb200_multi_pfbwt_file", "pfpb200_multi_pfbwt_ranks",
           "pfpb200_check_dict_order",
           "pfpb200_bwtparse_device", "pfpb200_bwtparse_host", "pfpb200_bwtparse_file",
           "pfpb200_unparse_device", "pfpb200_unparse_file",
           "pfpb200_pfbwt_device", "pfpb200_pfbwt_file", "pfpb200_bigbwt_file",
           "pfpb200_launch_count", "pfpb200_last_error", "pfpb200_abi_version"]


def load_library():
    """dlopen libpfpb200.so and declare prototypes.  Raises if it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ImportError(f"{LIB_PATH} not built: run `python -c 'import __graft_entry__ as g; g.build()'`")
    L = C.CDLL(LIB_PATH)
    vp, u64, u32 = C.c_void_p, C.c_uint64, C.c_uint32
    L.pfpb200_create.argtypes = [C.c_int, C.POINTER(vp)]
    L.pfpb200_create.restype = C.c_int
    L.pfpb200_destroy.argtypes = [vp]
    L.pfpb200_destroy.restype = None
    L.pfpb200_set_stream.argtypes = [vp, vp]
    L.pfpb200_set_stream.restype = C.c_int
    L.pfpb200_parse_device.argtypes = [vp, vp, u64, C.POINTER(Opts), C.POINTER(Outputs), C.POINTER(Stats)]
    L.pfpb200_parse_device.restype = C.c_int
    L.pfpb200_parse_host.argtypes = [vp, vp, u64, C.POINTER(Opts), C.POINTER(Outputs), C.POINTER(Stats)]
    L.pfpb200_parse_host.restype = C.c_int
    L.pfpb200_parse_file.argtypes = [vp, C.c_char_p, C.POINTER(Opts), C.POINTER(Stats)]
    L.pfpb200_parse_file.restype = C.c_int
    L.pfpb200_fasta_extract.argtypes = [vp, u64, vp, C.POINTER(C.c_int)]
    L.pfpb200_fasta_extract.restype = u64
    L.pfpb200_scan_triggers.argtypes = [vp, vp, u64, u64, u64, u64, u32, u32, C.POINTER(vp),
                                        C.POINTER(u64), C.POINTER(C.c_float)]
    L.pfpb200_scan_triggers.restype = C.c_int
    L.pfpb200_memcpy_d2h.argtypes = [vp, vp, vp, u64]
    L.pfpb200_memcpy_d2h.restype = C.c_int
    L.pfpb200_strerror.argtypes = [C.c_int]
    L.pfpb200_strerror.restype = C.c_char_p
    L.pfpb200_last_error.argtypes = [vp]
    L.pfpb200_last_error.restype = C.c_char_p
    L.pfpb200_abi_version.restype = C.c_int
    L.pfpb200_launch_count.argtypes = [vp]
    L.pfpb200_launch_count.restype = C.c_uint32
    L.pfpb200_bwtparse_device.argtypes = [vp, vp, u64, vp, vp, C.POINTER(BwtParseResult)]
    L.pfpb200_bwtparse_device.restype = C.c_int
    L.pfpb200_bwtparse_host.argtypes = [vp, vp, u64, vp, vp, vp, vp, vp, C.POINTER(BwtParseResult)]
    L.pfpb200_bwtparse_host.restype = C.c_int
    L.pfpb200_bwtparse_file.argtypes = [vp, C.c_char_p, C.c_int, C.c_int, C.POINTER(BwtParseResult)]
    L.pfpb200_bwtparse_file.restype = C.c_int
    L.pfpb200_multi_create.argtypes = [C.c_int, C.POINTER(C.c_int), C.POINTER(vp)]
    L.pfpb200_multi_create.restype = C.c_int
    L.pfpb200_multi_destroy.argtypes = [vp]
    L.pfpb200_multi_destroy.restype = None
    L.pfpb200_multi_parse_host.argtypes = [vp, vp, u64, C.POINTER(Opts), C.POINTER(Outputs), C.POINTER(Stats)]
    L.pfpb200_multi_parse_host.restype = C.c_int
    L.pfpb200_multi_parse_file.argtypes = [vp, C.c_char_p, C.POINTER(Opts), C.POINTER(Stats)]
    L.pfpb200_multi_parse_file.restype = C.c_int
    L.pfpb200_multi_last_error.argtypes = [vp]
    L.pfpb200_multi_last_error.restype = C.c_char_p
    L.pfpb200_multi_phase_ms.argtypes = [vp, C.POINTER(C.c_float), C.c_int]
    L.pfpb200_multi_phase_ms.restype = C.c_int
    L.pfpb200_multi_pfbwt_file.argtypes = [vp, C.c_char_p, u32, u32, C.POINTER(PfbwtResult)]
    L.pfpb200_multi_pfbwt_file.restype = C.c_int
    L.pfpb200_multi_pfbwt_ranks.argtypes = [vp, C.POINTER(PfbwtRank), C.c_int]
    L.pfpb200_multi_pfbwt_ranks.restype = C.c_int
    _lib = L
    return L


def fasta_extract(file_bytes) -> tuple[bytes, bool]:
    """Host-side FASTA/FASTQ -> text (kseq semantics); needs the library but no GPU."""
    L = load_library()
    a = np.frombuffer(bytes(file_bytes), dtype=np.uint8)
    out = np.empty(a.size + 1, dtype=np.uint8)
    tr = C.c_int(0)
    n = L.pfpb200_fasta_extract(a.ctypes.data if a.size else None, a.size, out.ctypes.data, C.byref(tr))
    return out[:n].tobytes(), bool(tr.value)


def read_input(path, fasta=False) -> tuple[bytes, bool]:
    """The text the parser sees for `path` (plain, FASTA/FASTQ, gzip-compressed FASTA); no GPU."""
    L = load_library()
    L.pfpb200_read_input.argtypes = [C.c_char_p, C.c_uint32, C.POINTER(C.c_void_p), C.POINTER(C.c_uint64),
                                     C.POINTER(C.c_int)]
    L.pfpb200_read_input.restype = C.c_int
    L.pfpb200_free_host.argtypes = [C.c_void_p]
    L.pfpb200_free_host.restype = None
    ptr, n, tr = C.c_void_p(), C.c_uint64(), C.c_int()
    rc = L.pfpb200_read_input(os.fsencode(path), F_FASTA if fasta else 0, C.byref(ptr), C.byref(n), C.byref(tr))
    if rc != 0:
        raise PfpError(rc, f"cannot read {path}")
    try:
        return C.string_at(ptr, n.value), bool(tr.value)
    finally:
        L.pfpb200_free_host(ptr)


def _flags(sai, fasta, compress, verbose=False, verify=False):
    return (F_SAI if sai else 0) | (F_FASTA if fasta else 0) | (F_COMPRESS if compress else 0) | \
        (F_VERBOSE if verbose else 0) | (F_VERIFY if verify else 0)


class Scanner:
    """One GPU's prefix-free parser: the drop-in for newscan.x / newscanNT.x / pscan.x."""

    def __init__(self, device: int = 0):
        self.L = load_library()
        h = C.c_void_p()
        rc = self.L.pfpb200_create(device, C.byref(h))
        if rc != 0:
            raise PfpError(rc, f"cannot create a context on CUDA device {device}: "
                               f"{self.L.pfpb200_strerror(rc).decode()}")
        self.h = h
        self.device = device
        self.stats = Stats()

    def close(self):
        if getattr(self, "h", None):
            self.L.pfpb200_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _check(self, rc):
        if rc != 0:
            raise PfpError(rc, self.L.pfpb200_last_error(self.h).decode(errors="replace"))

    def set_stream(self, cuda_stream_ptr: int | None):
        self._check(self.L.pfpb200_set_stream(self.h, C.c_void_p(cuda_stream_ptr or 0)))

    # -- text already in HBM (torch uint8 CUDA tensor); returns device pointers + sizes ---------
    def parse_device(self, text, w=10, p=100, sai=True, compress=False, verify=False) -> Outputs:
        assert text.is_cuda and text.dtype.itemsize == 1 and text.is_contiguous()
        o = Opts(w, p, _flags(sai, False, compress, verify=verify), 0)
        out = Outputs()
        self._check(self.L.pfpb200_parse_device(self.h, C.c_void_p(text.data_ptr()), text.numel(),
                                                C.byref(o), C.byref(out), C.byref(self.stats)))
        return out

    def to_host(self, dev_ptr, nbytes) -> bytes:
        if not dev_ptr or nbytes == 0:
            return b""
        buf = np.empty(nbytes, dtype=np.uint8)
        self._check(self.L.pfpb200_memcpy_d2h(self.h, C.c_void_p(buf.ctypes.data), C.c_void_p(dev_ptr),
                                              nbytes))
        return buf.tobytes()

    def fetch(self, out: Outputs) -> PfpFiles:
        """Copy the device outputs of parse_device to host bytes."""
        P, d = out.n_phrases, out.n_distinct
        g = self.to_host
        return PfpFiles(dict=g(out.dict, out.dict_bytes), occ=g(out.occ, 4 * d),
                        parse=g(out.parse, 4 * P), last=g(out.last, P),
                        sai=g(out.sai, 5 * P), stats=self.stats.as_dict())

    # -- text in host memory -----------------------------------------------------------------------
    def parse_host(self, text, w=10, p=100, sai=True, compress=False, copy=True, verify=False) -> PfpFiles:
        a = np.frombuffer(text, dtype=np.uint8) if isinstance(text, (bytes, bytearray, memoryview)) \
            else np.ascontiguousarray(text, dtype=np.uint8)
        o = Opts(w, p, _flags(sai, False, compress, verify=verify), 0)
        out = Outputs()
        self._check(self.L.pfpb200_parse_host(self.h, C.c_void_p(a.ctypes.data if a.size else 0), a.size,
                                              C.byref(o), C.byref(out), C.byref(self.stats)))
        if not copy:
            return out
        P, d = out.n_phrases, out.n_distinct
        s = C.string_at
        return PfpFiles(dict=s(out.dict, out.dict_bytes), occ=s(out.occ, 4 * d), parse=s(out.parse, 4 * P),
                        last=s(out.last, P), sai=s(out.sai, 5 * P) if out.sai else b"",
                        stats=self.stats.as_dict())

    def parse_host_ptr(self, ptr: int, n: int, w=10, p=100, sai=True) -> Outputs:
        """Host pointer (e.g. pinned torch tensor) in, pinned host pointers out; no Python copies."""
        o = Opts(w, p, _flags(sai, False, False), 0)
        out = Outputs()
        self._check(self.L.pfpb200_parse_host(self.h, C.c_void_p(ptr), n, C.byref(o), C.byref(out),
                                              C.byref(self.stats)))
        return out

    # -- file in, files out: what `bigbwt` runs -------------------------------------------------------
    def parse_file(self, path, w=10, p=100, sai=False, fasta=False, compress=False, nseg=0) -> dict:
        o = Opts(w, p, _flags(sai, fasta, compress), nseg)
        self._check(self.L.pfpb200_parse_file(self.h, os.fsencode(path), C.byref(o), C.byref(self.stats)))
        return self.stats.as_dict()

    # -- the stage after the parse: bwtparse (bwtparse.c) ---------------------------------------------
    def bwtparse_device(self, parse_ptr: int, n: int, last_ptr: int, sai_ptr: int | None = None) -> BwtParseResult:
        """Device pointers in (e.g. the Outputs of parse_device on this scanner), device pointers out."""
        r = BwtParseResult()
        self._check(self.L.pfpb200_bwtparse_device(self.h, C.c_void_p(parse_ptr), n, C.c_void_p(last_ptr),
                                                   C.c_void_p(sai_ptr or 0), C.byref(r)))
        return r

    def bwtparse_host(self, parse: bytes, last: bytes, sai: bytes | None = None) -> BwtParseFiles:
        """.parse / .last / .sai bytes in, .ilist / .bwlast / .bwsai bytes out."""
        pa = np.frombuffer(parse, dtype=np.uint32)
        la = np.frombuffer(last, dtype=np.uint8)
        n = pa.size
        sa = np.frombuffer(sai, dtype=np.uint8) if sai else None
        il = np.empty(n + 1, dtype=np.uint32)
        bl = np.empty(n + 1, dtype=np.uint8)
        bs = np.empty(5 * (n + 1), dtype=np.uint8) if sai else None
        r = BwtParseResult()
        self._check(self.L.pfpb200_bwtparse_host(self.h, C.c_void_p(pa.ctypes.data if n else 0), n,
                                                 C.c_void_p(la.ctypes.data if n else 0),
                                                 C.c_void_p(sa.ctypes.data) if sai else None,
                                                 C.c_void_p(il.ctypes.data), C.c_void_p(bl.ctypes.data),
                                                 C.c_void_p(bs.ctypes.data) if sai else None, C.byref(r)))
        return BwtParseFiles(il.tobytes(), bl.tobytes(), bs.tobytes() if sai else b"", r.as_dict())

    def bwtparse_file(self, basename, sai=False, nseg=0) -> dict:
        r = BwtParseResult()
        self._check(self.L.pfpb200_bwtparse_file(self.h, os.fsencode(basename), 1 if sai else 0, nseg, C.byref(r)))
        return r.as_dict()

    # -- the last stage: pfbwt (pfbwt.cpp) ------------------------------------------------------------------
    def pfbwt_device(self, dict_ptr, dict_bytes, occ_ptr, n_words, ilist_ptr, bwlast_ptr, bwsai_ptr, parse_size,
                     w=10, flags=0) -> PfbwtResult:
        """Device pointers in (outputs of parse_device and bwtparse_device on this scanner), device pointers out."""
        self.L.pfpb200_pfbwt_device.argtypes = [C.c_void_p, C.c_void_p, C.c_uint64, C.c_void_p, C.c_uint64, C.c_void_p,
                                                C.c_void_p, C.c_void_p, C.c_uint64, C.c_uint32, C.c_uint32,
                                                C.POINTER(PfbwtResult)]
        self.L.pfpb200_pfbwt_device.restype = C.c_int
        r = PfbwtResult()
        self._check(self.L.pfpb200_pfbwt_device(self.h, C.c_void_p(dict_ptr), dict_bytes, C.c_void_p(occ_ptr), n_words,
                                                C.c_void_p(ilist_ptr), C.c_void_p(bwlast_ptr), C.c_void_p(bwsai_ptr or 0),
                                                parse_size, w, flags, C.byref(r)))
        return r

    def pfbwt_file(self, basename, w=10, flags=0) -> dict:
        self.L.pfpb200_pfbwt_file.argtypes = [C.c_void_p, C.c_char_p, C.c_uint32, C.c_uint32, C.POINTER(PfbwtResult)]
        self.L.pfpb200_pfbwt_file.restype = C.c_int
        r = PfbwtResult()
        self._check(self.L.pfpb200_pfbwt_file(self.h, os.fsencode(basename), w, flags, C.byref(r)))
        return r.as_dict()

    def bigbwt_file(self, path, w=10, p=100, fasta=False, flags=0, keep=False) -> dict:
        """The whole pipeline for a file: <path>.bwt (+ .sa / .ssa / .esa) written, stages in HBM."""
        self.L.pfpb200_bigbwt_file.argtypes = [C.c_void_p, C.c_char_p, C.POINTER(Opts), C.c_uint32, C.c_int,
                                               C.POINTER(Stats), C.POINTER(BwtParseResult), C.POINTER(PfbwtResult)]
        self.L.pfpb200_bigbwt_file.restype = C.c_int
        o = Opts(w, p, _flags(True, fasta, False), 0)
        bp, r = BwtParseResult(), PfbwtResult()
        self._check(self.L.pfpb200_bigbwt_file(self.h, os.fsencode(path), C.byref(o), flags, 1 if keep else 0,
                                               C.byref(self.stats), C.byref(bp), C.byref(r)))
        return {"parse": self.stats.as_dict(), "bwtparse": bp.as_dict(), "pfbwt": r.as_dict()}

    def bwt_of_text(self, text, w=10, p=100, flags=0):
        """The whole pipeline on one context, nothing leaves HBM in between: parse -> bwtparse -> pfbwt.
        `text`: CUDA uint8 tensor.  Returns (PfbwtResult, Outputs of the parse, BwtParseResult)."""
        out = self.parse_device(text, w, p, sai=True)
        bp = self.bwtparse_device(out.parse, out.n_phrases, out.last, out.sai)
        r = self.pfbwt_device(out.dict, out.dict_bytes, out.occ, out.n_distinct, bp.ilist, bp.bwlast, bp.bwsai,
                              bp.n_out, w, flags)
        return r, out, bp

    # -- the inverse of the parse: unparse (unparse.c) ---------------------------------------------------
    def unparse_device(self, dict_ptr: int, dict_bytes: int, parse_ptr: int, n: int, strip_w: int = 0):
        """(device pointer, length, ms) of the text rebuilt from .dicz (strip_w = 0) or .dict (strip_w = w)
        bytes and the parse, all in HBM."""
        self.L.pfpb200_unparse_device.argtypes = [C.c_void_p, C.c_void_p, C.c_uint64, C.c_uint32, C.c_void_p, C.c_uint64,
                                                  C.POINTER(C.c_void_p), C.POINTER(C.c_uint64), C.POINTER(C.c_float)]
        self.L.pfpb200_unparse_device.restype = C.c_int
        ptr, nt, ms = C.c_void_p(), C.c_uint64(), C.c_float()
        self._check(self.L.pfpb200_unparse_device(self.h, C.c_void_p(dict_ptr), dict_bytes, strip_w, C.c_void_p(parse_ptr),
                                                  n, C.byref(ptr), C.byref(nt), C.byref(ms)))
        return ptr.value, nt.value, ms.value

    def unparse_file(self, basename, outname=None) -> dict:
        self.L.pfpb200_unparse_file.argtypes = [C.c_void_p, C.c_char_p, C.c_char_p, C.POINTER(C.c_uint64),
                                                C.POINTER(C.c_uint64), C.POINTER(C.c_float)]
        self.L.pfpb200_unparse_file.restype = C.c_int
        nw, nt, ms = C.c_uint64(), C.c_uint64(), C.c_float()
        self._check(self.L.pfpb200_unparse_file(self.h, os.fsencode(basename), os.fsencode(outname) if outname else None,
                                                C.byref(nw), C.byref(nt), C.byref(ms)))
        return {"n_words": nw.value, "n_text": nt.value, "ms": ms.value}

    def check_dict_order(self, dict_dev, seps_dev) -> int:
        """Adjacent pairs of the .dict stream (CUDA uint8 tensor) that are not strictly increasing;
        seps_dev: int64 CUDA tensor with the positions of the 0x01 terminators.  The library works on
        its own stream: synchronise the stream that produced the tensors first."""
        self.L.pfpb200_check_dict_order.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint64,
                                                    C.POINTER(C.c_uint64)]
        self.L.pfpb200_check_dict_order.restype = C.c_int
        bad = C.c_uint64()
        self._check(self.L.pfpb200_check_dict_order(self.h, C.c_void_p(dict_dev.data_ptr()),
                                                    C.c_void_p(seps_dev.data_ptr()), seps_dev.numel(), C.byref(bad)))
        return bad.value

    # -- K0 alone: FASTA bytes in HBM -> text in HBM ------------------------------------------------------
    def fasta_extract_device(self, file_dev):
        """(text bytes or None, supported) for FASTA bytes held in a CUDA uint8 tensor."""
        self.L.pfpb200_fasta_extract_device.argtypes = [C.c_void_p, C.c_void_p, C.c_uint64, C.POINTER(C.c_void_p),
                                                        C.POINTER(C.c_uint64), C.POINTER(C.c_int)]
        self.L.pfpb200_fasta_extract_device.restype = C.c_int
        ptr, n, ok = C.c_void_p(), C.c_uint64(), C.c_int()
        self._check(self.L.pfpb200_fasta_extract_device(self.h, C.c_void_p(file_dev.data_ptr() if file_dev.numel() else 0),
                                                        file_dev.numel(), C.byref(ptr), C.byref(n), C.byref(ok)))
        if not ok.value:
            return None, False
        return self.to_host(ptr.value, n.value), True

    # -- K1 alone ---------------------------------------------------------------------------------------
    def scan_triggers(self, buf, w=10, p=100, buf_pos0=0, own_lo=0, own_hi=None):
        """Trigger end positions (global, ascending, numpy u64) of a shard in a CUDA uint8 tensor."""
        n = buf.numel()
        if own_hi is None:
            own_hi = buf_pos0 + n
        ptr, cnt, ms = C.c_void_p(), C.c_uint64(), C.c_float()
        self._check(self.L.pfpb200_scan_triggers(self.h, C.c_void_p(buf.data_ptr()), n, buf_pos0, own_lo,
                                                 own_hi, w, p, C.byref(ptr), C.byref(cnt), C.byref(ms)))
        k = cnt.value
        pos = np.frombuffer(self.to_host(ptr.value, 8 * k), dtype=np.uint64)
        return pos, ms.value


PHASES = ("start", "h2d", "scan", "seams", "words", "splitters", "route", "exchange", "merge", "ranks_back",
          "remap", "d2h")


class MultiScanner:
    """Several GPUs of one box behind one call (pfpb200_multi_*): the drop-in for `newscan.x -t T`.
    One process, one host thread per GPU inside the library; no torch, no NCCL."""

    def __init__(self, gpu_ids):
        self.L = load_library()
        ids = (C.c_int * len(gpu_ids))(*gpu_ids)
        h = C.c_void_p()
        rc = self.L.pfpb200_multi_create(len(gpu_ids), ids, C.byref(h))
        if rc != 0:
            raise PfpError(rc, f"cannot create contexts on CUDA devices {list(gpu_ids)}: "
                               f"{self.L.pfpb200_strerror(rc).decode()}")
        self.h, self.gpu_ids, self.stats = h, list(gpu_ids), Stats()

    def close(self):
        if getattr(self, "h", None):
            self.L.pfpb200_multi_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _check(self, rc):
        if rc != 0:
            raise PfpError(rc, self.L.pfpb200_multi_last_error(self.h).decode(errors="replace"))

    def parse_host(self, text, w=10, p=100, sai=True, compress=False, verify=False, copy=True):
        a = np.frombuffer(text, dtype=np.uint8) if isinstance(text, (bytes, bytearray, memoryview)) \
            else np.ascontiguousarray(text, dtype=np.uint8)
        return self.parse_host_ptr(a.ctypes.data if a.size else 0, a.size, w, p, sai, compress, verify, copy)

    def parse_host_ptr(self, ptr, n, w=10, p=100, sai=True, compress=False, verify=False, copy=False):
        o = Opts(w, p, _flags(sai, False, compress, verify=verify), 0)
        out = Outputs()
        self._check(self.L.pfpb200_multi_parse_host(self.h, C.c_void_p(ptr), n, C.byref(o), C.byref(out),
                                                    C.byref(self.stats)))
        if not copy:
            return out
        P, d = out.n_phrases, out.n_distinct
        s = C.string_at
        return PfpFiles(dict=s(out.dict, out.dict_bytes), occ=s(out.occ, 4 * d), parse=s(out.parse, 4 * P),
                        last=s(out.last, P), sai=s(out.sai, 5 * P) if out.sai else b"",
                        stats=self.stats.as_dict())

    def parse_file(self, path, w=10, p=100, sai=False, fasta=False, compress=False, nseg=0) -> dict:
        o = Opts(w, p, _flags(sai, fasta, compress), nseg)
        self._check(self.L.pfpb200_multi_parse_file(self.h, os.fsencode(path), C.byref(o), C.byref(self.stats)))
        return self.stats.as_dict()

    def pfbwt_file(self, basename, w=10, flags=0) -> dict:
        """`pfbwt.x -w W [-S | -s -e] <basename>` sharded over the ranks: reads .dict .occ .ilist .bwlast
        [.bwsai], writes the same .bwt [.sa | .ssa .esa] as Scanner.pfbwt_file.  Returns the summed counts,
        the slowest rank's times and, under "ranks", each rank's suffixes, chars and times."""
        r = PfbwtResult()
        self._check(self.L.pfpb200_multi_pfbwt_file(self.h, os.fsencode(basename), w, flags, C.byref(r)))
        d = r.as_dict()
        buf = (PfbwtRank * len(self.gpu_ids))()
        k = self.L.pfpb200_multi_pfbwt_ranks(self.h, buf, len(self.gpu_ids))
        d["ranks"] = [buf[i].as_dict() for i in range(k)]
        return d

    def phase_ms(self):
        """{phase: [ms of rank 0, rank 1, ...]} of the last parse."""
        n = len(self.gpu_ids) * len(PHASES)
        buf = (C.c_float * n)()
        k = self.L.pfpb200_multi_phase_ms(self.h, buf, n)
        return {ph: [buf[r * len(PHASES) + i] for r in range(k // len(PHASES))] for i, ph in enumerate(PHASES)}
