"""pfp_arith.h (shared by the device kernels and the host): the division-free forms against plain
`%` arithmetic -- newscan.cpp:194-202 (window hash mod 1999999973) and :344,367 (hash % p == 0)."""
import ctypes as C
import os
import subprocess
import tempfile

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PW = 1999999973

SRC = r"""
#include "pfp_arith.h"
uint32_t t_reduce(uint64_t t) { return pfp_reduce_pw(t); }
uint32_t t_roll(uint32_t h, uint32_t cin, uint32_t cout, uint32_t negw) { return pfp_roll(h, cin, cout, negw); }
uint32_t t_push(uint32_t h, uint32_t c) { return pfp_push(h, c); }
int t_trig(uint32_t r, uint32_t w, uint32_t p) { pfp_scan_consts c = pfp_make_scan_consts(w, p);
    return pfp_is_trigger(r, c.pinv, c.pshift, c.plimit); }
uint32_t t_negw(uint32_t w) { return pfp_make_scan_consts(w, 100).negw; }
"""


@pytest.fixture(scope="module")
def lib():
    tmp = tempfile.mkdtemp(prefix="pfparith_")
    src, so = os.path.join(tmp, "a.c"), os.path.join(tmp, "a.so")
    with open(src, "w") as f:
        f.write(SRC)
    subprocess.check_call(["gcc", "-O2", "-shared", "-fPIC", "-I", os.path.join(ROOT, "big-bwt_b200", "csrc"),
                           "-o", so, src])
    L = C.CDLL(so)
    L.t_reduce.argtypes = [C.c_uint64]; L.t_reduce.restype = C.c_uint32
    L.t_roll.argtypes = [C.c_uint32] * 4; L.t_roll.restype = C.c_uint32
    L.t_push.argtypes = [C.c_uint32] * 2; L.t_push.restype = C.c_uint32
    L.t_trig.argtypes = [C.c_uint32] * 3; L.t_trig.restype = C.c_int
    L.t_negw.argtypes = [C.c_uint32]; L.t_negw.restype = C.c_uint32
    return L


def test_reduce_below_2_41(lib):
    rng = np.random.default_rng(1)
    vals = [0, 1, PW - 1, PW, PW + 1, 2 * PW - 1, 2 * PW, (1 << 41) - 1, (1 << 40), 255 * PW + 7]
    vals += [int(x) for x in rng.integers(0, 1 << 41, 20000, dtype=np.uint64)]
    vals += [k * PW + d for k in (1, 2, 1000, 1099) for d in (-1, 0, 1)]
    for t in vals:
        if 0 <= t < (1 << 41):
            assert lib.t_reduce(t) == t % PW, t


@pytest.mark.parametrize("w", [4, 6, 10, 16, 32])
def test_roll_is_the_reference_update(lib, w):
    """h' = (256 h + c_in - c_out 256^w) mod PW, as KR_window::addchar computes it."""
    rng = np.random.default_rng(w)
    negw = lib.t_negw(w)
    assert negw == (PW - pow(256, w, PW)) % PW
    for _ in range(20000):
        h, cin, cout = int(rng.integers(0, PW)), int(rng.integers(0, 256)), int(rng.integers(0, 256))
        want = (256 * h + cin - cout * pow(256, w, PW)) % PW
        assert lib.t_roll(h, cin, cout, negw) == want
    for h in (0, PW - 1):
        for cin in (0, 255):
            for cout in (0, 255):
                assert lib.t_roll(h, cin, cout, negw) == (256 * h + cin - cout * pow(256, w, PW)) % PW
                assert lib.t_push(h, cin) == (256 * h + cin) % PW


@pytest.mark.parametrize("p", [10, 11, 16, 50, 64, 100, 500, 1000, 1024, 99991, 1 << 20])
def test_divisibility_test(lib, p):
    rng = np.random.default_rng(p)
    vals = [0, 1, p - 1, p, p + 1, PW - 1, (PW // p) * p, (PW // p) * p - 1, 0xFFFFFFFF // p * p]
    vals += [int(x) for x in rng.integers(0, PW, 20000)]
    vals += [int(x) * p for x in rng.integers(0, PW // p, 5000)]
    for r in vals:
        assert bool(lib.t_trig(r, 10, p)) == (r % p == 0), (r, p)


# ---- the interval form of the scan (kr_scan_iv_k): both tables modelled in numpy over ALL 4^10 windows ----
def _interval_tables(w, p):
    """What dna_etab_k builds: per 5-symbol block x the exact partial hashes Ah (x as the w-5 older
    symbols of a window, 5 places up) and Bl (x as the 5 newest), and E = (a16 + 2) << 16 | b16 with
    a16 = floor(Ah u 2^16 / PW), b16 = floor(Bl u 2^16 / PW), u = p^-1 mod PW."""
    letters = np.array([65, 67, 84, 71], dtype=np.int64)
    x = np.arange(1024, dtype=np.int64)
    bl = np.zeros(1024, dtype=np.int64)
    ah = np.zeros(1024, dtype=np.int64)
    for j in range(5):
        c = letters[(x >> (2 * j)) & 3]
        if w - 5 + j >= 0:
            bl = (bl * 256 + c) % PW
        if w - 10 + j >= 0:
            ah = (ah * 256 + c) % PW
    ah = (ah * pow(256, 5, PW)) % PW
    u = pow(p, -1, PW)
    a_s = np.array([(int(a) * u) % PW for a in ah], dtype=np.int64)
    b_s = np.array([(int(b) * u) % PW for b in bl], dtype=np.int64)
    e = ((((a_s << 16) // PW + 2) & 0xFFFF) << 16) | ((b_s << 16) // PW)
    theta = ((((PW - 1) // p) + 1) << 16) // PW
    return ah, bl, e.astype(np.uint64), (theta + 4) << 16


@pytest.mark.parametrize("w,p", [(4, 10), (5, 11), (6, 50), (7, 99991), (8, 16), (9, 1000), (10, 10), (10, 100),
                                 (10, 65536), (10, 1999999), (10, PW - 1)])
def test_interval_form_candidates_cover_every_trigger(w, p):
    ah, bl, e, cthr = _interval_tables(w, p)
    assert cthr < 1 << 32
    idx = np.arange(1 << 20, dtype=np.int64)             # a window of 10 symbols, oldest in the lowest bits
    hi, lo = idx & 1023, idx >> 10
    letters = np.array([65, 67, 84, 71], dtype=np.int64)
    h = np.zeros_like(idx)
    for k in range(10 - w, 10):                           # the last w symbols are the window
        h = (h * 256 + letters[(idx >> (2 * k)) & 3]) % PW
    assert np.array_equal((ah[hi] + bl[lo]) % PW, h)      # linearity: the exact tables of the second stage
    trig = (h % p) == 0
    t = ((e[lo] << np.uint64(16)) + e[hi]) & np.uint64(0xFFFFFFFF)
    cand = t < np.uint64(cthr)
    assert not np.any(trig & ~cand)                       # no trigger is missed by the 16-bit interval test
    assert cand.sum() - trig.sum() <= 200                 # and next to nothing else passes it


def _interval_tables4(w, p):
    """What dna_etab4_k builds for 11 <= w <= 16: per 4-symbol block x and role r (the block ends 4 r
    symbols before the window's end) the exact partial hash F[r][x] and f16 = floor(F u 2^16 / PW)."""
    letters = np.array([65, 67, 84, 71], dtype=np.int64)
    x = np.arange(256, dtype=np.int64)
    F = np.zeros((4, 256), dtype=np.int64)
    for r in range(4):
        for j in range(4):
            dist = 4 * r + (3 - j)
            if dist < w:
                F[r] = (F[r] + letters[(x >> (2 * j)) & 3] * pow(256, dist, PW)) % PW
    u = pow(p, -1, PW)
    f16 = np.array([[((int(a) * u) % PW << 16) // PW for a in F[r]] for r in range(4)], dtype=np.int64)
    lo = (f16[1] << 16) | f16[0]
    hi = (((f16[3] + 5) & 0xFFFF) << 16) | f16[2]
    theta = ((((PW - 1) // p) + 1) << 16) // PW
    return F, lo, hi, (theta + 7) << 16


@pytest.mark.parametrize("w,p", [(11, 100), (12, 50), (13, 1000), (14, 10), (15, 500), (16, 100), (16, 10), (16, 65536)])
def test_interval_form_four_blocks_candidates_cover_every_trigger(w, p):
    F, lo, hi, cthr = _interval_tables4(w, p)
    assert cthr < 1 << 32
    rng = np.random.default_rng(1000 * w + p)
    n = 4_000_000
    codes = rng.integers(0, 4, (n, 16))                                   # 16 symbols, oldest first
    letters = np.array([65, 67, 84, 71], dtype=np.int64)
    h = np.zeros(n, dtype=np.int64)
    for k in range(16 - w, 16):
        h = (h * 256 + letters[codes[:, k]]) % PW
    xs = [sum(codes[:, 15 - 4 * r - (3 - j)] << (2 * j) for j in range(4)) for r in range(4)]    # block of role r
    assert np.array_equal((F[0][xs[0]] + F[1][xs[1]] + F[2][xs[2]] + F[3][xs[3]]) % PW, h)       # linearity
    trig = (h % p) == 0
    t = ((lo[xs[0]] << 16) + lo[xs[1]] + (hi[xs[2]] << 16) + hi[xs[3]]) & 0xFFFFFFFF
    cand = t < cthr
    assert not np.any(trig & ~cand)
    assert cand.sum() - trig.sum() <= 2000
