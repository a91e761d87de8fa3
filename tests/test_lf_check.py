"""The linear LF-walk check of bwtparse's outputs (oracle/lf_check.c) on the CPU: it accepts the outputs of
the unmodified bwtparse and of the numpy restatement, and rejects each kind of damage it is meant to see."""
import numpy as np

from oracle import bwtparse_oracle as bo
from oracle import lf_check
from test_oracle_golden import _bwtparse_golden


def _damaged(c, rng):
    """(what, ilist, bwlast, bwsai) with one defect each"""
    il = np.frombuffer(c["ilist"], np.uint32).copy()
    bl = np.frombuffer(c["bwlast"], np.uint8).copy()
    bs = np.frombuffer(c["bwsai"], np.uint8).copy()
    i, j = sorted(rng.choice(il.size, 2, replace=False))
    sw = il.copy()
    sw[i], sw[j] = sw[j], sw[i]
    yield "swapped ilist entries", sw, bl, bs
    k = int(rng.integers(bl.size))
    b2 = bl.copy()
    b2[k] ^= 0x20
    yield "changed bwlast byte", il, b2, bs
    k = int(rng.integers(1, bl.size))                        # a row with a suffix-array value > 0
    s2 = bs.copy()
    s2[5 * k] ^= 1
    yield "changed bwsai value", il, bl, s2


def test_accepts_reference_outputs_and_rejects_damage():
    rng = np.random.default_rng(3)
    for name, c in _bwtparse_golden().items():
        assert lf_check.check(c["parse"], c["last"], c["sai"], c["ilist"], c["bwlast"], c["bwsai"]) == "", name
        assert lf_check.check(c["parse"], c["last"], None, c["ilist"], c["bwlast"], None) == "", name
        for what, il, bl, bs in _damaged(c, rng):
            assert lf_check.check(c["parse"], c["last"], c["sai"], il, bl, bs) != "", (name, what)


def test_accepts_oracle_outputs_of_synthetic_parses():
    rng = np.random.default_rng(4)
    for t in (np.array([1, 2]), np.concatenate([[1], np.tile([2, 3, 4], 500)]),
              np.concatenate([[1], rng.integers(2, 9, 3000)])):
        parse = t.astype(np.uint32).tobytes()
        last = rng.integers(65, 91, t.size).astype(np.uint8).tobytes()
        sai = rng.integers(0, 256, 5 * t.size).astype(np.uint8).tobytes()
        il, bl, bs = bo.bwtparse(parse, last, sai)
        assert lf_check.check(parse, last, sai, il, bl, bs) == ""
        bad = np.frombuffer(il, np.uint32).copy()
        bad[-1], bad[-2] = bad[-2], bad[-1]
        assert lf_check.check(parse, last, sai, bad, bl, bs) != ""
