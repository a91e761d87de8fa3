"""The sharded pfbwt writing every rank's piece in windows (pfpb200_multi_pfbwt_file with
PFPB200_PFBWT_BUDGET per rank, MultiScanner.pfbwt_file, `gpupfbwt.x -g`): the same .bwt / .sa / .ssa /
.esa as the reference and as the one-GPU pfbwt in one piece, byte for byte, whatever the windows.  Device 0
listed several times runs every protocol path on one GPU: the run samples across window borders inside a
rank, across rank borders (the part files and the records dropped when a run crosses), empty ranks, groups
larger than a window and the split key form."""
import ctypes as C
import glob
import os
import shutil
import subprocess
import tempfile

import numpy as np
import pytest

from oracle import pfbwt_oracle as po
from test_oracle_golden import _pfbwt_golden
from test_pfbwt_windows_gpu import WINDOW_BYTES, out_bytes

RANK_LISTS = [[0, 0], [0, 0, 0], [0] * 5]
EXTS = {0: ("bwt",), 1: ("bwt", "sa"), 6: ("bwt", "ssa", "esa")}   # flags 0, -S, -s -e
INPUTS = ("dict", "occ", "ilist", "bwlast", "bwsai")


def test_windows_without_handle_fails(pkg):
    L = pkg.pfp.load_library()
    buf = (C.c_uint64 * 4)(7, 7, 7, 7)
    assert L.pfpb200_multi_pfbwt_windows(None, buf, 4) == -1                   # PFPB200_E_ARG
    assert list(buf) == [7, 7, 7, 7]


@pytest.fixture(scope="module")
def sc(pkg):
    s = pkg.pfp.Scanner(0)
    yield s
    s.close()


@pytest.fixture
def tmp():
    d = tempfile.mkdtemp(prefix="pfbwtmultiwin_")
    yield d
    os.chmod(d, 0o755)
    shutil.rmtree(d, ignore_errors=True)


def _read(base, exts):
    out = {}
    for e in exts:
        with open(f"{base}.{e}", "rb") as f:
            out[e] = f.read()
    return out


def _parts(base):
    return glob.glob(glob.escape(base) + ".ssa.*") + glob.glob(glob.escape(base) + ".esa.*")


def run_multi(ms, monkeypatch, base, w, flags, budget):
    """the sharded pfbwt on <base>.* with a per-rank budget (None: unset); the files and the result"""
    if budget is None:
        monkeypatch.delenv("PFPB200_PFBWT_BUDGET", raising=False)
    else:
        monkeypatch.setenv("PFPB200_PFBWT_BUDGET", str(budget))
    try:
        r = ms.pfbwt_file(base, w, flags)
    finally:
        monkeypatch.delenv("PFPB200_PFBWT_BUDGET", raising=False)
    assert not _parts(base)                                   # the part files are gone
    assert r["easy"] + r["hard"] == r["n_bwt"] and sum(x["chars"] for x in r["ranks"]) == r["n_bwt"]
    return _read(base, EXTS[flags]), r


def budget_for(ms, monkeypatch, base, w, flags, windows):
    """a per-rank budget of about 1 / windows of what the largest piece's output needs"""
    _, r = run_multi(ms, monkeypatch, base, w, flags, None)
    assert all(x["windows"] == (1 if x["suffixes"] else 0) for x in r["ranks"])
    need = max(out_bytes(x["chars"], x["hard"], flags) for x in r["ranks"])
    return max(1, need // windows)


def one_gpu(sc, base, w, flags):
    """the one-GPU pfbwt's files, in one piece"""
    r = sc.pfbwt_file(base, w, flags)
    assert r["windows"] == 1
    return _read(base, EXTS[flags])


def parse_chain(sc, base, text, w, p):
    with open(base, "wb") as f:
        f.write(bytes(text))
    sc.parse_file(base, w, p, sai=True)
    sc.bwtparse_file(base, sai=True)


def piece_borders_inside_runs(bwt, ranks):
    offs = np.cumsum([x["chars"] for x in ranks if x["chars"]])[:-1]
    return sum(1 for o in offs if bwt[o - 1] == bwt[o])


@pytest.mark.gpu
@pytest.mark.parametrize("windows", [1, 4, 16, "group"])
@pytest.mark.parametrize("ids", RANK_LISTS, ids=lambda x: f"{len(x)}ranks")
def test_golden_cases_in_windows_per_rank(pkg, monkeypatch, tmp, ids, windows):
    """The reference's intermediate files in, every rank's piece in windows out: every file equals the
    reference's, at one window, about 4 and about 16 windows per rank, and one group per window."""
    ms = pkg.pfp.MultiScanner(ids)
    try:
        for name, c in _pfbwt_golden().items():
            chars = len(c["text"]) + 1
            if windows == "group" and chars > 20_000:
                continue
            base = os.path.join(tmp, name)
            for ext in INPUTS:
                with open(f"{base}.{ext}", "wb") as f:
                    f.write(c[ext])
            for flags in EXTS:
                budget = (None if windows == 1 else 1 if windows == "group" else
                          budget_for(ms, monkeypatch, base, c["w"], flags, windows))
                got, r = run_multi(ms, monkeypatch, base, c["w"], flags, budget)
                for ext in EXTS[flags]:
                    assert got[ext] == c[ext], (name, ids, windows, flags, ext)
                assert r["n_bwt"] == chars
                most = max(x["windows"] for x in r["ranks"])
                if windows == 1:
                    assert most == 1
                else:
                    assert most > 1, (name, ids, windows, flags)
                if windows == 16:
                    assert most >= 4, (name, ids, flags, most)
    finally:
        ms.close()


@pytest.mark.gpu
@pytest.mark.parametrize("w,p", [(6, 20), (10, 100), (16, 50)])
def test_pangenome_multi_in_windows_equals_single_in_one_piece(pkg, sc, monkeypatch, tmp, w, p):
    text = pkg.synth.pangenome_text(60_000, 12, 40 + w).numpy()
    base = os.path.join(tmp, "pan")
    parse_chain(sc, base, text, w, p)
    ms = pkg.pfp.MultiScanner([0, 0, 0])
    try:
        for flags in EXTS:
            want = one_gpu(sc, base, w, flags)
            got, r = run_multi(ms, monkeypatch, base, w, flags, budget_for(ms, monkeypatch, base, w, flags, 6))
            assert max(x["windows"] for x in r["ranks"]) > 1
            assert got == want, (w, flags)
    finally:
        ms.close()


def _tandem_text(pkg, unit_len, copies, seed):
    unit = pkg.synth.random_dna(unit_len, seed).numpy().tobytes()
    return (pkg.synth.random_dna(20_000, seed + 1).numpy().tobytes() + unit * copies +
            pkg.synth.random_dna(20_000, seed + 2).numpy().tobytes())


@pytest.mark.gpu
def test_runs_across_window_and_rank_borders(pkg, sc, monkeypatch, tmp):
    """Tandem repeats: BWT runs longer than a window cross window borders inside a rank and the borders
    between ranks.  At a rank border inside a run, the next piece's first -s record and the previous
    piece's last -e record both go; the files equal the reference and the one-GPU output."""
    text = _tandem_text(pkg, 211, 3000, 21)
    want = po.pfbwt(text)
    base = os.path.join(tmp, "tr")
    parse_chain(sc, base, text, 10, 100)
    se = pkg.pfp.PFBWT_SSA | pkg.pfp.PFBWT_ESA
    assert one_gpu(sc, base, 10, se) == {e: want[e] for e in EXTS[se]}
    a = np.frombuffer(want["bwt"], np.uint8)
    assert int(np.diff(np.flatnonzero(np.concatenate([[True], a[1:] != a[:-1], [True]]))).max()) > 2 * 997
    inside = 0
    for ids in ([0, 0, 0], [0] * 7):
        ms = pkg.pfp.MultiScanner(ids)
        try:
            for cap in (None, 997, 131):
                got, r = run_multi(ms, monkeypatch, base, 10, se, None if cap is None else WINDOW_BYTES * cap)
                for ext in EXTS[se]:
                    assert got[ext] == want[ext], (ids, cap, ext)
                if cap is not None:
                    assert max(x["windows"] for x in r["ranks"]) > 1, (ids, cap)
                inside += piece_borders_inside_runs(got["bwt"], r["ranks"])
        finally:
            ms.close()
    assert inside >= 1                                        # a rank border inside a run of the BWT


@pytest.mark.gpu
def test_long_n_runs_leave_ranks_empty_with_windows_on_the_others(pkg, sc, monkeypatch, tmp):
    rng = np.random.default_rng(11)
    parts = []
    for i in range(6):
        parts += [pkg.synth.random_dna(3_000, 100 + i).numpy(), np.full(int(rng.integers(20_000, 40_000)), ord("N"), np.uint8)]
    base = os.path.join(tmp, "nruns")
    parse_chain(sc, base, np.concatenate(parts), 10, 100)
    ms = pkg.pfp.MultiScanner([0] * 5)
    try:
        for flags in EXTS:
            want = one_gpu(sc, base, 10, flags)
            got, r = run_multi(ms, monkeypatch, base, 10, flags, budget_for(ms, monkeypatch, base, 10, flags, 4))
            assert got == want, flags
            assert any(x["suffixes"] == 0 and x["windows"] == 0 for x in r["ranks"])
            assert max(x["windows"] for x in r["ranks"]) > 1
    finally:
        ms.close()


@pytest.mark.gpu
def test_group_larger_than_a_ranks_window(pkg, sc, monkeypatch, tmp):
    """Words with thousands of occurrences and windows of 50 chars: such a group takes a window of its own."""
    text = _tandem_text(pkg, 157, 2000, 31)
    want = po.pfbwt(text)
    base = os.path.join(tmp, "big")
    parse_chain(sc, base, text, 10, 100)
    assert np.frombuffer(_read(base, ["occ"])["occ"], np.uint32).max() > 1000
    ms = pkg.pfp.MultiScanner([0, 0, 0])
    try:
        for flags in (pkg.pfp.PFBWT_SA, pkg.pfp.PFBWT_SSA | pkg.pfp.PFBWT_ESA):
            got, r = run_multi(ms, monkeypatch, base, 10, flags, WINDOW_BYTES * 50)
            assert 1 < sum(x["windows"] for x in r["ranks"]) < len(text) // 50
            for ext in EXTS[flags]:
                assert got[ext] == want[ext], (flags, ext)
    finally:
        ms.close()


@pytest.mark.gpu
def test_split_key_form_in_windows(pkg, monkeypatch, tmp):
    monkeypatch.setenv("PFPB200_MULTI_SPLIT_KEY", "1")
    ms = pkg.pfp.MultiScanner([0, 0, 0])
    try:
        for name in ("pangenome_20k_x6_w10_p100", "low_complexity_w4_p11"):
            c = _pfbwt_golden()[name]
            base = os.path.join(tmp, name)
            for ext in INPUTS:
                with open(f"{base}.{ext}", "wb") as f:
                    f.write(c[ext])
            for flags in EXTS:
                got, r = run_multi(ms, monkeypatch, base, c["w"], flags, budget_for(ms, monkeypatch, base, c["w"], flags, 5))
                assert max(x["windows"] for x in r["ranks"]) > 1
                for ext in EXTS[flags]:
                    assert got[ext] == c[ext], (name, flags, ext)
    finally:
        ms.close()


@pytest.mark.gpu
@pytest.mark.skipif(hasattr(os, "geteuid") and os.geteuid() == 0, reason="root writes into read-only directories")
def test_no_part_files_after_a_write_error(pkg, monkeypatch, tmp):
    """The output directory read-only (the final files already there and writable): the ranks cannot
    create their part files, the call fails with PFPB200_E_IO and leaves no part file behind."""
    P = pkg.pfp
    c = _pfbwt_golden()["pangenome_20k_x6_w10_p100"]
    base = os.path.join(tmp, "ro")
    for ext in INPUTS:
        with open(f"{base}.{ext}", "wb") as f:
            f.write(c[ext])
    se = P.PFBWT_SSA | P.PFBWT_ESA
    ms = P.MultiScanner([0, 0, 0])
    try:
        run_multi(ms, monkeypatch, base, c["w"], se, None)
        os.chmod(tmp, 0o555)
        with pytest.raises(P.PfpError) as e:
            ms.pfbwt_file(base, c["w"], se)
        assert e.value.code == -2                                  # PFPB200_E_IO
        assert not _parts(base)
        os.chmod(tmp, 0o755)
        got, _ = run_multi(ms, monkeypatch, base, c["w"], se, 4096)
        assert got == {e: c[e] for e in EXTS[se]}
    finally:
        os.chmod(tmp, 0o755)
        ms.close()


def _devs(n):
    import torch
    k = torch.cuda.device_count()
    return ",".join(map(str, range(n))) if k >= n else ",".join(["0"] * n)


@pytest.mark.gpu
def test_cli_device_list_with_a_budget(pkg, sc, tmp):
    """`gpupfbwt.x -g 0,0,0` with a small per-rank budget writes the files of the one-GPU CLI and prints
    the windows of every rank; `gpubigbwt.x -g` prints them as well."""
    text = pkg.synth.pangenome_text(40_000, 8, 77).numpy()
    base = os.path.join(tmp, "cli")
    parse_chain(sc, base, text, 10, 100)
    cli = pkg.pfp.PFBWT_CLI_PATH
    env = dict(os.environ, PFPB200_PFBWT_BUDGET=str(WINDOW_BYTES * 2000))
    for flags, exts in ((["-S"], ("bwt", "sa")), (["-s", "-e"], ("bwt", "ssa", "esa"))):
        subprocess.run([cli, "-w", "10", *flags, base], check=True, stdout=subprocess.PIPE)
        want = _read(base, exts)
        for e in exts:
            os.remove(f"{base}.{e}")
        r = subprocess.run([cli, "-w", "10", *flags, "-g", _devs(3), base], check=True, stdout=subprocess.PIPE,
                           text=True, env=env)
        assert _read(base, exts) == want
        assert r.stdout.count("(rank ") == 3
        line = [x for x in r.stdout.splitlines() if x.startswith("Plan: output windows per rank: ")]
        assert len(line) == 1
        counts = [int(x) for x in line[0].rsplit(": ", 1)[1].split(",")]
        assert len(counts) == 3 and max(counts) > 1
        assert not _parts(base)
    path = os.path.join(tmp, "big")
    with open(path, "wb") as f:
        f.write(text.tobytes())
    r = subprocess.run([pkg.pfp.BIGBWT_CLI_PATH, path, "-g", _devs(2)], check=True, stdout=subprocess.PIPE, text=True,
                       env=env)
    line = [x for x in r.stdout.splitlines() if x.startswith("Plan: output windows per rank: ")]
    assert len(line) == 1 and len(line[0].rsplit(": ", 1)[1].split(",")) == 2
