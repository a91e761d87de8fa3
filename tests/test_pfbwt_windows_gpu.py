"""pfbwt's outputs in windows (pfpb200_pfbwt_file, pfpb200_bigbwt_file): when the BWT and its suffix-array
outputs do not fit the device memory left once the plan is done, they are produced one run of whole
groups of equal dictionary suffixes at a time and written to the files at their offsets.
PFPB200_PFBWT_BUDGET=<bytes> makes kilobyte inputs take that path (windows of the most chars whose
output fits the budget); every windowed case asserts through pfpb200_pfbwt_plan that it ran in more than one window, and compares the
files byte for byte with the reference's (golden outputs of the unmodified chain, or the suffix array of
the text)."""
import ctypes as C
import os
import shutil
import subprocess
import tempfile

import numpy as np
import pytest

from oracle import pfbwt_oracle as po
from test_oracle_golden import _pfbwt_golden
from test_pfbwt_gpu import reference_chain, write_fasta

WINDOW_BYTES = 32           # device bytes per BWT char of a window with a suffix array whose chars are all hard
EXTS = {0: ("bwt",), 1: ("bwt", "sa"), 6: ("bwt", "ssa", "esa")}   # flags 0, -S, -s -e


def out_bytes(c, hard, flags):
    """device bytes of the output of c BWT chars with at most `hard` hard occurrences (pb_out_bytes, pfp_pfbwt.cu)"""
    merge = 25 * min(c, hard, 1 << 30)
    sample = 22 * c if flags & 6 else 0
    return c * (2 + (5 if flags else 0)) + max(merge, sample)


@pytest.fixture(scope="module")
def sc(pkg):
    s = pkg.pfp.Scanner(0)
    yield s
    s.close()


@pytest.fixture
def tmp():
    d = tempfile.mkdtemp(prefix="pfbwtwin_")
    yield d
    shutil.rmtree(d, ignore_errors=True)


def _read(base, ext):
    with open(base + "." + ext, "rb") as f:
        return f.read()


def run_pfbwt(sc, monkeypatch, base, w, flags, budget):
    """pfbwt_file on <base>.* with the budget knob (None: unset); the outputs and the call's result"""
    if budget is None:
        monkeypatch.delenv("PFPB200_PFBWT_BUDGET", raising=False)
    else:
        monkeypatch.setenv("PFPB200_PFBWT_BUDGET", str(budget))
    r = sc.pfbwt_file(base, w, flags)
    monkeypatch.delenv("PFPB200_PFBWT_BUDGET", raising=False)
    return {ext: _read(base, ext) for ext in EXTS[flags]}, r


def budget_for(sc, monkeypatch, base, w, flags, windows):
    """a budget of about 1 / windows of what the whole output needs (from a one-window run's counts)"""
    _, r = run_pfbwt(sc, monkeypatch, base, w, flags, None)
    assert r["windows"] == 1
    return max(1, out_bytes(r["n_bwt"], r["hard"], flags) // windows)


def test_plan_without_context_fails(pkg):
    L = pkg.pfp.load_library()
    n, pk = C.c_uint64(7), C.c_uint64(7)
    assert L.pfpb200_pfbwt_plan(None, C.byref(n), C.byref(pk)) == -1          # PFPB200_E_ARG
    assert (n.value, pk.value) == (7, 7)


@pytest.mark.gpu
@pytest.mark.parametrize("windows", [1, 4, 16, "group"])
def test_golden_cases_in_windows(pkg, sc, monkeypatch, tmp, windows):
    """The reference's intermediate files in, windowed outputs out: every file equals the reference's, in
    one window, about 4, about 16, and one group per window (budget 1 byte: the smaller cases only)."""
    for name, c in _pfbwt_golden().items():
        chars = len(c["text"]) + 1
        if windows == "group" and chars > 20_000:
            continue
        base = os.path.join(tmp, name)
        for ext in ("dict", "occ", "ilist", "bwlast", "bwsai"):
            with open(base + "." + ext, "wb") as f:
                f.write(c[ext])
        for flags in (0, pkg.pfp.PFBWT_SA, pkg.pfp.PFBWT_SSA | pkg.pfp.PFBWT_ESA):
            budget = (None if windows == 1 else 1 if windows == "group" else
                      budget_for(sc, monkeypatch, base, c["w"], flags, windows))
            got, r = run_pfbwt(sc, monkeypatch, base, c["w"], flags, budget)
            for ext in EXTS[flags]:
                assert got[ext] == c[ext], (name, windows, flags, ext)
            assert r["n_bwt"] == chars and r["easy"] + r["hard"] == chars
            if windows == 1:
                assert r["windows"] == 1
            else:
                assert r["windows"] > 1, (name, windows, flags)
            if windows == 16:
                assert r["windows"] >= 4, (name, flags, r["windows"])


@pytest.mark.gpu
@pytest.mark.parametrize("base_len,haps,w,p", [(60_000, 20, 6, 20), (150_000, 10, 10, 100), (40_000, 8, 16, 50)])
def test_pangenome_files_in_windows_vs_suffix_array_of_the_text(pkg, sc, monkeypatch, tmp, base_len, haps, w, p):
    """gpuscan -> bwtparse -> windowed pfbwt through the files, against the suffix array of the text."""
    text = pkg.synth.pangenome_text(base_len, haps, 90 + haps).numpy().tobytes()
    want = po.pfbwt(text)
    base = os.path.join(tmp, "pg")
    with open(base, "wb") as f:
        f.write(text)
    sc.parse_file(base, w, p, sai=True)
    sc.bwtparse_file(base, sai=True)
    for flags, k in ((pkg.pfp.PFBWT_SA, 5), (pkg.pfp.PFBWT_SSA | pkg.pfp.PFBWT_ESA, 13), (0, 3)):
        got, r = run_pfbwt(sc, monkeypatch, base, w, flags, budget_for(sc, monkeypatch, base, w, flags, k))
        assert r["windows"] > 1
        for ext in EXTS[flags]:
            assert got[ext] == want[ext], (w, flags, ext)


def _tandem_text(pkg, unit_len, copies, seed):
    unit = pkg.synth.random_dna(unit_len, seed).numpy().tobytes()
    return (pkg.synth.random_dna(20_000, seed + 1).numpy().tobytes() + unit * copies +
            pkg.synth.random_dna(20_000, seed + 2).numpy().tobytes())


def _longest_run(bwt):
    a = np.frombuffer(bwt, np.uint8)
    starts = np.flatnonzero(np.concatenate([[True], a[1:] != a[:-1], [True]]))
    return int(np.diff(starts).max())


@pytest.mark.gpu
def test_window_borders_inside_bwt_runs(pkg, sc, monkeypatch, tmp):
    """Tandem repeats: BWT runs longer than twice a window, so window borders fall inside runs; the run
    samples across them (-s: the char in front of a window, -e: the pending run end) equal the one-window
    output and the reference, over a sweep of budgets."""
    text = _tandem_text(pkg, 211, 3000, 21)
    want = po.pfbwt(text)
    longest = _longest_run(want["bwt"])
    base = os.path.join(tmp, "tr")
    with open(base, "wb") as f:
        f.write(text)
    sc.parse_file(base, 10, 100, sai=True)
    sc.bwtparse_file(base, sai=True)
    se = pkg.pfp.PFBWT_SSA | pkg.pfp.PFBWT_ESA
    one, r = run_pfbwt(sc, monkeypatch, base, 10, se, None)
    assert r["windows"] == 1 and one["ssa"] == want["ssa"] and one["esa"] == want["esa"]
    for cap in (longest // 3, longest // 5 + 7, 997, 131):
        assert longest > 2 * cap
        got, r = run_pfbwt(sc, monkeypatch, base, 10, se, WINDOW_BYTES * cap)
        assert r["windows"] > 1, cap
        assert got == one, cap


@pytest.mark.gpu
def test_group_larger_than_the_budget(pkg, sc, monkeypatch, tmp):
    """Words with thousands of occurrences and windows of 50 chars: such a group gets a window of its own
    (its merge larger than the window), and the outputs are right."""
    text = _tandem_text(pkg, 157, 2000, 31)
    want = po.pfbwt(text)
    base = os.path.join(tmp, "big")
    with open(base, "wb") as f:
        f.write(text)
    sc.parse_file(base, 10, 100, sai=True)
    sc.bwtparse_file(base, sai=True)
    occ = np.frombuffer(_read(base, "occ"), np.uint32)
    assert occ.max() > 1000
    for flags in (pkg.pfp.PFBWT_SA, pkg.pfp.PFBWT_SSA | pkg.pfp.PFBWT_ESA):
        got, r = run_pfbwt(sc, monkeypatch, base, 10, flags, WINDOW_BYTES * 50)
        assert 1 < r["windows"] < len(text) // 50
        for ext in EXTS[flags]:
            assert got[ext] == want[ext], (flags, ext)


INTERMEDIATE = ("dict", "occ", "parse", "last", "sai", "ilist", "bwlast", "bwsai")


@pytest.mark.gpu
def test_gpubigbwt_streamed_parse_and_windows_match_the_reference_chain(pkg, sc, monkeypatch, tmp):
    """gpubigbwt.x with both knobs set: the streamed parse through the files, bwtparse, windowed pfbwt.
    Every file equals the unmodified chain's; without -k no intermediate file is left."""
    ref = reference_chain()
    chars = len(ref["text"]) + 1
    env = dict(os.environ, PFPB200_PARSE_BUDGET=str(8 * (len(ref["text"]) // 5)),
               PFPB200_PFBWT_BUDGET=str(WINDOW_BYTES * (chars // 6)))   # below the 7 B per char of any SA output
    for flags, exts in ((["-S"], ("bwt", "sa")), (["-s", "-e"], ("bwt", "ssa", "esa"))):
        for keep in (True, False):
            path = os.path.join(tmp, "k.fa" if keep else "nk.fa")
            write_fasta(pkg, path, ref["text"])
            r = subprocess.run([pkg.pfp.BIGBWT_CLI_PATH, path, "-f", *flags] + (["-k"] if keep else []), check=True,
                               stdout=subprocess.PIPE, text=True, env=env)
            assert "GPU: parse" in r.stdout and "Plan: parse" in r.stdout
            for ext in exts:
                assert _read(path, ext) == ref[ext], (flags, keep, ext)
            for ext in INTERMEDIATE:
                if keep:
                    assert _read(path, ext) == ref[ext], (flags, ext)
                else:
                    assert not os.path.exists(path + "." + ext), (flags, ext)
    # the library call reports both plans
    path = os.path.join(tmp, "lib.fa")
    write_fasta(pkg, path, ref["text"])
    monkeypatch.setenv("PFPB200_PARSE_BUDGET", env["PFPB200_PARSE_BUDGET"])
    monkeypatch.setenv("PFPB200_PFBWT_BUDGET", env["PFPB200_PFBWT_BUDGET"])
    d = sc.bigbwt_file(path, 10, 100, fasta=True, flags=pkg.pfp.PFBWT_SA)
    assert d["parse"]["chunks"] > 0 and d["pfbwt"]["windows"] > 1
    assert d["pfbwt"]["peak_device_bytes"] > 0
    assert _read(path, "bwt") == ref["bwt"] and _read(path, "sa") == ref["sa"]
    assert not any(os.path.exists(path + "." + ext) for ext in INTERMEDIATE)
