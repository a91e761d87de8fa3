"""bwtparse of a parse whose in-HBM suffix sort does not fit (pfpb200_bwtparse_file, DESIGN.md §6e): the
bounded path keeps a few bytes per phrase resident, sorts in windows of whole symbol ranges and groups of
suffixes, and writes .ilist / .bwlast / .bwsai in windows.  PFPB200_BWTPARSE_BUDGET=<bytes> makes kilobyte
parses take it.  Every bounded case asserts through pfpb200_bwtparse_plan that round 1 ran in more than one
window, and compares the files byte for byte: with the golden outputs of the unmodified bwtparse, with
the numpy restatement of bwtparse.c, and with the in-HBM path."""
import os
import re
import shutil
import subprocess
import tempfile

import numpy as np
import pytest

from oracle import bwtparse_oracle as bo
from oracle import lf_check
from test_oracle_golden import _bwtparse_golden
from test_pfbwt_gpu import reference_chain, write_fasta

pytestmark = pytest.mark.gpu

OUTS = ("ilist", "bwlast", "bwsai")
INTERMEDIATE = ("dict", "occ", "parse", "last", "sai", "ilist", "bwlast", "bwsai")
INHBM_PER_ROW = 74          # device bytes per row of the in-HBM path with .sai (DESIGN.md §6e), for scaling budgets


@pytest.fixture(scope="module")
def sc(pkg):
    s = pkg.pfp.Scanner(0)
    yield s
    s.close()


@pytest.fixture
def tmp():
    d = tempfile.mkdtemp(prefix="bwtparsewin_")
    yield d
    shutil.rmtree(d, ignore_errors=True)


def _read(base, ext):
    with open(base + "." + ext, "rb") as f:
        return f.read()


def write_inputs(base, parse, last, sai, nseg=0):
    """<base>.parse and .last / .sai, in nseg segment files <base>.<i>.last|sai when nseg > 0"""
    with open(base + ".parse", "wb") as f:
        f.write(parse)
    n = len(last)
    cuts = [n * i // nseg for i in range(nseg + 1)] if nseg else [0, n]
    for ext, data, unit in (("last", last, 1), ("sai", sai, 5)):
        if data is None:
            continue
        for i in range(len(cuts) - 1):
            name = f"{base}.{i}.{ext}" if nseg else f"{base}.{ext}"
            with open(name, "wb") as f:
                f.write(data[unit * cuts[i]:unit * cuts[i + 1]])


def run(sc, monkeypatch, base, sai, nseg=0, budget=None):
    """bwtparse_file under the budget (None: unset) -> (outputs, result with the plan)"""
    if budget is None:
        monkeypatch.delenv("PFPB200_BWTPARSE_BUDGET", raising=False)
    else:
        monkeypatch.setenv("PFPB200_BWTPARSE_BUDGET", str(budget))
    try:
        r = sc.bwtparse_file(base, sai=sai, nseg=nseg)
    finally:
        monkeypatch.delenv("PFPB200_BWTPARSE_BUDGET", raising=False)
    return {ext: _read(base, ext) for ext in OUTS if sai or ext != "bwsai"}, r


def min_budget(pkg, sc, monkeypatch, base, sai, nseg=0):
    """the smallest budget the bounded path takes, from the message of the call that is one byte short"""
    with pytest.raises(pkg.pfp.PfpError) as e:
        run(sc, monkeypatch, base, sai, nseg, budget=1)
    assert e.value.code == -4                                          # PFPB200_E_NOMEM
    need = int(re.search(r"need at least (\d+) bytes", str(e.value)).group(1))
    with pytest.raises(pkg.pfp.PfpError):
        run(sc, monkeypatch, base, sai, nseg, budget=need - 1)
    return need


def budgets(pkg, sc, monkeypatch, base, sai, n, nseg=0):
    """the smallest budget (one symbol or group per window), and the resident arrays plus about 1/16 and
    1/4 of the memory the in-HBM path adds to them"""
    lo = min_budget(pkg, sc, monkeypatch, base, sai, nseg)
    extra = max(INHBM_PER_ROW * (n + 1) - lo, 0)
    return [lo, lo + extra // 16, lo + extra // 4]


def check_bounded(pkg, sc, monkeypatch, base, sai, want, n, nseg=0):
    for b in budgets(pkg, sc, monkeypatch, base, sai, n, nseg):
        got, r = run(sc, monkeypatch, base, sai, nseg, budget=b)
        assert r["windows"] > 1, (base, b)
        assert r["n_out"] == n + 1 and r["peak_device_bytes"] > 0
        for ext in got:
            assert got[ext] == want[ext], (base, b, ext)


@pytest.mark.parametrize("sai", [True, False])
@pytest.mark.parametrize("nseg", [0, 3])
def test_golden_cases_bounded(pkg, sc, monkeypatch, tmp, sai, nseg):
    """every golden case, through the files, at three budgets: the unmodified bwtparse's outputs"""
    for name, c in _bwtparse_golden().items():
        base = os.path.join(tmp, f"{name}_{int(sai)}_{nseg}")
        write_inputs(base, c["parse"], c["last"], c["sai"] if sai else None, nseg)
        check_bounded(pkg, sc, monkeypatch, base, sai, c, len(c["last"]), nseg)


@pytest.mark.parametrize("base_len,haps,w,p", [(200_000, 12, 10, 100), (100_000, 30, 6, 20), (400_000, 4, 4, 10)])
def test_parse_device_parses_bounded(pkg, sc, monkeypatch, tmp, base_len, haps, w, p):
    """parses of pan-genome texts: the bounded path equals the numpy restatement and the in-HBM path"""
    text = pkg.synth.pangenome_text(base_len, haps, 60 + haps, device="cuda")
    files = sc.fetch(sc.parse_device(text, w, p, sai=True))
    base = os.path.join(tmp, "pg")
    write_inputs(base, files.parse, files.last, files.sai)
    il, bl, bs = bo.bwtparse(files.parse, files.last, files.sai)
    full, r = run(sc, monkeypatch, base, True)
    assert r["windows"] == 1                                           # unbudgeted: the in-HBM path
    assert full == {"ilist": il, "bwlast": bl, "bwsai": bs}
    check_bounded(pkg, sc, monkeypatch, base, True, full, len(files.last))


def _synthetic(kind, rng):
    if kind == "periodic":                                             # many rounds, groups far larger than a window
        t = np.concatenate([[1], np.tile([2, 3, 4, 2, 5], 4000)])
    elif kind == "one_symbol":                                         # one symbol holds most occurrences
        t = rng.choice(np.arange(2, 40), 30_000, p=None)
        t[rng.random(t.size) < 0.9] = 7
        t = np.concatenate([[1], t])
    elif kind == "n2":
        t = np.array([1, 2])
    else:                                                              # a long run of one symbol
        t = np.concatenate([[1], np.full(20_000, 3), rng.integers(2, 6, 3000)])
    t = t.astype(np.uint32)
    n = t.size
    return t.tobytes(), rng.integers(65, 91, n).astype(np.uint8).tobytes(), rng.integers(0, 256, 5 * n).astype(np.uint8).tobytes()


@pytest.mark.parametrize("kind", ["periodic", "one_symbol", "n2", "run"])
def test_synthetic_parses_bounded(pkg, sc, monkeypatch, tmp, kind):
    parse, last, sai = _synthetic(kind, np.random.default_rng(len(kind)))
    base = os.path.join(tmp, kind)
    write_inputs(base, parse, last, sai)
    il, bl, bs = bo.bwtparse(parse, last, sai)
    want = {"ilist": il, "bwlast": bl, "bwsai": bs}
    n = len(last)
    if n > 2:
        check_bounded(pkg, sc, monkeypatch, base, True, want, n)
    else:                                                              # n = 2: one symbol per window at the smallest budget
        got, r = run(sc, monkeypatch, base, True, budget=min_budget(pkg, sc, monkeypatch, base, True))
        assert r["windows"] == 2 and got == want
    assert lf_check.check_files(base) == ""


def reference_budget(pkg, sc, monkeypatch, tmp):
    """a budget that takes the bounded path in several windows for the parse of reference_chain()"""
    ref = reference_chain()
    base = os.path.join(tmp, "budget")
    write_inputs(base, ref["parse"], ref["last"], ref["sai"])
    n = len(ref["last"])
    lo = min_budget(pkg, sc, monkeypatch, base, True)
    return lo + max(INHBM_PER_ROW * (n + 1) - lo, 0) // 8


def test_cli_bounded_matches_reference_and_feeds_pfbwt(pkg, sc, monkeypatch, tmp):
    """gpubwtparse.x under the budget: the Plan line, the unmodified bwtparse's files, and gpupfbwt.x on
    them gives the reference's .bwt / .sa"""
    ref = reference_chain()
    base = os.path.join(tmp, "cli")
    for ext in ("dict", "occ", "parse", "last", "sai"):
        with open(base + "." + ext, "wb") as f:
            f.write(ref[ext])
    env = dict(os.environ, PFPB200_BWTPARSE_BUDGET=str(reference_budget(pkg, sc, monkeypatch, tmp)))
    r = subprocess.run([pkg.pfp.BWTPARSE_CLI_PATH, base, "-s"], check=True, stdout=subprocess.PIPE, text=True, env=env)
    m = re.search(r"^Plan: bwtparse (\d+) windows, peak [0-9.]+ GB$", r.stdout, re.M)
    assert m and int(m.group(1)) > 1, r.stdout
    assert "ilist positions written" in r.stdout and "GPU bwtparse:" in r.stdout
    for ext in OUTS:
        assert _read(base, ext) == ref[ext], ext
    subprocess.run([pkg.pfp.PFBWT_CLI_PATH, "-w", str(ref["w"]), base, "-S"], check=True, stdout=subprocess.PIPE)
    for ext in ("bwt", "sa"):
        assert _read(base, ext) == ref[ext], ext
    r = subprocess.run([pkg.pfp.BWTPARSE_CLI_PATH, base, "-s"], check=True, stdout=subprocess.PIPE, text=True)
    assert re.search(r"^Plan: bwtparse 1 windows, peak [0-9.]+ GB$", r.stdout, re.M), r.stdout


def test_bigbwt_all_three_bounded(pkg, sc, monkeypatch, tmp):
    """gpubigbwt.x with the parse streamed, bwtparse bounded and pfbwt in windows, with and without -k, and
    over two ranks (-g 0,0): every file equals the unmodified chain's"""
    ref = reference_chain()
    n = len(ref["last"])
    chars = len(ref["text"]) + 1
    env = dict(os.environ, PFPB200_PARSE_BUDGET=str(8 * (len(ref["text"]) // 5)),
               PFPB200_BWTPARSE_BUDGET=str(reference_budget(pkg, sc, monkeypatch, tmp)),
               PFPB200_PFBWT_BUDGET=str(32 * (chars // 6)))
    for extra in ([], ["-k"], ["-g", "0,0"]):
        path = os.path.join(tmp, "b%d.fa" % len(extra))
        write_fasta(pkg, path, ref["text"])
        r = subprocess.run([pkg.pfp.BIGBWT_CLI_PATH, path, "-f", "-S", *extra], check=True, stdout=subprocess.PIPE,
                           text=True, env=env)
        m = re.search(r"^Plan: bwtparse (\d+) windows, peak [0-9.]+ GB$", r.stdout, re.M)
        assert m and int(m.group(1)) > 1, (extra, r.stdout)
        assert "GPU: parse" in r.stdout
        for ext in ("bwt", "sa"):
            assert _read(path, ext) == ref[ext], (extra, ext)
        for ext in INTERMEDIATE:
            if extra == ["-k"]:
                assert _read(path, ext) == ref[ext], ext
            else:
                assert not os.path.exists(path + "." + ext), (extra, ext)
    # the library call reports the plan of each step
    path = os.path.join(tmp, "lib.fa")
    write_fasta(pkg, path, ref["text"])
    for k in ("PFPB200_PARSE_BUDGET", "PFPB200_BWTPARSE_BUDGET", "PFPB200_PFBWT_BUDGET"):
        monkeypatch.setenv(k, env[k])
    d = sc.bigbwt_file(path, ref["w"], ref["p"], fasta=True, flags=pkg.pfp.PFBWT_SA)
    assert d["parse"]["chunks"] > 0 and d["bwtparse"]["windows"] > 1 and d["pfbwt"]["windows"] > 1
    assert d["bwtparse"]["peak_device_bytes"] > 0 and d["bwtparse"]["n_out"] == n + 1
    assert _read(path, "bwt") == ref["bwt"] and _read(path, "sa") == ref["sa"]


def test_unbudgeted_small_inputs_run_in_hbm(pkg, sc, monkeypatch, tmp):
    ref = reference_chain()
    base = os.path.join(tmp, "u")
    write_inputs(base, ref["parse"], ref["last"], ref["sai"])
    got, r = run(sc, monkeypatch, base, True)
    assert r["windows"] == 1 and r["peak_device_bytes"] > 0
    assert got == {ext: ref[ext] for ext in OUTS}
    path = os.path.join(tmp, "u.fa")
    write_fasta(pkg, path, ref["text"])
    for k in ("PFPB200_PARSE_BUDGET", "PFPB200_BWTPARSE_BUDGET", "PFPB200_PFBWT_BUDGET"):
        monkeypatch.delenv(k, raising=False)
    d = sc.bigbwt_file(path, ref["w"], ref["p"], fasta=True, flags=pkg.pfp.PFBWT_SA)
    assert d["bwtparse"]["windows"] == 1 and d["parse"]["chunks"] == 0


def test_plan_null_context(pkg):
    import ctypes as C
    L = pkg.pfp.load_library()
    n = C.c_uint64(0)
    assert L.pfpb200_bwtparse_plan(None, C.byref(n), None) == -1       # PFPB200_E_ARG
