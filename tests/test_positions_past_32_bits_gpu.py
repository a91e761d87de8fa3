"""Suffix-array values and BWT positions that need more than 32 bits.

Part A (small, every GPU run).  pfbwt reads .bwsai only to compute suffix-array values (bwsai[ip] - len,
and bwsai[0] - w for the EOF suffix), so adding a constant C to every .bwsai value leaves .bwt unchanged
and adds C to every .sa value and to the value of every .ssa / .esa record, whose position stays.  With
C = 2^31 - m and 2^32 - m (m: half the text length) the values straddle the int32 and uint32 limits; with
C = 2^40 - 1 - max(bwsai) all five bytes are in use at the top of the range.  The expected files are the
unshifted ones (pinned to the reference by the other tests) shifted on the host in numpy uint64, and for
-S also the reference's algorithm restated in Python integers (oracle/pfbwt_oracle.py) on the shifted
.bwsai.  Every output path takes them: pfbwt_device in one window, pfbwt_file in about 4 windows and in
one group per window, the sharded pfbwt on 2 and 3 ranks in windows, and gpupfbwt.x with and without -g.
bwtparse copies .sai values into .bwsai: shifted .sai in, shifted .bwsai out.

Part B (full size, gated by free device memory and disk like test_fullsize_gpu.py).  One text longer
than 2^32, config 2 with ten more haplotypes (40 Mbp x 110, 4.4e9 chars), through the whole chain in five
arms run one after another, each deleting its outputs before the next:
  1. parse_device -> bwtparse_device -> pfbwt_device -S in HBM; the .sa values checked in linear time
     against the text (oracle/sa_check.py) on the device, once the library's buffers are released;
  2. the same chain with -s -e: .ssa / .esa equal the run starts / ends of arm 1's checked BWT and SA
     (skipped when the one-window output does not fit the free device memory, see the test);
  3. pfbwt_file in at least 4 windows, -S and -s -e: the files equal arms 1 and 2 (sha256);
  4. MultiScanner([0, 0]).pfbwt_file with a per-rank budget, -S and -s -e: the same files;
  5. gpubigbwt.x -S on the text file, the parse streamed in at least 4 chunks and pfbwt in at least 4
     windows: the .sai the streamed parse writes across chunk borders, bwtparse from the files and the
     windowed pfbwt give arm 1's .bwt / .sa.
Measured on one B200 (1000 W power limit; profiles/r11_positions_past_32_bits.log): the dictionary is
0.89 GB, so the one-GPU pfbwt applies; 105 M of the 4.4 G SA values and 1.9 M of the 81 M run starts are
>= 2^32.  In arms 1 and 2 the library's arena takes the card's free memory, so arm 1 copies .sa and .bwt
to the host (26 GB of RAM) before it closes the library; its checks then peak at 104 GB of device memory.
pfbwt's own peaks: arm 3 70 GB, arm 4 44 and 43 GB per rank, arm 5 61 GB (parse 6.5 GB).  .bwt and .sa
take 26 GB of disk.  Wall times: arms 1-5 40, 11, 43, 44 and 44 s; Part A and the checker's self-test
19 s in all.
"""
import hashlib
import os
import re
import shutil
import subprocess
import tempfile
import time

import numpy as np
import pytest
import torch

from oracle import bwtparse_oracle as bo
from oracle import pfbwt_oracle as po
from oracle import sa_check
from test_oracle_golden import _bwtparse_golden, _pfbwt_golden
from test_pfbwt_multi_windows_gpu import budget_for as multi_budget_for, run_multi
from test_pfbwt_windows_gpu import _tandem_text, budget_for, out_bytes, run_pfbwt

EXTS = {1: ("bwt", "sa"), 6: ("bwt", "ssa", "esa")}       # flags -S, -s -e
INPUTS = ("dict", "occ", "ilist", "bwlast", "bwsai")
TOP = (1 << 40) - 1


def get5(b):
    a = np.frombuffer(b, np.uint8).reshape(-1, 5).astype(np.uint64)
    return sum(a[:, j] << np.uint64(8 * j) for j in range(5))


def put5(v):
    v = np.asarray(v, np.uint64)
    return np.stack([(v >> np.uint64(8 * j)) & np.uint64(255) for j in range(5)], axis=1).astype(np.uint8).tobytes()


def shifted(b, c):
    """every 5-byte value of b plus c"""
    v = get5(b)
    assert int(v.max()) + c <= TOP
    return put5(v + np.uint64(c))


def shifted_records(b, c):
    """(BWT position, SA value) records with c added to the values"""
    v = get5(b).reshape(-1, 2)
    v[:, 1] += np.uint64(c)
    return put5(v.reshape(-1))


def shifts(n_text, bwsai):
    m = n_text // 2
    return {"int32": (1 << 31) - m, "uint32": (1 << 32) - m, "top": TOP - int(get5(bwsai).max())}


def expected(case, c, flags):
    want = case["want"]
    if flags == 1:
        return {"bwt": want["bwt"], "sa": shifted(want["sa"], c)}
    return {"bwt": want["bwt"], "ssa": shifted_records(want["ssa"], c), "esa": shifted_records(want["esa"], c)}


# ---- checker self-test (CPU) ------------------------------------------------------------------------------
def _reference_arrays(text):
    want = po.pfbwt(text)
    n = len(text)
    sa = torch.from_numpy(np.concatenate([[n], get5(want["sa"]).astype(np.int64)]))
    return torch.frombuffer(bytearray(text), dtype=torch.uint8), sa, torch.frombuffer(bytearray(want["bwt"]), dtype=torch.uint8), want


def _checker_texts():
    rng = np.random.default_rng(7)
    acgt = np.frombuffer(b"ACGT", np.uint8)
    rand = acgt[rng.integers(0, 4, 3000)].tobytes()
    periodic = b"ACGTTGCAA" * 400 + b"ACG"
    runs = b"".join(bytes([int(acgt[rng.integers(0, 4)])]) * int(rng.integers(1, 200)) for _ in range(60))
    return {"random": rand, "periodic": periodic, "runs": runs}


@pytest.mark.parametrize("kind", ["random", "periodic", "runs"])
def test_linear_checks_accept_the_suffix_array_and_reject_corruptions(tmp_path, kind):
    """oracle/sa_check.py accepts the suffix array and BWT of the text (chunk sizes that do and do not
    divide the rows) and rejects each corruption: two adjacent rows swapped, a repeated value, a value
    off by one either way, a changed BWT char, the EOF char on another row."""
    text = _checker_texts()[kind]
    T, sa, bwt, want = _reference_arrays(text)
    n = len(text)
    for chunk in (n + 1, 1000, 97):
        assert sa_check.linear_checks(T, sa, bwt, chunk=chunk) == [], (kind, chunk)
    path = str(tmp_path / "x.sa")
    with open(path, "wb") as f:
        f.write(want["sa"])
    assert torch.equal(sa_check.load_sa(path, n, "cpu", chunk=333), sa)
    assert sa_check.encode5(sa[1:]).numpy().tobytes() == want["sa"]
    eof = int(torch.nonzero(sa == 0)[0])
    rows = [1, n // 2, n - 1, eof]

    def bad(s, b):
        return sa_check.linear_checks(T, s, b, chunk=97)
    for i in rows:                                   # rows i, i + 1 swapped, with their BWT chars
        i = min(i, n - 1)
        s, b = sa.clone(), bwt.clone()
        s[[i, i + 1]] = s[[i + 1, i]]
        b[[i, i + 1]] = b[[i + 1, i]]
        assert any("out of order" in f for f in bad(s, b)), (kind, "swap", i)
        s = sa.clone()
        s[i] = s[i + 1]                              # a repeated value
        assert bad(s, bwt) == ["the suffix array is not a permutation of [0, n]"], (kind, "repeat", i)
        for d in (-1, 1):
            s = sa.clone()
            s[i] = s[i] + d if 0 <= int(s[i]) + d <= n else s[i] - d
            assert bad(s, bwt), (kind, "off by one", i, d)
        b = bwt.clone()
        if i != eof:
            b[i] = ord("A") if int(b[i]) != ord("A") else ord("C")
            assert any("bwt[i]" in f for f in bad(sa, b)), (kind, "char", i)
    for j in sorted({0, eof - 1, min(eof + 1, n)} - {eof}):   # the EOF char moved to another row
        b = bwt.clone()
        b[[eof, j]] = b[[j, eof]]
        assert any("EOF" in f for f in bad(sa, b)), (kind, "eof", j)


# ---- Part A: shifted .bwsai on every output path ----------------------------------------------------------
@pytest.fixture(scope="module")
def sc(pkg):
    s = pkg.pfp.Scanner(0)
    yield s
    s.close()


@pytest.fixture(scope="module")
def mtmp():
    d = tempfile.mkdtemp(prefix="pos40_")
    yield d
    shutil.rmtree(d, ignore_errors=True)


def _read(base, ext):
    with open(f"{base}.{ext}", "rb") as f:
        return f.read()


def _text_case(sc, d, name, text, w, p):
    """the chain's files of a text (gpuscan -> bwtparse through the files) and the reference outputs"""
    base = os.path.join(d, name)
    with open(base, "wb") as f:
        f.write(text)
    sc.parse_file(base, w, p, sai=True)
    sc.bwtparse_file(base, sai=True)
    files = {e: _read(base, e) for e in INPUTS + ("parse", "last", "sai")}
    return {"w": w, "n": len(text), "files": files, "want": po.pfbwt(text)}


@pytest.fixture(scope="module")
def cases(pkg, sc, mtmp):
    out = {}
    for name, c in _pfbwt_golden().items():
        out[name] = {"w": c["w"], "n": len(c["text"]), "files": {e: c[e] for e in INPUTS},
                     "want": {e: c[e] for e in ("bwt", "sa", "ssa", "esa")}}
    text = pkg.synth.pangenome_text(60_000, 12, 46).numpy().tobytes()
    out["pangenome_60k_x12"] = _text_case(sc, mtmp, "pg", text, 10, 100)
    out["tandem_211x3000"] = _text_case(sc, mtmp, "tr", _tandem_text(pkg, 211, 3000, 21), 10, 100)
    return out


TEXT_CASES = ["pangenome_60k_x12", "tandem_211x3000"]
CASE_NAMES = sorted(_pfbwt_golden()) + TEXT_CASES


def _dev(b):
    return torch.from_numpy(np.frombuffer(b, dtype=np.uint8).copy()).cuda()


def _write_inputs(base, case, c):
    for e in INPUTS:
        with open(f"{base}.{e}", "wb") as f:
            f.write(shifted(case["files"][e], c) if e == "bwsai" else case["files"][e])


def _files(base, flags):
    return {e: _read(base, e) for e in EXTS[flags]}


@pytest.mark.gpu
@pytest.mark.parametrize("name", CASE_NAMES)
def test_shifted_bwsai_in_hbm_one_window(pkg, sc, cases, name):
    """pfbwt_device: .bwt unchanged, every .sa / .ssa / .esa value + C; -S equals the restated algorithm
    on the shifted .bwsai."""
    case = cases[name]
    f = case["files"]
    for label, c in shifts(case["n"], f["bwsai"]).items():
        bws = shifted(f["bwsai"], c)
        t = {k: _dev(bws if k == "bwsai" else f[k]) for k in INPUTS}
        torch.cuda.synchronize()
        args = (t["dict"].data_ptr(), len(f["dict"]), t["occ"].data_ptr(), len(f["occ"]) // 4, t["ilist"].data_ptr(),
                t["bwlast"].data_ptr(), t["bwsai"].data_ptr(), len(f["ilist"]) // 4, case["w"])
        for flags in EXTS:
            r = sc.pfbwt_device(*args, flags=flags)
            got = {"bwt": sc.to_host(r.bwt, r.n_bwt)}
            if flags == 1:
                got["sa"] = sc.to_host(r.sa, 5 * r.n_sa)
            else:
                got["ssa"], got["esa"] = sc.to_host(r.ssa, 10 * r.n_ssa), sc.to_host(r.esa, 10 * r.n_esa)
            want = expected(case, c, flags)
            for e in EXTS[flags]:
                assert got[e] == want[e], (name, label, flags, e)
        alg = po.pfbwt_algorithm(f["dict"], f["occ"], f["ilist"], f["bwlast"], bws, case["w"])
        assert alg["bwt"] == case["want"]["bwt"] and alg["sa"] == expected(case, c, 1)["sa"], (name, label)


@pytest.mark.gpu
@pytest.mark.parametrize("windows", [4, "group"])
@pytest.mark.parametrize("name", CASE_NAMES)
def test_shifted_bwsai_file_in_windows(pkg, sc, cases, monkeypatch, mtmp, name, windows):
    """pfbwt_file in about 4 windows, and one group per window (budget 1, the smaller cases): the window
    offsets and the .sa file offsets carry the shifted values to their places."""
    case = cases[name]
    if windows == "group" and case["n"] > 20_000:
        pytest.skip("one group per window: the smaller cases only")
    base = os.path.join(mtmp, "f_" + name)
    for label, c in shifts(case["n"], case["files"]["bwsai"]).items():
        _write_inputs(base, case, c)
        for flags in EXTS:
            budget = 1 if windows == "group" else budget_for(sc, monkeypatch, base, case["w"], flags, 4)
            got, r = run_pfbwt(sc, monkeypatch, base, case["w"], flags, budget)
            assert r["windows"] > 1, (name, label, flags)
            assert got == expected(case, c, flags), (name, label, flags)


@pytest.mark.gpu
@pytest.mark.parametrize("ids", [[0, 0], [0, 0, 0]], ids=lambda x: f"{len(x)}ranks")
def test_shifted_bwsai_sharded_in_windows(pkg, cases, monkeypatch, mtmp, ids):
    """The sharded pfbwt with a per-rank budget of about 4 windows: each rank's global offset and the
    merge of the ranks' sample part files keep the shifted values."""
    ms = pkg.pfp.MultiScanner(ids)
    try:
        for name in CASE_NAMES:
            case = cases[name]
            base = os.path.join(mtmp, f"m{len(ids)}_" + name)
            for label, c in shifts(case["n"], case["files"]["bwsai"]).items():
                _write_inputs(base, case, c)
                for flags in EXTS:
                    budget = multi_budget_for(ms, monkeypatch, base, case["w"], flags, 4)
                    got, r = run_multi(ms, monkeypatch, base, case["w"], flags, budget)
                    assert max(x["windows"] for x in r["ranks"]) > 1, (name, label, flags)
                    assert got == expected(case, c, flags), (name, ids, label, flags)
    finally:
        ms.close()


@pytest.mark.gpu
def test_shifted_bwsai_cli(pkg, cases, mtmp):
    """gpupfbwt.x -S, and gpupfbwt.x -g 0,0 -s -e, on shifted files at the top of the 40-bit range."""
    case = cases["pangenome_60k_x12"]
    c = shifts(case["n"], case["files"]["bwsai"])["top"]
    base = os.path.join(mtmp, "cli")
    _write_inputs(base, case, c)
    for flags, args in ((1, ["-S"]), (6, ["-g", "0,0", "-s", "-e"])):
        subprocess.run([pkg.pfp.PFBWT_CLI_PATH, "-w", str(case["w"]), *args, base], check=True, stdout=subprocess.PIPE)
        assert _files(base, flags) == expected(case, c, flags), args


BWTPARSE_NAMES = sorted(_bwtparse_golden()) + TEXT_CASES


@pytest.mark.gpu
@pytest.mark.parametrize("name", BWTPARSE_NAMES)
def test_bwtparse_shifted_sai(pkg, sc, cases, name):
    """bwtparse_host(parse, last, sai + C): .bwsai = the unshifted .bwsai + C except row 1, the row of
    parse suffix 0, which stays 0; .ilist / .bwlast unchanged; equal to the restated bwtparse."""
    if name in TEXT_CASES:
        f, n_text = cases[name]["files"], cases[name]["n"]
    else:
        f = _bwtparse_golden()[name]
        n_text = int(get5(f["sai"]).max())                   # the end of the last phrase: about the text
    base = sc.bwtparse_host(f["parse"], f["last"], f["sai"])
    assert base.bwsai == f["bwsai"]
    unshifted = get5(f["bwsai"])
    assert unshifted[1] == 0
    for label, c in shifts(n_text, f["sai"]).items():
        sai = shifted(f["sai"], c)
        got = sc.bwtparse_host(f["parse"], f["last"], sai)
        want = unshifted + np.uint64(c)
        want[1] = 0
        assert got.ilist == base.ilist and got.bwlast == base.bwlast, (name, label)
        assert got.bwsai == put5(want), (name, label)
        assert (got.ilist, got.bwlast, got.bwsai) == bo.bwtparse(f["parse"], f["last"], sai), (name, label)


# ---- Part B: a text longer than 2^32 through the whole chain ---------------------------------------------
N_HAP, BASE_LEN, SEED, W, P = 110, 40_000_000, 2, 10, 100
FILE_ARM_DISK = 35 << 30


def _need(gb):
    torch.cuda.empty_cache()
    free, _ = torch.cuda.mem_get_info()
    if free < gb * (1 << 30):
        pytest.skip(f"needs {gb} GB of free device memory, {free / (1 << 30):.0f} GB free")


def _need_disk(d, nbytes):
    free = shutil.disk_usage(d).free
    if free < nbytes:
        pytest.skip(f"needs {nbytes / (1 << 30):.0f} GB of disk in {d}, {free / (1 << 30):.0f} GB free")


def _device_used():
    free, total = torch.cuda.mem_get_info()
    return total - free


class _DevBytes:
    """a device buffer of the library as a torch uint8 tensor without a copy"""
    def __init__(self, ptr, n):
        self.__cuda_array_interface__ = {"shape": (n,), "typestr": "|u1", "data": (ptr, False), "version": 3}


def _view(ptr, n):
    return torch.as_tensor(_DevBytes(ptr, n), device="cuda")


def _sha_dev(t, step=1 << 30):
    h = hashlib.sha256()
    for a in range(0, t.numel(), step):
        h.update(t[a:a + step].cpu().numpy().tobytes())
    return h.hexdigest()


def _sha_file(path):
    h = hashlib.sha256()
    with open(path, "rb") as f:
        while True:
            b = f.read(64 << 20)
            if not b:
                return h.hexdigest()
            h.update(b)


def _text(pkg):
    return pkg.synth.pangenome_text(BASE_LEN, N_HAP, SEED, device="cuda")


def _run_samples(bwt, sa, at_end, chunk=1 << 26):
    """sha256 and count of the (position, value) records of the run starts (at_end 0) / ends (1) of the
    BWT, as .ssa / .esa hold them, and how many of their positions are >= 2^32"""
    n1 = bwt.numel()
    h, k, high = hashlib.sha256(), 0, 0
    for a in range(0, n1, chunk):
        b = min(n1, a + chunk)
        m = torch.ones(b - a, dtype=torch.bool, device=bwt.device)   # the first / last row: a run border
        if at_end:
            e = min(b + 1, n1)
            m[:e - a - 1] = bwt[a:e - 1] != bwt[a + 1:e]
        else:
            lo = max(a, 1)
            m[lo - a:] = bwt[lo:b] != bwt[lo - 1:b - 1]
        pos = torch.nonzero(m).flatten() + a
        rec = torch.stack([pos, sa[pos]], dim=1).reshape(-1)
        h.update(sa_check.encode5(rec).cpu().numpy().tobytes())
        k += pos.numel()
        high += int((pos >= (1 << 32)).sum())
    return h.hexdigest(), k, high


@pytest.fixture(scope="module")
def big():
    return {}


@pytest.fixture(scope="module")
def bigdir():
    d = tempfile.mkdtemp(prefix="pos40_big_")
    yield d
    shutil.rmtree(d, ignore_errors=True)


def _log(big, arm, **kw):
    big.setdefault("log", []).append(dict(arm=arm, **kw))
    print({"arm": arm, **kw}, flush=True)


@pytest.mark.gpu
def test_fullsize_arm1_sa_in_hbm_checked_in_linear_time(pkg, big):
    _need(110)
    ram = os.sysconf("SC_AVPHYS_PAGES") * os.sysconf("SC_PAGE_SIZE")
    if ram < (40 << 30):
        pytest.skip(f"needs 40 GB of free host memory, {ram / (1 << 30):.0f} GB free")
    t0 = time.perf_counter()
    text = _text(pkg)
    n = text.numel()
    assert n > (1 << 32)
    sc = pkg.pfp.Scanner(0)
    try:
        r, out, bp = sc.bwt_of_text(text, W, P, flags=pkg.pfp.PFBWT_SA)
        torch.cuda.synchronize()
        assert r.n_bwt == n + 1 and r.n_sa == n and r.n_bwt > (1 << 32)
        assert out.dict_bytes < (1 << 30)
        lib_used = _device_used()                        # the library's arena, the text
        # the arena holds most of the card: the outputs go to the host until the library is closed
        sa5 = torch.empty(5 * r.n_sa, dtype=torch.uint8)
        bwt = torch.empty(r.n_bwt, dtype=torch.uint8)
        for host, ptr in ((sa5, r.sa), (bwt, r.bwt)):
            v = _view(ptr, host.numel())
            for a in range(0, host.numel(), 1 << 30):
                host[a:a + (1 << 30)].copy_(v[a:a + (1 << 30)])
        big.update(n=n, n_bwt=r.n_bwt, hard=r.hard, dict_bytes=out.dict_bytes, psize=bp.n_out)
    finally:
        sc.close()
    big["sha_sa"] = hashlib.sha256(sa5.numpy()).hexdigest()
    bwt = bwt.cuda()
    sa = torch.empty(n + 1, dtype=torch.int64, device="cuda")
    sa[0] = n
    step = 1 << 26
    for a in range(0, n, step):
        b = min(n, a + step)
        sa[1 + a:1 + b] = sa_check.decode5(sa5[5 * a:5 * b].cuda())
    del sa5
    torch.cuda.empty_cache()
    others = _device_used() - torch.cuda.memory_reserved()
    torch.cuda.reset_peak_memory_stats()
    big["sha_bwt"] = _sha_dev(bwt)
    sa_max = int(sa[1:].max())
    assert sa_max >= (1 << 32)
    fails = sa_check.linear_checks(text, sa, bwt)
    assert fails == [], fails
    big["past_2_32"] = int((sa[1:] >= (1 << 32)).sum())
    for at_end, e in ((0, "ssa"), (1, "esa")):
        big[f"sha_{e}"], big[f"n_{e}"], big[f"high_{e}"] = _run_samples(bwt, sa, at_end)
    assert big["high_ssa"] > 0 and big["high_esa"] > 0
    checks = others + torch.cuda.max_memory_reserved()
    _log(big, 1, n_text=n, n_bwt=r.n_bwt, max_bwt_position=r.n_bwt - 1, max_sa_value=sa_max,
         sa_values_past_2_32=big["past_2_32"], dict_bytes=big["dict_bytes"], parse_size=big["psize"],
         runs=big["n_ssa"], run_starts_past_2_32=big["high_ssa"], run_ends_past_2_32=big["high_esa"],
         device_GB={"library_arena_and_text": round(lib_used / 1e9, 1), "checks": round(checks / 1e9, 1)}, wall_s=round(time.perf_counter() - t0, 1))
    del text, sa, bwt
    torch.cuda.empty_cache()


def _need_arm1(big):
    if "sha_ssa" not in big:
        pytest.skip("arm 1 did not run")


@pytest.mark.gpu
def test_fullsize_arm2_sampled_sa_in_hbm(pkg, big):
    """pfbwt_device holds the whole -s -e output in one window: 29 B per BWT char (127.6 GB here) on top
    of the word structure, so this arm fits only a B200 with nearly all its memory free.  It completed
    when run on its own; after the rest of the GPU suite in the same process it failed with E_NOMEM, and
    so did pfbwt_file forced into one window in a fresh process with 190.8 GB free.  It skips then, and
    arms 3 and 4 check the same .ssa / .esa in windows."""
    _need_arm1(big)
    se = pkg.pfp.PFBWT_SSA | pkg.pfp.PFBWT_ESA
    _need(-(-out_bytes(big["n_bwt"], big["hard"], se) // (1 << 30)))
    t0 = time.perf_counter()
    text = _text(pkg)
    sc = pkg.pfp.Scanner(0)
    try:
        try:
            r, _, _ = sc.bwt_of_text(text, W, P, flags=se)
        except pkg.pfp.PfpError as e:
            if e.code != -4:                                  # PFPB200_E_NOMEM
                raise
            pytest.skip(f"the one-window -s -e output does not fit the free device memory: {e}")
        torch.cuda.synchronize()
        peak = _device_used()
        del text
        assert (r.n_ssa, r.n_esa) == (big["n_ssa"], big["n_esa"])
        assert _sha_dev(_view(r.bwt, r.n_bwt)) == big["sha_bwt"]
        assert _sha_dev(_view(r.ssa, 10 * r.n_ssa)) == big["sha_ssa"]
        assert _sha_dev(_view(r.esa, 10 * r.n_esa)) == big["sha_esa"]
        top = int(sa_check.decode5(_view(r.ssa, 10 * r.n_ssa)[-10:]).max())
    finally:
        sc.close()
    torch.cuda.empty_cache()
    _log(big, 2, n_ssa=r.n_ssa, n_esa=r.n_esa, last_ssa_record_max=top, device_GB=round(peak / 1e9, 1),
         wall_s=round(time.perf_counter() - t0, 1))


def _check_files(big, base, flags, arm, what):
    got = {e: _sha_file(f"{base}.{e}") for e in EXTS[flags]}
    for e in EXTS[flags]:
        assert got[e] == big[f"sha_{e}"], (arm, what, e)
        os.remove(f"{base}.{e}")


@pytest.fixture(scope="module")
def big_inputs(pkg, big, bigdir):
    """.dict .occ .ilist .bwlast .bwsai of the text, written once for arms 3 and 4"""
    _need_arm1(big)
    _need(20)
    _need_disk(bigdir, FILE_ARM_DISK)
    base = os.path.join(bigdir, "big")
    text = _text(pkg)
    sc = pkg.pfp.Scanner(0)
    try:
        out = sc.parse_device(text, W, P, sai=True)
        del text
        bp = sc.bwtparse_device(out.parse, out.n_phrases, out.last, out.sai)
        for ext, ptr, nb in (("dict", out.dict, out.dict_bytes), ("occ", out.occ, 4 * out.n_distinct),
                             ("ilist", bp.ilist, 4 * bp.n_out), ("bwlast", bp.bwlast, bp.n_out),
                             ("bwsai", bp.bwsai, 5 * bp.n_out)):
            v = _view(ptr, nb)
            with open(f"{base}.{ext}", "wb") as f:
                for a in range(0, nb, 1 << 30):
                    f.write(v[a:a + (1 << 30)].cpu().numpy().tobytes())
    finally:
        sc.close()
    torch.cuda.empty_cache()
    return base


@pytest.mark.gpu
def test_fullsize_arm3_files_in_windows(pkg, big, big_inputs, monkeypatch):
    _need(75)
    t0 = time.perf_counter()
    peak, windows = 0, []
    sc = pkg.pfp.Scanner(0)
    try:
        for flags in EXTS:
            monkeypatch.setenv("PFPB200_PFBWT_BUDGET", str(out_bytes(big["n_bwt"], big["hard"], flags) // 5))
            r = sc.pfbwt_file(big_inputs, W, flags)
            monkeypatch.delenv("PFPB200_PFBWT_BUDGET")
            assert r["windows"] >= 4 and r["n_bwt"] == big["n_bwt"], flags
            peak, windows = max(peak, r["peak_device_bytes"]), windows + [r["windows"]]
            _check_files(big, big_inputs, flags, 3, flags)
    finally:
        sc.close()
    _log(big, 3, windows=windows, device_peak_GB=round(peak / 1e9, 1), wall_s=round(time.perf_counter() - t0, 1))


@pytest.mark.gpu
def test_fullsize_arm4_sharded_in_windows(pkg, big, big_inputs, monkeypatch):
    _need(90)
    t0 = time.perf_counter()
    peaks, windows = [], []
    ms = pkg.pfp.MultiScanner([0, 0])
    try:
        for flags in EXTS:
            monkeypatch.setenv("PFPB200_PFBWT_BUDGET", str(out_bytes(big["n_bwt"], big["hard"], flags) // 10))
            r = ms.pfbwt_file(big_inputs, W, flags)
            monkeypatch.delenv("PFPB200_PFBWT_BUDGET")
            assert r["n_bwt"] == big["n_bwt"] and min(x["windows"] for x in r["ranks"]) >= 2, r["ranks"]
            peaks.append([x["peak_bytes"] for x in r["ranks"]])
            windows.append([x["windows"] for x in r["ranks"]])
            _check_files(big, big_inputs, flags, 4, flags)
    finally:
        ms.close()
    _log(big, 4, windows_per_rank=windows, rank_peaks_GB=[[round(p / 1e9, 1) for p in x] for x in peaks],
         wall_s=round(time.perf_counter() - t0, 1))


@pytest.mark.gpu
def test_fullsize_arm5_gpubigbwt_streamed_parse_and_windows(pkg, big, bigdir):
    _need_arm1(big)
    _need(70)
    _need_disk(bigdir, FILE_ARM_DISK)
    t0 = time.perf_counter()
    path = os.path.join(bigdir, "text")
    text = _text(pkg)
    with open(path, "wb") as f:
        for a in range(0, text.numel(), 1 << 30):
            f.write(text[a:a + (1 << 30)].cpu().numpy().tobytes())
    del text
    torch.cuda.empty_cache()
    n = big["n"]
    env = dict(os.environ, PFPB200_PARSE_BUDGET=str(8 * (n // 5)),
               PFPB200_PFBWT_BUDGET=str(out_bytes(big["n_bwt"], big["hard"], 1) // 5))
    r = subprocess.run([pkg.pfp.BIGBWT_CLI_PATH, path, "-w", str(W), "-p", str(P), "-S"], check=True,
                       stdout=subprocess.PIPE, text=True, env=env)
    os.remove(path)
    m = re.search(r"Plan: parse (\d+) chunks .*, peak ([\d.]+) GB; pfbwt (\d+) windows, peak ([\d.]+) GB", r.stdout)
    assert m, r.stdout
    chunks, windows = int(m.group(1)), int(m.group(3))
    assert chunks >= 4 and windows >= 4, r.stdout
    _check_files(big, path, 1, 5, "gpubigbwt")
    _log(big, 5, parse_chunks=chunks, parse_peak_GB=float(m.group(2)), pfbwt_windows=windows,
         pfbwt_peak_GB=float(m.group(4)), wall_s=round(time.perf_counter() - t0, 1))
