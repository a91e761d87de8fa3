"""The last stage sharded over several ranks (pfpb200_multi_pfbwt_file, MultiScanner.pfbwt_file,
`gpupfbwt.x -g`, `gpubigbwt.x -g`): the same .bwt / .sa / .ssa / .esa as the single-GPU pfbwt, byte
for byte, for every number of ranks.  Device 0 listed several times runs every protocol path of the
sharded suffix sort on one GPU (the ranks share it; peer loads and stores are then local)."""
import os
import shutil
import subprocess
import tempfile

import numpy as np
import pytest

from test_oracle_golden import _pfbwt_golden

pytestmark = pytest.mark.gpu

RANK_LISTS = [[0], [0, 0], [0, 0, 0], [0, 0, 0, 0, 0]]
INPUTS = ("dict", "occ", "ilist", "bwlast", "bwsai")


@pytest.fixture(scope="module")
def sc(pkg):
    s = pkg.pfp.Scanner(0)
    yield s
    s.close()


@pytest.fixture
def tmp():
    d = tempfile.mkdtemp(prefix="pfbwtmulti_")
    yield d
    shutil.rmtree(d, ignore_errors=True)


def _flag_sets(P):
    return [(P.PFBWT_SA, ("bwt", "sa")), (P.PFBWT_SSA | P.PFBWT_ESA, ("bwt", "ssa", "esa")), (0, ("bwt",))]


def _read(base, exts):
    out = {}
    for e in exts:
        with open(f"{base}.{e}", "rb") as f:
            out[e] = f.read()
    return out


def _write_inputs(base, c):
    for e in INPUTS:
        with open(f"{base}.{e}", "wb") as f:
            f.write(c[e])


def _parse_chain(sc, base, text, w, p):
    """text -> .dict .occ .parse .last .sai (parse) -> .ilist .bwlast .bwsai (bwtparse), on one GPU"""
    with open(base, "wb") as f:
        f.write(bytes(text))
    sc.parse_file(base, w, p, sai=True)
    sc.bwtparse_file(base, sai=True)


def _single_vs_multi(pkg, sc, base, w, ids, split=False, monkeypatch=None):
    """every flag set: single-GPU files, then the sharded run on `ids`, byte-identical; returns the ranks"""
    if split:
        monkeypatch.setenv("PFPB200_MULTI_SPLIT_KEY", "1")
    ms = pkg.pfp.MultiScanner(ids)
    ranks = None
    try:
        for flags, exts in _flag_sets(pkg.pfp):
            sc.pfbwt_file(base, w, flags)
            want = _read(base, exts)
            for e in exts:
                os.remove(f"{base}.{e}")
            r = ms.pfbwt_file(base, w, flags)
            got = _read(base, exts)
            for e in exts:
                assert got[e] == want[e], f"{base} ranks {ids} flags {flags}: .{e}"
            assert r["n_bwt"] == len(want["bwt"]) and r["easy"] + r["hard"] == r["n_bwt"]
            assert len(r["ranks"]) == len(ids) and sum(x["chars"] for x in r["ranks"]) == r["n_bwt"]
            ranks = r["ranks"]
    finally:
        ms.close()
    return ranks


def _distinct_first_keys(d: bytes) -> int:
    """distinct first keys of the dictionary's positions: h0 dense-coded symbols, cut behind the terminator"""
    present = sorted(set(b for b in d if b > 1))
    code = {0: 1, 1: 1}
    for i, b in enumerate(present):
        code[b] = i + 2
    bs = (len(present) + 1).bit_length()
    h0 = min(32, 64 // bs)
    keys = set()
    for t in range(len(d)):
        k, live = 0, d[t] > 1
        for i in range(h0):
            c = 0
            if live:
                b = d[t + i] if t + i < len(d) else 0
                c = code[b]
                live = b > 1
            k = (k << bs) | c
        keys.add(k)
    return len(keys)


@pytest.mark.parametrize("split", [False, True], ids=["one-key", "two-sorts"])
@pytest.mark.parametrize("ids", RANK_LISTS, ids=lambda x: f"{len(x)}ranks")
def test_golden_cases_through_files(pkg, tmp, monkeypatch, ids, split):
    """The stored outputs of the unmodified reference chain (tests/golden/golden_pfbwt.npz), -S and -s -e."""
    if split:
        monkeypatch.setenv("PFPB200_MULTI_SPLIT_KEY", "1")
    P = pkg.pfp
    ms = P.MultiScanner(ids)
    try:
        for name, c in _pfbwt_golden().items():
            base = os.path.join(tmp, name)
            _write_inputs(base, c)
            for flags, exts in ((P.PFBWT_SA, ("bwt", "sa")), (P.PFBWT_SSA | P.PFBWT_ESA, ("bwt", "ssa", "esa"))):
                r = ms.pfbwt_file(base, c["w"], flags)
                got = _read(base, exts)
                for e in exts:
                    assert got[e] == c[e], f"{name} ranks {ids} flags {flags}: .{e}"
                assert r["n_bwt"] == len(c["bwt"]) and r["dict_bytes"] == len(c["dict"])
    finally:
        ms.close()


@pytest.mark.parametrize("split", [False, True], ids=["one-key", "two-sorts"])
@pytest.mark.parametrize("w,p", [(6, 20), (10, 100), (16, 50)])
def test_pangenome_multi_equals_single(pkg, sc, tmp, monkeypatch, w, p, split):
    text = pkg.synth.pangenome_text(60_000, 12, 40 + w).numpy()
    base = os.path.join(tmp, "pan")
    _parse_chain(sc, base, text, w, p)
    for ids in ([0, 0], [0, 0, 0, 0]):
        _single_vs_multi(pkg, sc, base, w, ids, split, monkeypatch)


@pytest.mark.parametrize("split", [False, True], ids=["one-key", "two-sorts"])
def test_long_n_runs_leave_ranks_empty(pkg, sc, tmp, monkeypatch, split):
    """Long runs of N put most dictionary suffixes under one first key: the splitters coincide and
    some ranks own no suffix at all."""
    rng = np.random.default_rng(11)
    parts = []
    for i in range(6):
        parts += [pkg.synth.random_dna(3_000, 100 + i).numpy(), np.full(int(rng.integers(20_000, 40_000)), ord("N"), np.uint8)]
    text = np.concatenate(parts)
    base = os.path.join(tmp, "nruns")
    _parse_chain(sc, base, text, 10, 100)
    ranks = _single_vs_multi(pkg, sc, base, 10, [0] * 5, split, monkeypatch)
    assert any(r["suffixes"] == 0 for r in ranks)


@pytest.mark.parametrize("split", [False, True], ids=["one-key", "two-sorts"])
def test_tandem_repeats_hard_groups_at_rank_borders(pkg, sc, tmp, monkeypatch, split):
    """A few units repeated thousands of times, lightly mutated: words with thousands of occurrences,
    big hard groups next to the rank borders, long runs of the BWT across them (-s / -e)."""
    rng = np.random.default_rng(5)
    units = [pkg.synth.random_dna(int(n), 200 + i).numpy() for i, n in enumerate((37, 91, 180))]
    chunks = []
    for _ in range(3_000):
        u = units[int(rng.integers(0, 3))].copy()
        if rng.random() < 0.05:
            u[int(rng.integers(0, len(u)))] = ord("ACGT"[int(rng.integers(0, 4))])
        chunks.append(u)
    text = np.concatenate(chunks)
    base = os.path.join(tmp, "tandem")
    _parse_chain(sc, base, text, 10, 100)
    inside_runs = 0
    for ids in ([0, 0, 0], [0] * 7):
        ranks = _single_vs_multi(pkg, sc, base, 10, ids, split, monkeypatch)
        assert sum(1 for r in ranks if r["chars"]) >= 2          # the BWT really is cut into pieces
        bwt = _read(base, ["bwt"])["bwt"]
        offs = np.cumsum([r["chars"] for r in ranks if r["chars"]])[:-1]
        inside_runs += sum(1 for o in offs if bwt[o - 1] == bwt[o])
    assert inside_runs >= 1                                       # a piece border inside a run of the BWT


def test_all_byte_values(pkg, sc, tmp, monkeypatch):
    """Text bytes 3..255 (and the terminators 0 / 1 in the dictionary): 8-bit codes, 8 symbols per key."""
    rng = np.random.default_rng(7)
    text = np.concatenate([rng.integers(3, 256, 40_000).astype(np.uint8), pkg.synth.random_dna(30_000, 9).numpy(),
                           rng.integers(3, 256, 20_000).astype(np.uint8)])
    base = os.path.join(tmp, "bytes")
    _parse_chain(sc, base, text, 4, 10)
    for split in (False, True):
        _single_vs_multi(pkg, sc, base, 4, [0, 0, 0, 0], split, monkeypatch)


def test_fewer_distinct_first_keys_than_ranks(pkg, sc, tmp, monkeypatch):
    """A two-phrase text whose dictionary has 15 distinct first keys, sorted by 16 ranks."""
    base = os.path.join(tmp, "tiny")
    _parse_chain(sc, base, b"AAAAT", 4, 13)
    with open(base + ".dict", "rb") as f:
        assert _distinct_first_keys(f.read()) < 16
    ranks = _single_vs_multi(pkg, sc, base, 4, [0] * 16, False, monkeypatch)
    assert sum(1 for r in ranks if r["suffixes"] == 0) >= 1


def _devs(n):
    import torch
    k = torch.cuda.device_count()
    return ",".join(map(str, range(n))) if k >= n else ",".join(["0"] * n)


def test_cli_gpupfbwt_device_list(pkg, sc, tmp):
    """`gpupfbwt.x -g 0,0,0` writes the files `gpupfbwt.x` writes with one device."""
    text = pkg.synth.pangenome_text(40_000, 8, 77).numpy()
    base = os.path.join(tmp, "cli")
    _parse_chain(sc, base, text, 10, 100)
    cli = pkg.pfp.PFBWT_CLI_PATH
    for flags, exts in ((["-S"], ("bwt", "sa")), (["-s", "-e"], ("bwt", "ssa", "esa"))):
        subprocess.run([cli, "-w", "10", *flags, base], check=True, stdout=subprocess.PIPE)
        want = _read(base, exts)
        for e in exts:
            os.remove(f"{base}.{e}")
        r = subprocess.run([cli, "-w", "10", *flags, "-g", _devs(3), base], check=True, stdout=subprocess.PIPE, text=True)
        assert "Hard bwt chars" in r.stdout and r.stdout.count("(rank ") == 3
        assert _read(base, exts) == want


def test_cli_gpubigbwt_device_list(pkg, tmp):
    """`gpubigbwt.x -g 0,0 -S -k`: parse and pfbwt sharded, bwtparse on the first device, through files --
    the same files as the one-device run; without -k the intermediate files are gone."""
    text = pkg.synth.pangenome_text(50_000, 10, 31).numpy().tobytes()
    one, two, plain = (os.path.join(tmp, n) for n in ("one", "two", "plain"))
    for pth in (one, two, plain):
        with open(pth, "wb") as f:
            f.write(text)
    cli = pkg.pfp.BIGBWT_CLI_PATH
    subprocess.run([cli, one, "-w", "10", "-p", "100", "-S", "-k"], check=True, stdout=subprocess.PIPE)
    r = subprocess.run([cli, two, "-w", "10", "-p", "100", "-S", "-k", "-g", _devs(2)], check=True,
                       stdout=subprocess.PIPE, text=True)
    assert "Hard bwt chars" in r.stdout
    for ext in ("bwt", "sa", "dict", "occ", "parse", "last", "sai", "ilist", "bwlast", "bwsai"):
        assert _read(two, [ext]) == _read(one, [ext]), ext
    subprocess.run([cli, plain, "-g", _devs(2)], check=True, stdout=subprocess.PIPE)
    assert _read(plain, ["bwt"]) == _read(one, ["bwt"])
    assert not os.path.exists(plain + ".dict") and not os.path.exists(plain + ".ilist")


def test_errors_match_the_single_path(pkg, sc, tmp):
    P = pkg.pfp
    c = _pfbwt_golden()["short_w4_p10"]
    base = os.path.join(tmp, "err")
    ms = P.MultiScanner([0, 0, 0])
    try:
        def both(w, flags):
            out = []
            for f in (lambda: sc.pfbwt_file(base, w, flags), lambda: ms.pfbwt_file(base, w, flags)):
                with pytest.raises(P.PfpError) as e:
                    f()
                out.append(e.value)
            return out
        _write_inputs(base, c)
        with open(base + ".occ", "wb") as f:                           # .occ does not match the dictionary
            f.write(c["occ"][:-4])
        one, multi = both(c["w"], 0)
        assert one.code == multi.code and str(one).split(": ")[-1] in str(multi)
        _write_inputs(base, c)
        os.remove(base + ".bwsai")                                     # -S without .bwsai
        one, multi = both(c["w"], P.PFBWT_SA)
        assert one.code == multi.code and "cannot open" in str(multi) and ".bwsai" in str(multi)
        os.remove(base + ".ilist")                                     # a missing file
        one, multi = both(c["w"], 0)
        assert one.code == multi.code and ".ilist" in str(multi)
        _write_inputs(base, c)
        one, multi = both(3, 0)                                        # w < 4
        assert one.code == multi.code and "at least 4" in str(multi)
        one, multi = both(c["w"], P.PFBWT_SA | P.PFBWT_SSA)            # -S with -s
        assert one.code == multi.code and "not both" in str(multi)
        r = subprocess.run([P.PFBWT_CLI_PATH, "-w", "4", "-g", "0,0", os.path.join(tmp, "missing")],
                           capture_output=True, text=True)
        assert r.returncode == 1 and "cannot open" in r.stderr
    finally:
        ms.close()
