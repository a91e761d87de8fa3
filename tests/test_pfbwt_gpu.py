"""The last stage on the GPU (pfpb200_pfbwt_*, SURVEY 8(f) row 2) against the reference's pfbwt:
byte-identical .bwt / .sa / .ssa / .esa -- golden outputs of the unmodified chain
(tests/golden/golden_pfbwt.npz), the whole pipeline parse -> bwtparse -> pfbwt in HBM against the
suffix array of the text, and gpupfbwt.x / gpubigbwt.x against the files of the unmodified chain."""
import os
import shutil
import subprocess
import tempfile

import numpy as np
import pytest
import torch

from oracle import pfbwt_oracle as po
from test_oracle_golden import _bwtparse_golden, _pfbwt_golden

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def sc(pkg):
    s = pkg.pfp.Scanner(0)
    yield s
    s.close()


def _dev(b):
    return torch.from_numpy(np.frombuffer(b, dtype=np.uint8).copy()).cuda()


def _fetch(sc, r):
    g = sc.to_host
    return {"bwt": g(r.bwt, r.n_bwt), "sa": g(r.sa, 5 * r.n_sa) if r.sa else b"",
            "ssa": g(r.ssa, 10 * r.n_ssa) if r.ssa else b"", "esa": g(r.esa, 10 * r.n_esa) if r.esa else b""}


def test_golden_cases(pkg, sc):
    P = pkg.pfp
    for name, c in _pfbwt_golden().items():
        t = {k: _dev(c[k]) for k in ("dict", "occ", "ilist", "bwlast", "bwsai")}
        torch.cuda.synchronize()
        args = (t["dict"].data_ptr(), len(c["dict"]), t["occ"].data_ptr(), len(c["occ"]) // 4, t["ilist"].data_ptr(),
                t["bwlast"].data_ptr(), t["bwsai"].data_ptr(), len(c["ilist"]) // 4, c["w"])
        got = _fetch(sc, sc.pfbwt_device(*args, flags=0))
        assert got["bwt"] == c["bwt"], f"{name}: .bwt"
        got = _fetch(sc, sc.pfbwt_device(*args, flags=P.PFBWT_SA))
        assert got["bwt"] == c["bwt"] and got["sa"] == c["sa"], f"{name}: -S"
        got = _fetch(sc, sc.pfbwt_device(*args, flags=P.PFBWT_SSA | P.PFBWT_ESA))
        assert got["bwt"] == c["bwt"] and got["ssa"] == c["ssa"] and got["esa"] == c["esa"], f"{name}: -s -e"


@pytest.mark.parametrize("base_len,haps,w,p", [(150_000, 10, 10, 100), (60_000, 20, 6, 20), (1_500_000, 1, 10, 100),
                                                (40_000, 8, 16, 50)])
def test_whole_pipeline_in_hbm_vs_suffix_array_of_the_text(pkg, sc, base_len, haps, w, p):
    """parse -> bwtparse -> pfbwt on ONE context: the text goes in, its BWT and suffix array come out,
    nothing leaves HBM in between.  Checked against the suffix array of the text (the result
    pfbwt.cpp defines; oracle/pfbwt_oracle.py, pinned to the reference binary)."""
    text = pkg.synth.pangenome_text(base_len, haps, 70 + haps, device="cuda")
    want = po.pfbwt(text.cpu().numpy().tobytes())
    r, out, bp = sc.bwt_of_text(text, w, p, flags=pkg.pfp.PFBWT_SA)
    got = _fetch(sc, r)
    assert r.n_bwt == text.numel() + 1 and r.easy + r.hard == r.n_bwt
    assert got["bwt"] == want["bwt"]
    assert got["sa"] == want["sa"]
    r, out, bp = sc.bwt_of_text(text, w, p, flags=pkg.pfp.PFBWT_SSA | pkg.pfp.PFBWT_ESA)
    got = _fetch(sc, r)
    assert got["bwt"] == want["bwt"] and got["ssa"] == want["ssa"] and got["esa"] == want["esa"]
    r, out, bp = sc.bwt_of_text(text, w, p, flags=0)
    assert _fetch(sc, r)["bwt"] == want["bwt"]


def test_text_with_long_runs_and_all_byte_values(pkg, sc):
    rng = np.random.default_rng(3)
    a = np.concatenate([rng.integers(3, 256, 50_000).astype(np.uint8), np.full(30_000, ord("N"), np.uint8),
                        pkg.synth.random_dna(40_000, 4).numpy(), np.full(5_000, ord("N"), np.uint8)])
    text = torch.from_numpy(a).cuda()
    want = po.pfbwt(a.tobytes())
    r, _, _ = sc.bwt_of_text(text, 10, 100, flags=pkg.pfp.PFBWT_SA)
    got = _fetch(sc, r)
    assert got["bwt"] == want["bwt"] and got["sa"] == want["sa"]


def test_tandem_repeats_words_with_thousands_of_occurrences(pkg, sc):
    """A unit repeated 6000 times: a handful of words carry thousands of occurrences each (the CTA
    path of the easy members, long per-member loops in the merge)."""
    unit = pkg.synth.random_dna(211, 12).numpy().tobytes()
    a = pkg.synth.random_dna(20_000, 13).numpy().tobytes() + unit * 6000 + pkg.synth.random_dna(20_000, 14).numpy().tobytes()
    text = torch.from_numpy(np.frombuffer(a, np.uint8).copy()).cuda()
    want = po.pfbwt(a)
    for w, p in ((10, 100), (4, 10)):
        r, out, _ = sc.bwt_of_text(text, w, p, flags=pkg.pfp.PFBWT_SA)
        got = _fetch(sc, r)
        assert got["bwt"] == want["bwt"] and got["sa"] == want["sa"], (w, p)
        occ = np.frombuffer(sc.to_host(out.occ, 4 * out.n_distinct), np.uint32)
        assert occ.max() > 1000
        r, _, _ = sc.bwt_of_text(text, w, p, flags=0)
        assert _fetch(sc, r)["bwt"] == want["bwt"]


def reference_chain(name="pangenome_20k_x6_w10_p100"):
    """Every file the unmodified chain newscanNT.x -s -> bwtparse -s -> pfbwtNT.x wrote for one stored
    text (tools/make_golden_bwtparse.py and tools/make_golden_pfbwt.py ran it on the same text)."""
    c = dict(_bwtparse_golden()[name])
    c.update(_pfbwt_golden()[name])
    return c


def write_fasta(pkg, path, text):
    """`text` as a one-record FASTA file: the text the tools extract from it is `text` again."""
    with open(path, "wb") as f:
        f.write(pkg.synth.to_fasta([np.frombuffer(text, np.uint8)]))


def test_cli_matches_reference(pkg):
    """gpupfbwt.x as the drop-in for pfbwtNT.x on the reference's own intermediate files, and the whole
    GPU chain gpuscan.x -> gpubwtparse.x -> gpupfbwt.x on the text: the .bwt / .sa / .ssa / .esa the
    all-reference chain wrote."""
    ref = reference_chain()
    w, p = str(ref["w"]), str(ref["p"])
    tmp = tempfile.mkdtemp(prefix="pfbwtcli_")
    try:
        drop, ours = os.path.join(tmp, "drop"), os.path.join(tmp, "ours.fa")
        for ext in ("dict", "occ", "ilist", "bwlast", "bwsai"):
            with open(drop + "." + ext, "wb") as f:
                f.write(ref[ext])
        write_fasta(pkg, ours, ref["text"])
        subprocess.run([pkg.pfp.CLI_PATH, ours, "-w", w, "-p", p, "-s", "-f"], check=True, stdout=subprocess.PIPE)
        subprocess.run([pkg.pfp.BWTPARSE_CLI_PATH, ours, "-s"], check=True, stdout=subprocess.PIPE)
        for flags, exts in ((["-S"], ("bwt", "sa")), (["-s", "-e"], ("bwt", "ssa", "esa")), ([], ("bwt",))):
            for base in (drop, ours):
                r = subprocess.run([pkg.pfp.PFBWT_CLI_PATH, "-w", w, *flags, base], check=True, stdout=subprocess.PIPE,
                                   text=True)
                assert "Easy bwt chars" in r.stdout and "Hard bwt chars" in r.stdout
                for ext in exts:
                    assert open(base + "." + ext, "rb").read() == ref[ext], (base, flags, ext)
        r = subprocess.run([pkg.pfp.PFBWT_CLI_PATH, "-w", "10", "-S", "-s", ours], capture_output=True, text=True)
        assert r.returncode == 1 and "not both" in r.stdout
        r = subprocess.run([pkg.pfp.PFBWT_CLI_PATH, "-w", "10", os.path.join(tmp, "missing")], capture_output=True, text=True)
        assert r.returncode == 1
    finally:
        shutil.rmtree(tmp, ignore_errors=True)


def test_gpubigbwt_one_process_matches_the_reference_chain(pkg):
    """gpubigbwt.x: file in, .bwt / .sa out, the three stages in HBM in one process -- against the
    files newscanNT.x + bwtparse + pfbwtNT.x wrote; with -k the intermediate files are the reference's too."""
    ref = reference_chain()
    assert (ref["w"], ref["p"]) == (10, 100)            # the defaults the run without -w / -p relies on
    tmp = tempfile.mkdtemp(prefix="bigbwtcli_")
    try:
        ours, plain = os.path.join(tmp, "ours.fa"), os.path.join(tmp, "plain.fa")
        for pth in (ours, plain):
            write_fasta(pkg, pth, ref["text"])
        r = subprocess.run([pkg.pfp.BIGBWT_CLI_PATH, ours, "-w", "10", "-p", "100", "-f", "-S", "-k"], check=True,
                           stdout=subprocess.PIPE, text=True)
        assert "Hard bwt chars" in r.stdout
        for ext in ("bwt", "sa", "dict", "occ", "parse", "last", "sai", "ilist", "bwlast", "bwsai"):
            assert open(ours + "." + ext, "rb").read() == ref[ext], ext
        subprocess.run([pkg.pfp.BIGBWT_CLI_PATH, plain, "-f"], check=True, stdout=subprocess.PIPE)
        assert open(plain + ".bwt", "rb").read() == ref["bwt"]
        assert not os.path.exists(plain + ".dict") and not os.path.exists(plain + ".sa")
    finally:
        shutil.rmtree(tmp, ignore_errors=True)


def test_errors(pkg, sc):
    c = next(iter(_pfbwt_golden().values()))
    t = {k: _dev(c[k]) for k in ("dict", "occ", "ilist", "bwlast", "bwsai")}
    torch.cuda.synchronize()
    with pytest.raises(pkg.pfp.PfpError) as e:                       # .occ does not match the dictionary
        sc.pfbwt_device(t["dict"].data_ptr(), len(c["dict"]), t["occ"].data_ptr(), len(c["occ"]) // 4 - 1,
                        t["ilist"].data_ptr(), t["bwlast"].data_ptr(), None, len(c["ilist"]) // 4, c["w"], 0)
    assert e.value.code == -1
    with pytest.raises(pkg.pfp.PfpError) as e:                       # -S without .bwsai
        sc.pfbwt_device(t["dict"].data_ptr(), len(c["dict"]), t["occ"].data_ptr(), len(c["occ"]) // 4,
                        t["ilist"].data_ptr(), t["bwlast"].data_ptr(), None, len(c["ilist"]) // 4, c["w"], pkg.pfp.PFBWT_SA)
    assert e.value.code == -1
