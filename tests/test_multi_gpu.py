"""The multi-GPU path behind the C ABI (pfpb200_multi_*, csrc/pfp_multi.cu; reference: newscan -t T /
pscan -t T, newscan.hpp:230-337, pscan.hpp:114-165): one process, one host thread per listed GPU,
peer-to-peer DMA between them.  A device may be listed several times, so the whole protocol --
shards, seams, routing, exchange, ranks back, assembly of the five streams -- runs on a 1-GPU box;
with two or more GPUs the same tests also run over real peer copies.  Bit-exact vs the oracle."""
import os
import shutil
import subprocess
import tempfile

import numpy as np
import pytest
import torch

from conftest import assert_same_files, golden
from oracle import pfp_oracle as orc

pytestmark = pytest.mark.gpu


def device_lists():
    n = torch.cuda.device_count() if torch.cuda.is_available() else 1
    out = [[0, 0], [0, 0, 0], [0, 0, 0, 0, 0]]
    if n >= 2:
        out += [[0, 1], [1, 0, 1]]
    if n >= 4:
        out += [[0, 1, 2, 3]]
    if n >= 8:
        out += [list(range(8))]
    return out


@pytest.fixture
def small_shards(monkeypatch):
    """Shards down to 4 KB and 256 bytes of reserved front, so that seams, empty shards and the
    growth of the front are exercised by inputs the oracle parses in milliseconds."""
    monkeypatch.setenv("PFPB200_MULTI_MIN_SHARD", "4096")
    monkeypatch.setenv("PFPB200_MULTI_FRONT", "256")


@pytest.mark.parametrize("ids", device_lists(), ids=lambda v: "g" + "".join(map(str, v)))
@pytest.mark.parametrize("w,p", [(10, 100), (4, 10), (16, 500), (40, 100)])
def test_multi_matches_oracle(pkg, small_shards, ids, w, p):
    text = pkg.synth.pangenome_text(30_000, 8, 171).numpy().tobytes()
    ms = pkg.pfp.MultiScanner(ids)
    try:
        got = ms.parse_host(text, w, p, sai=True)
        assert_same_files(got, orc.parse(text, w, p), f"multi {ids} w{w} p{p}")
        st = got.stats
        assert st["n_text"] == len(text) and st["n_phrases"] == got.n_phrases and st["launches"] > 0
        # a second parse on the same handle (buffers reused), other parameters, no .sai
        got2 = ms.parse_host(text, w, p, sai=False)
        assert got2.sai == b"" and got2.parse == got.parse and got2.dict == got.dict
    finally:
        ms.close()


def test_multi_long_run_across_seams_and_front_growth(pkg, small_shards):
    """A run of N covering two whole shards: they own no phrase, and the phrase straddling into
    the next shard starts far more bytes before it than the reserved front."""
    a = pkg.synth.random_dna(20_000, 172).numpy().tobytes()
    text = a + b"N" * 45_000 + a[:15_000]
    for ids in ([0, 0, 0, 0], [0] * 7):
        ms = pkg.pfp.MultiScanner(ids)
        try:
            assert_same_files(ms.parse_host(text, 10, 100), orc.parse(text, 10, 100), f"N run {len(ids)} shards")
        finally:
            ms.close()


def test_multi_tiny_empty_and_truncated_inputs(pkg, small_shards):
    ms = pkg.pfp.MultiScanner([0, 0, 0])
    try:
        for text in (b"", b"ACG", b"ACGTTGCAACG", b"A" * 5000, b"ACGT" * 3000):
            assert_same_files(ms.parse_host(text, 10, 100), orc.parse(text, 10, 100), f"tiny {len(text)}")
        # the input ends at the first byte <= 0x02 (newscan.cpp:364), wherever the shard borders are
        t = pkg.synth.random_dna(40_000, 173).numpy().tobytes()
        for cut in (100, 13_400, 26_667, 39_999):
            text = t[:cut] + b"\x01" + t[cut:]
            got = ms.parse_host(text, 10, 100)
            assert_same_files(got, orc.parse(text, 10, 100), f"invalid byte at {cut}")
            assert got.stats["n_text"] == cut
    finally:
        ms.close()


def test_multi_compress_verify_and_errors(pkg, small_shards):
    text = pkg.synth.pangenome_text(20_000, 6, 174).numpy().tobytes()
    ms = pkg.pfp.MultiScanner([0, 0, 0])
    try:
        want = orc.parse(text, 10, 100)
        got = ms.parse_host(text, 10, 100, compress=True, verify=True)
        assert got.dict == orc.dicz_of(want.dict, 10) and got.parse == want.parse and got.occ == want.occ
        with pytest.raises(pkg.pfp.PfpError) as e:
            ms.parse_host(text, 3, 100)
        assert e.value.code == -1
        assert_same_files(ms.parse_host(text, 10, 100), want, "after an error")
    finally:
        ms.close()


def test_multi_verify_catches_forced_collisions(pkg, small_shards, monkeypatch):
    """2-bit fingerprints (test hook): the shards' local dedup and the owners' merge both have
    collisions; with PFPB200_F_VERIFY the parse stops instead of merging different words."""
    monkeypatch.setenv("PFPB200_TEST_WEAK_FP", "1")
    text = pkg.synth.pangenome_text(20_000, 6, 175).numpy().tobytes()
    ms = pkg.pfp.MultiScanner([0, 0])
    try:
        with pytest.raises(pkg.pfp.PfpError) as e:
            ms.parse_host(text, 10, 100, verify=True)
        assert e.value.code == -6
    finally:
        ms.close()


def test_multi_64mb_equals_single_gpu(pkg):
    """Production shard sizes (no test overrides): 64 MB over 2, 3 and 4 shards against the
    single-GPU parser, and the phase timeline is filled in."""
    t = pkg.synth.pangenome_text(4_000_000, 16, 176)
    host = t.numpy()
    sc = pkg.pfp.Scanner(0)
    want = sc.fetch(sc.parse_device(t.cuda(), 10, 100, sai=True))
    sc.close()
    n = torch.cuda.device_count()
    for ids in ([0, 0], [0, 0, 0], list(range(min(n, 4))) if n > 1 else [0, 0, 0, 0]):
        ms = pkg.pfp.MultiScanner(ids)
        try:
            assert_same_files(ms.parse_host(host, 10, 100), want, f"64 MB over {ids}")
            ph = ms.phase_ms()
            assert len(ph["merge"]) == len(ids) and all(v > 0 for v in ph["words"])
        finally:
            ms.close()


def test_cli_multi_gpu_files_match_reference(pkg):
    """`gpuscan.x -g 0,0,0` (or real GPUs) writes the files the unmodified newscanNT.x wrote for the
    stored plain and FASTA inputs (tests/golden, cases pangenome_plain / pangenome_fasta: the same
    text), through gzip too, and `-t 2` segments concatenate to the same streams.  Shards down to
    4 KB (the small_shards settings) so that these 36 KB inputs are cut at several seams."""
    n = torch.cuda.device_count()
    devs = ",".join(map(str, range(n))) if n > 1 else "0,0,0"
    env = dict(os.environ, PFPB200_MULTI_MIN_SHARD="4096", PFPB200_MULTI_FRONT="256")
    run = lambda cmd: subprocess.run(cmd, check=True, stdout=subprocess.PIPE, text=True, env=env)  # noqa: E731
    plain, fasta = golden().case("pangenome_plain"), golden().case("pangenome_fasta")
    tmp = tempfile.mkdtemp(prefix="pfpmulti_")
    try:
        for c, extra in ((plain, []), (fasta, ["-f"])):
            ours = os.path.join(tmp, c["name"])
            with open(ours, "wb") as f:
                f.write(c["input"])
            r = run([pkg.pfp.CLI_PATH, ours, "-w", str(c["w"]), "-p", str(c["p"]), "-s", "-g", devs, "-v"] + extra)
            assert "merge" in r.stdout          # the per-GPU timeline of -v
            assert_same_files(orc.collect_files(ours), c, f"cli -g {devs} {c['name']}")
        # gzip-compressed FASTA goes through the host reader (zlib, as the reference's gzread)
        import gzip
        gzp = os.path.join(tmp, "ours.gz")
        with gzip.open(gzp, "wb") as f:
            f.write(fasta["input"])
        run([pkg.pfp.CLI_PATH, gzp, "-w", str(fasta["w"]), "-p", str(fasta["p"]), "-s", "-f", "-g", devs])
        assert_same_files(orc.collect_files(gzp), fasta, "cli multi gzip")
        seg = os.path.join(tmp, "seg")
        with open(seg, "wb") as f:
            f.write(plain["input"])
        run([pkg.pfp.CLI_PATH, seg, "-w", str(plain["w"]), "-p", str(plain["p"]), "-s", "-g", devs, "-t", "2"])
        assert_same_files(orc.collect_files(seg, nseg=2), plain, "cli -t 2")
    finally:
        shutil.rmtree(tmp, ignore_errors=True)
