"""Parity of the CUDA path (through the C ABI) with the oracle / the reference's golden outputs.
Bit-exact: every byte of .dict .occ .parse .last .sai."""
import os
import shutil
import subprocess
import tempfile

import numpy as np
import pytest
import torch

from conftest import assert_same_files, golden, golden_dicz, golden_names
from oracle import pfbwt_oracle as po
from oracle import pfp_oracle as orc

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def sc(pkg):
    s = pkg.pfp.Scanner(0)
    yield s
    s.close()


def unparse(dict_bytes: bytes, parse_bytes: bytes, w: int) -> bytes:
    """Rebuild the text from .dict + .parse (what the reference's unparse.c does)."""
    words = dict_bytes[:-1].split(b"\x01")[:-1]
    ranks = np.frombuffer(parse_bytes, dtype=np.uint32)
    parts = []
    for j, r in enumerate(ranks):
        wd = words[r - 1]
        parts.append(wd if j == 0 else wd[w:])
    full = b"".join(parts)
    return full[1:len(full) - w]


@pytest.mark.parametrize("name", golden_names())
def test_golden(pkg, sc, name):
    c = golden().case(name)
    text = pkg.pfp.fasta_extract(c["input"])[0] if c["fasta"] else c["input"]
    got = sc.parse_host(text, c["w"], c["p"], sai=True)
    assert_same_files(got, c, name)


@pytest.mark.parametrize("w,p", [(10, 100), (4, 10), (6, 50), (16, 500), (32, 1000), (13, 37),
                                 (19, 64), (27, 100), (40, 100), (100, 50)])
def test_trigger_scan_vs_oracle(pkg, sc, w, p):
    n = 300_000
    text = pkg.synth.random_dna(n, 21).numpy()
    for off in (0, 1, 7, 15):          # misaligned shard starts
        buf = torch.from_numpy(np.concatenate([np.zeros(off, np.uint8), text])).cuda()
        got, _ = sc.scan_triggers(buf[off:], w, p)
        want = orc.triggers(text.tobytes(), w, p)
        assert np.array_equal(got, want), f"w={w} p={p} off={off}: {len(got)} vs {len(want)}"


@pytest.mark.parametrize("w,p", [(4, 10), (5, 11), (6, 64), (7, 16), (8, 33), (9, 1000), (10, 10), (10, 100),
                                 (10, 65536), (10, 99991), (10, 1999999), (10, 3999999946),
                                 (11, 100), (12, 50), (13, 1000), (14, 10), (15, 500), (16, 100), (16, 500), (16, 65536)])
def test_interval_form_scan_vs_oracle_and_other_forms(pkg, w, p):
    """K1's interval form (kr_scan_ivf_k: two 5-symbol blocks for w <= 10, four 4-symbol blocks for
    w <= 16) against the oracle and against the rolling form, on DNA with rows that leave the interval
    form (N runs, lower case, a newline) and at misaligned starts.  p >= PW (the case (10, 3999999946))
    has no inverse: the library falls back to the rolling form."""
    n = 700_000
    text = pkg.synth.random_dna(n, 77 + w).numpy().copy()
    text[100_000:103_000] = ord("N")
    text[300_010:300_050] |= 0x20            # lower case
    text[500_000] = ord("\n")
    text[n - 5] = ord("N")
    want = orc.triggers(text.tobytes(), w, p)
    for mode in ("", "rolling"):
        old = os.environ.get("PFPB200_K1")
        if mode:
            os.environ["PFPB200_K1"] = mode
        else:
            os.environ.pop("PFPB200_K1", None)
        try:
            s = pkg.pfp.Scanner(0)
        finally:
            if old is None:
                os.environ.pop("PFPB200_K1", None)
            else:
                os.environ["PFPB200_K1"] = old
        try:
            for off in (0, 5, 16):
                buf = torch.from_numpy(np.concatenate([np.zeros(off, np.uint8), text])).cuda()
                got, _ = s.scan_triggers(buf[off:], w, p)
                assert np.array_equal(got, want), f"mode={mode or 'interval'} w={w} p={p} off={off}: {len(got)} vs {len(want)}"
        finally:
            s.close()


def test_trigger_scan_shard_with_halo(pkg, sc):
    """A shard [lo,hi) scanned from a buffer with a left halo gives exactly the global triggers
    in [lo,hi) (pscan.hpp:44-108 semantics, sequential first-window rule)."""
    w, p, n = 10, 100, 500_000
    text = pkg.synth.random_dna(n, 22).numpy()
    want = orc.triggers(text.tobytes(), w, p)
    whole = torch.from_numpy(text).cuda()
    cuts = [0, 100_003, 250_000, 250_001, 499_990, n]
    got_all = []
    for lo, hi in zip(cuts[:-1], cuts[1:]):
        b0 = max(0, lo - (w - 1))
        got, _ = sc.scan_triggers(whole[b0:hi], w, p, buf_pos0=b0, own_lo=lo, own_hi=hi)
        got_all.append(got)
    assert np.array_equal(np.concatenate(got_all), want)


@pytest.mark.parametrize("seed,n,w,p", [(31, 1000, 10, 100), (32, 40_000, 10, 100), (33, 1_000_000, 10, 100),
                                         (34, 300_000, 4, 10), (35, 300_000, 6, 50), (36, 500_000, 16, 500),
                                         (37, 500_000, 32, 1000), (38, 200_000, 19, 77), (39, 65_537, 10, 100)])
def test_random_dna_vs_oracle(pkg, sc, seed, n, w, p):
    text = pkg.synth.random_dna(n, seed).numpy().tobytes()
    assert_same_files(sc.parse_host(text, w, p), orc.parse(text, w, p), f"seed{seed}")


@pytest.mark.parametrize("w,p", [(10, 100), (6, 50), (16, 500), (32, 1000)])
def test_pangenome_vs_oracle(pkg, sc, w, p):
    text = pkg.synth.pangenome_text(100_000, 20, 41).numpy().tobytes()
    got = sc.parse_host(text, w, p)
    want = orc.parse(text, w, p)
    assert_same_files(got, want, f"pangenome w{w} p{p}")
    assert got.stats["n_distinct"] == want.n_distinct and got.stats["sum_word_len"] == want.sum_word_len


def test_all_byte_values_vs_oracle(sc):
    rng = np.random.default_rng(51)
    text = rng.integers(3, 256, 400_000, dtype=np.uint8).tobytes()
    assert_same_files(sc.parse_host(text, 10, 100), orc.parse(text, 10, 100), "bytes")
    assert_same_files(sc.parse_host(text, 5, 17), orc.parse(text, 5, 17), "bytes w5")


def test_long_phrases_vs_oracle(pkg, sc):
    """Phrases beyond 64 KB take the one-CTA-per-phrase fingerprint path; long shared prefixes
    stress the ranking rounds."""
    a = pkg.synth.random_dna(50_000, 61).numpy().tobytes()
    b = pkg.synth.random_dna(50_000, 62).numpy().tobytes()
    text = a + b"N" * 200_000 + b + b"N" * 70_000 + a[:1000] + b"N" * 200_000 + b[:3000]
    assert_same_files(sc.parse_host(text, 10, 100), orc.parse(text, 10, 100), "long")
    text2 = b"A" * 150_000
    assert_same_files(sc.parse_host(text2, 10, 100), orc.parse(text2, 10, 100), "allA")


def test_low_complexity_vs_oracle(sc):
    rng = np.random.default_rng(71)
    unit = b"ACACACACGT"
    text = unit * 3000 + bytes(rng.choice(np.frombuffer(b"AC", np.uint8), 50_000)) + unit * 2000
    for (w, p) in [(10, 100), (4, 10), (8, 16)]:
        assert_same_files(sc.parse_host(text, w, p), orc.parse(text, w, p), f"lowcx w{w}")


def test_dictionary_table_resize_retry(pkg):
    """The dictionary table is sized from the previous parse's distinct/phrase ratio; an input
    with far more distinct words than that guess must trigger the overflow retry and still be exact."""
    s = pkg.pfp.Scanner(0)
    rep = (pkg.synth.random_dna(2000, 77).numpy().tobytes()) * 400        # ~1% distinct
    assert_same_files(s.parse_host(rep, 10, 100), orc.parse(rep, 10, 100), "repetitive")
    rnd = pkg.synth.random_dna(800_000, 78).numpy().tobytes()              # ~100% distinct
    assert_same_files(s.parse_host(rnd, 10, 100), orc.parse(rnd, 10, 100), "random after repetitive")
    assert_same_files(s.parse_host(rep, 10, 100), orc.parse(rep, 10, 100), "repetitive again")
    s.close()


def test_invalid_byte_truncates(sc):
    text = b"ACGT" * 5000 + b"\x01" + b"ACGT" * 100
    got = sc.parse_host(text, 10, 100)
    assert_same_files(got, orc.parse(text, 10, 100), "invalid")
    assert got.stats["n_text"] == 20000


def test_device_entry_matches_host_entry(pkg, sc):
    t = pkg.synth.pangenome_text(50_000, 10, 81)
    want = sc.parse_host(t.numpy().tobytes(), 10, 100)
    out = sc.parse_device(t.cuda(), 10, 100, sai=True)
    got = sc.fetch(out)
    assert_same_files(got, want, "device entry")
    out = sc.parse_device(t.cuda(), 10, 100, sai=False)
    assert not out.sai


def test_stream_k2_misaligned_buffers_and_dense_triggers(pkg, sc):
    """The streaming K2 pass (pfp_stream.cu): device buffers that start at every alignment within
    16 bytes, phrases crossing run / warp / tile borders, runs holding many phrases (small p) and
    tiles holding none (N runs)."""
    a = pkg.synth.random_dna(150_000, 131).numpy()
    text = np.concatenate([a, np.full(100_000, ord("N"), np.uint8), a[:70_000],
                           np.frombuffer(b"ACGTTGCA" * 4000, np.uint8), a[5_000:90_000]])
    for (w, p) in [(10, 100), (4, 10), (7, 11), (32, 50), (16, 1000)]:
        want = orc.parse(text.tobytes(), w, p)
        for off in (0, 3, 9):
            buf = torch.from_numpy(np.concatenate([np.full(off, 65, np.uint8), text])).cuda()
            got = sc.fetch(sc.parse_device(buf[off:], w, p, sai=True))
            assert_same_files(got, want, f"stream w{w} p{p} off{off}")


def test_stream_k2_equals_per_phrase_k2_64mb(pkg):
    """Same files from the streaming K2 and from the per-phrase K2 kernels it replaced
    (PFPB200_LEGACY_K2=1), at a size the oracle is too slow for."""
    t = pkg.synth.pangenome_text(4_000_000, 16, 133).cuda()
    res = []
    for legacy in ("0", "1"):
        os.environ["PFPB200_LEGACY_K2"] = legacy
        try:
            s = pkg.pfp.Scanner(0)
        finally:
            os.environ.pop("PFPB200_LEGACY_K2", None)
        res.append(s.fetch(s.parse_device(t, 10, 100, sai=True)))
        s.close()
    assert_same_files(res[0], res[1], "stream vs per-phrase K2")


@pytest.mark.parametrize("w,p", [(10, 500), (16, 1000), (10, 100)])
def test_rank_lcp_walks_on_large_families(pkg, w, p):
    """Families of near-identical long words (many haplotypes, large p): tie groups of 33..256 words
    are ranked by LCP walks against the group's head (rank_lcp_k).  Against the oracle, and against
    the chunk-pass kernel it replaced (PFPB200_RANK_CHUNK_PASSES=1)."""
    text = pkg.synth.pangenome_text(150_000, 150, 136).numpy().tobytes()
    want = orc.parse(text, w, p)
    for chunk_passes in ("0", "1"):
        os.environ["PFPB200_RANK_CHUNK_PASSES"] = chunk_passes
        try:
            s = pkg.pfp.Scanner(0)
        finally:
            os.environ.pop("PFPB200_RANK_CHUNK_PASSES", None)
        assert_same_files(s.parse_host(text, w, p), want, f"families w{w} p{p} chunk_passes={chunk_passes}")
        s.close()


@pytest.mark.parametrize("name", sorted(golden_dicz()))
def test_compress_mode_dicz_golden(pkg, sc, name):
    """-c against the .dicz the unmodified newscanNT.x -c wrote (tools/make_golden_dicz.py)."""
    meta, dicz = golden_dicz()[name]
    c = golden().case(name)
    text = pkg.pfp.fasta_extract(c["input"])[0] if c["fasta"] else c["input"]
    comp = sc.parse_host(text, c["w"], c["p"], compress=True)
    assert comp.dict == dicz, f"{name}: .dicz differs ({len(comp.dict)} vs {len(dicz)} bytes)"
    assert comp.parse == c["parse"] and comp.occ == c["occ"] and comp.last == c["last"]


def test_compress_mode_dicz(pkg, sc):
    """-c at a larger size: words lose their last w bytes and the leading 0x02 (newscan.cpp:410-413;
    the rule is pinned to newscanNT.x -c by test_oracle_dicz_matches_golden)."""
    text = pkg.synth.pangenome_text(30_000, 5, 82).numpy().tobytes()
    w = 10
    plain = sc.parse_host(text, w, 100)
    comp = sc.parse_host(text, w, 100, compress=True)
    assert comp.dict == orc.dicz_of(plain.dict, w) and comp.parse == plain.parse and comp.occ == plain.occ


@pytest.mark.parametrize("w,p,n", [(9000, 100, 400_000), (8192, 50, 300_000), (7000, 500, 600_000),
                                   (40, 10, 300), (40, 10, 41), (33, 11, 2000), (65536, 100, 200_000)])
def test_huge_windows_and_tiny_inputs_per_phrase_k2(pkg, sc, w, p, n):
    """The per-phrase K2 path (w > 32): every phrase is longer than one fingerprint segment when
    w >= 8192, and on tiny inputs most phrases end within the last bytes of the buffer -- both
    used to overflow the list of phrases handed to the long-phrase kernel."""
    text = pkg.synth.random_dna(n, 140 + w % 7).numpy().tobytes()
    assert_same_files(sc.parse_host(text, w, p), orc.parse(text, w, p), f"w{w} p{p} n{n}")


def test_verify_flag_catches_forced_collisions(pkg):
    """PFPB200_F_VERIFY compares every phrase with its dictionary word byte for byte
    (newscan.cpp:282-286).  With the fingerprints cut to 2 bits (test hook) almost all phrases
    collide: without the flag the merge is silent, with it the parse must stop with E_COLLISION;
    with full fingerprints the flag changes nothing."""
    text = pkg.synth.pangenome_text(30_000, 6, 83).numpy().tobytes()
    want = orc.parse(text, 10, 100)
    s = pkg.pfp.Scanner(0)
    assert_same_files(s.parse_host(text, 10, 100, verify=True), want, "verify on")
    assert_same_files(s.fetch(s.parse_device(torch.from_numpy(np.frombuffer(text, np.uint8).copy()).cuda(),
                                             10, 100, verify=True)), want, "verify on, device entry")
    s.close()
    os.environ["PFPB200_TEST_WEAK_FP"] = "1"
    try:
        weak = pkg.pfp.Scanner(0)
    finally:
        os.environ.pop("PFPB200_TEST_WEAK_FP", None)
    with pytest.raises(pkg.pfp.PfpError) as e:
        weak.parse_host(text, 10, 100, verify=True)
    assert e.value.code == -6
    weak.close()


def test_bad_arguments(pkg, sc):
    with pytest.raises(pkg.pfp.PfpError) as e:
        sc.parse_host(b"ACGT" * 100, w=3, p=100)
    assert e.value.code == -1
    with pytest.raises(pkg.pfp.PfpError):
        sc.parse_host(b"ACGT" * 100, w=10, p=9)


def test_round_trip_properties_32mb(pkg, sc):
    """Size-independent properties at a size the oracle is too slow for in a unit test."""
    w, p = 10, 100
    t = pkg.synth.pangenome_text(2_000_000, 16, 91)
    text = t.numpy().tobytes()
    got = sc.parse_host(text, w, p)
    words = got.dict[:-1].split(b"\x01")[:-1]
    assert got.dict[-1:] == b"\x00" and len(words) == got.n_distinct
    assert all(words[i] < words[i + 1] for i in range(len(words) - 1)), "dictionary not sorted/unique"
    occ = np.frombuffer(got.occ, np.uint32)
    ranks = np.frombuffer(got.parse, np.uint32)
    assert occ.sum() == got.n_phrases
    assert np.array_equal(np.bincount(ranks, minlength=len(words) + 1)[1:], occ)
    assert unparse(got.dict, got.parse, w) == text
    sai = np.frombuffer(got.sai, np.uint8).reshape(-1, 5).astype(np.uint64)
    pos = sum(sai[:, i] << np.uint64(8 * i) for i in range(5))
    assert pos[-1] == len(text) + w and np.all(np.diff(pos.astype(np.int64)) > 0)
    tb = np.frombuffer(text, np.uint8)
    last = np.frombuffer(got.last, np.uint8)
    assert np.array_equal(last[:-1], tb[pos[:-1].astype(np.int64) - 1 - w]) and last[-1] == tb[-1]


def test_cli_files_and_bwt_match_reference(pkg):
    """gpuscan.x as the drop-in for newscan.x: byte-identical to the files newscanNT.x -s -f wrote for a
    stored FASTA (tests/golden, case pangenome_fasta), also as -t 3 segments and through gzip; and
    gpubwtparse.x + gpupfbwt.x turn them into the BWT and suffix array of the text (bigbwt -f -S)."""
    c = golden().case("pangenome_fasta")
    w, p = str(c["w"]), str(c["p"])
    tmp = tempfile.mkdtemp(prefix="pfpcli_")
    try:
        ours, seg = os.path.join(tmp, "ours.fa"), os.path.join(tmp, "seg.fa")
        for pth in (ours, seg):
            with open(pth, "wb") as f:
                f.write(c["input"])
        subprocess.run([pkg.pfp.CLI_PATH, ours, "-w", w, "-p", p, "-s", "-f"], check=True, stdout=subprocess.PIPE)
        assert_same_files(orc.collect_files(ours), c, "cli")
        subprocess.run([pkg.pfp.BWTPARSE_CLI_PATH, ours, "-s"], check=True, stdout=subprocess.PIPE)
        subprocess.run([pkg.pfp.PFBWT_CLI_PATH, "-w", w, ours, "-S"], check=True, stdout=subprocess.PIPE)
        want = po.pfbwt(orc.fasta_extract(c["input"])[0])
        for ext in ("bwt", "sa"):
            assert open(ours + "." + ext, "rb").read() == want[ext], ext
        # segmented .last/.sai (-t 3) concatenate to the same streams
        subprocess.run([pkg.pfp.CLI_PATH, seg, "-w", w, "-p", p, "-s", "-f", "-t", "3"], check=True,
                       stdout=subprocess.PIPE)
        assert_same_files(orc.collect_files(seg, nseg=3), c, "cli -t 3")
        # gzip-compressed FASTA, as the reference's kseq/gzread takes it
        import gzip
        gz = os.path.join(tmp, "ours.gz")
        with gzip.open(gz, "wb") as f:
            f.write(c["input"])
        subprocess.run([pkg.pfp.CLI_PATH, gz, "-w", w, "-p", p, "-s", "-f"], check=True, stdout=subprocess.PIPE)
        assert_same_files(orc.collect_files(gz), c, "cli gzip")
    finally:
        shutil.rmtree(tmp, ignore_errors=True)


def test_config1_yeast_shaped_fasta_to_bwt(pkg):
    """BASELINE config 1 (`bigbwt yeast.fasta -w 10 -p 100`; the bundled file is not in the repository,
    so a stand-in of its shape: 17 records, 12.16 Mbp, 60-column FASTA).  gpuscan.x, gpubwtparse.x and
    gpupfbwt.x write the files of newscanNT.x -s -f, bwtparse -s and pfbwtNT.x -S (sha256 in
    tests/golden/config1_sha256.json), and the .bwt is the BWT of the extracted text -- the check
    `bigbwt -c` does (bigbwt:176-195; on the extracted text, SURVEY App. B3)."""
    import hashlib
    import json
    with open(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "config1_sha256.json")) as f:
        want_sha = json.load(f)["sha256"]
    recs = [r.numpy() for r in pkg.synth.yeast_like_records(1)]
    assert len(recs) == 17 and 12_000_000 < sum(r.size for r in recs) < 12_300_000
    fa = b"".join(pkg.synth.to_fasta_np(r, f"{nm} stand-in").tobytes() for r, nm in zip(recs, pkg.synth.YEAST_NAMES))
    tmp = tempfile.mkdtemp(prefix="pfpyeast_")
    try:
        ours = os.path.join(tmp, "ours.fa")
        with open(ours, "wb") as f:
            f.write(fa)
        run = lambda cmd: subprocess.run(cmd, check=True, stdout=subprocess.PIPE, stderr=subprocess.STDOUT)  # noqa: E731
        run([pkg.pfp.CLI_PATH, ours, "-w", "10", "-p", "100", "-s", "-f"])
        run([pkg.pfp.BWTPARSE_CLI_PATH, ours, "-s"])
        run([pkg.pfp.PFBWT_CLI_PATH, "-w", "10", ours, "-S"])
        for ext, sha in want_sha.items():
            with open(ours + "." + ext, "rb") as f:
                assert hashlib.sha256(f.read()).hexdigest() == sha, f".{ext} differs from the reference's"
        text, trunc = pkg.pfp.read_input(ours, fasta=True)
        assert not trunc and text == b"".join(r.tobytes() for r in recs)
        assert open(ours + ".bwt", "rb").read() == po.pfbwt(text)["bwt"], "BWT differs from the suffix array of the text"
    finally:
        shutil.rmtree(tmp, ignore_errors=True)
