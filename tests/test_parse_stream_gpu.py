"""The streamed parse of pfpb200_parse_file: inputs larger than the device memory pass through HBM in
chunks against one dictionary.  PFPB200_PARSE_BUDGET=<bytes> makes megabyte inputs take that path
(chunks of budget / 8 new bytes); every case asserts that it did, and compares the five files byte for
byte with the one-shot parse_file of the same input and, where the case is golden, with the files the
unmodified newscanNT.x wrote."""
import gzip
import os
import shutil
import subprocess
import tempfile

import numpy as np
import pytest

from conftest import assert_same_files, golden, golden_names
from oracle import pfp_oracle as orc

pytestmark = pytest.mark.gpu

BYTES_PER_BYTE = 8          # chunk = budget / 8 new input bytes (pfp_chunked.cu)


def budget_for(nbytes, chunks):
    """a budget whose chunks take about nbytes / chunks new bytes each"""
    return BYTES_PER_BYTE * max(256, -(-max(nbytes, 1) // chunks))


@pytest.fixture(scope="module")
def sc(pkg):
    s = pkg.pfp.Scanner(0)
    yield s
    s.close()


@pytest.fixture
def tmp():
    d = tempfile.mkdtemp(prefix="pfpstream_")
    yield d
    shutil.rmtree(d, ignore_errors=True)


def _files(path, sai=True, nseg=0, compress=False):
    f = orc.collect_files(path, nseg=nseg, sai=sai) if not compress else None
    if compress:                                         # .dicz in place of .dict
        os.replace(path + ".dicz", path + ".dict")
        f = orc.collect_files(path, nseg=nseg, sai=sai)
    return f


def parse(sc, monkeypatch, tmp, name, data, w, p, budget=None, sai=True, fasta=False, nseg=0, compress=False,
          verify=False):
    """data -> <tmp>/<name>/in, parsed by parse_file (with the budget knob if given): (files, stats)"""
    d = os.path.join(tmp, name + ("_stream" if budget else "_oneshot"))
    os.makedirs(d, exist_ok=True)
    path = os.path.join(d, "in")
    with open(path, "wb") as f:
        f.write(data)
    if budget:
        monkeypatch.setenv("PFPB200_PARSE_BUDGET", str(budget))
    else:
        monkeypatch.delenv("PFPB200_PARSE_BUDGET", raising=False)
    st = sc.parse_file(path, w, p, sai=sai, fasta=fasta, nseg=nseg, compress=compress, verify=verify)
    monkeypatch.delenv("PFPB200_PARSE_BUDGET", raising=False)
    return _files(path, sai=sai, nseg=nseg, compress=compress), st


def same_as_oneshot(sc, monkeypatch, tmp, name, data, w, p, chunks, min_chunks=3, **kw):
    want, st1 = parse(sc, monkeypatch, tmp, name, data, w, p, **kw)
    assert st1["chunks"] == 0, "the one-shot path must stay the one-shot path"
    got, st2 = parse(sc, monkeypatch, tmp, name, data, w, p, budget=budget_for(len(data), chunks), **kw)
    assert min_chunks <= st2["chunks"] <= 50, f"{name}: {st2['chunks']} chunks"
    assert_same_files(got, want, name)
    for k in ("n_text", "n_phrases", "n_distinct", "sum_word_len", "dict_bytes", "alg_bytes"):
        assert st2[k] == st1[k], f"{name}: stats {k}"
    return st2


@pytest.mark.parametrize("chunks", [4, 16])
@pytest.mark.parametrize("name", golden_names())
def test_golden_streamed(pkg, sc, monkeypatch, tmp, name, chunks):
    c = golden().case(name)
    got, st = parse(sc, monkeypatch, tmp, name, c["input"], c["w"], c["p"],
                    budget=budget_for(len(c["input"]), chunks), fasta=c["fasta"])
    assert 0 < st["chunks"] <= 50
    if st["n_text"] >= max(256 * chunks, len(c["input"]) // 2):     # (a cut or headers leave less text)
        assert st["chunks"] >= 3
    assert_same_files(got, c, name)


@pytest.mark.parametrize("w,p", [(4, 10), (10, 100), (16, 500), (32, 1000), (40, 100)])
def test_pangenome_streamed(pkg, sc, monkeypatch, tmp, w, p):
    """w = 40 takes the per-phrase K2 kernels"""
    text = np.concatenate([r.numpy() for r in pkg.synth.pangenome_records(200_000, 8, 71)]).tobytes()
    same_as_oneshot(sc, monkeypatch, tmp, f"pan_w{w}_p{p}", text, w, p, chunks=12)


def test_run_of_n_across_chunks(pkg, sc, monkeypatch, tmp):
    """one phrase spans several chunks: the carry grows"""
    a = pkg.synth.random_dna(30_000, 3).numpy().tobytes()
    b = pkg.synth.random_dna(30_000, 4).numpy().tobytes()
    data = a + b"N" * 50_000 + b
    st = same_as_oneshot(sc, monkeypatch, tmp, "nrun", data, 10, 100, chunks=11)   # 10 KB chunks: N over 5
    assert st["chunks"] >= 10


def test_text_without_trigger(pkg, sc, monkeypatch, tmp):
    for ch in b"ACGTN":
        data = bytes([ch]) * 20_000
        if orc.parse(data, 10, 100).n_phrases == 1:
            break
    else:
        pytest.skip("every constant text has a trigger")
    st = same_as_oneshot(sc, monkeypatch, tmp, "notrigger", data, 10, 100, chunks=8)
    assert st["n_phrases"] == 1


@pytest.mark.parametrize("data", [b"", b"ACGTA", b"ACGTACGTA"])
def test_empty_and_shorter_than_w(pkg, sc, monkeypatch, tmp, data):
    st = same_as_oneshot(sc, monkeypatch, tmp, f"tiny{len(data)}", data, 10, 100, chunks=4, min_chunks=1)
    assert st["chunks"] == 1


def test_all_byte_values(pkg, sc, monkeypatch, tmp):
    rng = np.random.default_rng(9)
    data = rng.integers(3, 256, 120_000, dtype=np.uint8).tobytes()
    same_as_oneshot(sc, monkeypatch, tmp, "bytes", data, 5, 17, chunks=10)


def test_invalid_byte_in_a_late_chunk(pkg, sc, monkeypatch, tmp):
    data = bytearray(pkg.synth.random_dna(100_000, 5).numpy().tobytes())
    data[83_001] = 1
    st = same_as_oneshot(sc, monkeypatch, tmp, "invalid", bytes(data), 10, 100, chunks=10)
    assert st["n_text"] == 83_001


def _fasta(pkg, single_line=False):
    recs = [r.numpy() for r in pkg.synth.pangenome_records(30_000, 5, 11)]
    out = []
    for k, r in enumerate(recs):
        s = bytearray(r.tobytes())
        s[1000:4000] = s[1000:4000].lower()                                  # lowercase stretch
        name = f">hap{k} " + "description " * (40 + 30 * k)                   # headers of 0.5 .. 2 KB
        if single_line:
            out.append(name.encode() + b"\n" + bytes(s) + b"\n")
        else:
            body = b"\n".join(bytes(s[i:i + 60]) for i in range(0, len(s), 60))
            out.append(name.encode() + b"\n" + body + b"\n")
    return b"".join(out)


@pytest.mark.parametrize("single_line", [False, True])
def test_fasta_headers_across_chunk_borders(pkg, sc, monkeypatch, tmp, single_line):
    data = _fasta(pkg, single_line)
    same_as_oneshot(sc, monkeypatch, tmp, f"fa{int(single_line)}", data, 10, 100, chunks=40, fasta=True)


def test_gzip_fasta_and_fastq_take_the_host_text(pkg, sc, monkeypatch, tmp):
    data = _fasta(pkg)
    same_as_oneshot(sc, monkeypatch, tmp, "fagz", gzip.compress(data), 10, 100, chunks=2, fasta=True)   # chunks of the inflated text
    seq = pkg.synth.random_dna(40_000, 6).numpy().tobytes()
    fq = b"".join(b"@r%d\n%s\n+\n%s\n" % (i, seq[i * 400:(i + 1) * 400], b"I" * 400) for i in range(100))
    same_as_oneshot(sc, monkeypatch, tmp, "fq", fq, 10, 100, chunks=5, fasta=True)


def test_k0_refuses_a_late_chunk(pkg, sc, monkeypatch, tmp):
    """a '\\r' far into the file: the streamed path starts again from the host reader's text"""
    data = _fasta(pkg)
    k = data.index(b"\n", len(data) * 3 // 4)
    data = data[:k] + b"\r" + data[k:]
    same_as_oneshot(sc, monkeypatch, tmp, "fa_cr", data, 10, 100, chunks=10, fasta=True)


def test_options_compress_segments_verify_and_no_sai(pkg, sc, monkeypatch, tmp):
    text = np.concatenate([r.numpy() for r in pkg.synth.pangenome_records(100_000, 6, 13)]).tobytes()
    same_as_oneshot(sc, monkeypatch, tmp, "c_t3", text, 10, 100, chunks=8, compress=True, nseg=3)
    same_as_oneshot(sc, monkeypatch, tmp, "verify", text, 10, 100, chunks=8, verify=True)
    same_as_oneshot(sc, monkeypatch, tmp, "nosai", text, 10, 100, chunks=8, sai=False)
    d = os.path.join(tmp, "c_t3_stream")
    assert not any(f.endswith(".part") for f in os.listdir(d)), "the unsegmented streams are removed"


def test_verify_catches_forced_collisions_across_chunks(pkg, monkeypatch, tmp):
    """2-bit fingerprints make different words meet in the global table; -V must stop the parse"""
    monkeypatch.setenv("PFPB200_TEST_WEAK_FP", "1")
    s = pkg.pfp.Scanner(0)
    try:
        text = pkg.synth.random_dna(60_000, 8).numpy().tobytes()
        with pytest.raises(pkg.pfp.PfpError) as e:
            parse(s, monkeypatch, tmp, "weak", text, 10, 100, budget=budget_for(len(text), 6), verify=True)
        assert e.value.code == -6
    finally:
        s.close()


def test_gpuscan_with_the_knob(pkg, tmp):
    text = np.concatenate([r.numpy() for r in pkg.synth.pangenome_records(100_000, 6, 17)])
    fa = pkg.synth.to_fasta_np(text, "all").tobytes()
    outs = {}
    for mode in ("oneshot", "stream"):
        d = os.path.join(tmp, mode)
        os.makedirs(d)
        path = os.path.join(d, "in.fa")
        with open(path, "wb") as f:
            f.write(fa)
        env = dict(os.environ)
        env.pop("PFPB200_PARSE_BUDGET", None)
        if mode == "stream":
            env["PFPB200_PARSE_BUDGET"] = str(budget_for(len(fa), 10))
        r = subprocess.run([pkg.pfp.CLI_PATH, path, "-w", "10", "-p", "100", "-s", "-f", "-v"], env=env, check=True,
                           stdout=subprocess.PIPE, text=True)
        plan = [l for l in r.stdout.splitlines() if l.startswith("Parse plan:")]
        assert plan and (("streamed in" in plan[0]) == (mode == "stream")), r.stdout
        counts = [l for l in r.stdout.splitlines() if l.startswith(("Total input", "Found", "Sum of", "Total number"))]
        outs[mode] = (orc.collect_files(path), counts)
    assert_same_files(outs["stream"][0], outs["oneshot"][0], "gpuscan.x")
    assert outs["stream"][1] == outs["oneshot"][1]


def test_peak_within_budget_plus_dictionary(pkg, sc, monkeypatch, tmp):
    text = np.concatenate([r.numpy() for r in pkg.synth.pangenome_records(500_000, 8, 23)]).tobytes()
    budget = budget_for(len(text), 30)
    _, st = parse(sc, monkeypatch, tmp, "peak", text, 10, 100, budget=budget)
    assert 3 <= st["chunks"] <= 50
    # the global dictionary: per word 36 B of arrays and a table of <= 4 slots of 16 B (capacities <= 2x),
    # the pool (<= 2x its bytes), and at the end the ranking scratch and .dict/.occ
    dict_mem = 256 * st["n_distinct"] + 4 * st["dict_bytes"] + (1 << 20)
    assert st["peak_device_bytes"] <= budget + dict_mem, (st["peak_device_bytes"], budget, dict_mem)


def test_config2_streamed_in_about_4_chunks(pkg, tmp):
    """config 2 (100 haplotypes x 40 Mbp, w 10 p 100) through the streamed path: sha256 of the five files
    == the unmodified newscanNT.x's (tests/golden/fullsize_sha256.json)"""
    import sys
    import torch
    free, _ = torch.cuda.mem_get_info()
    if free < 40 * (1 << 30):
        pytest.skip("needs 40 GB of free device memory")
    sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tools"))
    import stream_check as sck
    path = os.path.join(tmp, "config2.txt")
    sck.write_config2(pkg, path, fasta=False)
    res = sck.check_file(pkg, path, "config2 w10 p100", chunks=4, fasta=False)
    assert res["ok"], res
