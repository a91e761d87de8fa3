"""CPU-side checks of the drop-in boundary: the library loads, exports every symbol the
public header declares, and refuses to work without a GPU (no CPU fallback)."""
import ctypes as C
import os
import re

import pytest
import torch

from conftest import ROOT, assert_same_files, golden, golden_names
from oracle import pfp_oracle as orc


def header_functions():
    src = open(os.path.join(ROOT, "include", "pfpb200.h")).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(pfpb200_\w+)\s*\(", src)))


def test_library_exports_every_declared_symbol(pkg):
    L = pkg.pfp.load_library()
    names = header_functions()
    assert len(names) >= 11
    for n in names:
        assert hasattr(L, n), f"libpfpb200.so does not export {n}"
    assert set(names) == set(pkg.pfp.SYMBOLS)
    assert L.pfpb200_abi_version() == 2


def test_struct_layouts_match_header(pkg):
    # sizes the C compiler gives the public structs (natural alignment, no packing)
    assert C.sizeof(pkg.pfp.Opts) == 16
    assert C.sizeof(pkg.pfp.Outputs) == 64
    assert C.sizeof(pkg.pfp.Stats) == 6 * 8 + 2 * 4 + 12 * 4


def test_strerror(pkg):
    L = pkg.pfp.load_library()
    assert L.pfpb200_strerror(0) == b"ok"
    assert b"CUDA" in L.pfpb200_strerror(-3)


@pytest.mark.skipif(torch.cuda.is_available(), reason="only meaningful on a box without a GPU")
def test_no_cpu_fallback(pkg):
    with pytest.raises(pkg.pfp.PfpError) as e:
        pkg.pfp.Scanner(0)
    assert e.value.code == -3


def test_cli_rejects_bad_arguments(pkg):
    import subprocess
    r = subprocess.run([pkg.pfp.CLI_PATH, "/nonexistent", "-w", "3"], capture_output=True, text=True)
    assert r.returncode == 1 and "Windows size must be at least 4" in r.stdout
    r = subprocess.run([pkg.pfp.CLI_PATH, "/nonexistent", "-p", "5"], capture_output=True, text=True)
    assert r.returncode == 1 and "Modulus must be at least 10" in r.stdout
    r = subprocess.run([pkg.pfp.CLI_PATH], capture_output=True, text=True)
    assert r.returncode == 1 and "Invalid number of arguments" in r.stdout


def test_clis_of_the_later_stages_check_their_arguments(pkg):
    """gpubwtparse.x / gpupfbwt.x / gpuunparse.x / gpubigbwt.x: the argument errors of the reference's
    tools (bwtparse.c:131-160, pfbwt.cpp:257-315, unparse.c:33-64, bigbwt:59-61), before any GPU work."""
    import subprocess
    P = pkg.pfp
    r = subprocess.run([P.BWTPARSE_CLI_PATH], capture_output=True, text=True)
    assert r.returncode == 1 and "Usage" in r.stdout and "permute also sa info" in r.stdout
    r = subprocess.run([P.PFBWT_CLI_PATH, "-w", "10", "-S", "-s", "x"], capture_output=True, text=True)
    assert r.returncode == 1 and "not both" in r.stdout
    r = subprocess.run([P.PFBWT_CLI_PATH, "-w", "3", "x"], capture_output=True, text=True)
    assert r.returncode == 1 and "Windows size must be at least 4" in r.stdout
    r = subprocess.run([P.PFBWT_CLI_PATH], capture_output=True, text=True)
    assert r.returncode == 1 and "Invalid number of arguments" in r.stdout
    r = subprocess.run([P.UNPARSE_CLI_PATH], capture_output=True, text=True)
    assert r.returncode == 1 and "Usage" in r.stdout
    r = subprocess.run([P.BIGBWT_CLI_PATH, "x", "-S", "-e"], capture_output=True, text=True)
    assert r.returncode == 1 and "not both" in r.stdout
    r = subprocess.run([P.BIGBWT_CLI_PATH, "x", "-p", "5"], capture_output=True, text=True)
    assert r.returncode == 1 and "Modulus must be at least 10" in r.stdout


@pytest.mark.skipif(torch.cuda.is_available(), reason="only meaningful on a box without a GPU")
def test_later_stage_clis_fail_loudly_without_a_gpu(pkg, tmp_path):
    import subprocess
    base = str(tmp_path / "x")
    for exe in (pkg.pfp.BWTPARSE_CLI_PATH, pkg.pfp.UNPARSE_CLI_PATH, pkg.pfp.BIGBWT_CLI_PATH):
        r = subprocess.run([exe, base], capture_output=True, text=True)
        assert r.returncode == 1 and "cannot use CUDA device" in r.stderr, exe
    r = subprocess.run([pkg.pfp.PFBWT_CLI_PATH, "-w", "10", base], capture_output=True, text=True)
    assert r.returncode == 1 and "cannot use CUDA device" in r.stderr


@pytest.mark.parametrize("name", [n for n in golden_names() if n.startswith(("fasta", "fastq", "pangenome_fasta"))])
def test_host_fasta_reader_matches_oracle(pkg, name):
    """The product's own kseq-equivalent reader (pfp_io.c) against the oracle's restatement,
    which tests/test_oracle_golden.py pins to the reference."""
    c = golden().case(name)
    want, want_tr = orc.fasta_extract(c["input"])
    got, got_tr = pkg.pfp.fasta_extract(c["input"])
    assert got == want and got_tr == want_tr


def test_read_input_plain_fasta_and_gzip(pkg, tmp_path):
    """pfpb200_read_input: the text the parser sees for a file -- bytes as they are, the kseq
    extraction of a FASTA file, and the same through gzip (the reference reads -f input with
    gzread, newscan.cpp:332-336).  Host only."""
    import gzip
    recs = [r.numpy() for r in pkg.synth.pangenome_records(5_000, 3, 17)]
    fa = pkg.synth.to_fasta(recs, width=60)
    want, _ = orc.fasta_extract(fa)
    plain, gz = tmp_path / "x.fa", tmp_path / "x.fa.gz"
    plain.write_bytes(fa)
    with gzip.open(gz, "wb") as f:
        f.write(fa)
    assert pkg.pfp.read_input(str(plain), fasta=True) == (want, False)
    assert pkg.pfp.read_input(str(gz), fasta=True) == (want, False)
    assert pkg.pfp.read_input(str(plain), fasta=False) == (fa, False)
    assert pkg.pfp.read_input(str(gz), fasta=False)[0] == gz.read_bytes()      # no -f: bytes, as ifstream reads them
    with pytest.raises(pkg.pfp.PfpError):
        pkg.pfp.read_input(str(tmp_path / "missing.fa"), fasta=True)


def test_gzip_fasta_text_equals_what_the_reference_parses(pkg, tmp_path):
    """The files newscanNT.x -f wrote for a stored FASTA (tests/golden, case pangenome_fasta) are the
    parse of the text read_input extracts from the same FASTA gzip-compressed.  Where oracle/_ref is
    built, also: newscanNT.x -f writes those files for x.fa.gz as for x.fa (the stored files come from
    the uncompressed file only)."""
    import gzip
    import subprocess
    c = golden().case("pangenome_fasta")
    a, b = tmp_path / "a.fa", tmp_path / "b.fa.gz"
    a.write_bytes(c["input"])
    with gzip.open(b, "wb") as f:
        f.write(c["input"])
    text, _ = pkg.pfp.read_input(str(b), fasta=True)
    want = orc.parse(text, c["w"], c["p"])
    for ext in ("dict", "occ", "parse", "last", "sai"):
        assert c[ext] == getattr(want, ext), ext
    if orc.have_ref():
        for pth in (a, b):
            subprocess.run([orc.ref_exe("newscanNT.x"), str(pth), "-w", str(c["w"]), "-p", str(c["p"]), "-s", "-f"],
                           check=True, stdout=subprocess.PIPE)
            assert_same_files(orc.collect_files(str(pth)), c, pth.name)
