"""The inverse of the parse on the GPU (pfpb200_unparse_*, SURVEY 8(f) row 4; reference unparse.c):
parse -> unparse gives the text back, from the -c dictionary (.dicz) and from the plain .dict, and
gpuunparse.x writes the file the reference's unparse writes."""
import os
import shutil
import subprocess
import tempfile

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def sc(pkg):
    s = pkg.pfp.Scanner(0)
    yield s
    s.close()


@pytest.mark.parametrize("w,p,n,haps", [(10, 100, 300_000, 8), (4, 10, 50_000, 3), (16, 500, 400_000, 6), (32, 50, 100_000, 4)])
def test_round_trip_from_dict_and_dicz(pkg, sc, w, p, n, haps):
    text = pkg.synth.pangenome_text(n, haps, 60 + w, device="cuda")
    want = text.cpu().numpy().tobytes()
    out = sc.parse_device(text, w, p, sai=False)                       # plain .dict: overlaps skipped on the fly
    ptr, nt, _ = sc.unparse_device(out.dict, out.dict_bytes, out.parse, out.n_phrases, strip_w=w)
    assert nt == len(want) and sc.to_host(ptr, nt) == want
    ptr2, nt2, _ = sc.unparse_device(out.dict, out.dict_bytes, out.parse, out.n_phrases, strip_w=w)   # own output recycled
    assert sc.to_host(ptr2, nt2) == want
    out = sc.parse_device(text, w, p, sai=False, compress=True)       # -c: out.dict holds the .dicz bytes
    ptr, nt, _ = sc.unparse_device(out.dict, out.dict_bytes, out.parse, out.n_phrases, strip_w=0)
    assert nt == len(want) and sc.to_host(ptr, nt) == want


def test_round_trip_text_with_all_byte_values(pkg, sc):
    rng = np.random.default_rng(5)
    a = rng.integers(3, 256, 200_000).astype(np.uint8)
    text = torch.from_numpy(a).cuda()
    out = sc.parse_device(text, 10, 100, sai=False)
    ptr, nt, _ = sc.unparse_device(out.dict, out.dict_bytes, out.parse, out.n_phrases, strip_w=10)
    assert sc.to_host(ptr, nt) == a.tobytes()


def test_round_trip_128mb_on_the_device(pkg, sc):
    """parse -> unparse == text, compared on the device (no host copy of the text)."""
    text = pkg.synth.pangenome_text(4_000_000, 32, 9, device="cuda")
    out = sc.parse_device(text, 10, 100, sai=True)
    ptr, nt, ms = sc.unparse_device(out.dict, out.dict_bytes, out.parse, out.n_phrases, strip_w=10)
    assert nt == text.numel()
    import sys
    sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tools"))
    from fullsize_check import view
    torch.cuda.synchronize()
    assert torch.equal(view(ptr, nt), text)


def test_invalid_word_id(pkg, sc):
    text = pkg.synth.random_dna(50_000, 3, device="cuda")
    out = sc.parse_device(text, 10, 100, sai=False)
    bad = torch.tensor([1, 2, out.n_distinct + 1], dtype=torch.int32, device="cuda")
    torch.cuda.synchronize()
    with pytest.raises(pkg.pfp.PfpError) as e:                          # unparse.c:120
        sc.unparse_device(out.dict, out.dict_bytes, bad.data_ptr(), 3, strip_w=10)
    assert e.value.code == -1


def test_cli_matches_reference_unparse(pkg):
    """gpuunparse.x on the -c files of gpuscan.x writes <base>.out (or -o) holding the text, as the
    reference's unparse does."""
    text = pkg.synth.pangenome_text(80_000, 7, 21).numpy().tobytes()
    tmp = tempfile.mkdtemp(prefix="unparsecli_")
    try:
        base = os.path.join(tmp, "t.txt")
        with open(base, "wb") as f:
            f.write(text)
        subprocess.run([pkg.pfp.CLI_PATH, base, "-w", "10", "-p", "100", "-c"], check=True, stdout=subprocess.PIPE)
        subprocess.run([pkg.pfp.UNPARSE_CLI_PATH, base], check=True, stdout=subprocess.PIPE, stderr=subprocess.PIPE)
        assert open(base + ".out", "rb").read() == text
        subprocess.run([pkg.pfp.UNPARSE_CLI_PATH, base, "-o", os.path.join(tmp, "named")], check=True,
                       stdout=subprocess.PIPE, stderr=subprocess.PIPE)
        assert open(os.path.join(tmp, "named"), "rb").read() == text
        r = subprocess.run([pkg.pfp.UNPARSE_CLI_PATH, os.path.join(tmp, "missing")], capture_output=True, text=True)
        assert r.returncode == 1
    finally:
        shutil.rmtree(tmp, ignore_errors=True)
