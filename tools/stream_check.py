#!/usr/bin/env python3
"""Full-size checks of the streamed parse_file (pfp_chunked.cu): BASELINE.json config 2 (4 GB pan-genome)
and config 4 (8 GB random ACGT) are written to files, plain and as 60-column FASTA, and parsed by
pfpb200_parse_file with PFPB200_PARSE_BUDGET set for about 4 and about 16 chunks.  The sha256 of each of
the five files must equal tests/golden/fullsize_sha256.json: the digests of the unmodified newscanNT.x on
the same text (tools/make_fullsize_digests.py; the FASTA form parses to the same text).
usage: stream_check.py [--config 2|4|all] [--chunks 4,16] [--forms plain,fasta] [--dir DIR]
Prints one JSON line per case; exit status 1 on any failure."""
import argparse, hashlib, json, os, shutil, sys, tempfile, time
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
import numpy as np
from fullsize_check import load_digests

BYTES_PER_BYTE = 8          # chunk = budget / 8 new input bytes (pfp_chunked.cu)
KEYS = {"2": "config2 w10 p100", "4": "config4 random 8 GB w10 p100"}


def write_config2(pkg, path, fasta):
    """100 haplotypes x 40 Mbp (seed 2), what fullsize_check.py parses in HBM"""
    with open(path, "wb") as f:
        for k, rec in enumerate(pkg.synth.pangenome_records(40_000_000, 100, 2, device="cuda")):
            a = rec.cpu().numpy()
            (pkg.synth.to_fasta_np(a, f"hap{k}") if fasta else a).tofile(f)


def write_config4(pkg, path, fasta):
    """8 GB of random ACGT (seed 4) in 1 GB pieces; as FASTA one record of 60-column lines"""
    n, step = 8_000_000_000, 960_000_000                 # a multiple of 60: lines do not straddle pieces
    with open(path, "wb") as f:
        if fasta:
            f.write(b">random\n")
        for o in range(0, n, step):
            a = pkg.synth.random_dna(min(step, n - o), 4, device="cuda", start=o).cpu().numpy()
            if fasta:
                a = pkg.synth.to_fasta_np(a, "x")[3:]     # body only
            a.tofile(f)


def sha_file(path):
    h = hashlib.sha256()
    with open(path, "rb") as f:
        for b in iter(lambda: f.read(1 << 26), b""):
            h.update(b)
    return h.hexdigest()


def check_file(pkg, path, key, chunks, fasta, sc=None):
    size = os.path.getsize(path)
    budget = BYTES_PER_BYTE * -(-size // chunks)
    os.environ["PFPB200_PARSE_BUDGET"] = str(budget)
    own = sc is None
    sc = sc or pkg.pfp.Scanner(0)
    try:
        t0 = time.perf_counter()
        st = sc.parse_file(path, 10, 100, sai=True, fasta=fasta)
        wall = time.perf_counter() - t0
    finally:
        del os.environ["PFPB200_PARSE_BUDGET"]
        if own:
            sc.close()
    want = load_digests()["cases"][key]["sha256"]
    got = {e: sha_file(f"{path}.{e}") for e in want}
    res = {"case": key, "form": "fasta" if fasta else "plain", "file_bytes": size, "budget": budget,
           "chunks": st["chunks"], "peak_device_bytes": st["peak_device_bytes"], "n_text": st["n_text"],
           "phrases": st["n_phrases"], "distinct": st["n_distinct"], "wall_s": round(wall, 3),
           "sec_read": round(st["sec_read"], 3), "sec_write": round(st["sec_write"], 3),
           "ms_gpu": round(st["ms_total"], 1), "sha256_vs_reference": {e: got[e] == want[e] for e in want}}
    res["ok"] = all(res["sha256_vs_reference"].values())
    for e in want:
        try:
            os.remove(f"{path}.{e}")
        except OSError:
            pass
    print(json.dumps(res), flush=True)
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--config", default="all", choices=["2", "4", "all"])
    ap.add_argument("--chunks", default="4,16")
    ap.add_argument("--forms", default="plain,fasta")
    ap.add_argument("--dir", default=None)
    a = ap.parse_args()
    from __graft_entry__ import load_package
    pkg = load_package()
    tmp = tempfile.mkdtemp(prefix="streamcheck_", dir=a.dir)
    ok = True
    try:
        for cfg in (["2", "4"] if a.config == "all" else [a.config]):
            for form in a.forms.split(","):
                fasta = form == "fasta"
                path = os.path.join(tmp, f"config{cfg}.{'fa' if fasta else 'txt'}")
                (write_config2 if cfg == "2" else write_config4)(pkg, path, fasta)
                for c in a.chunks.split(","):
                    ok &= check_file(pkg, path, KEYS[cfg], int(c), fasta)["ok"]
                os.remove(path)
    finally:
        shutil.rmtree(tmp, ignore_errors=True)
    sys.exit(0 if ok else 1)


if __name__ == "__main__":
    main()
