#!/usr/bin/env python3
"""Full-size check of the sharded pfbwt (pfpb200_multi_pfbwt_file): the files it wrote, checked on the
device in linear time against the text, and, where the unmodified reference chain's digests exist, by
sha256.  Every rank writes its piece in windows sized by its budget (DESIGN.md §6d); each run logs every
rank's windows, device peak and times.

  --config 2  BASELINE config 2 (100 haplotypes x 40 Mbp, w=10 p=100, 814 MB dictionary) with the rank
              list --ranks (default 0,0: two ranks on one GPU; 0,0,0,0 runs four on one card).  .bwt
              (4,000,000,199 B) and .sa (20,000,000,990 B) must match tests/golden/fullsize_sha256.json
              "config2 w10 p100" -> "pipeline".
  --config 3  BASELINE config 3 (1000 haplotypes x 64 Mbp, dictionary about 11.5 GB): needs 8 GPUs of
              180 GB; with fewer it prints a "not run" line.
  --config 4  BASELINE config 4 (8 GB of random ACGT, 8.8 GB dictionary): parse and bwtparse on GPU 0,
              pfbwt -S on the visible GPUs.  No reference digest exists; the linear checks decide.
  --flags se  `-s -e` instead of `-S`: the one-GPU pfpb200_pfbwt_file runs on the same inputs first, and
              the sharded .ssa / .esa must equal its files (sha256); .bwt is checked as with -S.
  --reps K    the sharded call K times; the per-rank medians of sort / emission wall clock and peaks.

The linear checks of the written .sa / .bwt are oracle/sa_check.py's (permutation, bwt[i] == T[sa[i] - 1],
the EOF row, Burkhardt-Kaerkkaeinen order of adjacent rows); they check the files, not a second suffix
sort.  A case that does not fit (device memory, disk, too few GPUs) prints a "not run" line with the
reason and exits 0; a failed check exits 1.
usage: pfbwt_multi_check.py --config {2,3,4} [--ranks 0,0,0,0] [--flags S|se] [--reps K] [--dir DIR]"""
import argparse
import hashlib
import json
import os
import shutil
import statistics
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch  # noqa: E402

from oracle.sa_check import linear_checks, load_sa  # noqa: E402


def emit(d):
    print(json.dumps(d), flush=True)


def sha(path):
    h = hashlib.sha256()
    with open(path, "rb") as f:
        while True:
            b = f.read(64 << 20)
            if not b:
                return h.hexdigest()
            h.update(b)


def prepare(pkg, sc, text, w, p, base):
    out = sc.parse_device(text, w, p, sai=True)
    bp = sc.bwtparse_device(out.parse, out.n_phrases, out.last, out.sai)
    for ext, ptr, nb in (("dict", out.dict, out.dict_bytes), ("occ", out.occ, 4 * out.n_distinct),
                         ("ilist", bp.ilist, 4 * bp.n_out), ("bwlast", bp.bwlast, bp.n_out),
                         ("bwsai", bp.bwsai, 5 * bp.n_out)):
        with open(f"{base}.{ext}", "wb") as f:
            f.write(sc.to_host(ptr, nb))
    return out.dict_bytes, bp.n_out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--config", required=True, choices=["2", "3", "4"])
    ap.add_argument("--ranks", default=None, help="rank list (config 2 default 0,0; configs 3 and 4 default all GPUs)")
    ap.add_argument("--flags", default="S", choices=["S", "se"])
    ap.add_argument("--reps", type=int, default=1)
    ap.add_argument("--dir", default=None)
    a = ap.parse_args()
    import __graft_entry__ as g
    pkg = g.load_package()
    P = pkg.pfp
    import subprocess
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,memory.total", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    n_gpu = torch.cuda.device_count()
    emit({"cards": q, "visible_gpus": n_gpu, "config": a.config})
    if a.config == "3":
        ids = [int(x) for x in a.ranks.split(",")] if a.ranks else list(range(n_gpu))
        if len(set(ids)) < 8:
            emit({"config": "3", "not_run": f"needs 8 GPUs of 180 GB (distinct devices); {len(set(ids))} listed"})
            return 0
        text_gen = lambda: pkg.synth.pangenome_text(64_000_000, 1000, 3, device="cuda")  # noqa: E731
    elif a.config == "4":
        ids = [int(x) for x in a.ranks.split(",")] if a.ranks else list(range(n_gpu))
        # per rank: the 8.8 GB dictionary, 8 B per byte / G of the rank block and the bytes per owned suffix
        # of DESIGN.md §6d
        if len(set(ids)) < 8:
            emit({"config": "4", "not_run": f"needs 8 GPUs of 180 GB (distinct devices); {len(set(ids))} listed"})
            return 0
        text_gen = lambda: pkg.synth.random_dna(8_000_000_000, 4, device="cuda")  # noqa: E731
    else:
        ids = [int(x) for x in a.ranks.split(",")] if a.ranks else [0, 0]
        text_gen = lambda: pkg.synth.pangenome_text(40_000_000, 100, 2, device="cuda")  # noqa: E731
    tmp = a.dir or tempfile.mkdtemp(prefix="pfbwtcheck_")
    os.makedirs(tmp, exist_ok=True)
    base = os.path.join(tmp, f"config{a.config}")
    rc = 0
    try:
        sc = P.Scanner(0)
        text = text_gen()
        n = text.numel()
        free_disk = shutil.disk_usage(tmp).free
        if free_disk < 7.5 * n:
            emit({"config": a.config, "not_run": f"needs {7.5 * n / 1e9:.0f} GB of disk, {free_disk / 1e9:.0f} GB free"})
            return 0
        dict_bytes, psize = prepare(pkg, sc, text, 10, 100, base)
        sc.close()
        del text
        torch.cuda.empty_cache()
        fails = []
        flags = P.PFBWT_SA if a.flags == "S" else P.PFBWT_SSA | P.PFBWT_ESA
        samples = ("ssa", "esa") if a.flags == "se" else ()
        single = {}
        if samples:                                               # the one-GPU files the sharded ones must equal
            t0 = time.perf_counter()
            # a context of its own; a budget of 48 GB, so that its outputs go in windows whatever its arena
            # holds (the one-window -s -e output of config 2 takes more than the card's memory)
            os.environ["PFPB200_PFBWT_BUDGET"] = str(48 << 30)
            sc = P.Scanner(0)
            r1 = sc.pfbwt_file(base, 10, flags)
            sc.close()
            del os.environ["PFPB200_PFBWT_BUDGET"]
            single = {e: sha(f"{base}.{e}") for e in samples}
            emit({"one_gpu_pfbwt_wall_s": round(time.perf_counter() - t0, 2), "windows": r1["windows"],
                  "peak_device_bytes": r1["peak_device_bytes"], "n_ssa": r1["n_ssa"], "n_esa": r1["n_esa"]})
            for e in ("bwt",) + samples:
                os.remove(f"{base}.{e}")
        torch.cuda.empty_cache()
        free_mem = torch.cuda.mem_get_info(0)[0]
        emit({"n_text": n, "dict_bytes": dict_bytes, "parse_size": psize, "ranks": ids, "flags": a.flags,
              "device0_free_GB": round(free_mem / 1e9, 1), "disk_free_GB": round(free_disk / 1e9, 1)})
        ms = P.MultiScanner(ids)
        runs = []
        for rep in range(a.reps):
            t0 = time.perf_counter()
            try:
                r = ms.pfbwt_file(base, 10, flags)
            except P.PfpError as e:
                if e.code == -4:                                  # E_NOMEM
                    emit({"config": a.config, "not_run": f"device memory: {e}"})
                    return 0
                raise
            wall = time.perf_counter() - t0
            runs.append(r)
            emit({"run": rep, "pfbwt_wall_s": round(wall, 2), "rounds": r["rounds"], "n_bwt": r["n_bwt"],
                  "hard": r["hard"], "n_ssa": r["n_ssa"], "n_esa": r["n_esa"], "ms_sort": round(r["ms_sa"], 1),
                  "ms_fill": round(r["ms_fill"], 1),
                  "per_rank": [{k: (round(v, 1) if isinstance(v, float) else v) for k, v in x.items()} for x in r["ranks"]]})
        ms.close()
        if a.reps > 1:
            med = lambda k, g: statistics.median(x["ranks"][g][k] for x in runs)  # noqa: E731
            emit({"medians_of_runs": a.reps,
                  "per_rank": [{"ms_sort": round(med("ms_sort", g), 1), "ms_emit": round(med("ms_emit", g), 1),
                                "ms_write": round(med("ms_write", g), 1), "peak_GB": round(med("peak_bytes", g) / 1e9, 2),
                                "windows": [x["ranks"][g]["windows"] for x in runs]} for g in range(len(ids))],
                  "spread_ms_sort": [[round(x["ranks"][g]["ms_sort"], 1) for x in runs] for g in range(len(ids))],
                  "spread_ms_emit": [[round(x["ranks"][g]["ms_emit"], 1) for x in runs] for g in range(len(ids))]})
        if a.config == "2":
            with open(os.path.join(ROOT, "tests", "golden", "fullsize_sha256.json")) as f:
                ref = json.load(f)["cases"]["config2 w10 p100"]["pipeline"]
            got = {e: sha(f"{base}.{e}") for e in ("bwt", "sa") if e == "bwt" or not samples}
            res = {e: got[e] == ref["sha256"][e] for e in got}
            emit({"sha256_vs_reference_chain": res, "bytes": {e: os.path.getsize(f"{base}.{e}") for e in got}})
            fails += [f".{e} sha256 differs from the reference chain" for e in res if not res[e]]
        if samples:
            same = {e: sha(f"{base}.{e}") == single[e] for e in samples}
            emit({"sha256_vs_one_gpu_pfbwt": same, "bytes": {e: os.path.getsize(f"{base}.{e}") for e in samples}})
            fails += [f".{e} differs from the one-GPU pfbwt's" for e in samples if not same[e]]
        else:
            t1 = time.perf_counter()
            T = text_gen()
            with open(base + ".bwt", "rb") as f:
                bwt = torch.frombuffer(bytearray(f.read()), dtype=torch.uint8).cuda()
            sa = load_sa(base + ".sa", n)
            lf = linear_checks(T, sa, bwt)
            emit({"linear_checks": "ok" if not lf else lf, "seconds": round(time.perf_counter() - t1, 1)})
            fails += lf
        emit({"config": a.config, "ok": not fails, "fails": fails})
        rc = 1 if fails else 0
    finally:
        if not a.dir:
            shutil.rmtree(tmp, ignore_errors=True)
    return rc


if __name__ == "__main__":
    sys.exit(main())
