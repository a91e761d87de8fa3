#!/usr/bin/env python3
"""Measurement and full-size check of the sharded pfbwt (pfpb200_multi_pfbwt_file) on BASELINE config 2
(100 haplotypes x 40 Mbp, w=10, p=100; its .dict is 814 MB).

The text is parsed and bwtparse'd on GPU 0 and the five inputs of pfbwt go to files.  Then the arms
run alternately, each in a process of its own (so that every arm has the whole GPU memory: the
contexts keep their scratch between calls): the single-GPU pfpb200_pfbwt_file and the sharded call
on each rank list -- [0] (the sharded path with one rank), [0,0,0,0] (four ranks time-sharing one
GPU) and 2 / 4 / 8 real GPUs where present.  In every process one warm-up call, then --steps timed
calls, every call reading and writing files.  After the first -S run of a sharded arm, the sha256
of .bwt and .sa is compared with the digests of the unmodified reference chain
(tests/golden/fullsize_sha256.json, "config2 w10 p100" -> "pipeline").

Prints the cards' names and power limits, then one JSON line per timed call and one summary line per
(arm, flags).  usage: pfbwt_multi_bench.py [--steps 2] [--reps 2] [--small] [--no-sa] [--lists 0 0,0,0,0 ...]"""
import argparse
import hashlib
import json
import os
import shutil
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


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


def run_arm(a):
    """one process: one arm, one warm-up call and a.steps timed calls per flag set"""
    import __graft_entry__ as g
    P = g.load_package().pfp
    ids = [int(x) for x in a.arm.split(",")] if a.arm != "single" else None
    obj = P.Scanner(0) if ids is None else P.MultiScanner(ids)
    sets = [(0, "bwt")] + ([] if a.no_sa else [(P.PFBWT_SA, "bwt -S")])
    for flags, name in sets:
        for step in range(a.steps + 1):
            t0 = time.perf_counter()
            r = obj.pfbwt_file(a.base, 10, flags)
            wall = (time.perf_counter() - t0) * 1e3
            row = {"arm": a.arm, "flags": name, "step": step, "wall_ms": round(wall, 1), "ms_sort": round(r["ms_sa"], 1),
                   "ms_fill": round(r["ms_fill"], 1), "rounds": r["rounds"], "n_bwt": r["n_bwt"], "hard": r["hard"],
                   "launches": r["launches"]}
            if ids is not None:
                row["per_rank"] = [{k: (round(v, 1) if isinstance(v, float) else v) for k, v in x.items()}
                                   for x in r["ranks"]]
            emit(row)
            if flags and ids is not None and a.digests and step == 0:
                with open(a.digests) as f:
                    dg = json.load(f)
                got = {"bwt": sha(a.base + ".bwt"), "sa": sha(a.base + ".sa")}
                emit({"arm": a.arm, "sha256_vs_reference_chain": {e: got[e] == dg[e] for e in got}})


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=2)
    ap.add_argument("--reps", type=int, default=2, help="alternations of the arms (processes per arm)")
    ap.add_argument("--small", action="store_true", help="1/16 of the text (rehearsal; no digests)")
    ap.add_argument("--no-sa", action="store_true", help="without the -S runs")
    ap.add_argument("--lists", nargs="*", default=None, help="rank lists, e.g. 0 0,0,0,0 0,1")
    ap.add_argument("--dir", default=None, help="directory for the files (default: a temporary one)")
    ap.add_argument("--arm", default=None, help=argparse.SUPPRESS)
    ap.add_argument("--base", default=None, help=argparse.SUPPRESS)
    ap.add_argument("--digests", default=None, help=argparse.SUPPRESS)
    a = ap.parse_args()
    if a.arm:
        return run_arm(a)
    import torch
    import __graft_entry__ as g
    pkg = g.load_package()
    P = pkg.pfp
    n_gpu = torch.cuda.device_count()
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    emit({"cards": q, "visible_gpus": n_gpu})
    lists = a.lists if a.lists else ["0", "0,0,0,0"] + [",".join(map(str, range(k))) for k in (2, 4, 8) if n_gpu >= k]
    tmp = a.dir or tempfile.mkdtemp(prefix="pfbwtmulti_")
    os.makedirs(tmp, exist_ok=True)
    base = os.path.join(tmp, "config2")
    scale = 16 if a.small else 1
    try:
        sc = P.Scanner(0)
        text = pkg.synth.pangenome_text(40_000_000 // scale, 100, 2, device="cuda")
        n = text.numel()
        out = sc.parse_device(text, 10, 100, sai=True)
        bp = sc.bwtparse_device(out.parse, out.n_phrases, out.last, out.sai)
        for ext, ptr, nb in (("dict", out.dict, out.dict_bytes), ("occ", out.occ, 4 * out.n_distinct),
                             ("ilist", bp.ilist, 4 * bp.n_out), ("bwlast", bp.bwlast, bp.n_out),
                             ("bwsai", bp.bwsai, 5 * bp.n_out)):
            with open(f"{base}.{ext}", "wb") as f:
                f.write(sc.to_host(ptr, nb))
        free = shutil.disk_usage(tmp).free
        emit({"workload": f"config 2: 100 haplotypes x {40_000_000 // scale} bp, w=10 p=100", "n_text": n,
              "dict_bytes": out.dict_bytes, "dict_words": out.n_distinct, "parse_size": bp.n_out,
              "disk_free_GB": round(free / 1e9, 1)})
        sc.close()
        del text
        torch.cuda.empty_cache()
        cmd = [sys.executable, os.path.abspath(__file__), "--base", base, "--steps", str(a.steps)]
        if a.no_sa or free < 6 * (n + 1) * 1.1:            # .bwt + .sa of one run
            cmd.append("--no-sa")
            if not a.no_sa:
                emit({"note": "-S runs not run: not enough disk for the 6 B per text byte of .bwt + .sa"})
        dfile = None
        if not a.small:
            with open(os.path.join(ROOT, "tests", "golden", "fullsize_sha256.json")) as f:
                dg = json.load(f)["cases"]["config2 w10 p100"]["pipeline"]["sha256"]
            dfile = base + ".digests.json"
            with open(dfile, "w") as f:
                json.dump(dg, f)
        rows = []
        for rep in range(a.reps):
            for arm in ["single"] + lists:
                c = cmd + ["--arm", arm] + (["--digests", dfile] if dfile and rep == 0 and arm != "single" else [])
                r = subprocess.run(c, capture_output=True, text=True)
                for line in r.stdout.splitlines():
                    print(line, flush=True)
                    d = json.loads(line)
                    if d.get("step"):
                        rows.append(d)
                if r.returncode != 0:
                    emit({"arm": arm, "error": r.stderr[-800:]})
        for arm in ["single"] + lists:
            for name in ("bwt", "bwt -S"):
                v = [x for x in rows if x["arm"] == arm and x["flags"] == name]
                if not v:
                    continue
                w = sorted(x["wall_ms"] for x in v)
                emit({"summary": name, "arm": arm, "n": len(v), "wall_ms_median": w[len(w) // 2],
                      "wall_ms_min": w[0], "wall_ms_max": w[-1],
                      "ms_sort_median": sorted(x["ms_sort"] for x in v)[len(v) // 2],
                      "ms_fill_median": sorted(x["ms_fill"] for x in v)[len(v) // 2]})
    finally:
        if not a.dir:
            shutil.rmtree(tmp, ignore_errors=True)


if __name__ == "__main__":
    main()
