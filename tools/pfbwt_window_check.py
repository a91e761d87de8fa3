#!/usr/bin/env python3
"""Full-size checks of pfbwt's windowed output (pfpb200_pfbwt_file, pfpb200_bigbwt_file; DESIGN.md §6c).

  parity   BASELINE.json config 2 (4 GB pan-genome, w 10 p 100) parsed and bwtparsed to files, then
           pfbwt_file -S in one window and in about --windows windows: the sha256 of .bwt and .sa must
           equal tests/golden/fullsize_sha256.json (the unmodified pfbwtNT.x -S on the same text);
           -s -e windowed must equal -s -e in one window.  Device peaks of both; the windowed ones must
           stay within the plan's part plus the budget.  Then gpubigbwt.x -f -S on the config 2 FASTA with
           the streamed parse forced (PFPB200_PARSE_BUDGET) and windows: the same digests.
  wall     pfbwt_file -S wall clock, one window against about --windows windows, alternated.
  big      gpubigbwt.x -f -s -e on a synthetic pan-genome of --big-haps x 40 Mbp (10 GB at 250; at 400 the
           dictionary, about 8 MB per haplotype, would need more than the device for its suffix sort):
           with --parent DIR (a build of the parent commit) the parent's gpubigbwt.x must fail; this
           build must finish, and its outputs are checked by properties: the .bwt byte histogram is the
           text's plus one EOF, .ssa and .esa have equal counts, strictly ascending positions below n + 1,
           and as many entries as .bwt has runs.  Skipped, and said so, when the disk is too small.
usage: pfbwt_window_check.py [--cases parity,wall,big] [--windows 8] [--dir DIR] [--parent DIR]
Prints one JSON line per case; exit status 1 on any failure."""
import argparse, json, os, shutil, subprocess, sys, tempfile, time
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
import numpy as np
from fullsize_check import load_digests
from stream_check import sha_file, write_config2

WINDOW_BYTES = 32           # device bytes per BWT char of a window with a suffix array whose chars are all hard (pb_out_bytes)
KEY = "config2 w10 p100"
GB = 1e9


def emit(d):
    print(json.dumps(d), flush=True)
    return d


def pfbwt(sc, base, flags, budget):
    if budget:
        os.environ["PFPB200_PFBWT_BUDGET"] = str(budget)
    try:
        t0 = time.perf_counter()
        r = sc.pfbwt_file(base, 10, flags)
        wall = time.perf_counter() - t0
    finally:
        os.environ.pop("PFPB200_PFBWT_BUDGET", None)
    return r, wall


def case_parity(pkg, tmp, windows, ok):
    ref = load_digests()["cases"][KEY]["pipeline"]["sha256"]
    base = os.path.join(tmp, "config2.txt")
    write_config2(pkg, base, False)
    n = os.path.getsize(base)
    sc = pkg.pfp.Scanner(0)
    try:
        sc.parse_file(base, 10, 100, sai=True)
        sc.bwtparse_file(base, sai=True)
        budget = WINDOW_BYTES * ((n + 1) // windows + 1)
        res = {}
        for flags, exts in ((pkg.pfp.PFBWT_SA, ("bwt", "sa")), (pkg.pfp.PFBWT_SSA | pkg.pfp.PFBWT_ESA, ("ssa", "esa"))):
            name = "-S" if flags == pkg.pfp.PFBWT_SA else "-s -e"
            for b in (None, budget):
                r, wall = pfbwt(sc, base, flags, b)
                dig = {e: sha_file(f"{base}.{e}") for e in exts}
                res[(name, b is None)] = (r, dig)
                d = {"case": "parity", "flags": name, "budget": b, "windows": r["windows"],
                     "peak_device_gb": round(r["peak_device_bytes"] / GB, 3), "wall_s": round(wall, 3),
                     "ms_gpu": round(r["ms_total"], 1), "chars": r["n_bwt"]}
                if flags == pkg.pfp.PFBWT_SA:
                    d["sha256_vs_reference"] = {e: dig[e] == ref[e] for e in exts}
                    d["ok"] = all(d["sha256_vs_reference"].values())
                else:
                    d["ok"] = True
                if b is not None:
                    d["ok"] &= r["windows"] > 1
                    one = res[(name, True)][0]
                    # the plan's part is at most the one-window peak less its held chars and SA values
                    # (6 B per char); the windows may add the budget on top of it
                    d["peak_reduction_gb"] = round((one["peak_device_bytes"] - r["peak_device_bytes"]) / GB, 3)
                    d["peak_within_budget"] = r["peak_device_bytes"] - b <= one["peak_device_bytes"] - 6 * (n + 1)
                    d["ok"] &= d["peak_within_budget"]
                    if flags != pkg.pfp.PFBWT_SA:
                        d["same_as_one_window"] = dig == res[(name, True)][1]
                        d["ok"] &= d["same_as_one_window"]
                ok &= emit(d)["ok"]
            for e in exts:
                os.remove(f"{base}.{e}")
        for e in ("dict", "occ", "parse", "last", "sai", "ilist", "bwlast", "bwsai"):
            os.remove(f"{base}.{e}")
    finally:
        sc.close()
    os.remove(base)
    # gpubigbwt.x on the FASTA with the streamed parse forced and windows
    fa = os.path.join(tmp, "config2.fa")
    write_config2(pkg, fa, True)
    env = dict(os.environ, PFPB200_PARSE_BUDGET=str(8 * (os.path.getsize(fa) // 4)),
               PFPB200_PFBWT_BUDGET=str(WINDOW_BYTES * ((n + 1) // windows + 1)))
    t0 = time.perf_counter()
    p = subprocess.run([pkg.pfp.BIGBWT_CLI_PATH, fa, "-f", "-S"], env=env, stdout=subprocess.PIPE, stderr=subprocess.STDOUT,
                       text=True)
    wall = time.perf_counter() - t0
    d = {"case": "gpubigbwt -f -S streamed parse + windows", "rc": p.returncode, "wall_s": round(wall, 3),
         "plan": [l for l in p.stdout.splitlines() if l.startswith("Plan:") or l.startswith("GPU:")]}
    if p.returncode == 0:
        d["sha256_vs_reference"] = {e: sha_file(f"{fa}.{e}") == ref[e] for e in ("bwt", "sa")}
        d["intermediate_left"] = [e for e in ("dict", "parse", "ilist") if os.path.exists(f"{fa}.{e}")]
        d["ok"] = all(d["sha256_vs_reference"].values()) and not d["intermediate_left"]
    else:
        d["ok"] = False
        d["tail"] = p.stdout[-600:]
    for e in ("bwt", "sa"):
        if os.path.exists(f"{fa}.{e}"):
            os.remove(f"{fa}.{e}")
    os.remove(fa)
    return emit(d)["ok"] and ok


def case_wall(pkg, tmp, windows, rounds):
    base = os.path.join(tmp, "config2w.txt")
    write_config2(pkg, base, False)
    n = os.path.getsize(base)
    sc = pkg.pfp.Scanner(0)
    t = {"one": [], "windows": []}
    try:
        sc.parse_file(base, 10, 100, sai=True)
        sc.bwtparse_file(base, sai=True)
        pfbwt(sc, base, pkg.pfp.PFBWT_SA, None)                                   # warm-up
        for _ in range(rounds):
            for arm, b in (("one", None), ("windows", WINDOW_BYTES * ((n + 1) // windows + 1))):
                r, wall = pfbwt(sc, base, pkg.pfp.PFBWT_SA, b)
                t[arm].append(round(wall, 3))
    finally:
        sc.close()
        shutil.rmtree(tmp, ignore_errors=True)
        os.makedirs(tmp, exist_ok=True)
    return emit({"case": "wall pfbwt_file -S config 2", "windows": windows, "one_window_s": t["one"],
                 "windowed_s": t["windows"], "median_one": float(np.median(t["one"])),
                 "median_windowed": float(np.median(t["windows"])), "ok": True})["ok"]


def case_big(pkg, tmp, haps, parent):
    need = haps * 40e6 * (1 + 1 + 1.3)            # FASTA, .bwt, intermediates and samples
    free = shutil.disk_usage(tmp).free
    if free < need:
        return emit({"case": "big", "skipped": f"disk: {free / GB:.0f} GB free, about {need / GB:.0f} GB needed",
                     "ok": True})["ok"]
    fa = os.path.join(tmp, "big.fa")
    hist = np.zeros(256, np.int64)
    with open(fa, "wb") as f:
        for k, rec in enumerate(pkg.synth.pangenome_records(40_000_000, haps, 7, device="cuda")):
            a = rec.cpu().numpy()
            hist += np.bincount(a, minlength=256)
            pkg.synth.to_fasta_np(a, f"hap{k}").tofile(f)
    n = int(hist.sum())
    res = {"case": "big gpubigbwt -f -s -e", "text_bytes": n, "fasta_bytes": os.path.getsize(fa)}
    if parent:
        p = subprocess.run([os.path.join(parent, "big-bwt_b200", "gpubigbwt.x"), fa, "-f", "-s", "-e"],
                           stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
        res["parent_rc"] = p.returncode
        res["parent_tail"] = p.stdout[-300:]
        for e in ("bwt", "ssa", "esa"):
            if os.path.exists(f"{fa}.{e}"):
                os.remove(f"{fa}.{e}")
    t0 = time.perf_counter()
    p = subprocess.run([pkg.pfp.BIGBWT_CLI_PATH, fa, "-f", "-s", "-e"], stdout=subprocess.PIPE, stderr=subprocess.STDOUT,
                       text=True)
    res["wall_s"] = round(time.perf_counter() - t0, 3)
    res["rc"] = p.returncode
    res["out"] = [l for l in p.stdout.splitlines() if l.startswith(("Plan:", "GPU:", "gpubigbwt"))]
    ok = p.returncode == 0 and (not parent or res["parent_rc"] != 0)
    if p.returncode == 0:
        bh = np.zeros(256, np.int64)
        runs, last, size = 0, -1, 0
        with open(fa + ".bwt", "rb") as f:
            for b in iter(lambda: f.read(1 << 28), b""):
                a = np.frombuffer(b, np.uint8)
                bh += np.bincount(a, minlength=256)
                runs += int(np.count_nonzero(a[1:] != a[:-1])) + (1 if a[0] != last else 0)
                last = int(a[-1])
                size += a.size
        want = hist.copy()
        want[0] += 1
        res["bwt_histogram_ok"] = bool((bh == want).all()) and size == n + 1

        def positions(ext):
            v = np.fromfile(f"{fa}.{ext}", np.uint8).reshape(-1, 10)[:, :5].astype(np.uint64)
            return (v * (np.uint64(1) << (np.arange(5, dtype=np.uint64) * np.uint64(8)))).sum(axis=1)
        ps, pe = positions("ssa"), positions("esa")
        res.update({"bwt_runs": runs, "n_ssa": int(ps.size), "n_esa": int(pe.size),
                    "ssa_ascending": bool((np.diff(ps.astype(np.int64)) > 0).all()) and int(ps.max()) < n + 1,
                    "esa_ascending": bool((np.diff(pe.astype(np.int64)) > 0).all()) and int(pe.max()) < n + 1})
        ok &= res["bwt_histogram_ok"] and res["n_ssa"] == res["n_esa"] == runs and res["ssa_ascending"] and res["esa_ascending"]
    res["ok"] = bool(ok)
    for e in ("bwt", "ssa", "esa"):
        if os.path.exists(f"{fa}.{e}"):
            os.remove(f"{fa}.{e}")
    os.remove(fa)
    return emit(res)["ok"]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--cases", default="parity,wall,big")
    ap.add_argument("--windows", type=int, default=8)
    ap.add_argument("--rounds", type=int, default=2)
    ap.add_argument("--big-haps", type=int, default=250)
    ap.add_argument("--dir", default=None)
    ap.add_argument("--parent", default=None, help="a build of the parent commit (for the big case)")
    a = ap.parse_args()
    from __graft_entry__ import load_package
    pkg = load_package()
    card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                          stdout=subprocess.PIPE, text=True).stdout.strip().splitlines()
    emit({"card": card[0] if card else "unknown"})
    tmp = tempfile.mkdtemp(prefix="pfbwtwin_", dir=a.dir)
    ok = True
    try:
        cases = a.cases.split(",")
        if "parity" in cases:
            ok &= case_parity(pkg, tmp, a.windows, True)
        if "wall" in cases:
            ok &= case_wall(pkg, tmp, a.windows, a.rounds)
        if "big" in cases:
            ok &= case_big(pkg, tmp, a.big_haps, a.parent)
    finally:
        shutil.rmtree(tmp, ignore_errors=True)
    sys.exit(0 if ok else 1)


if __name__ == "__main__":
    main()
