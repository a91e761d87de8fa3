#!/usr/bin/env python3
"""Measurements of the streamed parse_file (pfp_chunked.cu) on one GPU.

--peaks: the one-shot path's device footprint per input byte (the arena's high-water mark over the
  file size, pfpb200_parse_plan) on config 2 as plain text and as 60-column FASTA and on config 4 --
  the figures behind the routing estimate in pfp_api.cu.
--bench: gpuscan.x -s -f on the config 2 FASTA (page-cache warm): the one-shot path against the streamed
  path at about 4 and about 16 chunks, alternated, medians of the wall clock, with the breakdown the
  library prints under PFPB200_TRACE (per-chunk K1/K2/K3, global insert, final rank, .parse rewrite).
Prints JSON lines, the first one naming the GPU and its power limit."""
import argparse, json, os, re, statistics, subprocess, sys, tempfile, shutil, time
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
import stream_check as sck


def card():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return r.stdout.strip().splitlines()[0] if r.returncode == 0 else "unknown"


def peaks(pkg, tmp):
    sc = pkg.pfp.Scanner(0)
    os.environ.pop("PFPB200_PARSE_BUDGET", None)
    for cfg, fasta in (("2", False), ("2", True), ("4", False)):
        path = os.path.join(tmp, f"c{cfg}.{'fa' if fasta else 'txt'}")
        (sck.write_config2 if cfg == "2" else sck.write_config4)(pkg, path, fasta)
        sc.parse_file(path, 10, 100, sai=True, fasta=fasta)          # warm-up: arena growth, table sizing hint
        st = sc.parse_file(path, 10, 100, sai=True, fasta=fasta)
        size = os.path.getsize(path)
        print(json.dumps({"peak": f"config{cfg}", "form": "fasta" if fasta else "plain", "file_bytes": size,
                          "chunks": st["chunks"], "peak_device_bytes": st["peak_device_bytes"],
                          "peak_per_input_byte": round(st["peak_device_bytes"] / size, 3)}), flush=True)
        for f in os.listdir(tmp):
            os.remove(os.path.join(tmp, f))
    sc.close()


def run_cli(pkg, path, budget):
    env = dict(os.environ)
    env.pop("PFPB200_PARSE_BUDGET", None)
    env["PFPB200_TRACE"] = "1"
    if budget:
        env["PFPB200_PARSE_BUDGET"] = str(budget)
    t0 = time.perf_counter()
    r = subprocess.run([pkg.pfp.CLI_PATH, path, "-w", "10", "-p", "100", "-s", "-f", "-v"], env=env,
                       capture_output=True, text=True, check=True)
    wall = time.perf_counter() - t0
    out = {"wall_s": wall}
    m = re.search(r"File read: ([\d.]+) s, file write: ([\d.]+) s", r.stdout)
    out["read_s"], out["write_s"] = float(m.group(1)), float(m.group(2))
    m = re.search(r"GPU parse: ([\d.]+) ms", r.stdout)
    out["gpu_ms"] = float(m.group(1))
    ch = [l for l in r.stderr.splitlines() if l.startswith("[pfpb200 stream] chunk")]
    if ch:
        num = lambda key: [float(re.search(key + r" ([\d.]+)", l).group(1)) for l in ch]
        out["chunks"] = len(ch)
        out["k1_ms"], out["k2_ms"], out["k3_ms"] = sum(num("K1")), sum(num("K2")), sum(num("K3"))
        out["insert_ms"], out["remap_ms"] = sum(num("insert")), sum(num("remap"))
        out["insert_over_k3_per_chunk"] = [round(a / b, 3) if b else None for a, b in zip(num("insert"), num("K3"))]
        e = [l for l in r.stderr.splitlines() if l.startswith("[pfpb200 stream] end")][0]
        out["rank_ms"] = float(re.search(r"rank ([\d.]+) ms", e).group(1))
        out["dict_ms"] = float(re.search(r"dict ([\d.]+) ms", e).group(1))
        out["parse_rewrite_s"] = float(re.search(r"rewrite ([\d.]+) s", e).group(1))
    return out


def bench(pkg, tmp, reps):
    path = os.path.join(tmp, "config2.fa")
    sck.write_config2(pkg, path, True)
    size = os.path.getsize(path)
    modes = {"one-shot": 0, "stream ~4 chunks": 8 * -(-size // 4), "stream ~16 chunks": 8 * -(-size // 16)}
    run_cli(pkg, path, 0)                                               # page cache warm
    res = {m: [] for m in modes}
    for _ in range(reps):
        for m, b in modes.items():
            res[m].append(run_cli(pkg, path, b))
    base = statistics.median(x["wall_s"] for x in res["one-shot"])
    for m, runs in res.items():
        med = {k: statistics.median(x[k] for x in runs) for k in runs[0] if not isinstance(runs[0][k], list)}
        med["wall_over_one_shot"] = round(med["wall_s"] / base, 3)
        if "insert_over_k3_per_chunk" in runs[0]:
            med["insert_over_k3_per_chunk"] = runs[len(runs) // 2]["insert_over_k3_per_chunk"]
        print(json.dumps({"bench": m, "reps": reps, "file_bytes": size, "median": med,
                          "wall_s_all": [round(x["wall_s"], 3) for x in runs]}), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--peaks", action="store_true")
    ap.add_argument("--bench", action="store_true")
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--dir", default=None)
    a = ap.parse_args()
    from __graft_entry__ import load_package
    pkg = load_package()
    print(json.dumps({"gpu": card()}), flush=True)
    tmp = tempfile.mkdtemp(prefix="streambench_", dir=a.dir)
    try:
        if a.peaks:
            peaks(pkg, tmp)
        if a.bench:
            bench(pkg, tmp, a.reps)
    finally:
        shutil.rmtree(tmp, ignore_errors=True)


if __name__ == "__main__":
    main()
