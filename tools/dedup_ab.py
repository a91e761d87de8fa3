"""Per-step stage times of one build of the package, for A/B runs of the dedup stage against another
checkout (each arm is its own process: run it alternately for the two trees).

  --root DIR         tree whose built package is loaded (default: this one)
  --workload bench   bench.py's workload: 100 haplotypes x 40 Mbp, w=10 p=100, seed 2
  --workload random  8 GB of uniform random ACGT (seed 4), w=10 p=100: nearly every phrase a new word

Prints one JSON line: the per-step ms_total, ms_dedup and the other stage times, their medians, the
sha256 of the five streams of the last step, and the card.  --profile FILE: afterwards one more step
under torch.profiler, per-kernel CUDA times written to FILE.
--summarize FILE...: pool the steps of such lines per workload and label; median, min and max of
each stage time."""
import argparse
import hashlib
import json
import os
import statistics
import subprocess
import sys

W, P = 10, 100
STREAMS = ("dict", "occ", "parse", "last", "sai")
STAGES = ("ms_total", "ms_scan", "ms_hash", "ms_dedup", "ms_rank", "ms_dict", "ms_remap")


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "unknown"


def summarize(paths):
    runs = {}
    for path in paths:
        with open(path) as f:
            for line in f:
                r = json.loads(line)
                arm = runs.setdefault((r["workload"], r["label"]), {"steps": 0, "sha": set(), "card": r["card"]})
                arm["steps"] += r["steps"]
                arm["sha"].add(json.dumps(r["sha256_16"], sort_keys=True))
                for k, v in r["runs"].items():
                    arm.setdefault(k, []).extend(v)
    for (wl, label), arm in sorted(runs.items()):
        st = {k: {"median": round(statistics.median(arm[k]), 4), "min": min(arm[k]), "max": max(arm[k])} for k in STAGES}
        print(json.dumps({"workload": wl, "label": label, "steps": arm["steps"], "card": arm["card"],
                          "sha256_16": [json.loads(x) for x in sorted(arm["sha"])], **st}))


def main():
    if len(sys.argv) > 1 and sys.argv[1] == "--summarize":
        return summarize(sys.argv[2:])
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--root", default=os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
    ap.add_argument("--workload", default="bench", choices=["bench", "random"])
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--label", default="")
    ap.add_argument("--profile", metavar="FILE")
    a = ap.parse_args()

    root = os.path.abspath(a.root)
    sys.path.insert(0, root)
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("dedup_ab.py: no CUDA device")
    from __graft_entry__ import load_package
    pkg = load_package()
    if a.workload == "bench":
        text = pkg.synth.pangenome_text(40_000_000, 100, 2, device="cuda")
    else:
        text = pkg.synth.random_dna(8_000_000_000, 4, device="cuda")
    torch.cuda.synchronize()
    sc = pkg.pfp.Scanner(0)
    for _ in range(a.warmup):
        sc.parse_device(text, W, P, sai=True)
    runs = {k: [] for k in STAGES}
    for _ in range(a.steps):
        out = sc.parse_device(text, W, P, sai=True)
        st = sc.stats.as_dict()
        for k in STAGES:
            runs[k].append(round(st[k], 4))
    files = sc.fetch(out)
    digest = {s: hashlib.sha256(bytes(getattr(files, s))).hexdigest()[:16] for s in STREAMS}
    del files
    line = {"label": a.label, "root": os.path.basename(root), "workload": a.workload, "steps": a.steps,
            "median": {k: round(statistics.median(v), 4) for k, v in runs.items()}, "runs": runs,
            "n_distinct": st["n_distinct"], "sha256_16": digest, "card": card()}
    print(json.dumps(line), flush=True)
    if a.profile:
        from torch.profiler import ProfilerActivity, profile
        sc.parse_device(text, W, P, sai=True)
        torch.cuda.synchronize()
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            sc.parse_device(text, W, P, sai=True)
            torch.cuda.synchronize()
        table = prof.key_averages().table(sort_by="cuda_time_total", row_limit=60, max_name_column_width=60)
        with open(a.profile, "w") as f:
            f.write(f"# {a.label} ({a.workload}): one step under torch.profiler; card: {line['card']}\n{table}\n")
    sc.close()


if __name__ == "__main__":
    main()
