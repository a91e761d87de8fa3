"""A/B of the ranking of tie groups of 2..32 words on the bench.py workload (100 haplotypes x 40 Mbp,
w=10 p=100, generated on the GPU with bench.py's seed): LCP walks (rank_small_lcp_k, the default)
against warp chunk passes (rank_window_k + rank_warp_k, PFPB200_RANK_WARP_PASSES=1).

Both arms are Scanner contexts of one process (the variable is read when a context is created),
warmed up, then run alternately A, B, A, B ...  Prints one JSON line per arm (median and spread of
ms_total and ms_rank), whether the sha256 of the five streams agree, and the card it ran on.
--profile DIR: afterwards one more step of each arm under torch.profiler, per-kernel CUDA times
written to DIR/rank_ab_kernels_<arm>.txt."""
import argparse
import hashlib
import json
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

W, P, SEED = 10, 100, 2          # bench.py's workload
ARMS = (("walks", "0"), ("warp_passes", "1"))
STREAMS = ("dict", "occ", "parse", "last", "sai")


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "unknown"


def spread(xs):
    return {"median": round(statistics.median(xs), 4), "min": round(min(xs), 4), "max": round(max(xs), 4)}


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--base-len", type=int, default=40_000_000)
    ap.add_argument("--haplotypes", type=int, default=100)
    ap.add_argument("--steps", type=int, default=10, help="timed steps per arm")
    ap.add_argument("--warmup", type=int, default=3, help="untimed steps per arm")
    ap.add_argument("--profile", metavar="DIR")
    a = ap.parse_args()

    import torch
    if not torch.cuda.is_available():
        raise SystemExit("rank_ab.py: no CUDA device")
    from __graft_entry__ import load_package
    pkg = load_package()
    text = pkg.synth.pangenome_text(a.base_len, a.haplotypes, SEED, device="cuda")
    torch.cuda.synchronize()

    sc = {}
    for arm, val in ARMS:
        os.environ["PFPB200_RANK_WARP_PASSES"] = val
        try:
            sc[arm] = pkg.pfp.Scanner(0)
        finally:
            os.environ.pop("PFPB200_RANK_WARP_PASSES", None)

    def step(arm):
        out = sc[arm].parse_device(text, W, P, sai=True)
        return out, sc[arm].stats.as_dict()

    digests = {}
    for arm, _ in ARMS:
        for _ in range(a.warmup):
            out, _st = step(arm)
        files = sc[arm].fetch(out)
        digests[arm] = {s: hashlib.sha256(bytes(getattr(files, s))).hexdigest() for s in STREAMS}
        del files
    runs = {arm: {"ms_total": [], "ms_rank": []} for arm, _ in ARMS}
    for _ in range(a.steps):
        for arm, _ in ARMS:
            _out, st = step(arm)
            runs[arm]["ms_total"].append(st["ms_total"])
            runs[arm]["ms_rank"].append(st["ms_rank"])
    gpu = card()
    for arm, val in ARMS:
        print(json.dumps({"arm": arm, "PFPB200_RANK_WARP_PASSES": val, "steps": a.steps,
                          "ms_total": spread(runs[arm]["ms_total"]), "ms_rank": spread(runs[arm]["ms_rank"]),
                          "card": gpu}))
    same = digests["walks"] == digests["warp_passes"]
    print(json.dumps({"streams_identical": same, "sha256_walks": digests["walks"],
                      "sha256_warp_passes": digests["warp_passes"]}))

    if a.profile:
        from torch.profiler import ProfilerActivity, profile
        os.makedirs(a.profile, exist_ok=True)
        for arm, _ in ARMS:
            step(arm)
            torch.cuda.synchronize()
            with profile(activities=[ProfilerActivity.CUDA]) as prof:
                step(arm)
                torch.cuda.synchronize()
            table = prof.key_averages().table(sort_by="cuda_time_total", row_limit=60, max_name_column_width=60)
            with open(os.path.join(a.profile, f"rank_ab_kernels_{arm}.txt"), "w") as f:
                f.write(f"# {arm}: one step of the bench workload under torch.profiler; card: {gpu}\n{table}\n")
            print(f"profile {arm}: {os.path.join(a.profile, f'rank_ab_kernels_{arm}.txt')}")
    for s in sc.values():
        s.close()
    if not same:
        raise SystemExit("rank_ab.py: the two arms wrote different streams")


if __name__ == "__main__":
    main()
