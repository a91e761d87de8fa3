#!/usr/bin/env python3
"""Full-size checks of bwtparse's bounded path (pfpb200_bwtparse_file; DESIGN.md §6e).

  a   BASELINE.json config 2 (4 GB pan-genome, w 10 p 100, 39.6 M phrases) parsed to files, then
      bwtparse_file -s in HBM and with PFPB200_BWTPARSE_BUDGET at about 4 and 16 round-1 windows: the
      sha256 of .ilist .bwlast .bwsai must equal tests/golden/fullsize_sha256.json (the unmodified
      bwtparse on the same text); wall clock of each.
  b   a seeded pan-genome-shaped parse of --b-phrases (2.16 G: .ilist values past 2^31), in HBM and
      bounded (budget: resident + 16 windows): the two sets of files must be equal.  Needs a nearly free
      card (the in-HBM path, by its allocation count, about 74 B per phrase).
  c   a seeded parse of --c-phrases (3.2 G), more than the in-HBM path can hold: without a budget the
      routing must take the bounded path; the LF-walk check (oracle/lf_check.c) must pass.  Peak and time.
Each arm measures what it needs (device memory, disk, host memory) first and skips, saying why, when it
is not there.  Prints one JSON line per arm; exit status 1 on any failure.
usage: bwtparse_window_check.py [--arms a,b,c] [--dir DIR] [--b-phrases N] [--c-phrases N]"""
import argparse, json, os, shutil, subprocess, sys, tempfile, time
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
import numpy as np
import torch
from fullsize_check import load_digests
from stream_check import sha_file, write_config2

KEY = "config2 w10 p100"
OUTS = ("ilist", "bwlast", "bwsai")
INHBM = 74                  # device bytes per phrase of the in-HBM path with .sai (bp_inhbm_bytes, pfp_bwtparse.cu)
RESIDENT = 19               # ... resident in the bounded path (bw_resident_bytes)
WINDOW = 37                 # ... of a sort window (bw_window_bytes)
GB = 1e9


def emit(d):
    print(json.dumps(d), flush=True)
    return d


def free_device():
    f, _ = torch.cuda.mem_get_info()
    return f


def free_disk(d):
    return shutil.disk_usage(d).free


def host_ram():
    with open("/proc/meminfo") as f:
        for line in f:
            if line.startswith("MemAvailable:"):
                return int(line.split()[1]) * 1024
    return 0


def budget_for(n, windows):
    return RESIDENT * (n + 1) + WINDOW * ((n + 1) // windows) + (8 << 20)


def bwtparse(sc, base, budget):
    if budget:
        os.environ["PFPB200_BWTPARSE_BUDGET"] = str(budget)
    try:
        t0 = time.perf_counter()
        r = sc.bwtparse_file(base, sai=True)
        wall = time.perf_counter() - t0
    finally:
        os.environ.pop("PFPB200_BWTPARSE_BUDGET", None)
    return r, wall


def digests(base):
    return {ext: sha_file(f"{base}.{ext}") for ext in OUTS}


def arm_a(pkg, tmp):
    ref = load_digests()["cases"][KEY]["pipeline"]["sha256"]
    if free_disk(tmp) < 12 * GB:
        return emit({"arm": "a", "skipped": f"{free_disk(tmp) / GB:.1f} GB free disk, 12 GB needed"})
    base = os.path.join(tmp, "config2.txt")
    write_config2(pkg, base, False)
    sc = pkg.pfp.Scanner(0)
    try:
        sc.parse_file(base, 10, 100, sai=True)
        n = os.path.getsize(base + ".parse") // 4
        out = {"arm": "a", "phrases": n, "runs": []}
        for windows in (None, 4, 16, None, 4, 16):        # alternated, twice
            r, wall = bwtparse(sc, base, budget_for(n, windows) if windows else None)
            got = digests(base)
            ok = all(got[e] == ref[e] for e in OUTS)
            out["runs"].append({"target_windows": windows, "windows": r["windows"], "rounds": r["rounds"],
                                "wall_s": round(wall, 3), "ms_total": round(r["ms_total"], 1),
                                "peak_gb": round(r["peak_device_bytes"] / GB, 3), "sha256_ok": ok})
        out["ok"] = all(x["sha256_ok"] for x in out["runs"]) and all(
            (x["windows"] == 1) == (x["target_windows"] is None) for x in out["runs"])
    finally:
        sc.close()
    return emit(out)


def write_synthetic(base, n, seed):
    """a pan-genome-shaped parse: 100 copies of a base phrase sequence over a dictionary of about n / 50
    words, each copy with 0.5 % of its phrases replaced by fresh words; T[0] = 1 is unique.  .last are
    letters, .sai ascending 5-byte positions."""
    g = torch.Generator(device="cuda")
    g.manual_seed(seed)
    copies = 100
    L = (n - 1 + copies - 1) // copies
    d = max(n // 50, 16)
    basev = torch.randint(2, d, (L,), device="cuda", generator=g, dtype=torch.int64)
    fresh = d
    step = 1 << 27
    with open(base + ".parse", "wb") as fp, open(base + ".last", "wb") as fl, open(base + ".sai", "wb") as fs:
        np.array([1], np.uint32).tofile(fp)
        written = 1
        for k in range(copies):
            for a in range(0, L, step):
                m = min(step, L - a, n - written)
                if m <= 0:
                    break
                t = basev[a:a + m].clone()
                mut = torch.rand(m, device="cuda", generator=g) < 0.005
                nm = int(mut.sum())
                t[mut] = torch.arange(fresh, fresh + nm, device="cuda")
                fresh += nm
                t.cpu().numpy().astype(np.uint32).tofile(fp)
                written += m
        total = written
        for a in range(0, total, step):
            m = min(step, total - a)
            torch.randint(65, 91, (m,), device="cuda", generator=g, dtype=torch.uint8).cpu().numpy().tofile(fl)
            p = torch.arange(a, a + m, device="cuda", dtype=torch.int64) * 100 + 99
            torch.stack([(p >> (8 * j)) & 255 for j in range(5)], 1).to(torch.uint8).cpu().numpy().tofile(fs)
    return total


def arm_b(pkg, tmp, n):
    need_dev, need_disk = INHBM * (n + 1) + (2 << 30), 2 * 25 * (n + 1) + (4 << 30)
    if free_device() < need_dev:
        return emit({"arm": "b", "skipped": f"{free_device() / GB:.1f} GB free on the device, {need_dev / GB:.1f} GB needed"})
    if free_disk(tmp) < need_disk:
        return emit({"arm": "b", "skipped": f"{free_disk(tmp) / GB:.1f} GB free disk, {need_disk / GB:.1f} GB needed"})
    base = os.path.join(tmp, "b")
    n = write_synthetic(base, n, 21)
    sc = pkg.pfp.Scanner(0)
    try:
        r1, w1 = bwtparse(sc, base, None)
        d1 = digests(base)
        for e in OUTS:
            os.unlink(f"{base}.{e}")
        r2, w2 = bwtparse(sc, base, budget_for(n, 16))
        d2 = digests(base)
    finally:
        sc.close()
    return emit({"arm": "b", "phrases": n, "inhbm": {"windows": r1["windows"], "wall_s": round(w1, 2),
                                                     "peak_gb": round(r1["peak_device_bytes"] / GB, 2)},
                 "bounded": {"windows": r2["windows"], "wall_s": round(w2, 2), "peak_gb": round(r2["peak_device_bytes"] / GB, 2)},
                 "ok": d1 == d2 and r1["windows"] == 1 and r2["windows"] > 1})


def arm_c(pkg, tmp, n):
    from oracle import lf_check
    need_dev, need_disk, need_ram = RESIDENT * (n + 1) + (8 << 30), 21 * (n + 1) + (4 << 30), 30 * (n + 1)
    if free_device() < need_dev:
        return emit({"arm": "c", "skipped": f"{free_device() / GB:.1f} GB free on the device, {need_dev / GB:.1f} GB needed"})
    if free_disk(tmp) < need_disk:
        return emit({"arm": "c", "skipped": f"{free_disk(tmp) / GB:.1f} GB free disk, {need_disk / GB:.1f} GB needed"})
    if host_ram() < need_ram:
        return emit({"arm": "c", "skipped": f"{host_ram() / GB:.1f} GB host memory available, {need_ram / GB:.1f} GB needed"})
    base = os.path.join(tmp, "c")
    n = write_synthetic(base, n, 31)
    sc = pkg.pfp.Scanner(0)
    try:
        r, wall = bwtparse(sc, base, None)
    finally:
        sc.close()
    t0 = time.perf_counter()
    msg = lf_check.check_files(base)
    return emit({"arm": "c", "phrases": n, "windows": r["windows"], "rounds": r["rounds"], "wall_s": round(wall, 2),
                 "peak_gb": round(r["peak_device_bytes"] / GB, 2), "lf_check_s": round(time.perf_counter() - t0, 1),
                 "lf_check": msg or "ok", "ok": r["windows"] > 1 and msg == ""})


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--arms", default="a,b,c")
    ap.add_argument("--dir", default=None)
    ap.add_argument("--b-phrases", type=int, default=2_160_000_000)
    ap.add_argument("--c-phrases", type=int, default=3_200_000_000)
    a = ap.parse_args()
    import __graft_entry__ as g
    pkg = g.load_package()
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    emit({"card": q.stdout.strip().splitlines()[0] if q.stdout.strip() else "unknown"})
    ok = True
    for arm in a.arms.split(","):
        tmp = tempfile.mkdtemp(prefix=f"bwtwin_{arm}_", dir=a.dir)
        try:
            r = {"a": lambda: arm_a(pkg, tmp), "b": lambda: arm_b(pkg, tmp, a.b_phrases),
                 "c": lambda: arm_c(pkg, tmp, a.c_phrases)}[arm]()
            ok &= r.get("ok", True)
        finally:
            shutil.rmtree(tmp, ignore_errors=True)
    sys.exit(0 if ok else 1)


if __name__ == "__main__":
    main()
