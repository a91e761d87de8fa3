#!/usr/bin/env python3
"""Full-size check of the sharded pfbwt (pfpb200_multi_pfbwt_file, `-S`): the files it wrote, checked on
the device in linear time against the text, and, where the unmodified reference chain's digests exist,
by sha256.

  --config 2  BASELINE config 2 (100 haplotypes x 40 Mbp, w=10 p=100, 814 MB dictionary) with the rank
              list --ranks (default 0,0: two ranks on one GPU; four ranks on one 180 GB card run out
              of device memory in the emission, each rank keeping its own word structure).  .bwt (4,000,000,199 B) and .sa
              (20,000,000,990 B) must match tests/golden/fullsize_sha256.json "config2 w10 p100" ->
              "pipeline".
  --config 4  BASELINE config 4 (8 GB of random ACGT, 8.8 GB dictionary): parse and bwtparse on GPU 0,
              pfbwt -S on the visible GPUs.  No reference digest exists; the linear checks decide.

The linear checks of the written .sa / .bwt (the suffix-array row 0 is the end-of-text suffix, which
.sa leaves out):
  * the suffix array is a permutation of [0, n];
  * bwt[i] == T[sa[i] - 1], and the EOF char 0 sits at the row of the suffix at position 0;
  * adjacent rows: T[sa[i]] < T[sa[i+1]], or they are equal and ISA[sa[i]+1] < ISA[sa[i+1]+1]
    (Burkhardt-Kaerkkaeinen), the end of the text smaller than every char.
This checks the files; it is not a second suffix sort.  A case that does not fit (device memory, disk,
too few GPUs) prints a "not run" line with the reason and exits 0; a failed check exits 1.
usage: pfbwt_multi_check.py --config {2,4} [--ranks 0,0,0,0] [--dir DIR]"""
import argparse
import hashlib
import json
import os
import shutil
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch  # noqa: E402

CHUNK = 1 << 28


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


def load_sa(path, n):
    """.sa (n values of 5 bytes, rows 1..n) -> int64 suffix array of rows 0..n on the device"""
    sa = torch.empty(n + 1, dtype=torch.int64, device="cuda")
    sa[0] = n
    w = torch.tensor([1 << (8 * j) for j in range(5)], dtype=torch.int64, device="cuda")
    with open(path, "rb") as f:
        i = 1
        while i <= n:
            k = min(CHUNK, n + 1 - i)
            b = torch.frombuffer(bytearray(f.read(5 * k)), dtype=torch.uint8).cuda().view(k, 5).to(torch.int64)
            sa[i:i + k] = (b * w).sum(1)
            i += k
    return sa


def linear_checks(T, sa, bwt):
    """T: text (uint8, n), sa: int64 (n + 1 rows), bwt: uint8 (n + 1) -- all on the device"""
    n = T.numel()
    fails = []
    if bwt.numel() != n + 1 or sa.numel() != n + 1:
        return [f"sizes: bwt {bwt.numel()}, sa {sa.numel()}, text {n}"]
    if int(sa.min()) < 0 or int(sa.max()) > n:
        return ["suffix array values outside [0, n]"]
    isa = torch.full((n + 2,), -1, dtype=torch.int64, device="cuda")
    for a in range(0, n + 1, CHUNK):
        b = min(n + 1, a + CHUNK)
        isa[sa[a:b]] = torch.arange(a, b, dtype=torch.int64, device="cuda")
    if bool((isa[:n + 1] < 0).any()):
        fails.append("the suffix array is not a permutation of [0, n]")
        return fails
    isa[n + 1] = -1
    Tx = torch.empty(n + 1, dtype=torch.int16, device="cuda")
    Tx[:n] = T.to(torch.int16)
    Tx[n] = -1                                                    # the end of the text: smaller than every char
    bad_bwt = bad_order = 0
    for a in range(0, n + 1, CHUNK):
        b = min(n + 1, a + CHUNK)
        s = sa[a:b]
        prev = torch.where(s > 0, Tx[(s - 1).clamp(min=0)], torch.zeros_like(s, dtype=torch.int16))
        bad_bwt += int((prev != bwt[a:b].to(torch.int16)).sum())
        e = min(b, n)                                             # rows a..e-1 against rows a+1..e
        if e > a:
            s0, s1 = sa[a:e], sa[a + 1:e + 1]
            c0, c1 = Tx[s0], Tx[s1]
            r0 = isa[(s0 + 1).clamp(max=n + 1)]
            r1 = isa[(s1 + 1).clamp(max=n + 1)]
            ok = (c0 < c1) | ((c0 == c1) & (r0 < r1))
            bad_order += int((~ok).sum())
    if bad_bwt:
        fails.append(f"bwt[i] != T[sa[i]-1] at {bad_bwt} rows")
    if bad_order:
        fails.append(f"adjacent rows out of order at {bad_order} places")
    return fails


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
    ap.add_argument("--config", required=True, choices=["2", "4"])
    ap.add_argument("--ranks", default=None, help="rank list (config 2 default 0,0; config 4 default all GPUs)")
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
    if a.config == "4":
        ids = [int(x) for x in a.ranks.split(",")] if a.ranks else list(range(n_gpu))
        # per rank: the 8.8 GB dictionary, 4 B of word ids per dictionary byte, 8 B per byte / G of the rank
        # block, about 80 B per owned suffix and 6 B per owned BWT char: it fits 180 GB from G = 8 on
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
        free_mem = torch.cuda.mem_get_info(0)[0]
        emit({"n_text": n, "dict_bytes": dict_bytes, "parse_size": psize, "ranks": ids,
              "device0_free_GB": round(free_mem / 1e9, 1), "disk_free_GB": round(free_disk / 1e9, 1)})
        ms = P.MultiScanner(ids)
        t0 = time.perf_counter()
        try:
            r = ms.pfbwt_file(base, 10, P.PFBWT_SA)
        except P.PfpError as e:
            if e.code == -4:                                      # E_NOMEM
                emit({"config": a.config, "not_run": f"device memory: {e}"})
                return 0
            raise
        wall = time.perf_counter() - t0
        ms.close()
        emit({"pfbwt_wall_s": round(wall, 2), "rounds": r["rounds"], "n_bwt": r["n_bwt"], "hard": r["hard"],
              "ms_sort": round(r["ms_sa"], 1), "ms_fill": round(r["ms_fill"], 1),
              "per_rank": [{k: (round(v, 1) if isinstance(v, float) else v) for k, v in x.items()} for x in r["ranks"]]})
        fails = []
        if a.config == "2":
            with open(os.path.join(ROOT, "tests", "golden", "fullsize_sha256.json")) as f:
                ref = json.load(f)["cases"]["config2 w10 p100"]["pipeline"]
            got = {e: sha(f"{base}.{e}") for e in ("bwt", "sa")}
            res = {e: got[e] == ref["sha256"][e] for e in got}
            emit({"sha256_vs_reference_chain": res, "bytes": {e: os.path.getsize(f"{base}.{e}") for e in got}})
            fails += [f".{e} sha256 differs from the reference chain" for e in res if not res[e]]
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
