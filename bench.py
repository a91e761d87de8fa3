#!/usr/bin/env python3
"""bench.py -- PFP parse GB/s (text in -> .dict/.occ/.parse/.last/.sai out), BASELINE.json's metric.

One "step" = one complete prefix-free parse of the workload text:
  value : device-resident (text already in HBM -> all five outputs in HBM), CUDA events
  e2e   : through the C-ABI host entry pfpb200_parse_host with pinned HOST buffers, the H2D copy
          of the text and the D2H copy of all outputs inside the timed region
Workload at N=1 = BASELINE.json configs[1]: 100 haplotypes of a 40 Mbp chromosome, 0.1 %
SNP/indel variation, w=10 p=100 (4 GB of text; synthetic, seeded, generated on the GPU).
`--impl reference` times the reference's own CPU scanner (oracle/_ref, unmodified) on a
bounded prefix of the same workload with all host threads.
"""
import argparse
import json
import os
import shutil
import subprocess
import sys
import tempfile
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

W, P = 10, 100
SEED = 2
METRIC = "pfp_parse_throughput"
UNIT = "GB/s"


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--base-len", type=int, default=40_000_000, help="chromosome length (bp)")
    ap.add_argument("--haplotypes", type=int, default=100, help="haplotypes per GPU")
    ap.add_argument("--workload", default="pangenome", choices=["pangenome", "random"])
    ap.add_argument("--cpu-haplotypes", type=int, default=4, help="prefix timed on the CPU")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-ref-full", action="store_true",
                    help="reference arm: skip the single run on the whole workload (N=1 only, about a minute)")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-parity", action="store_true", help="skip the byte-exact output check after the timed region")
    ap.add_argument("--e2e-steps", type=int, default=10)
    ap.add_argument("--no-t2", action="store_true", help="skip the file-to-files wall clock of gpuscan.x (N=1 only)")
    ap.add_argument("--no-pipeline", action="store_true", help="skip the text -> BWT leg (parse + bwtparse + pfbwt, N=1 only)")
    ap.add_argument("--merge", default="partition", choices=["partition", "replicate"],
                    help="multi-GPU dictionary merge: range-partitioned all-to-all or replicated all-gather")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the five streams of the last timed step to DIR/<stream>.npy; covers the "
                         "single-GPU path only (refused with --gpus > 1)")
    a = ap.parse_args()
    if a.steps < 1 or a.warmup < 0:
        ap.error("--steps must be at least 1 and --warmup at least 0")
    if a.dump_outputs and a.gpus != 1:
        ap.error("--dump-outputs needs --gpus 1")
    return a


def workload_name(a, world=None):
    world = world or a.gpus
    if a.workload == "random":
        return f"uniform random ACGT, {a.base_len * a.haplotypes * world / 1e9:.2f} GB, w={W} p={P}, -s"
    return (f"{a.haplotypes * world} haplotypes x {a.base_len / 1e6:g} Mbp, 0.1% SNP/indel "
            f"({a.base_len * a.haplotypes * world / 1e9:.2f} GB text), w={W} p={P}, -s")


def workload_config(a, world=None):
    """`config` of the JSON line: the same dict from both arms (the reference arm measures the
    same workload; how much of it one of its steps covers is in its cpu_baseline.sample)."""
    world = world or a.gpus
    per_gpu = a.base_len * a.haplotypes
    return {"workload": workload_name(a, world),
            "l2": "inputs larger than L2 (no flush needed)" if per_gpu > 256e6 else "input smaller than L2",
            "parallelism": f"{world} shard(s) of {per_gpu / 1e9:.2f} GB, one process per GPU" +
                           (f", {a.merge} dictionary merge" if world > 1 else "")}


# ------------------------------------------------------------------------------------------------
# clocks: sample nvidia-smi while the timed region runs
# ------------------------------------------------------------------------------------------------
class ClockSampler:
    """SM clock + throttle reasons through NVML every 5 ms while the timed region runs."""
    REASONS = {0x4: "sw_power_cap", 0x8: "hw_slowdown", 0x20: "sw_thermal_slowdown",
               0x40: "hw_thermal_slowdown"}

    def __init__(self, index):
        self.index = index
        self.samples, self.reasons, self.max_mhz = [], set(), None
        self.stop_flag = threading.Event()
        self.thread = None
        self.err = None

    def start(self):
        try:
            import pynvml
            pynvml.nvmlInit()
            vis = os.environ.get("CUDA_VISIBLE_DEVICES")
            idx = int(vis.split(",")[self.index]) if vis and vis.split(",")[self.index].isdigit() else self.index
            self.h = pynvml.nvmlDeviceGetHandleByIndex(idx)
            self.nv = pynvml
            self.max_mhz = float(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))
        except Exception as e:  # noqa: BLE001
            self.err = f"nvml unavailable: {e}"
            return
        self.thread = threading.Thread(target=self._run, daemon=True)
        self.thread.start()

    def _run(self):
        nv = self.nv
        while not self.stop_flag.is_set():
            try:
                self.samples.append(float(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM)))
                try:
                    r = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                except Exception:  # noqa: BLE001
                    r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for bit, name in self.REASONS.items():
                    if r & bit:
                        self.reasons.add(name)
            except Exception as e:  # noqa: BLE001
                self.err = str(e)
                return
            time.sleep(0.005)

    def stop(self):
        self.stop_flag.set()
        if self.thread:
            self.thread.join(timeout=2)
        sm = sorted(self.samples)
        out = {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": self.max_mhz,
               "samples": len(sm), "reasons": sorted(self.reasons)}
        if self.err:
            out["note"] = self.err
        return out


# ------------------------------------------------------------------------------------------------
# the reference's CPU scanner on a bounded prefix of the workload
# ------------------------------------------------------------------------------------------------
def cpu_sample_text(a, synth):
    """First --cpu-haplotypes haplotypes of the workload (same seeds => same bytes), on the CPU."""
    import torch
    if a.workload == "random":
        n = min(a.base_len * a.cpu_haplotypes, a.base_len * a.haplotypes)
        return synth.random_dna(n, SEED).numpy(), f"first {n / 1e6:.0f} MB of the text"
    dev = "cuda" if torch.cuda.is_available() else "cpu"
    h = min(a.cpu_haplotypes, a.haplotypes)
    t = synth.pangenome_text(a.base_len, h, SEED, device=dev).cpu().numpy()
    return t, f"first {h} haplotypes ({t.size / 1e6:.0f} MB of text) of the same workload"


def run_reference_scanner(text_np, threads, tmpdir, reps):
    """Time oracle/_ref pscan (the reference's scaling multi-thread scanner, plain text) or, if it
    is missing, the oracle port.  Returns (best-effort list of seconds, kind, description)."""
    from oracle import pfp_oracle as orc
    path = os.path.join(tmpdir, "sample.txt")
    text_np.tofile(path)
    exe = None
    for cand in ("pscan_fast.x", "pscan.x"):
        if orc.have_ref(cand):
            exe = orc.ref_exe(cand)
            break
    secs = []
    if exe:
        cmd = [exe, path, "-w", str(W), "-p", str(P), "-s", "-t", str(threads)]
        for _ in range(reps):
            t0 = time.perf_counter()
            subprocess.run(cmd, check=True, stdout=subprocess.DEVNULL, stderr=subprocess.DEVNULL)
            secs.append(time.perf_counter() - t0)
        return secs, "reference", f"{os.path.basename(exe)} -t {threads} (unmodified reference, oracle/_ref)", threads
    data = text_np.tobytes()
    for _ in range(reps):
        t0 = time.perf_counter()
        orc.parse(data, W, P)
        secs.append(time.perf_counter() - t0)
    return secs, "port", "oracle/pfp_oracle.c (single thread)", 1


def run_newscan_fasta(text_np, threads, tmpdir):
    """`newscan.x <fasta> -f -t T` -- the command `bigbwt -f -t T` issues and BASELINE.json names --
    once, on the sample wrapped as one 60-column FASTA record.  Its threads are serialised by a
    global mutex and a serial prescan (SURVEY 3.3), which is why pscan is the headline baseline."""
    from oracle import pfp_oracle as orc
    from __graft_entry__ import load_package
    exe = next((orc.ref_exe(c) for c in ("newscan_fast.x", "newscan.x") if orc.have_ref(c)), None)
    if exe is None:
        return None
    path = os.path.join(tmpdir, "sample.fa")
    load_package().synth.to_fasta_np(text_np, "sample").tofile(path)
    cmd = [exe, path, "-w", str(W), "-p", str(P), "-s", "-f", "-t", str(threads)]
    t0 = time.perf_counter()
    r = subprocess.run(cmd, stdout=subprocess.DEVNULL, stderr=subprocess.DEVNULL)
    dt = time.perf_counter() - t0
    if r.returncode != 0:
        return {"cmd": f"{os.path.basename(exe)} -f -t {threads}", "failed": r.returncode}
    return {"cmd": f"{os.path.basename(exe)} -f -t {threads}", "value": text_np.size / dt / 1e9, "unit": UNIT,
            "seconds": dt, "text_bytes": int(text_np.size)}


def reference_arm(a, synth):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import torch
    threads = os.cpu_count() or 1
    text, sample = cpu_sample_text(a, synth)
    tmp = tempfile.mkdtemp(prefix="pfpbench_")
    full = newscan = None
    try:
        secs, kind, how, cores = run_reference_scanner(text, threads, tmp, a.warmup + a.steps)
        if kind == "reference":
            newscan = run_newscan_fasta(text, threads, tmp)
        # one run on the WHOLE workload (the same 4 GB the GPU arm parses) when it is one GPU's
        if kind == "reference" and a.gpus == 1 and not a.no_ref_full and a.workload == "pangenome":
            dev = "cuda" if torch.cuda.is_available() else "cpu"
            whole = synth.pangenome_text(a.base_len, a.haplotypes, SEED, device=dev).cpu().numpy()
            fs, _, fhow, _ = run_reference_scanner(whole, threads, tmp, 1)
            full = {"value": whole.size / fs[0] / 1e9, "unit": UNIT, "seconds": fs[0],
                    "text_bytes": int(whole.size), "cmd": fhow, "steps": 1}
            del whole
    finally:
        shutil.rmtree(tmp, ignore_errors=True)
    timed = secs[a.warmup:]
    total = sum(timed)
    val = text.size * len(timed) / total / 1e9
    line = {
        "metric": METRIC, "value": val, "unit": UNIT, "n_gpus": a.gpus, "steps": a.steps,
        "warmup": a.warmup, "ms_per_step": 1e3 * total / len(timed), "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "u8/u32/u64 integer", "data": "synthetic",
        "impl": "reference",
        "config": workload_config(a),
        "cpu_baseline": {"value": val, "unit": UNIT, "cores": cores, "kind": kind,
                         "sample": f"{how}; every step = {sample}; wall clock of the scanner process"},
        "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
        "whole_workload_once": full, "newscan_fasta_once": newscan,
    }
    print(json.dumps(line))


# ------------------------------------------------------------------------------------------------
# our arm
# ------------------------------------------------------------------------------------------------
def load_peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md)"


def scan_kernel_name():
    """K1 of the benchmarked configuration (w=10): the interval form unless PFPB200_K1=rolling / table."""
    mode = os.environ.get("PFPB200_K1")
    return "kr_scan_k<10>" if mode == "rolling" else "kr_scan_dna_k<10>" if mode == "table" else "kr_scan_ivf_k"


def load_traffic(n_text):
    """dram bytes per launch of the scan kernel from the committed ncu --set full capture."""
    try:
        with open(os.path.join(ROOT, "profiles", "traffic.json")) as f:
            t = json.load(f)
        per_byte = t[scan_kernel_name().split("<")[0]]["dram_bytes_per_text_byte"]
        return per_byte * n_text
    except Exception:
        return None


# ------------------------------------------------------------------------------------------------
# byte-exact check of the code path that was just timed (outside the timed region)
# ------------------------------------------------------------------------------------------------
PARITY_BASE, PARITY_HAP, PARITY_NRUN = 4_000_000, 100, 3 << 20


def parity_text_and_cuts(synth, world, dev):
    """400 MB pan-genome (100 haplotypes x 4 Mbp, own seed) with a 3 MB run of N, cut into `world`
    uneven shards.  With 3 or more shards, shard 1 is 1 MB long and lies INSIDE the run: it owns no
    phrase at all, and the phrase straddling into shard 2 crosses two seams and starts 2 MB before
    it -- more than the megabyte a rank reserves in front of its shard."""
    import torch
    t = synth.pangenome_text(PARITY_BASE, PARITY_HAP, SEED + 7, device=dev)
    n = t.numel()
    cuts = [0] + [n * k // world + 1237 * k for k in range(1, world)] + [n]
    if world >= 3:
        cuts[2] = cuts[1] + (1 << 20)
    c1 = cuts[1] if world > 1 else n // 2
    t[c1 - (1 << 20): c1 - (1 << 20) + PARITY_NRUN] = ord("N")
    return t, cuts


def parity_check(job, pkg, synth, world, rank, local, dev, merge):
    """Parse the parity text through the SAME ShardedParser object (same merge mode, same peer
    exchange) that was timed and compare all five streams byte for byte: at N > 1 with a 1-GPU
    pfpb200_parse_device of the whole text on rank 0, at N = 1 with the CPU oracle (the checker,
    pinned to the reference's newscanNT.x by tests/test_oracle_golden.py)."""
    import hashlib
    import torch
    text, cuts = parity_text_and_cuts(synth, world, dev)
    job.set_text(text[cuts[rank]:cuts[rank + 1]].clone() if world > 1 else text)
    job.parse_device(W, P, sai=True)
    if world > 1:
        got = job.gather_files()
    else:
        f = job.scanner.fetch(job.out)
        got = {k: getattr(f, k) for k in ("dict", "occ", "parse", "last", "sai")}
    if rank != 0:
        return None
    if world > 1:
        sc = pkg.pfp.Scanner(local)
        f = sc.fetch(sc.parse_device(text, W, P, sai=True))
        want = {k: getattr(f, k) for k in got}
        sc.close()
        against = "pfpb200_parse_device of the whole text on one GPU (rank 0)"
    else:
        from oracle import pfp_oracle as orc
        f = orc.parse(text.cpu().numpy(), W, P)
        want = {k: getattr(f, k) for k in got}
        against = "oracle/pfp_oracle.c on the host (CPU restatement of newscan.cpp, the checker)"
    bad = [k for k in got if got[k] != want[k]]
    return {"ok": not bad, "bytes": sum(len(v) for v in got.values()), "text_bytes": int(text.numel()),
            "shard_cuts": cuts, "n_run_bytes": PARITY_NRUN, "mismatch": bad, "against": against,
            "phrases": len(got["parse"]) // 4, "distinct": len(got["occ"]) // 4,
            "sha256": {k: hashlib.sha256(v).hexdigest()[:16] for k, v in got.items()}}


# ------------------------------------------------------------------------------------------------
# --dump-outputs: what the timed path handed its caller, for comparing two builds output by output
# ------------------------------------------------------------------------------------------------
DUMP_MAX_ELEMS, DUMP_SEED = 1 << 20, 12345     # at most 5 x 8 MB of float64


def dump_outputs(files, out_dir):
    """Each of the five streams as DIR/<stream>.npy: .dict and .last bytes as float32, .occ and .parse
    ranks and the 5-byte .sai positions as float64 (all exact).  A stream longer than DUMP_MAX_ELEMS
    is replaced by the elements at a sorted sample of positions drawn with DUMP_SEED, which depends on
    nothing but the stream's length.  Returns {stream: [full length, elements stored]}."""
    import numpy as np
    sai = np.frombuffer(files.sai, np.uint8).reshape(-1, 5)
    streams = {"dict": (np.frombuffer(files.dict, np.uint8), np.float32),
               "occ": (np.frombuffer(files.occ, np.uint32), np.float64),
               "parse": (np.frombuffer(files.parse, np.uint32), np.float64),
               "last": (np.frombuffer(files.last, np.uint8), np.float32),
               "sai": (sai, np.float64)}
    os.makedirs(out_dir, exist_ok=True)
    info = {}
    for name, (a, dtype) in streams.items():
        n = len(a)
        if n > DUMP_MAX_ELEMS:
            a = a[np.sort(np.random.default_rng(DUMP_SEED).choice(n, DUMP_MAX_ELEMS, replace=False))]
        if name == "sai":
            a = sum(a[:, i].astype(np.uint64) << np.uint64(8 * i) for i in range(5)) if len(a) else a[:, 0]
        np.save(os.path.join(out_dir, name + ".npy"), a.astype(dtype))
        info[name] = [n, len(a)]
    return info


# ------------------------------------------------------------------------------------------------
# T2 (SURVEY 8d): page-cache-warm FASTA file -> five files closed, wall clock of the gpuscan.x process
# ------------------------------------------------------------------------------------------------
def pipeline_to_bwt(pkg, device, text, steps=3, cpu_sample_bytes=0):
    """The whole bigbwt pipeline on the GPU with the text resident in HBM: parse -> bwtparse -> pfbwt
    (pfpb200_parse_device / _bwtparse_device / _pfbwt_device on one context, nothing leaves HBM in
    between).  Wall clock of the three calls + each stage's CUDA-event time; reported beside the
    metric, not part of it."""
    import torch
    try:
        sc = pkg.pfp.Scanner(device)
        runs = []
        for _ in range(steps + 1):
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            r, out, bp = sc.bwt_of_text(text, W, P, flags=0)
            wall = time.perf_counter() - t0
            runs.append({"seconds": wall, "ms_parse": sc.stats.ms_total, "ms_bwtparse": bp.ms_total,
                         "ms_pfbwt": r.ms_total, "ms_pfbwt_suffix_sort": r.ms_sa, "ms_pfbwt_emit": r.ms_fill,
                         "doubling_rounds": {"bwtparse": bp.rounds, "pfbwt": r.rounds},
                         "easy_chars": r.easy, "hard_chars": r.hard, "bwt_bytes": r.n_bwt})
        # the reference's own later stages on a bounded sample (first haplotype), host cores, for the ratio
        cpu = None
        ref_dir = os.path.join(ROOT, "oracle", "_ref")
        if cpu_sample_bytes and os.path.exists(os.path.join(ref_dir, "pfbwtNT.x")):
            sub = text[:cpu_sample_bytes].clone()
            o2 = sc.parse_device(sub, W, P, sai=True)
            f = sc.fetch(o2)
            tmp = tempfile.mkdtemp(prefix="pfppipe_")
            try:
                base = os.path.join(tmp, "x")
                for ext in ("dict", "occ", "parse", "last", "sai"):
                    with open(base + "." + ext, "wb") as fh:
                        fh.write(getattr(f, ext))
                t0 = time.perf_counter()
                subprocess.run([os.path.join(ref_dir, "bwtparse"), base, "-s"], check=True, stdout=subprocess.DEVNULL)
                t1 = time.perf_counter()
                subprocess.run([os.path.join(ref_dir, "pfbwtNT.x"), "-w", str(W), base], check=True, stdout=subprocess.DEVNULL)
                t2 = time.perf_counter()
                r2, _, _ = sc.bwt_of_text(sub, W, P, flags=0)
                same = open(base + ".bwt", "rb").read() == sc.to_host(r2.bwt, r2.n_bwt)
                cpu = {"kind": "reference", "cores": 1, "value": sub.numel() / (t2 - t0) / 1e9, "unit": "GB/s of text",
                       "bwtparse_s": t1 - t0, "pfbwt_s": t2 - t1, "bwt_identical": same,
                       "sample": f"bwtparse -s + pfbwtNT.x (unmodified, oracle/_ref) on the GPU parse of the first {sub.numel()} bytes of the text"}
            finally:
                shutil.rmtree(tmp, ignore_errors=True)
        sc.close()
        torch.cuda.empty_cache()
        med = sorted(runs[1:], key=lambda d: d["seconds"])[len(runs[1:]) // 2]
        med["cpu_baseline"] = cpu
        med["value"] = text.numel() / med["seconds"] / 1e9
        med["unit"] = "GB/s of text, text in HBM -> BWT in HBM"
        med["steps"] = steps
        med["how"] = "Scanner.bwt_of_text: pfpb200_parse_device -> pfpb200_bwtparse_device -> pfpb200_pfbwt_device"
        return med
    except Exception as e:  # noqa: BLE001  (a failure here must not take the metric's line down)
        return {"error": str(e)[:300]}


def t2_file_to_files(a, pkg, synth, dev):
    """Writes the workload as a one-record-per-haplotype, 60-column FASTA (what `bigbwt -f` is
    given), runs `gpuscan.x <file> -w 10 -p 100 -s -f` twice as a subprocess -- process start, CUDA
    context creation, streaming read, K0, parse, streaming write all inside the wall clock -- and
    reports the faster run with the tool's own breakdown."""
    import re
    tmp = tempfile.mkdtemp(prefix="pfpt2_")
    try:
        path = os.path.join(tmp, "workload.fa")
        t0 = time.perf_counter()
        n_text = 0
        with open(path, "wb") as f:
            for k, rec in enumerate(synth.pangenome_records(a.base_len, a.haplotypes, SEED, device=dev)):
                r = rec.cpu().numpy()
                n_text += r.size
                synth.to_fasta_np(r, f"hap{k}").tofile(f)
        gen_s = time.perf_counter() - t0
        fsize = os.path.getsize(path)
        runs = []
        for _ in range(2):
            t0 = time.perf_counter()
            r = subprocess.run([pkg.pfp.CLI_PATH, path, "-w", str(W), "-p", str(P), "-s", "-f"],
                               stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True)
            dt = time.perf_counter() - t0
            if r.returncode != 0:
                return {"failed": r.returncode, "stderr": r.stderr[-300:]}
            io = re.search(r"File read: ([0-9.]+) s, file write: ([0-9.]+) s", r.stdout)
            gp = re.search(r"GPU parse: ([0-9.]+) ms", r.stdout)
            runs.append({"seconds": dt, "read_s": float(io.group(1)) if io else None,
                         "write_s": float(io.group(2)) if io else None,
                         "gpu_parse_ms": float(gp.group(1)) if gp else None})
        best = min(runs, key=lambda x: x["seconds"])
        out_bytes = sum(os.path.getsize(path + "." + e) for e in ("dict", "occ", "parse", "last", "sai"))
        # the whole pipeline as one process: FASTA in, .bwt out (gpubigbwt.x = bigbwt's three stages in HBM)
        to_bwt = None
        if not a.no_pipeline and n_text <= (6 << 30):
            t0 = time.perf_counter()
            r = subprocess.run([pkg.pfp.BIGBWT_CLI_PATH, path, "-w", str(W), "-p", str(P), "-f"],
                               stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True)
            dt = time.perf_counter() - t0
            if r.returncode == 0:
                gp = re.search(r"GPU: parse ([0-9.]+) ms, bwtparse ([0-9.]+) ms \(\d+ rounds\), pfbwt ([0-9.]+) ms", r.stdout)
                to_bwt = {"seconds": dt, "value": n_text / dt / 1e9, "unit": UNIT, "bwt_bytes": os.path.getsize(path + ".bwt"),
                          "gpu_ms": [float(x) for x in gp.groups()] if gp else None,
                          "how": "wall clock of the gpubigbwt.x process: FASTA file -> parse -> bwtparse -> pfbwt -> .bwt file"}
            else:
                to_bwt = {"failed": r.returncode, "stderr": r.stderr[-300:]}
        return {"file_to_bwt": to_bwt,
                "value": n_text / best["seconds"] / 1e9, "unit": UNIT, "seconds": best["seconds"],
                "read_and_k0_s": best["read_s"], "gpu_parse_ms": best["gpu_parse_ms"], "write_s": best["write_s"],
                "other_s": best["seconds"] - (best["read_s"] or 0) - (best["write_s"] or 0) - (best["gpu_parse_ms"] or 0) / 1e3,
                "fasta_bytes": fsize, "text_bytes": n_text, "output_bytes": out_bytes, "runs": len(runs),
                "how": "wall clock of the gpuscan.x process (start, CUDA context, streaming read + K0, parse, streaming "
                       "write) on a page-cache-warm 60-column FASTA of the workload; 'other' = process start + CUDA init",
                "fasta_generation_s": gen_s}
    finally:
        shutil.rmtree(tmp, ignore_errors=True)


def main():
    a = parse_args()
    from __graft_entry__ import load_package
    pkg = load_package()
    synth = pkg.synth
    if a.impl == "reference":
        return reference_arm(a, synth)

    import torch
    import torch.distributed as dist
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device -- this framework has no CPU path")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    from bigbwt_b200 import shards
    job = shards.ShardedParser(local, world, rank, mode=a.merge)

    # ---- workload: this rank's shard of the text, generated in HBM ------------------------------
    if a.workload == "random":
        n_local = a.base_len * a.haplotypes
        text = synth.random_dna(n_local, SEED + 1000 * rank, device=dev)
    else:
        text = synth.pangenome_text(a.base_len, a.haplotypes, SEED, device=dev,
                                    first_hap=rank * a.haplotypes)
    torch.cuda.synchronize()
    n_local = text.numel()
    job.set_text(text)
    n_total = job.n_global

    stream = torch.cuda.Stream(device=dev)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def one_step():
        with torch.cuda.stream(stream):
            return job.parse_device(W, P, sai=True)

    for _ in range(a.warmup):
        one_step()
    barrier()
    clocks = ClockSampler(local)
    clocks.start()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    launches = 0
    scan_ms, stage_ms = [], {}
    barrier()
    ev0.record(stream)
    for _ in range(a.steps):
        st = one_step()
        launches += st["launches"]
        scan_ms.append(st["ms_scan"])
        for k, v in st.items():
            if k.startswith("ms_"):
                stage_ms[k] = stage_ms.get(k, 0.0) + v / a.steps
    ev1.record(stream)
    barrier()
    clk = clocks.stop()
    ms = ev0.elapsed_time(ev1)
    if world > 1:
        t = torch.tensor([ms], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t.item())
    value = n_total * a.steps / (ms * 1e-3) / 1e9
    last_stats = st
    per_rank = None
    if world > 1:                      # every rank's phase timeline (who waits for whom)
        gathered = [None] * world
        dist.all_gather_object(gathered, {k: round(v, 3) for k, v in stage_ms.items() if k.startswith("ms_phase_")})
        per_rank = {k: [g.get(k, 0.0) for g in gathered] for k in gathered[0]}
    dumped = None
    if a.dump_outputs:                 # before the legs below run the parser again
        dumped = dump_outputs(job.scanner.fetch(job.out), a.dump_outputs)

    # ---- the stages after the parse (SURVEY 8f rows 2-3), N = 1: text in HBM -> BWT in HBM ---------
    pipeline = None
    if world == 1 and not a.no_pipeline and a.workload == "pangenome" and n_local <= (6 << 30):
        pipeline = pipeline_to_bwt(pkg, local, text, cpu_sample_bytes=0 if a.no_cpu_baseline else min(n_local, a.base_len))

    # ---- e2e: host buffers in, host buffers out ------------------------------------------------
    e2e = None
    host = None
    if not a.no_e2e:
        host = torch.empty(n_local, dtype=torch.uint8, pin_memory=True)
        host.copy_(text)
        torch.cuda.synchronize()
        job.release_text()
        del text
        torch.cuda.empty_cache()
        h2d = d2h = 0
        es = max(1, a.e2e_steps)
        ms_h2d, ms_d2h = [], []
        for _ in range(2):
            job.parse_host(host, W, P, sai=True)
        barrier()
        t0 = time.perf_counter()
        for _ in range(es):
            st2 = job.parse_host(host, W, P, sai=True)
            h2d, d2h = st2["h2d_bytes"], st2["d2h_bytes"]
            ms_h2d.append(st2.get("ms_h2d", 0.0))
            ms_d2h.append(st2.get("ms_d2h", 0.0))
        barrier()
        dt = time.perf_counter() - t0
        if world > 1:
            t = torch.tensor([dt], device=dev, dtype=torch.float64)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            dt = float(t.item())
        e2e = {"value": n_total * es / dt / 1e9, "unit": UNIT, "h2d_bytes_per_step": h2d,
               "d2h_bytes_per_step": d2h, "steps": es, "warmup": 2, "ms_per_step": 1e3 * dt / es,
               "ms_h2d": sum(ms_h2d) / es, "ms_d2h": sum(ms_d2h) / es,
               "h2d_gbs": (h2d / (sum(ms_h2d) / es) / 1e6) if sum(ms_h2d) > 0 else None,
               "how": "pfpb200_parse_host: pinned host text -> H2D -> parse -> D2H of all five outputs"}
        job.release_text()
        torch.cuda.empty_cache()

    # ---- parity of the timed code path (outside every timed region) -------------------------------
    parity = None
    if not a.no_parity:
        parity = parity_check(job, pkg, synth, world, rank, local, dev, a.merge)

    t2 = None
    if world == 1 and not a.no_t2 and a.workload == "pangenome":
        job.release_text()
        torch.cuda.empty_cache()
        t2 = t2_file_to_files(a, pkg, synth, dev)

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    # ---- roofline of the dominant kernel (K1 scan): 1 byte read + 1 bit written per position ---
    peak, peak_src = load_peaks()
    scan_ms_avg = sum(scan_ms) / len(scan_ms)
    scan_bytes = n_local * (1.0 + 1.0 / 8.0)
    achieved = scan_bytes / (scan_ms_avg * 1e-3) / 1e9
    traffic = load_traffic(n_local)
    roofline = {"kernel": scan_kernel_name(), "bound": "hbm", "achieved": achieved, "peak": peak,
                "unit": "GB/s", "frac": achieved / peak, "traffic": traffic, "peak_source": peak_src,
                "alg_bytes_per_launch": scan_bytes, "ms_per_launch": scan_ms_avg,
                "share_of_step": scan_ms_avg / (ms / a.steps),
                "whole_path": {"alg_bytes_per_step": last_stats["alg_bytes"],
                               "achieved": last_stats["alg_bytes"] * a.steps / (ms * 1e-3) / 1e9,
                               "frac": last_stats["alg_bytes"] * a.steps / (ms * 1e-3) / 1e9 / (peak * world)}}

    # ---- CPU baseline: the reference's scanner on a bounded prefix, host cores of this box ------
    cpu = None
    if not a.no_cpu_baseline and world == 1:
        threads = os.cpu_count() or 1
        text_np, sample = cpu_sample_text(a, synth)
        tmp = tempfile.mkdtemp(prefix="pfpbench_")
        try:
            secs, kind, how, cores = run_reference_scanner(text_np, threads, tmp, 1)
        finally:
            shutil.rmtree(tmp, ignore_errors=True)
        cpu = {"value": text_np.size / secs[0] / 1e9, "unit": UNIT, "cores": cores, "kind": kind,
               "sample": f"{how}; {sample}; wall clock {secs[0]:.2f} s"}

    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": a.steps,
        "warmup": a.warmup, "ms_per_step": ms / a.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "u8/u32/u64 integer", "data": "synthetic",
        "config": workload_config(a, world),
        "workload_stats": {"text_bytes_total": n_total, "text_bytes_per_gpu": n_local,
                           "phrases": last_stats["n_phrases"], "distinct": last_stats["n_distinct"],
                           "dict_bytes": last_stats["dict_bytes"], "rank_rounds": last_stats["rank_rounds"]},
        "roofline": roofline, "cpu_baseline": cpu, "e2e": e2e, "gpu_launches": launches, "clocks": clk,
        "stages_ms": stage_ms,
    }
    if per_rank:
        line["per_rank_phase_ms"] = per_rank
    if parity is not None:
        line["parity_check"] = parity
    if t2 is not None:
        line["t2_file_to_files"] = t2
    if pipeline is not None:
        line["pipeline_to_bwt"] = pipeline
    if dumped is not None:
        line["dump_outputs"] = {"dir": a.dump_outputs, "length_and_stored": dumped}
    print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()
    if parity is not None and not parity["ok"]:
        raise SystemExit(f"bench.py: parity check FAILED: {parity['mismatch']} differ")


if __name__ == "__main__":
    main()
