#!/usr/bin/env python
"""bench.py -- GB/s scanned by the match loop of stealth/grab (reference grab.cc:175-213) on a B200.

  python bench.py [--gpus N --steps K --warmup W]                 our engine (1 process per GPU)
  python bench.py --impl reference [...]                          grab master (PCRE2-JIT shim) on the host cores
  python bench.py [...] --dump-outputs DIR                        also writes the records of the last timed step as .npy

One JSON line on stdout (rank 0).  The headline (`value`, `roofline`, `e2e`, `cpu_baseline`) is BASELINE.json configs[1]:
a literal (-S semantics) over a synthetic corpus of 1 MiB files, 64 GiB per GPU, device resident, all offsets (-O -l).
`configs` carries the same measurements for every BASELINE config (SURVEY.md 8(d) C1..C5), each with its own pattern,
corpus shape, scan mode, kernel GB/s and fraction of the measured HBM peak, read probe of the same buffer, resolve
time, parity against the oracle on regenerated sample files and the unmodified reference on the host cores.

Contract notes:
  value    whole-job GB/s with the corpus already in HBM (inputs 64 GiB >> 126 MB L2, so no flush needed)
  e2e      the same metric through gscan_scan_batch() with HOST buffers: H2D + scan + D2H inside the timed region
  roofline scan kernel only: algorithmic bytes (1 B read per corpus byte, SURVEY.md 8(d)) / CUDA-event kernel time
  cpu_baseline  the unmodified reference (oracle/_ref/grab_ref) timed on this box's host cores on a bounded sample
A parity MISMATCH anywhere drops `value`, sets "invalid" and makes the exit code non-zero.
"""
import argparse
import ctypes
import json
import os
import shutil
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

GiB = 1 << 30
MiB = 1 << 20
PATTERN = "foobardoesexist"      # literal; planted once per 64 files (= per 64 MiB) + natural hits (none expected)
NEEDLE_EVERY = 64
SEED = 2
FILE_LEN = 1 << 20
DUMP_BYTES = 60 * MiB  # what --dump-outputs writes at most (64 MB with the .npy headers)
REF_BIN = os.path.join(ROOT, "oracle", "_ref", "grab_ref")
ENGINE_LABEL = "grab master + PCRE2 10.42 JIT via oracle/shim (NOT hyperscan: no -H source or library available)"


def ctypes_memmove(dst, src, n):
    ctypes.memmove(ctypes.c_void_p(dst), ctypes.c_void_p(src), n)


def log(*a):
    print(*a, file=sys.stderr, flush=True)


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md recipe):
    one nvidia-smi process looping every 20 ms, started just before and stopped just after."""

    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap,power.draw")

    def __init__(self, index):
        self.index, self.rows, self.p = index, [], None

    def start(self):
        try:
            self.p = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits",
                                       "-lms", "20"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL)
            time.sleep(0.15)  # first sample lands before the timed region starts
        except Exception:
            self.p = None

    def stop(self):
        if not self.p:
            return
        time.sleep(0.03)
        self.p.terminate()
        try:
            out = self.p.communicate(timeout=5)[0].decode()
        except Exception:
            out = ""
        for line in out.splitlines():
            r = [x.strip() for x in line.split(",")]
            if len(r) >= 6 and r[0].isdigit():
                self.rows.append(r)

    def summary(self):
        if not self.rows:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["unavailable"]}
        sm = sorted(int(r[0]) for r in self.rows)
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(r[2 + i].lower().startswith("active") for r in self.rows)]
        pw = [float(r[6]) for r in self.rows if len(r) > 6 and r[6].replace(".", "", 1).isdigit()]
        return {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": int(self.rows[0][1]) if self.rows[0][1].isdigit() else None,
                "reasons": reasons, "samples": len(self.rows), "power_w_max": max(pw) if pw else None}


# ------------------------------------------------------------------------------------------------
# the five BASELINE.json configs (SURVEY.md 8(d)).  Shapes are per GPU; files are sharded by rank (weak scaling).
# ------------------------------------------------------------------------------------------------
def baseline_configs():
    import corpus
    return [
        {"key": "configs[0]", "what": "literal 'foobardoesnotexist' over one 256 MiB file, first match only (-s): a full scan, 0 matches",
         "pattern": "foobardoesnotexist", "literal": True, "mode": "FIRST", "seed": 1, "file_len": 256 * MiB, "n_files": 1,
         "needle": None, "cpu_args": ["-s"], "cpu_cores": 1, "cpu_bytes": 256 * MiB},
        {"key": "configs[1]", "what": "literal (-S semantics) over a corpus of 1 MiB files, 64 GiB per GPU, all offsets (-O -l)",
         "pattern": PATTERN, "literal": True, "mode": "ALL", "seed": SEED, "file_len": FILE_LEN, "n_files": 65536,
         "needle": PATTERN, "cpu_args": ["-r", "-O", "-l"], "cpu_cores": None, "cpu_bytes": 16 * GiB},
        {"key": "configs[2]", "what": "PCRE alternation foo|bar|baz|quux (non-capturing spelling: with capturing parentheses the reference prints "
                                      "nothing, SURVEY.md Q2) over the 64 GiB corpus, all offsets (-O -l)",
         "pattern": "foo|bar|baz|quux", "literal": False, "mode": "ALL", "seed": SEED, "file_len": FILE_LEN, "n_files": 65536,
         "needle": PATTERN, "cpu_args": ["-r", "-O", "-l"], "cpu_cores": None, "cpu_bytes": 16 * GiB},
        {"key": "configs[3]", "what": "char-class run [A-Za-z0-9_]{16,} over 128 GiB sharded across 8 GPUs = 16 GiB of 1 MiB files per GPU",
         "pattern": "[A-Za-z0-9_]{16,}", "literal": False, "mode": "ALL", "seed": SEED, "file_len": FILE_LEN, "n_files": 16384,
         "needle": PATTERN, "cpu_args": ["-r", "-O", "-l"], "cpu_cores": None, "cpu_bytes": 16 * GiB},
        {"key": "configs[4]", "what": "100 literals (3-5 lowercase letters, seeded) over 256 GiB of 16 KiB files across 8 GPUs = 2 097 152 files "
                                      "/ 32 GiB per GPU; at N > 1 the (file id, offset) records are gathered on rank 0 over NCCL inside the timed region",
         "pattern": corpus.literals100(), "literal": False, "mode": "ALL", "seed": 5, "file_len": 16384, "n_files": 2097152,
         "needle": None, "cpu_args": ["-r", "-O", "-l"], "cpu_cores": None, "cpu_bytes": 2 * GiB, "gather": True},
    ]


def _parity_job(job):
    """(seed, file_id, file_len, needle, pattern, literal, mode) -> (file_id, [starts]) from the oracle on the regenerated
    file (worker process: tests/corpus.py twin of the device generator + oracle/libgrab_oracle.so)."""
    import corpus
    import oracle_py as O
    seed, fid, flen, needle, pattern, literal, mode = job
    data = corpus.synth_file(seed, fid, flen, needle.encode() if needle else None, NEEDLE_EVERY if needle else 0).tobytes()
    o = O.Regex(pattern, literal=literal)
    return fid, [s for s, _ in o.scan_window(data, mode={"ALL": O.MODE_ALL, "FIRST": O.MODE_FIRST}[mode])]


def _range_job(job):
    import corpus
    seed, fid, off, n = job
    return off, corpus.synth_range(seed, fid, off, n).tobytes()


def oracle_parity(cfg, first_id, got, pool, n_sample=64):
    """Compares the GPU records of `n_sample` seeded files (plus every needle file among the first 4096) with the oracle on
    the CPU-regenerated bytes.  Returns (ok, files checked)."""
    import numpy as np
    n = cfg["n_files"]
    if cfg["file_len"] >= 64 * MiB:
        # one big file: regenerate it piecewise in parallel, scan once
        import oracle_py as O
        ok = True
        for f in range(n):
            parts = dict(pool.map(_range_job, [(cfg["seed"], first_id + f, o, min(4 * MiB, cfg["file_len"] - o)) for o in range(0, cfg["file_len"], 4 * MiB)]))
            data = b"".join(parts[o] for o in sorted(parts))
            want = [s for s, _ in O.Regex(cfg["pattern"], literal=cfg["literal"]).scan_window(
                data, mode={"ALL": O.MODE_ALL, "FIRST": O.MODE_FIRST}[cfg["mode"]])]
            if cfg["literal"]:  # second opinion that shares no code with the oracle
                first = data.find(cfg["pattern"].encode())
                ok = ok and ((first < 0 and not want) or (want and want[0] == first))
            ok = ok and want == got.get(first_id + f, [])
        return ok, n
    rng = np.random.default_rng(cfg["seed"] * 1000 + first_id % 997)
    ids = set(int(x) for x in rng.choice(n, size=min(n_sample, n), replace=False))
    ids |= {0, n - 1}
    if cfg["needle"]:
        ids |= set(range(NEEDLE_EVERY // 2, min(n, 512), NEEDLE_EVERY))
    jobs = [(cfg["seed"], first_id + f, cfg["file_len"], cfg["needle"], cfg["pattern"], cfg["literal"], cfg["mode"]) for f in sorted(ids)]
    ok = True
    for fid, want in pool.imap_unordered(_parity_job, jobs, chunksize=1):
        if want != got.get(fid, []):
            ok = False
            log("bench: PARITY MISMATCH %s file %d: oracle %s... engine %s..." % (cfg["key"], fid, want[:4], got.get(fid, [])[:4]))
    return ok, len(jobs)


class records_by_file:
    """The engine's records (sorted by file id, then offset) looked up per file without building a dict of millions."""

    def __init__(self, r):
        self.fid, self.start = r["file_id"], r["start"]

    def get(self, f, default=None):
        import numpy as np
        lo, hi = np.searchsorted(self.fid, f, side="left"), np.searchsorted(self.fid, f, side="right")
        return self.start[lo:hi].tolist() if hi > lo else ([] if default is None else default)

    def __len__(self):
        return len(self.fid)


def dump_records(r, out_dir, prefix, max_bytes):
    """The records a caller of the scan receives, one float64 array per field (exact: offsets and ids stay below 2**53),
    so that two builds can be compared field for field.  Above `max_bytes` a fixed-seed sample of the records is written,
    with the sampled row numbers as `sample_rows`."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    fields = ("file_id", "start", "match_len")
    rows = None
    if len(r) * 8 * len(fields) > max_bytes:
        keep = max_bytes // (8 * (len(fields) + 1))
        rows = np.sort(np.random.default_rng(0).choice(len(r), size=keep, replace=False))
        r = r[rows]
        np.save(os.path.join(out_dir, prefix + "sample_rows.npy"), rows.astype(np.float64))
    for f in fields:
        np.save(os.path.join(out_dir, prefix + f + ".npy"), r[f].astype(np.float64))
    log("bench: wrote %d%s records to %s" % (len(r), "" if rows is None else " sampled", out_dir))


# ------------------------------------------------------------------------------------------------
# CPU reference (the unmodified grab sources, oracle/_ref/grab_ref)
# ------------------------------------------------------------------------------------------------
def usable_cores():
    try:
        return len(os.sched_getaffinity(0))
    except Exception:
        return os.cpu_count() or 1


def reference_cores():
    # grab pins thread i to CPU i (main.cc:200-215): every CPU 0..n-1 must be in our affinity mask
    try:
        aff = sorted(os.sched_getaffinity(0))
        n = 0
        while n < len(aff) and aff[n] == n:
            n += 1
        return max(1, n)
    except Exception:
        return usable_cores()


def tmp_base(need_bytes):
    """tmpfs if it has room for the sample (page cache warm by construction), else the default temp dir."""
    try:
        st = os.statvfs("/dev/shm")
        if st.f_bavail * st.f_frsize > need_bytes * 1.25 + GiB:
            return "/dev/shm"
    except Exception:
        pass
    return None


def _gen_file(args):
    import corpus
    d, seed, fid, flen, needle = args
    corpus.synth_file(seed, fid, flen, needle.encode() if needle else None, NEEDLE_EVERY if needle else 0).tofile(os.path.join(d, "f%07d" % fid))
    return fid


def materialise(cfg, n_files, first_id=0, from_device=None, pool=None):
    """Writes files [first_id, first_id + n_files) of a config's corpus under a tmp dir; returns the path."""
    flen = cfg["file_len"]
    d = tempfile.mkdtemp(prefix="gscan_bench_", dir=tmp_base(n_files * flen))
    if from_device is not None:
        ctx, dptr = from_device
        step = max(1, (256 * MiB) // flen)
        for lo in range(0, n_files, step):
            k = min(step, n_files - lo)
            blob = ctx.d2h(dptr + lo * flen, k * flen)
            for i in range(k):
                blob[i * flen:(i + 1) * flen].tofile(os.path.join(d, "f%07d" % (first_id + lo + i)))
    else:
        jobs = [(d, cfg["seed"], first_id + f, flen, cfg["needle"]) for f in range(n_files)]
        if pool is None:
            import multiprocessing as mp
            with mp.Pool(min(64, usable_cores())) as p:
                list(p.imap_unordered(_gen_file, jobs, chunksize=8))
        else:
            list(pool.imap_unordered(_gen_file, jobs, chunksize=8))
    return d


def time_reference(cfg, path, cores, repeats=1):
    """One grab_ref run per repeat over `path`, stdout -> /dev/null; returns the list of wall times."""
    args = [REF_BIN] + (["-n", str(cores)] if cores > 1 else []) + list(cfg["cpu_args"]) + [cfg["pattern"], path]
    out = []
    for _ in range(repeats):
        t0 = time.perf_counter()
        p = subprocess.run(args, stdout=subprocess.DEVNULL, stderr=subprocess.PIPE)
        dt = time.perf_counter() - t0
        if p.returncode != 0:
            raise RuntimeError("grab_ref failed: %s" % p.stderr.decode()[:200])
        out.append(dt)
    return out


def median(v):
    v = sorted(v)
    return v[len(v) // 2]


def cpu_arm(cfg, ctx_dptr, pool, repeats=3, with_one_core=True):
    """The reference on this box's host cores for one config: a bounded sample of the same corpus on tmpfs."""
    if not os.path.exists(REF_BIN):
        return {"value": None, "unit": "GB/s", "cores": 0, "kind": "reference", "sample": "oracle/_ref/grab_ref missing"}
    flen = cfg["file_len"]
    nf = max(1, min(cfg["n_files"], cfg["cpu_bytes"] // flen))
    base = tmp_base(nf * flen)
    if base is None and nf * flen > 4 * GiB:  # no roomy tmpfs: keep the sample small
        nf = max(1, (4 * GiB) // flen)
    d = materialise(cfg, nf, from_device=ctx_dptr)
    try:
        cores = cfg["cpu_cores"] or reference_cores()
        path = os.path.join(d, "f%07d" % 0) if cfg["n_files"] == 1 else d
        time_reference(cfg, path, cores, 1)  # warm-up (page cache, binary)
        ts = time_reference(cfg, path, cores, repeats)
        res = {"value": nf * flen / median(ts) / 1e9, "best": nf * flen / min(ts) / 1e9, "unit": "GB/s", "cores": cores, "kind": "reference",
               "sample": "grab_ref %s%s over %d file(s) x %d B = %.2f GiB on %s, page cache warm, median of %d runs" %
                         ("-n %d " % cores if cores > 1 else "", " ".join(cfg["cpu_args"]), nf, flen, nf * flen / GiB, "tmpfs" if d.startswith("/dev/shm") else "tmp", repeats)}
        if with_one_core and cores > 1:
            sub = max(1, min(nf, (1 * GiB) // flen))
            sd = os.path.join(d, "one")
            os.mkdir(sd)
            for f in sorted(os.listdir(d))[:sub]:
                if f != "one":
                    os.link(os.path.join(d, f), os.path.join(sd, f))
            res["one_core_value"] = sub * flen / min(time_reference(cfg, sd, 1, 2)) / 1e9
        return res
    finally:
        shutil.rmtree(d, ignore_errors=True)


def run_reference(a, rank, world):
    """--impl reference: configs[1] on the host cores, each step one pass over a bounded sample of the corpus."""
    if rank != 0:
        return
    cfg = baseline_configs()[1]
    line = {"impl": "reference", "metric": "GB/s scanned", "unit": "GB/s", "n_gpus": a.gpus, "steps": a.steps, "warmup": a.warmup,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u8", "data": "synthetic"}
    if not os.path.exists(REF_BIN):
        line["unavailable"] = "oracle/_ref/grab_ref is not built (needs /root/reference at build time)"
        print(json.dumps(line))
        return
    n_files = a.ref_files
    if tmp_base(n_files * FILE_LEN) is None:
        n_files = min(n_files, 4096)
    d = materialise(cfg, n_files)
    try:
        cores = reference_cores()
        time_reference(cfg, d, cores, max(1, a.warmup))
        ts = time_reference(cfg, d, cores, a.steps)
        sub = os.path.join(d, "one")
        os.mkdir(sub)
        for f in sorted(os.listdir(d))[:1024]:
            if f != "one":
                os.link(os.path.join(d, f), os.path.join(sub, f))
        one = None if a.quick else min(time_reference(cfg, sub, 1, 2))
    finally:
        shutil.rmtree(d, ignore_errors=True)
    nbytes = n_files * FILE_LEN
    dt = sum(ts) / len(ts)
    gbs = nbytes / dt / 1e9
    line.update({
        "value": gbs, "ms_per_step": dt * 1e3, "median_value": nbytes / median(ts) / 1e9, "best_value": nbytes / min(ts) / 1e9,
        "config": {"workload": "BASELINE configs[1]: literal over a corpus of 1 MiB files; reference arm scans a bounded sample",
                   "pattern": PATTERN, "files": n_files, "file_bytes": FILE_LEN, "mode": "-n %d -r -O -l" % cores, "engine": ENGINE_LABEL},
        "cpu_baseline": {"value": gbs, "unit": "GB/s", "cores": cores, "kind": "reference",
                         "sample": "%d files x 1 MiB (%.1f GiB) on tmpfs, page cache warm, mean of %d steps; 1-core (1 GiB): %s GB/s" %
                                   (n_files, nbytes / GiB, a.steps, ("%.2f" % (1024 * FILE_LEN / one / 1e9)) if one else "n/a")},
        "e2e": {"value": gbs, "unit": "GB/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    })
    print(json.dumps(line))


def e2e_all_ranks(scan, want_bytes, steps, world, rank, torch, dist, device, sync_all):
    """The timed end-to-end region at N > 1: every rank runs `scan()` (one gscan_scan_batch over its host sample) `steps`
    times between barriers.  Returns (seconds per step of the slowest rank, records per step on this rank, results equal
    `want_bytes` on every rank), or None when any rank could not run it (scan is None there, or it raised): every rank
    reaches every collective whatever happens on the others, so a local failure can drop the number but never hang the job."""
    failed, bad, n_rec = (1.0 if scan is None else 0.0), 0.0, 0
    sync_all()
    t0 = time.perf_counter()
    try:
        if not failed:
            out = None
            for _ in range(steps):
                out = scan()
            n_rec = len(out)
            bad = 0.0 if out.tobytes() == want_bytes else 1.0
    except Exception as ex:  # noqa: BLE001
        failed = 1.0
        sys.stderr.write("bench: e2e leg failed on rank %d: %r\n" % (rank, ex))
    if device == "cuda":
        torch.cuda.synchronize()
    dt = (time.perf_counter() - t0) / max(steps, 1)
    sync_all()
    t = torch.tensor([dt, bad, failed], dtype=torch.float64, device=device)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    if float(t[2].item()) != 0.0:
        return None
    return float(t[0].item()), n_rec, float(t[1].item()) == 0.0


def load_traffic(kernel_key, bytes_per_launch):
    """dram__bytes_read.sum + dram__bytes_write.sum per launch of this kernel from a committed ncu capture of the SAME
    workload (profiles/r02_traffic.json, written by tools/ncu_traffic.py from an `ncu --set full` run); None when no
    capture of exactly this launch size exists -- never a scaled constant."""
    try:
        t = json.load(open(os.path.join(ROOT, "profiles", "r02_traffic.json")))
        e = t.get(kernel_key)
        if e and int(e["algorithmic_bytes_per_launch"]) == int(bytes_per_launch):
            return float(e["dram_bytes_per_launch"]), e.get("source")
    except Exception:
        pass
    return None, None


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--corpus-gib", type=float, default=64.0, help="device-resident corpus per GPU (scales every config)")
    ap.add_argument("--e2e-gib", type=float, default=4.0, help="host-resident sample for the end-to-end leg")
    ap.add_argument("--ref-files", type=int, default=16384, help="files of the corpus the CPU reference arm scans per step")
    ap.add_argument("--config-steps", type=int, default=5, help="timed steps of each entry of `configs`")
    ap.add_argument("--only", default="", help="comma list of config indices to run in `configs` (default: all)")
    ap.add_argument("--quick", action="store_true", help="skip the cpu baselines and the e2e legs")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the records of the headline's last timed step to DIR/<field>.npy "
                    "(float64; a seeded sample of the records above %d MiB in all)" % (DUMP_BYTES // MiB))
    a = ap.parse_args()
    if a.steps < 1:
        ap.error("--steps must be at least 1")

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if a.impl == "reference":
        return run_reference(a, rank, world)
    # stdout carries exactly one JSON line: whatever libraries print there (NCCL's version banner ignores NCCL_DEBUG_FILE)
    # goes to stderr instead -- the real stdout is kept aside for the line
    sys.stdout.flush()
    json_fd = os.dup(1)
    os.dup2(2, 1)

    import multiprocessing as mp
    pool = mp.get_context("spawn").Pool(min(32, max(2, usable_cores() // max(world, 1))))  # before CUDA is touched: parity workers

    import numpy as np
    import torch
    import torch.distributed as dist
    import grab_b200 as G
    from grab_b200 import shard

    torch.cuda.set_device(local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        # stdout carries exactly one JSON line: NCCL's own log (version banner, NCCL_DEBUG output) goes to stderr
        os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    ctx = G.Context(local_rank)
    modes = {"ALL": G.MODE_ALL, "FIRST": G.MODE_FIRST, "LINE": G.MODE_LINE}

    free_b, _ = torch.cuda.mem_get_info()
    scale = min(1.0, a.corpus_gib / 64.0)
    buf_bytes = int(64 * GiB * scale)
    if buf_bytes > free_b - 12 * GiB:
        # the corpus is never shrunk to fit: the arguments alone fix the workload, so that runs stay comparable
        sys.exit("bench: a %.1f GiB corpus and 12 GiB of working memory do not fit in the %.1f GiB free on GPU %d: "
                 "pass a smaller --corpus-gib" % (buf_bytes / GiB, free_b / GiB, local_rank))
    dptr = ctx.device_alloc(buf_bytes)
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    peak = float(peaks.get("hbm_gbs", 6650.0))
    peak_src = "MEASURED_PEAKS.json hbm_gbs (copy, burst)" if peaks else "fallback 6650 GB/s"

    def sync_all():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    def max_over_ranks(x):
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def all_ok(ok):
        if world == 1:
            return ok
        t = torch.tensor([0.0 if ok else 1.0], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item()) == 0.0

    cfgs = baseline_configs()
    for c in cfgs:  # scale the shapes with --corpus-gib (tests, small GPUs); 1.0 at the default
        if c["n_files"] > 1:
            c["n_files"] = max(64, int(c["n_files"] * scale))
    resident = {"key": None}

    def make_resident(cfg):
        """Device corpus of a config: files [rank * n, (rank + 1) * n) of its seeded corpus (weak scaling, reference main.cc:94)."""
        n, first_id = cfg["n_files"], rank * cfg["n_files"]
        key = (cfg["seed"], cfg["file_len"], cfg["needle"], first_id)  # rank r's shard starts at file r * n: part of the identity
        if resident["key"] != key or resident.get("n", 0) < n:
            ctx.synth_corpus(dptr, cfg["seed"], first_id, n, cfg["file_len"],
                             needle=cfg["needle"].encode() if cfg["needle"] else None, needle_every=NEEDLE_EVERY if cfg["needle"] else 0)
            resident.update(key=key, n=n)
        return first_id

    # ---------------------------------------------------------------------------------------
    # headline: configs[1]
    # ---------------------------------------------------------------------------------------
    H = cfgs[1]
    n_files = H["n_files"]
    corpus_bytes = n_files * FILE_LEN
    first_id = make_resident(H)
    pat = G.Pattern(H["pattern"], literal=True)
    batch = ctx.batch_create(G.Context.device_units(dptr, n_files, FILE_LEN, first_file_id=first_id))
    state = {"counts": None, "pending": None}

    def step():
        # the one collective of the path: an NCCL all-gather of the per-rank match counts, once per step.  It is
        # enqueued right after the scan and collected one step later (the last one before the timed region ends), so
        # its launch/completion latency and the rank skew it exposes overlap the next scan instead of adding to it
        r = ctx.batch_scan(pat, batch, G.MODE_ALL, copy=False)  # a view of the pinned result buffer: no per-record host work
        h = shard.gather_counts_start(len(r))
        if state["pending"] is not None:
            state["counts"] = state["pending"].finish()
        state["pending"] = h
        return r

    def drain():
        if state["pending"] is not None:
            state["counts"] = state["pending"].finish()
            state["pending"] = None

    for _ in range(max(a.warmup, 1)):
        step()
    drain()

    # ---- timed region: K resident steps ----
    sampler = ClockSampler(local_rank)
    kernel_ms, step_ms, launches = [], [], 0
    sampler.start()
    sync_all()
    t0 = time.perf_counter()
    tp = t0
    for _ in range(a.steps):
        r = step()
        st = ctx.stats()
        kernel_ms.append(st["scan_kernel_ms"])
        launches += st["total_launches"]
        tn = time.perf_counter()
        step_ms.append((tn - tp) * 1e3)
        tp = tn
    drain()  # every step's all-gather has completed inside the timed region
    sync_all()
    dt = max_over_ranks(time.perf_counter() - t0)
    sampler.stop()
    ms_per_step = dt / a.steps * 1e3
    value = world * corpus_bytes / (dt / a.steps) / 1e9

    # ---- parity gate (outside the timed region, on the records of the last timed step): every planted needle +
    # the oracle on >= 64 regenerated files ----
    import corpus
    r = r.copy()
    if a.dump_outputs:
        dump_records(r, a.dump_outputs, "" if world == 1 else "rank%d_" % rank, DUMP_BYTES // world)
    ids = np.arange(first_id, first_id + n_files)
    planted = ids[ids % NEEDLE_EVERY == NEEDLE_EVERY // 2]
    want = {int(f): corpus.needle_offset(SEED, int(f), FILE_LEN, len(PATTERN)) for f in planted}
    got = records_by_file(r)
    parity = all(o in got.get(f, []) for f, o in want.items())
    ok, n_checked = oracle_parity(H, first_id, got, pool)
    parity = all_ok(parity and ok)
    extra = len(got) - len(want)

    # ---- roofline of the scan kernel ----
    k_ms = float(np.mean(kernel_ms))
    achieved = corpus_bytes / (k_ms * 1e-3) / 1e9
    probe_ms = min(ctx.read_probe(dptr, corpus_bytes)[0] for _ in range(3))
    traffic, traffic_src = load_traffic("configs[1]", corpus_bytes)
    roofline = {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "traffic": traffic,
                "traffic_source": traffic_src, "peak_source": peak_src,
                "kernel": "scan_kernel<FixedEngine<D,1>>", "kernel_ms": k_ms, "kernel_ms_median": float(np.median(kernel_ms)),
                "algorithmic_bytes_per_launch": corpus_bytes, "read_probe_gbs": corpus_bytes / (probe_ms * 1e-3) / 1e9}

    line = {"metric": "GB/s scanned", "value": value, "unit": "GB/s", "n_gpus": world, "steps": a.steps, "warmup": a.warmup,
            "ms_per_step": ms_per_step, "ms_per_step_median": float(np.median(step_ms)), "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u8",
            "data": "synthetic",
            "config": {"workload": "BASELINE configs[1]: literal (-S) over %.1f GiB/GPU synthetic corpus of 1 MiB files, all offsets (-O -l)" % (corpus_bytes / GiB),
                       "pattern": H["pattern"], "files_per_gpu": int(n_files), "file_bytes": FILE_LEN, "mode": "ALL",
                       "sharding": "files by rank, no data-path collective; one all-gather of match counts per step",
                       "l2": "inputs larger than L2 (%.0f GiB vs 126 MB), no flush" % (corpus_bytes / GiB)},
            "roofline": roofline, "clocks": sampler.summary(), "gpu_launches": launches,
            "parity": "ok" if parity else "MISMATCH", "parity_files_checked": int(n_checked + len(want)),
            "matches_per_step": int(state["counts"].sum()), "natural_hits": int(extra)}

    # ---------------------------------------------------------------------------------------
    # e2e: host buffers through gscan_scan_batch (H2D + scan + D2H inside the timed region)
    # ---------------------------------------------------------------------------------------
    e_files = int(min(a.e2e_gib * GiB, corpus_bytes) // FILE_LEN)
    if not a.quick:
        hptr, scan = None, None
        try:
            hptr = G.lib().gscan_host_alloc(e_files * FILE_LEN)
            if not hptr:
                raise RuntimeError("pinned allocation failed")
            G.lib().gscan_memcpy_d2h(ctx._h, hptr, dptr, e_files * FILE_LEN)
            hunits = np.zeros(e_files, dtype=G.UNIT_DTYPE)
            hunits["ptr"] = hptr + np.arange(e_files, dtype=np.uint64) * np.uint64(FILE_LEN)
            hunits["len"] = FILE_LEN
            hunits["file_id"] = first_id + np.arange(e_files, dtype=np.uint32)
            for _ in range(2):
                ctx.scan_units(pat, hunits)
            scan = lambda: ctx.scan_units(pat, hunits)  # noqa: E731
        except Exception as ex:  # noqa: BLE001
            log("bench: e2e leg failed on rank %d: %r" % (rank, ex))
        want_b = r[r["file_id"] < first_id + e_files].tobytes()
        if world == 1:
            res = None
            if scan is not None:
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                for _ in range(a.steps):
                    re2e = scan()
                torch.cuda.synchronize()
                res = ((time.perf_counter() - t0) / a.steps, len(re2e), re2e.tobytes() == want_b)
        else:
            res = e2e_all_ranks(scan, want_b, a.steps, world, rank, torch, dist, "cuda", sync_all)
        if res is not None:
            e_dt, n_rec, ok = res
            if not ok:
                line["parity"] = "MISMATCH(e2e)"
            line["e2e"] = {"value": world * e_files * FILE_LEN / e_dt / 1e9, "unit": "GB/s",
                           "h2d_bytes_per_step": int(world * (e_files * FILE_LEN + e_files * 32)),
                           "d2h_bytes_per_step": int(world * (n_rec * 16 + 24)),
                           "sample": "%d files x 1 MiB in pinned host memory per rank, %d rank(s), slowest rank" % (e_files, world)}
        if world == 1 and scan is not None:
            # the same call on PAGEABLE host memory (what the CLI's mmap windows are): staged by the engine's helper lanes
            pag = np.empty(e_files * FILE_LEN, dtype=np.uint8)
            ctypes_memmove(pag.ctypes.data, hptr, e_files * FILE_LEN)
            punits = hunits.copy()
            punits["ptr"] = pag.ctypes.data + np.arange(e_files, dtype=np.uint64) * np.uint64(FILE_LEN)
            ctx.scan_units(pat, punits)
            t0 = time.perf_counter()
            for _ in range(5):
                rp = ctx.scan_units(pat, punits)
            p_dt = (time.perf_counter() - t0) / 5
            if rp.tobytes() != want_b:
                line["parity"] = "MISMATCH(e2e pageable)"
            line["e2e"]["pageable_host_value"] = e_files * FILE_LEN / p_dt / 1e9
            del pag
        if hptr:
            G.lib().gscan_host_free(hptr)
    batch.free()

    # ---------------------------------------------------------------------------------------
    # every BASELINE config: kernel GB/s, fraction of the HBM peak, read probe, resolve, parity, CPU arm
    # ---------------------------------------------------------------------------------------
    only = set(int(x) for x in a.only.split(",") if x.strip() != "") if a.only else None
    entries = []
    for ci, cfg in enumerate(cfgs):
        if only is not None and ci not in only:
            continue
        n, flen = cfg["n_files"], cfg["file_len"]
        nbytes = n * flen
        fid0 = make_resident(cfg)
        p = G.Pattern(cfg["pattern"], literal=cfg["literal"])
        b = ctx.batch_create(G.Context.device_units(dptr, n, flen, first_file_id=fid0))
        mode = modes[cfg["mode"]]
        gather = bool(cfg.get("gather")) and world > 1
        pend = {"h": None, "last": None}

        def one_step():
            rr = ctx.batch_scan(p, b, mode, copy=False)
            if gather:
                # records of all ranks to rank 0 over NCCL, merged by file id: started after the scan, collected one
                # step later (the last one inside the timed region), like the count exchange of the headline
                h = shard.gather_matches_start(rr, dst=0, device_records=ctx.last_device_matches())
                if pend["h"] is not None:
                    pend["last"] = pend["h"].finish()
                pend["h"] = h
            return rr

        def drain_c():
            if pend["h"] is not None:
                pend["last"] = pend["h"].finish()
                pend["h"] = None

        for _ in range(2):
            rr = one_step()
        drain_c()
        rr = rr.copy()
        got_c = records_by_file(rr)
        ok, nchk = oracle_parity(cfg, fid0, got_c, pool)
        if gather and rank == 0 and pend["last"] is not None:
            mine = pend["last"][(pend["last"]["file_id"] >= fid0) & (pend["last"]["file_id"] < fid0 + n)]
            ok = ok and mine.tobytes() == rr.tobytes() and bool(np.all(np.diff(pend["last"]["file_id"].astype(np.int64)) >= 0))
        ok = all_ok(ok)
        kms, rms, nl = [], [], 0
        sync_all()
        t0 = time.perf_counter()
        for _ in range(a.config_steps):
            one_step()
            st = ctx.stats()
            kms.append(st["scan_kernel_ms"])
            rms.append(st["resolve_ms"])
            nl += st["total_launches"]
        drain_c()
        sync_all()
        c_dt = max_over_ranks(time.perf_counter() - t0) / a.config_steps
        k = float(np.mean(kms))
        pr_ms = min(ctx.read_probe(dptr, nbytes)[0] for _ in range(2))
        info = p.info
        tr, tr_src = load_traffic(cfg["key"], nbytes)
        e = {"config": cfg["key"], "what": cfg["what"], "pattern": cfg["pattern"] if len(cfg["pattern"]) <= 48 else cfg["pattern"][:45] + "...",
             "mode": cfg["mode"], "files_per_gpu": int(n), "file_bytes": int(flen), "bytes_per_gpu": int(nbytes), "steps": a.config_steps,
             "value": world * nbytes / c_dt / 1e9, "ms_per_step": c_dt * 1e3,
             "kernel_gbs": nbytes / (k * 1e-3) / 1e9, "kernel_ms": k, "kernel_ms_median": float(np.median(kms)), "frac": nbytes / (k * 1e-3) / 1e9 / peak,
             "read_probe_gbs": nbytes / (pr_ms * 1e-3) / 1e9, "resolve_ms": float(np.mean(rms)), "gpu_launches": int(nl),
             "matches_per_step": int(len(rr)), "engine": int(info["engine"]), "traffic": tr, "traffic_source": tr_src,
             "parity": "ok" if ok else "MISMATCH", "parity_files_checked": int(nchk)}
        if gather:
            e["gather"] = "records of %d ranks merged by file id on rank 0 (NCCL all-gather), started after each scan and collected one step later, inside the timed region" % world
            if rank == 0 and pend["last"] is not None:
                e["gathered_records"] = int(len(pend["last"]))
        if rank == 0 and not a.quick and world == 1:
            try:
                e["cpu_baseline"] = cpu_arm(cfg, (ctx, dptr), pool)
            except Exception as ex:  # noqa: BLE001
                e["cpu_baseline"] = {"value": None, "error": repr(ex)[:200]}
        entries.append(e)
        if not ok:
            line["parity"] = "MISMATCH(%s)" % cfg["key"]
        b.free()
        log("bench: %s %-24s kernel %7.0f GB/s (%.2f of peak), step %7.0f GB/s, resolve %.2f ms, parity %s" %
            (cfg["key"], e["pattern"][:24], e["kernel_gbs"], e["frac"], e["value"], e["resolve_ms"], e["parity"]))
    line["configs"] = entries
    for e in entries:  # the headline's cpu_baseline is configs[1]'s CPU arm
        if e["config"] == "configs[1]" and "cpu_baseline" in e:
            line["cpu_baseline"] = e["cpu_baseline"]
    line["cpu_engine"] = ENGINE_LABEL

    pool.terminate()
    ctx.device_free(dptr)
    ctx.close()
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    bad = line["parity"] != "ok"
    if bad:
        line["invalid"] = "parity gate failed: %s -- no value reported" % line["parity"]
        line["value"] = None
    if rank == 0:
        os.write(json_fd, (json.dumps(line) + "\n").encode())
    if bad:
        sys.exit(3)


if __name__ == "__main__":
    main()
