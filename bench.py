#!/usr/bin/env python
"""bench.py — BASELINE.json's metric: MB/s ingested end to end, TF-IDF (benchmarks/tf-idf-dampr.py)
on synthetic Zipf text, through the Dampr DSL on the B200 engine.

    python bench.py --gpus 1 --steps K --warmup W            # this engine
    python bench.py --impl reference --gpus 1 ...             # the reference's own CPU runner

A step = one complete run of the TF-IDF graph (len + tokenise/count + fold + cross + sink_tsv) over
the whole corpus (10 GB, V = 1e6, split evenly over the ranks: strong scaling).
  value / e2e   whole-job MB/s END TO END: the text starts in page-locked HOST memory, the host->device copies,
                every kernel, the exchange, the device->host fetch of the result table and the sink files
                are inside the timed region (max over ranks). This is BASELINE.json's metric.
  device_resident  the same job with the text already resident in HBM when the step starts (explains e2e:
                the difference is PCIe).
  roofline      the tokenise+combine kernel (dominant): algorithmic bytes = 1 B per input byte
                (SURVEY §8(d)), CUDA-event duration measured inside the timed steps, peak = measured HBM
                copy bandwidth (MEASURED_PEAKS.json).
  parity        after the timed loops the SAME graph runs on a line-aligned sample of the same corpus on the
                GPU(s) and through the CPU checker (the real reference from oracle/_ref when present, else
                oracle/cpu_runner.py); the sorted sink lines must be byte-identical or the run fails.
  extra         (1 GPU) the north-star's own stage and the other BASELINE configs: partition+sort of 1e8 and
                6.25e8 16-byte records (32*N/t against the HBM peak), merge / reduce, config 2 end to end,
                config 5 joins, the file-path e2e.
  cpu_baseline  the CPU arm on a bounded sample of the same corpus, all host cores.
"""
import argparse
import hashlib
import json
import math
import os
import re
import shutil
import subprocess
import sys
import tempfile
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import numpy as np

RX = re.compile(r"[^\w]+")
MB = 1e6
METRIC = "MB/s ingested end-to-end, TF-IDF 10 GB synthetic text, 1/2/4/8 GPU"
MEAN_LINE = 99.94  # mean synthetic line: 99.94 B at V = 1e6 (measured)
REF_TIMEOUT = 120  # seconds one run of the reference may take before the arm gives up on it


_T0 = time.time()


def progress(msg):
    """phase log on stderr (the JSON line is the only thing on stdout)"""
    print("[bench %7.1fs] %s" % (time.time() - _T0, msg), file=sys.stderr, flush=True)


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--gb", type=float, default=float(os.environ.get("DAMPR_BENCH_GB", "10")),
                    help="corpus size in GB (10 = the BASELINE config)")
    ap.add_argument("--vocab", type=int, default=1000000)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extra", action="store_true", help="skip the kv / join / file-path extras (1 GPU)")
    ap.add_argument("--no-parity", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the TF-IDF table of the last timed end-to-end step to DIR/*.npy (see dump_outputs)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    return args


def dist_env():
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    return rank, world, local


class ClockSampler(threading.Thread):
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        threading.Thread.__init__(self)
        self.daemon = True
        self.gpu = gpu_index
        self.samples = []
        self.stop_flag = threading.Event()

    def run(self):
        """In-process NVML sampling (spawning nvidia-smi every 200 ms stalls CUDA calls of this process
        for tens of ms); nvidia-smi is the fallback when pynvml is missing."""
        try:
            import pynvml
            pynvml.nvmlInit()
            h = pynvml.nvmlDeviceGetHandleByIndex(self.gpu)
            mx = pynvml.nvmlDeviceGetMaxClockInfo(h, pynvml.NVML_CLOCK_SM)
            R = pynvml
            bits = [("hw_slowdown", R.nvmlClocksThrottleReasonHwSlowdown),
                    ("hw_thermal_slowdown", R.nvmlClocksThrottleReasonHwThermalSlowdown),
                    ("sw_thermal_slowdown", R.nvmlClocksThrottleReasonSwThermalSlowdown),
                    ("sw_power_cap", R.nvmlClocksThrottleReasonSwPowerCap)]
            while not self.stop_flag.is_set():
                sm = pynvml.nvmlDeviceGetClockInfo(h, pynvml.NVML_CLOCK_SM)
                rs = pynvml.nvmlDeviceGetCurrentClocksThrottleReasons(h)
                row = [str(self.gpu), str(sm), str(mx), "", hex(rs)]
                row += ["Active" if rs & b else "Not Active" for _n, b in bits]
                self.samples.append(row)
                # NVML queries and CUDA calls share a driver lock: sample sparsely (2 Hz) so the
                # sampler itself does not stall the allocation calls of the timed steps
                self.stop_flag.wait(0.5)
            return
        except Exception:
            pass
        while not self.stop_flag.is_set():
            try:
                out = subprocess.run(["nvidia-smi", "-i", str(self.gpu), "--query-gpu=" + self.Q,
                                      "--format=csv,noheader,nounits"], capture_output=True, text=True,
                                     timeout=5).stdout.strip()
                if out:
                    self.samples.append([x.strip() for x in out.split(",")])
            except Exception:
                pass
            self.stop_flag.wait(0.2)

    def summary(self):
        sm = [float(s[1]) for s in self.samples if len(s) > 2 and s[1].replace(".", "").isdigit()]
        mx = [float(s[2]) for s in self.samples if len(s) > 2 and s[2].replace(".", "").isdigit()]
        reasons = set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for s in self.samples:
            for nm, v in zip(names, s[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(self.samples)}


def tfidf_job(Dampr, source_dataset, out_dir):
    """benchmarks/tf-idf-dampr.py:9-21 verbatim, on a given input dataset."""
    docs = Dampr.read_input(source_dataset)
    doc_freq = docs.flat_map(lambda x: set(RX.split(x.lower()))).count(reduce_buffer=float("inf"))
    idf = doc_freq.cross_right(docs.len(),
                               lambda df, total: (df[0], df[1], math.log(1 + (float(total) / df[1]))),
                               memory=True)
    return idf.sink_tsv(out_dir).run()


def measured_peak():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured"
    except Exception:
        return 6650.0, "fallback"


# ---- the CPU arms: the real reference (oracle/_ref, a separate process) or the oracle port ------------------------
def have_reference():
    return os.path.isdir(os.path.join(ROOT, "oracle", "_ref", "dampr"))


def run_cpu_tfidf(path, out_dir, n_procs, kind):
    """One TF-IDF run of the CPU arm on `path`; returns wall seconds (process start -> exit for the reference,
    like benchmarks/run.sh times it)."""
    shutil.rmtree(out_dir, ignore_errors=True)
    if kind == "reference":
        t0 = time.time()
        # the reference hangs when one of its workers dies (SURVEY B6): bound the run
        # own process group: on a timeout the reference's forked workers are killed with it
        proc = subprocess.Popen([sys.executable, os.path.join(ROOT, "oracle", "ref_tfidf.py"), path, out_dir, str(n_procs)],
                                cwd=tempfile.gettempdir(), stdout=subprocess.DEVNULL, stderr=subprocess.PIPE, text=True,
                                start_new_session=True)
        try:
            _out, err = proc.communicate(timeout=REF_TIMEOUT)
        except subprocess.TimeoutExpired:
            import signal
            try:
                os.killpg(proc.pid, signal.SIGKILL)
            except Exception:
                proc.kill()
            proc.wait()
            raise RuntimeError("the reference did not finish within %d s on this box" % REF_TIMEOUT)
        sec = time.time() - t0
        if proc.returncode != 0:
            raise RuntimeError("reference run failed: %s" % (err or "")[-2000:])
        return sec
    from oracle import cpu_runner
    sec, _n_terms, _n_lines = cpu_runner.timed_tfidf(path, out_dir, n_procs)
    return sec


_REF_STATE = {"broken": None, "procs": None}


def reference_procs(ncores):
    """settings.max_processes the unmodified reference finishes with on this box. Measured on the 128-core GPU boxes
    (gpurun_out/r2_refdiag.log): with its default (= all cores) the reference never returns — 48 MB of text, no output,
    no error, the open-file limit raised — while 32 and 8 worker processes finish in about a second. So the arm
    probes, on an 8 MB sample and with a short timeout, all cores first and then 64 / 32 / 16 / 8, and keeps the
    largest count that finishes. (The chunking of the script still follows cpu_count(); only the worker pool is capped.)"""
    global REF_TIMEOUT
    if _REF_STATE["procs"] is not None or _REF_STATE["broken"]:
        return _REF_STATE["procs"]
    from oracle import gen
    tmp = tempfile.mkdtemp(prefix="dampr_refprobe_")
    try:
        path = os.path.join(tmp, "probe.txt")
        data = np.frombuffer(gen.text(4321, 80000, V=50000), dtype=np.uint8)
        with open(path, "wb") as f:
            f.write(pad_sample(data, 0, lcm(64, ncores)))
        cands = []
        for c in (ncores, 64, 32, 16, 8, 1):
            if c <= ncores and c not in cands:
                cands.append(c)
        saved = REF_TIMEOUT
        REF_TIMEOUT = 12   # a count that works needs 1-2 s for the 8 MB sample
        try:
            for c in cands:
                try:
                    run_cpu_tfidf(path, os.path.join(tmp, "idfs"), c, "reference")
                    _REF_STATE["procs"] = c
                    break
                except Exception as e:
                    progress("reference with %d worker processes: %s" % (c, str(e)[:120]))
        finally:
            REF_TIMEOUT = saved
        if _REF_STATE["procs"] is None:
            _REF_STATE["broken"] = "the reference finished with no worker count tried (%s)" % cands
    finally:
        shutil.rmtree(tmp, ignore_errors=True)
    return _REF_STATE["procs"]


def cpu_arm(path, out_dir, n_procs):
    """The CPU arm on `path`: the unmodified reference when oracle/_ref is present and finishes on this box, else the
    oracle port. Returns (seconds, kind, note, processes used)."""
    if have_reference() and not _REF_STATE["broken"]:
        procs = reference_procs(n_procs)
        if procs:
            try:
                return run_cpu_tfidf(path, out_dir, procs, "reference"), "reference", None, procs
            except Exception as e:
                _REF_STATE["broken"] = str(e)[:300]
                progress("the reference failed here (%s): falling back to the oracle port" % _REF_STATE["broken"])
    return run_cpu_tfidf(path, out_dir, n_procs, "port"), "port", _REF_STATE["broken"], n_procs


def read_sink_lines(out_dir):
    lines = []
    for fn in sorted(os.listdir(out_dir)):
        with open(os.path.join(out_dir, fn), "rb") as f:
            lines.extend(f.read().split(b"\n"))
    return sorted(l for l in lines if l)


DUMP_LIMIT = 64 << 20  # bytes of .npy data dump_outputs writes at most


def dump_outputs(out_dir, dump_dir, suffix=""):
    """The sink_tsv table a TF-IDF step wrote to `out_dir` (term, document frequency, idf), as float64 columns in term
    order: term_hash.npy (the first 52 bits of the term's blake2b digest, exact in a float64), doc_freq.npy, idf.npy.
    A table larger than DUMP_LIMIT is cut to a seeded sample of rows (the same rows for the same table size)."""
    lines = read_sink_lines(out_dir)
    cols = {"term_hash": np.empty(len(lines)), "doc_freq": np.empty(len(lines)), "idf": np.empty(len(lines))}
    for i, l in enumerate(lines):
        term, df, idf = l.split(b"\t")
        cols["term_hash"][i] = int.from_bytes(hashlib.blake2b(term, digest_size=8).digest(), "little") >> 12
        cols["doc_freq"][i] = int(df)
        cols["idf"][i] = float(idf)
    rows = DUMP_LIMIT // (8 * len(cols))
    if len(lines) > rows:
        keep = np.sort(np.random.default_rng(0).choice(len(lines), rows, replace=False))
        cols = {k: v[keep] for k, v in cols.items()}
    os.makedirs(dump_dir, exist_ok=True)
    for name, col in cols.items():
        np.save(os.path.join(dump_dir, name + suffix + ".npy"), col)
    return len(lines)


def warm_page_cache(path):
    with open(path, "rb") as f:  # like benchmarks/run.sh:3
        while f.read(1 << 24):
            pass


def lcm(a, b):
    return a * b // math.gcd(a, b)


def cut_at_line(arr, nbytes):
    """Largest prefix <= nbytes that ends at a newline."""
    nbytes = min(nbytes, len(arr))
    if nbytes == len(arr):
        return arr
    tail = arr[max(0, nbytes - 65536):nbytes]
    idx = np.flatnonzero(tail == 10)
    cut = nbytes - (len(tail) - 1 - int(idx[-1])) if len(idx) else nbytes
    return arr[:cut]


def pad_sample(sample, before, mult):
    """bytes: `sample` with its last line extended by the generator's filler words so that before + len is a
    multiple of `mult` (the reference's float chunk size must be integral, SURVEY §8(a) T1)."""
    from oracle import gen
    tail, _ = gen.pad_tail(before + len(sample), mult)
    data = sample.tobytes() if hasattr(sample, "tobytes") else bytes(sample)
    return data[:-1] + tail if tail else data


def reference_arm(args):
    """--impl reference: the reference's own CPU implementation of the path on the host cores, on a bounded
    sample of the same workload per step. Loads nothing of this repository's native code."""
    from oracle import gen
    ncores = os.cpu_count() or 1
    kind = "reference" if have_reference() else "port"
    total_bytes = int(args.gb * 1e9)
    sample_target = int(min(total_bytes, max(32e6, 4e6 * ncores)))
    tmp = tempfile.mkdtemp(prefix="dampr_refarm_")
    try:
        path = os.path.join(tmp, "sample.txt")
        n_lines = max(1, int(sample_target / MEAN_LINE))
        gen.text_to_file(path, 1234, n_lines, V=args.vocab, procs=ncores)
        # the reference chunks by st_size / cpu_count (a float): make it integral
        with open(path, "rb") as f:
            data = np.frombuffer(f.read(), dtype=np.uint8)
        with open(path, "wb") as f:
            f.write(pad_sample(data, 0, lcm(64, ncores)))
        del data
        nbytes = os.path.getsize(path)
        warm_page_cache(path)
        times = []
        budget = 240.0
        note = None
        for i in range(args.warmup + args.steps):
            sec, kind, note, used = cpu_arm(path, os.path.join(tmp, "idfs"), ncores)
            if i == 0 and sec * (args.warmup + args.steps) > budget and nbytes > 48e6:
                # the box is slower than planned: shrink the per-step sample so the whole run stays bounded
                keep = int(max(32e6, nbytes * budget / (sec * (args.warmup + args.steps))))
                with open(path, "rb") as f:
                    data = np.frombuffer(f.read(), dtype=np.uint8)
                with open(path, "wb") as f:
                    f.write(pad_sample(cut_at_line(data, keep), 0, lcm(64, ncores)))
                del data
                nbytes = os.path.getsize(path)
                warm_page_cache(path)
            if i >= args.warmup:
                times.append(sec)
        val = nbytes * len(times) / sum(times) / MB
        sample = "%d-byte line-aligned prefix of the synthetic corpus per step (oracle/gen.py, seed 1234, V=%d), %d worker processes on %d cores" % (
            nbytes, args.vocab, used, ncores)
        how = ("the unmodified reference (pip install of /root/reference under oracle/_ref), benchmarks/tf-idf-dampr.py "
               "statements, wall time of the whole python process" if kind == "reference"
               else "oracle/cpu_runner.py (port of the reference's runner; %s)" % (
                   ("the reference under oracle/_ref failed on this box: " + note) if note else "oracle/_ref is absent"))
        line = {"impl": "reference", "metric": METRIC, "value": val, "unit": "MB/s", "n_gpus": args.gpus,
                "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * sum(times) / len(times),
                "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "u8", "data": "synthetic",
                "config": {"workload": "benchmarks/tf-idf-dampr.py on synthetic Zipf(1.1) text, V=%d: %s" % (args.vocab, sample),
                           "sample": sample, "how": how},
                "cpu_baseline": {"value": val, "unit": "MB/s", "cores": used, "kind": kind, "sample": sample},
                "e2e": {"value": val, "unit": "MB/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
        print(json.dumps(line))
    finally:
        shutil.rmtree(tmp, ignore_errors=True)
    return 0


# ---- parity of the timed graph: GPU result vs the CPU checker on a sample of the same corpus ---------------------
def parity_check(Dampr, MemoryText, host_text, rank, world, use_dist, dist, out_root):
    """Runs the TF-IDF graph on a line-aligned sample (every rank takes a prefix of its shard) through the
    engine — all ranks, with the exchange — and through the CPU checker on the concatenation of the samples;
    the sorted sink lines must be byte-identical. Returns the `parity` object (rank 0) or None."""
    ncores = os.cpu_count() or 1
    mult = lcm(64, ncores)
    per_rank = int(min(len(host_text), (48e6 if world == 1 else 24e6)))
    sample = cut_at_line(host_text, per_rank)
    lens = [len(sample)]
    if use_dist:
        lens = [None] * world
        dist.all_gather_object(lens, len(sample))
    before = sum(lens[:rank])
    if rank == world - 1:
        data = pad_sample(sample, before, mult)
    else:
        data = sample.tobytes()
    arr = np.frombuffer(data, dtype=np.uint8)
    shared = os.path.join(tempfile.gettempdir(), "dampr_parity_%s" % os.environ.get("MASTER_PORT", str(os.getppid())))
    if rank == 0:
        shutil.rmtree(shared, ignore_errors=True)
        os.makedirs(shared)
    if use_dist:
        dist.barrier()
    with open(os.path.join(shared, "sample-%03d.txt" % rank), "wb") as f:
        f.write(data)
    out_dir = os.path.join(shared, "gpu_idfs")
    tfidf_job(Dampr, MemoryText(arr), out_dir)
    if use_dist:
        dist.barrier()
    if rank != 0:
        return None
    corpus = os.path.join(shared, "corpus.txt")
    with open(corpus, "wb") as f:
        for r in range(world):
            with open(os.path.join(shared, "sample-%03d.txt" % r), "rb") as g:
                shutil.copyfileobj(g, f)
    nbytes = os.path.getsize(corpus)
    got = read_sink_lines(out_dir)
    progress("parity: GPU side done (%d lines), running the CPU checker on %d bytes" % (len(got), nbytes))
    _sec, kind, _note, _used = cpu_arm(corpus, os.path.join(shared, "cpu_idfs"), ncores)
    progress("parity: checker (%s) done" % kind)
    exp = read_sink_lines(os.path.join(shared, "cpu_idfs"))
    equal = got == exp
    second = None
    if kind == "reference":
        # the port is the second checker (independent of the reference's float chunking)
        run_cpu_tfidf(corpus, os.path.join(shared, "cpu2_idfs"), ncores, "port")
        second = read_sink_lines(os.path.join(shared, "cpu2_idfs")) == got
    res = {"checked_bytes": nbytes, "equal": bool(equal and (second is not False)), "n_terms": len(got),
           "sha256_sorted_lines": hashlib.sha256(b"\n".join(got)).hexdigest(),
           "checker": ("the unmodified reference (oracle/_ref)" if kind == "reference" else "oracle/cpu_runner.py"),
           "second_checker_equal": second, "ranks": world,
           "what": "sorted sink_tsv lines of the same TF-IDF graph on a %d-byte line-aligned sample "
                   "(prefix of every rank's shard), byte-identical" % nbytes}
    if not res["equal"]:
        bad = [l for l in got if l not in set(exp)][:5]
        res["first_differences"] = [b.decode("utf-8", "replace") for b in bad]
    shutil.rmtree(shared, ignore_errors=True)
    return res


# ---- extras (1 GPU): the north-star's own stage and the other BASELINE configs ------------------------------------
def kv_extras(ctx_unused, args):
    sys.path.insert(0, os.path.join(ROOT, "tools"))
    import kv_bench
    from dampr_b200 import device as dev
    from dampr_b200 import runner as runner_mod
    ctx = runner_mod.get_ctx()
    extra = {}

    def guarded(name, fn):
        progress("extra: " + name)
        try:
            t0 = time.time()
            extra[name] = fn()
            if isinstance(extra[name], dict):
                extra[name]["bench_wall_s"] = round(time.time() - t0, 2)
        except Exception as e:  # an extra must never take the headline line down
            extra[name] = {"error": "%s: %s" % (type(e).__name__, str(e)[:300])}
            progress("extra %s failed: %s: %s" % (name, type(e).__name__, str(e)[:300]))

    guarded("kv_partition_sort_1e8_K=N", lambda: kv_bench.sort_case(ctx, 100_000_000, 100_000_000, label="K=N"))
    guarded("kv_partition_sort_1e8_K=1e7", lambda: kv_bench.sort_case(ctx, 100_000_000, 10_000_000, label="K=1e7"))
    guarded("kv_partition_sort_6.25e8_K=N", lambda: kv_bench.sort_case(ctx, 625_000_000, 625_000_000, label="K=N"))
    guarded("kv_partition_sort_6.25e8_K=1e7", lambda: kv_bench.sort_case(ctx, 625_000_000, 10_000_000, label="K=1e7"))
    guarded("kv_sort_reduce_6.25e8_K=1e7", lambda: kv_bench.reduce_case(ctx, 625_000_000, 10_000_000, label="config 2 on device"))
    guarded("kv_merge_8runs_1e8", lambda: kv_bench.merge_case(ctx, 100_000_000, 100_000_000, 8, -1))
    guarded("kv_merge_reduce_8runs_1e8_K=1e7", lambda: kv_bench.merge_case(ctx, 100_000_000, 10_000_000, 8, dev.OP_SUM_I64))
    guarded("kv_reduce_by_key_sorted_1e8_K=1e7", lambda: kv_bench.reduce_sorted_case(ctx, 100_000_000, 10_000_000))
    guarded("config2_e2e", lambda: kv_bench.config2_e2e(ctx))
    guarded("config4_scaled", lambda: kv_bench.config4_scaled(ctx))
    guarded("config5", lambda: kv_bench.config5(ctx))
    guarded("config5_dsl", lambda: kv_bench.config5_dsl(ctx))
    return extra


def file_e2e(Dampr, host_text, out_root, steps=2):
    """The script under test takes a PATH: Dampr.text(path) -> page cache -> pinned ring -> device. Timed on a
    file holding a 2.5 GB line-aligned prefix of the corpus (written and page-cache-warmed before timing)."""
    progress("extra: file_e2e")
    part = cut_at_line(host_text, int(2.5e9))
    path = os.path.join(out_root, "corpus_prefix.txt")
    part.tofile(path)
    warm_page_cache(path)
    nbytes = os.path.getsize(path)

    def one(i):
        out_dir = os.path.join(out_root, "file_idfs_%d" % i)
        docs = Dampr.text(path, nbytes / (os.cpu_count() or 1) + 1)
        doc_freq = docs.flat_map(lambda x: set(RX.split(x.lower()))).count(reduce_buffer=float("inf"))
        idf = doc_freq.cross_right(docs.len(), lambda df, total: (df[0], df[1], math.log(1 + (float(total) / df[1]))),
                                   memory=True)
        idf.sink_tsv(out_dir).run()
        shutil.rmtree(out_dir, ignore_errors=True)

    one(-1)
    t0 = time.perf_counter()
    for i in range(steps):
        one(i)
    sec = (time.perf_counter() - t0) / steps
    out = {"value": nbytes / sec / MB, "unit": "MB/s", "bytes": nbytes, "ms_per_step": 1e3 * sec,
           "what": "Dampr.text(path, st_size/cpu_count + 1) ... sink_tsv(dir).run(): file in the page cache -> "
                   "copy threads pread() into the pinned ring -> device -> sink files"}
    # the same job with the opt-in cuFile (GPUDirect Storage) ingest: dampr_set_option("file_cufile", 1)
    from dampr_b200 import device as dev
    try:
        dev.set_option("file_cufile", 1)
        one(-2)
        t0 = time.perf_counter()
        for i in range(steps):
            one(100 + i)
        sec2 = (time.perf_counter() - t0) / steps
        out["cufile"] = {"value": nbytes / sec2 / MB, "unit": "MB/s", "ms_per_step": 1e3 * sec2,
                         "what": "file bytes -> device through cuFileRead (8 host threads, 16 MB reads); without the "
                                 "nvidia-fs driver cuFile runs in its compatibility mode (its own bounce buffers)"}
    except Exception as e:
        out["cufile"] = {"error": "%s: %s" % (type(e).__name__, str(e)[:200])}
    finally:
        dev.set_option("file_cufile", 0)
    os.remove(path)
    return out


def main():
    args = parse_args()
    rank, world, local = dist_env()
    if world != max(1, args.gpus) and world > 1:
        args.gpus = world
    if args.impl == "reference":
        if rank != 0:
            return 0
        return reference_arm(args)

    total_bytes = int(args.gb * 1e9)
    shard_bytes = total_bytes // world
    n_lines = int(shard_bytes / MEAN_LINE)

    from dampr_b200 import device as dev
    from dampr_b200 import synth, settings

    settings.device = local
    try:
        ctx = dev.Ctx(local)
    except dev.DeviceError as e:
        raise SystemExit("bench.py needs a CUDA device (no CPU fallback): %s" % e)

    use_dist = world > 1
    dist = None
    if use_dist:
        import torch
        import torch.distributed as dist
        torch.cuda.set_device(local)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))

    # ---- synthetic corpus: generated on the device, mirrored into page-locked host memory -------------
    progress("rank %d/%d: generating %.2f GB of text" % (rank, world, shard_bytes / 1e9))
    vocab = synth.make_vocab(args.vocab)
    cdf = synth.make_cdf(args.vocab)
    tb = ctx.synth_text(1234 + rank, n_lines, vocab[0], vocab[1], cdf)
    nbytes = tb.n
    pin = dev.PinnedBuffer(nbytes)
    ctx.check(ctx.lib.dampr_textbuf_download(ctx.h, tb.h, 0, pin.array.ctypes.data, nbytes))
    host_text = pin.array[:nbytes]

    ncores = os.cpu_count() or 1
    workload = "benchmarks/tf-idf-dampr.py on %.2f GB synthetic Zipf(1.1) text, V=%d, %d GPU(s)" % (
        nbytes * world / 1e9, args.vocab, world)

    from dampr_b200 import Dampr
    from dampr_b200 import runner as runner_mod
    from dampr_b200.plan import MemoryText, DeviceText

    out_root = tempfile.mkdtemp(prefix="dampr_bench_r%d_" % rank)

    def barrier():
        ctx.sync()
        if use_dist:
            dist.barrier()

    def step(resident, i):
        out_dir = os.path.join(out_root, "idfs_%s_%d" % ("dev" if resident else "host", i))
        src = DeviceText(tb) if resident else MemoryText(host_text)
        tfidf_job(Dampr, src, out_dir)
        return out_dir

    def max_over_ranks(x):
        if not use_dist:
            return x
        t = torch.tensor([x], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def sink_digest(out_dir):
        """order-independent digest of this rank's sink lines: (lines, sum of 64-bit line hashes mod 2^64)"""
        n, acc = 0, 0
        for fn in os.listdir(out_dir):
            with open(os.path.join(out_dir, fn), "rb") as f:
                for l in f:
                    n += 1
                    acc = (acc + int.from_bytes(hashlib.blake2b(l, digest_size=8).digest(), "little")) & 0xFFFFFFFFFFFFFFFF
        return n, acc

    # ---- warm-up immediately before each timed loop (no host-side pause in between) -------------------
    sampler = ClockSampler(local)
    if not os.environ.get("DAMPR_BENCH_NOSAMPLER"):
        sampler.start()
    verbose = bool(os.environ.get("DAMPR_BENCH_VERBOSE"))
    progress("warm-up + timed loops")
    for i in range(args.warmup):
        ts = time.perf_counter()
        shutil.rmtree(step(True, -1 - i), ignore_errors=True)
        if verbose:
            print("warmup resident %d: %.1f ms %s" % (i, 1e3 * (time.perf_counter() - ts),
                                                      [round(ms, 1) for _s, ms in runner_mod.LAST_STATS.ms]), file=sys.stderr)

    # ---- timed: device-resident input ("device_resident") ------------------------------------------------
    runner_ctx = runner_mod.get_ctx(local)
    barrier()
    runner_ctx.timings_reset()
    t0 = time.perf_counter()
    dev_steps = []
    d_dev = None
    for i in range(args.steps):
        ts = time.perf_counter()
        d_dev = step(True, i)
        dev_steps.append([round(1e3 * (time.perf_counter() - ts), 1)] +
                         [round(ms, 1) for _s, ms in runner_mod.LAST_STATS.ms])
    barrier()
    t_dev = max_over_ranks(time.perf_counter() - t0)
    ktimes = runner_ctx.timings()
    for i in range(args.warmup):
        ts = time.perf_counter()
        shutil.rmtree(step(False, -1 - i), ignore_errors=True)
        if verbose:
            print("warmup e2e %d: %.1f ms %s" % (i, 1e3 * (time.perf_counter() - ts),
                                                 [round(ms, 1) for _s, ms in runner_mod.LAST_STATS.ms]), file=sys.stderr)

    # ---- timed: host-resident input (the metric) -----------------------------------------------------------
    barrier()
    l0 = runner_ctx.launches()
    t0 = time.perf_counter()
    e2e_steps = []
    d = None
    for i in range(args.steps):
        ts = time.perf_counter()
        d = step(False, i)
        e2e_steps.append([round(1e3 * (time.perf_counter() - ts), 1)] +
                         [round(ms, 1) for _s, ms in runner_mod.LAST_STATS.ms])
    barrier()
    t_e2e = max_over_ranks(time.perf_counter() - t0)
    launches = runner_ctx.launches() - l0
    stats = runner_mod.LAST_STATS.stages if runner_mod.LAST_STATS else []
    e2e_stage_ms = [round(ms, 2) for _s, ms in (runner_mod.LAST_STATS.ms if runner_mod.LAST_STATS else [])]
    sampler.stop_flag.set()
    if sampler.is_alive():
        sampler.join(timeout=5)
    if os.environ.get("DAMPR_BENCH_PROFILE") and rank == 0:
        # development aid: where the host time of a device-resident step goes (after the timed loops)
        import cProfile
        import io
        import pstats
        pr = cProfile.Profile()
        pr.enable()
        for i in range(5):
            step(True, 100 + i)
        pr.disable()
        for key in ("cumulative", "tottime"):
            sio = io.StringIO()
            pstats.Stats(pr, stream=sio).sort_stats(key).print_stats(35)
            print(sio.getvalue()[:7000], file=sys.stderr)
    elif os.environ.get("DAMPR_BENCH_PROFILE"):
        for i in range(5):
            step(True, 100 + i)

    # ---- full-size consistency: both timed variants produced the same result on every rank, the line
    # totals add up over the ranks -------------------------------------------------------------------------
    n_terms, dig_host = sink_digest(d)
    n_terms_dev, dig_dev = sink_digest(d_dev)
    full = {"rank_terms": n_terms, "host_vs_resident_equal": bool(dig_host == dig_dev and n_terms == n_terms_dev)}
    if use_dist:
        t = torch.tensor([n_terms, int(full["host_vs_resident_equal"])], dtype=torch.int64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.SUM)
        full = {"terms_all_ranks": int(t[0].item()), "host_vs_resident_equal": bool(int(t[1].item()) == world)}
        n_terms_total = int(t[0].item())
    else:
        n_terms_total = n_terms
    if args.dump_outputs:
        dumped = dump_outputs(d, args.dump_outputs, "" if world == 1 else "_rank%d" % rank)
        progress("dumped the %d-row TF-IDF table of the last timed step to %s" % (dumped, args.dump_outputs))

    total = nbytes * world
    value_dev = total * args.steps / t_dev / MB
    e2e = total * args.steps / t_e2e / MB
    tc = [ms for name, ms in ktimes if name == "text_count"]
    peak, peak_kind = measured_peak()
    roof = None
    if tc:
        per_launch_ms = sum(tc) / len(tc)
        per_launch_bytes = nbytes * args.steps / len(tc)
        ach = per_launch_bytes / (per_launch_ms * 1e-3) / 1e9
        traffic, traffic_src, issue = None, None, None
        try:
            tj = None
            for fn in ("text_traffic.json", "r01_text_traffic.json"):
                fp = os.path.join(ROOT, "profiles", fn)
                if os.path.exists(fp):
                    with open(fp) as f:
                        tj = json.load(f)
                    break
            # dram__bytes_read+write of one ncu --set full capture of this kernel, scaled from the
            # captured launch (250 MB of the same corpus) to this launch's bytes
            traffic = tj["dram_bytes_per_input_byte"] * per_launch_bytes
            traffic_src = "ncu capture scaled per input byte: " + tj["source"]
            # what actually bounds this kernel: instruction issue. smsp__inst_executed of the same capture
            # per input byte against 4 schedulers x SMs x SM clock (one warp instruction per cycle each)
            wipb = tj.get("warp_instructions_per_input_byte")
            clk = (sampler.summary().get("sm_mhz") or 0) * 1e6
            if wipb and clk:
                issue_peak = 4 * ctx.num_sms() * clk / wipb / 1e9
                issue = {"bound": "issue", "warp_instructions_per_byte": wipb, "peak": issue_peak, "unit": "GB/s",
                         "frac": ach / issue_peak}
        except Exception:
            pass
        roof = {"bound": "hbm", "achieved": ach, "peak": peak, "unit": "GB/s", "frac": ach / peak,
                "traffic": traffic, "traffic_source": traffic_src,
                "kernel": "text_count2_kernel<NONWORD_LOWER_SET> (csrc/text2.cu)",
                "algorithmic_bytes_per_launch": per_launch_bytes, "ms_per_launch": per_launch_ms,
                "peak_source": peak_kind + " (MEASURED_PEAKS.json hbm_gbs)", "issue_roofline": issue}

    # ---- parity of the timed graph against the CPU checker (all ranks take part) ----------------------------
    parity = None
    progress("timed loops done: e2e %.1f ms/step, resident %.1f ms/step" % (1e3 * t_e2e / args.steps, 1e3 * t_dev / args.steps))
    if not args.no_parity:
        progress("parity check")
        try:
            parity = parity_check(Dampr, MemoryText, host_text, rank, world, use_dist, dist, out_root)
        except Exception as e:
            parity = {"equal": False, "error": "%s: %s" % (type(e).__name__, str(e)[:500])}
        if parity is not None:
            parity["full_size"] = full

    d2h = int(n_terms_total) * (24 if world == 1 else 32)
    line = {"metric": METRIC, "value": e2e, "unit": "MB/s",
            "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": 1e3 * t_e2e / args.steps, "higher_is_better": True, "scaling": "strong",
            "vs_baseline": None, "dtype": "u8", "data": "synthetic",
            "config": {"workload": workload, "bytes_per_rank": nbytes, "lines_per_rank": n_lines,
                       "l2": "inputs (%.1f GB per rank) are larger than L2" % (nbytes / 1e9),
                       "value_is": "end to end: text in page-locked host memory -> H2D -> kernels -> exchange -> result "
                                   "table D2H -> sink files, all inside the timed region",
                       "stages": [[s.split("`")[1][:40] if "`" in s else s, h] for s, h, _d in stats],
                       "e2e_stage_ms": e2e_stage_ms},
            "e2e": {"value": e2e, "unit": "MB/s", "h2d_bytes_per_step": nbytes * world,
                    # result table per term: 16-byte key string + 8-byte count (single GPU; the synthetic
                    # corpus has no hashed tokens), plus the 8-byte code after the exchange (multi GPU)
                    "d2h_bytes_per_step": d2h, "ms_per_step": 1e3 * t_e2e / args.steps, "step_ms": e2e_steps},
            "device_resident": {"value": value_dev, "unit": "MB/s", "ms_per_step": 1e3 * t_dev / args.steps,
                                "step_ms_total_then_stages": dev_steps,
                                "what": "the same job with the text already in HBM when the step starts"},
            "gpu_launches": int(launches), "clocks": sampler.summary(), "roofline": roof, "parity": parity}

    if rank == 0 and world == 1 and not args.no_extra:
        tb.free()
        extra = kv_extras(ctx, args)
        try:
            extra["file_e2e"] = file_e2e(Dampr, host_text, out_root)
        except Exception as e:
            extra["file_e2e"] = {"error": "%s: %s" % (type(e).__name__, str(e)[:300])}
        line["extra"] = extra

    if rank == 0 and not args.no_cpu_baseline:
        progress("cpu_baseline")
        tmp = tempfile.mkdtemp(prefix="dampr_cpu_")
        try:
            sample = cut_at_line(host_text, int(min(nbytes, max(32e6, 4e6 * ncores))))
            path = os.path.join(tmp, "sample.txt")
            with open(path, "wb") as f:
                f.write(pad_sample(sample, 0, lcm(64, ncores)))
            sbytes = os.path.getsize(path)
            warm_page_cache(path)
            cpu_arm(path, os.path.join(tmp, "idfs"), ncores)  # warm-up (imports, fork, page cache)
            sec, kind, _note, used = cpu_arm(path, os.path.join(tmp, "idfs"), ncores)
            line["cpu_baseline"] = {"value": sbytes / sec / MB, "unit": "MB/s", "cores": used, "kind": kind,
                                    "sample": "%d-byte line-aligned prefix of the corpus, %d worker processes on %d cores (%s)" % (
                                        sbytes, used, ncores, "the unmodified reference, oracle/_ref; with all cores as workers "
                                        "it never returns on this box" if kind == "reference"
                                        else "oracle/cpu_runner.py, a leaner port of the reference's runner")}
        finally:
            shutil.rmtree(tmp, ignore_errors=True)
    shutil.rmtree(out_root, ignore_errors=True)
    progress("done")
    if rank == 0:
        print(json.dumps(line))
    ok = True
    if parity is not None and not parity.get("equal", False):
        ok = False
        print("PARITY FAILURE: %s" % json.dumps(parity)[:2000], file=sys.stderr)
    if use_dist:
        dist.barrier()
        dist.destroy_process_group()
    return 0 if ok else 3


if __name__ == "__main__":
    sys.exit(main())
