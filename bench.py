#!/usr/bin/env python
"""
bench.py — benchmark of the read -> feature -> count path on every workload BASELINE.json names.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--reads R] [--configs a,b,...] [--scale S]
                    [--dump-outputs DIR]

Headline (the JSON line's own metric/value/e2e/roofline, comparable across rounds): BASELINE.json configs[1],
synthetic 100 M x 50 bp reads per GPU vs a 2 000-guide library, --st 0 --l 20 --m 1 --ph 30; weak scaling over GPUs.
One "step" = one pass of the hot path over the whole synthetic sample.
  value     M reads/s with the sample resident in HBM (f2q_submit_device); device-timed, max over ranks
  e2e       the same through the C-ABI call a user makes with HOST buffers (f2q_submit from pinned memory):
            H2D of every byte + D2H of the counts inside the timed region
  roofline  achieved HBM GB/s of the fused streaming kernel = algorithmic bytes (2L+18 per read) / its CUDA-event time
  cpu_baseline  the oracle port (oracle/f2q_oracle.c, the reference's algorithm in C) on a bounded sample, 1 core
  parity    the benchmarked stream itself: the GPU's counts of the CPU-baseline sample == the oracle's (asserted)

`other_configs` (same run, same JSON line) holds the other BASELINE shapes, each with value / ms_per_step / per-kernel ms /
roofline.frac / e2e and a parity block (GPU == oracle on a >= 1 M-read slice of that very stream; with N > 1 also the
--fs-style record-aligned shards of the slice over ALL ranks, merged over NCCL, == the oracle):
  north_star  50 bp reads vs 100 000 guides, m = 1 (the target shape of BASELINE.json's north_star), weak
  config3     1e9 x 75 bp reads vs 100 000 guides, m = 2, STRONG-scaled (1e9 / N reads per GPU), generated per chunk by K0
  config4     Extract + Count Bar-seq, 500 M x 75 bp reads between --us/--ds with 1 mismatch each, STRONG-scaled; at N > 1
              the per-rank key tables are merged (f2q_ec_merge: all-gather over NCCL + merge on the device) inside the timed step
  config5a/b  48 samples x 1.5 M x 75 bp, 10 000 'X:Y' dual keys + their singles, m = 1: fixed positions / delimiters;
              samples over GPUs, no collective
--impl reference times the reference's CPU algorithm (the oracle port on all host threads, file-parallel like the reference's
multiprocessing mode) and, when it imports on the box, the UNMODIFIED Python reference from baseline/_ref on a small slice.
Data are synthetic (K0 generator, csrc/synth_gen.h, bit-identical to 2fast2q_b200/synth.py).
"""
from __future__ import annotations

import argparse
import importlib
import json
import os
import statistics
import subprocess
import sys
import threading
import time

import numpy as np

_JSON_OUT = None


def emit(obj):
    out = _JSON_OUT or sys.stdout
    out.write(json.dumps(obj) + "\n")
    out.flush()


ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

READ_LEN, FEAT_LEN, N_GUIDES, CONFIG = 50, 20, 2000, 2
REC = 2 * READ_LEN + 18
WORKLOAD = "config2: synthetic 50bp reads vs 2000-guide library, --st 0 --l 20 --m 1 --ph 30"


def env_int(k, d):
    try:
        return int(os.environ.get(k, d))
    except ValueError:
        return d


def log(*a):
    print("[bench]", *a, file=sys.stderr, flush=True)


class ClockSampler:
    """samples SM clocks / throttle reasons during the timed regions (B200_PROFILING.md recipe) with an `nvidia-smi`
    subprocess polling every 20 ms.  Deliberately NOT in-process NVML: measured on this pool, one NVML query from a thread
    of the benchmark process blocks its CUDA launches for ~15 ms, three times the length of a whole resident pass."""
    Q = "index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
        "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, gpu_index, uuid=None):
        self.gpu, self.uuid, self.rows, self.p = gpu_index, uuid, [], None

    def start(self):
        sel = f"GPU-{self.uuid}" if self.uuid and not str(self.uuid).startswith("GPU-") else (self.uuid or str(self.gpu))
        try:
            self.p = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "20",
                                       "-i", str(sel)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
            time.sleep(0.5)                                        # let it come up before the timed region starts
        except OSError:
            self.p = None

    def _read(self):
        for line in self.p.stdout:
            self.rows.append([time.perf_counter()] + [x.strip() for x in line.split(",")])

    def stop(self, windows=()):
        """windows: (t0, t1) perf_counter intervals of the timed regions; samples inside them are counted separately"""
        if not self.p:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.05)
        self.p.terminate()
        try:
            self.p.wait(timeout=2)
        except subprocess.TimeoutExpired:
            self.p.kill()
        sm, mx, reasons, inside = [], [], set(), [0] * len(windows)
        for r in self.rows:
            if len(r) < 9:
                continue
            try:
                sm.append(float(r[2])); mx.append(float(r[3]))
            except ValueError:
                continue
            for k, (a, b) in enumerate(windows):
                if a <= r[0] <= b + 0.02:
                    inside[k] += 1
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm), "samples_in_timed_regions": inside,
                "source": "nvidia-smi -lms 20 from just before the headline resident timed region to the end of the last timed region"}


def measured_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def committed_traffic():
    """dram bytes per read of the dominant kernel from the committed ncu --set full capture (profiles/), scaled to this launch"""
    try:
        return json.load(open(os.path.join(ROOT, "profiles", "tile_kernel_traffic.json")))
    except Exception:
        return None


DUMP_LIMIT = 64 << 20                # bytes of all arrays --dump-outputs writes
DUMP_ARRAY_ELEMS = 1 << 21           # a larger array keeps a fixed, seeded sample of its rows


class OutputDump:
    """--dump-outputs DIR: what the last timed step of each leg handed to its caller, as DIR/<name>.npy, so that two builds
    can be compared output for output (the inputs are seeded: the same arguments give the same inputs).  Counts and
    statistics are float64, exact below 2**53; an array of more than DUMP_ARRAY_ELEMS elements keeps the rows of a fixed,
    seeded sample, in their original order."""

    def __init__(self, path):
        self.dir, self.nbytes = path, 0
        os.makedirs(path, exist_ok=True)

    @staticmethod
    def rows(n, row_elems):
        keep = max(1, DUMP_ARRAY_ELEMS // max(1, row_elems))
        if n <= keep:
            return np.arange(n)
        return np.sort(np.random.default_rng(0).choice(n, keep, replace=False))

    def save(self, name, a):
        a = np.asarray(a, dtype=np.float64)
        if a.size > DUMP_ARRAY_ELEMS:
            a = a[self.rows(a.shape[0], a.size // a.shape[0])]
        if self.nbytes + a.nbytes > DUMP_LIMIT:
            raise RuntimeError(f"--dump-outputs: {name} would take the dump past {DUMP_LIMIT >> 20} MB")
        self.nbytes += a.nbytes
        np.save(os.path.join(self.dir, name + ".npy"), a)

    def save_stats(self, name, stats):
        """one stats dict (or a list of them, one per sample) in STAT_NAMES order"""
        self.save(name, [list(s.values()) for s in stats] if isinstance(stats, list) else list(stats.values()))

    def save_table(self, name, table):
        """an Extract+Count key table: one row per key in byte order — count, key length, the key's bytes (0-padded)"""
        keys = sorted(table)
        width = max((len(k) for k in keys), default=0)
        idx = self.rows(len(keys), 2 + width)
        a = np.zeros((len(idx), 2 + width))
        for r, i in enumerate(idx):
            k = keys[i]
            a[r, 0], a[r, 1] = table[k], len(k)
            a[r, 2:2 + len(k)] = np.frombuffer(k, dtype=np.uint8)
        self.save(name, a)


def library():
    synth = importlib.import_module("2fast2q_b200.synth")        # generator spec + library builder (not the oracle)
    return synth.make_library(CONFIG, N_GUIDES, FEAT_LEN), synth.default_spec(CONFIG)


# ------------------------------------------------------------------------------------------------------------
# the reference arm
# ------------------------------------------------------------------------------------------------------------
def real_reference(keys, names, spec, reads, cores, timeout_s=240):
    """the UNMODIFIED Python reference (its fast2q package placed by hand in the git-ignored baseline/_ref) through its own CLI on a
    slice of the config-2 stream written as `cores` files (file-parallel = its best case, SURVEY.md §8d)"""
    import shutil
    import tempfile
    ref = os.path.join(ROOT, "baseline", "_ref")
    if not os.path.isdir(os.path.join(ref, "fast2q")):
        return {"unavailable": "baseline/_ref/fast2q is absent (place the unmodified reference package there)"}
    synth = importlib.import_module("2fast2q_b200.synth")
    tmp = tempfile.mkdtemp(prefix="f2q_ref_")
    try:
        src, out = os.path.join(tmp, "in"), os.path.join(tmp, "out")
        os.makedirs(src); os.makedirs(out)
        per = max(1, reads // cores)
        for t in range(cores):
            synth.fixed_reads(keys, t * per, per, **spec).tofile(os.path.join(src, "s%03d.fastq" % t))
        with open(os.path.join(tmp, "lib.csv"), "w") as f:
            f.write("".join(f"{n},{k.decode()}\n" for n, k in zip(names, keys)))
        stubs = os.path.join(ROOT, "tests", "golden", "_stubs")                # colorama / matplotlib, cosmetic on the counting path
        env = dict(os.environ, PYTHONPATH=os.pathsep.join([stubs, ref]), PYTHONWARNINGS="ignore",
                   NUMBA_CACHE_DIR=os.path.join(tmp, "nc"))
        cmd = [sys.executable, "-m", "fast2q", "-c", "--s", src, "--g", os.path.join(tmp, "lib.csv"), "--o", out, "--pb",
               "--cp", str(cores), "--m", "1", "--ph", "30", "--st", "0", "--l", str(FEAT_LEN)]
        t0 = time.perf_counter()
        p = subprocess.run(cmd, env=env, cwd=tmp, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, timeout=timeout_s)
        dt = time.perf_counter() - t0
        if p.returncode != 0:
            return {"unavailable": "reference CLI exited %d: %s" % (p.returncode, p.stdout.strip().splitlines()[-1][:200] if p.stdout.strip() else "")}
        import glob
        comp = glob.glob(os.path.join(out, "2FAST2Q_output_*", "compiled.csv"))
        if not comp:
            return {"unavailable": "reference CLI wrote no compiled.csv"}
        total = 0
        with open(comp[0]) as f:
            for line in f:
                if not line.startswith("#"):
                    total += sum(int(x) for x in line.strip().split(",")[1:])
        return {"value": cores * per / dt / 1e6, "unit": "M reads/s", "cores": cores, "kind": "reference",
                "sample": f"unmodified fast2q.py CLI (numba) on {cores} files x {per} reads of the config-2 stream, --cp {cores}, CLI wall time "
                          f"{dt:.1f} s incl. interpreter start + numba JIT; aligned reads counted {total}"}
    except subprocess.TimeoutExpired:
        return {"unavailable": f"reference CLI did not finish within {timeout_s} s"}
    except Exception as e:                                         # noqa: BLE001 — a baseline, not the product
        return {"unavailable": f"{type(e).__name__}: {e}"}
    finally:
        shutil.rmtree(tmp, ignore_errors=True)


def run_reference(args, rank, world):
    """the reference's CPU algorithm on all host threads: the oracle port (the timed arm), beside it the real Python reference"""
    if rank != 0:
        return
    from oracle import oracle as O                               # the reference arm IS the oracle port (task statement ④)
    synth = importlib.import_module("2fast2q_b200.synth")
    (names, keys), spec = library()
    cores = os.cpu_count() or 1
    threads = max(1, min(cores, 64))
    per = args.ref_reads_per_thread
    cfg = O.make_config(miss=1, phred=30, length=FEAT_LEN, start="0")
    O.lib()
    shards = [synth.fixed_reads(keys, t * per, per, **spec) for t in range(threads)]      # distinct reads per thread
    from concurrent.futures import ThreadPoolExecutor

    def work(a):
        return O.count(cfg, keys, a)

    def step():
        with ThreadPoolExecutor(threads) as ex:
            res = list(ex.map(work, shards))                       # ctypes releases the GIL: real thread parallelism
        tot = np.zeros(len(keys), dtype=np.uint64)
        for c, _ in res:
            tot += c                                               # merge_feature_dicts, fast2q.py:439-445
        return tot

    for _ in range(args.warmup):
        step()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        step()
    dt = (time.perf_counter() - t0) / args.steps
    v = threads * per / dt / 1e6
    sample = f"{threads} threads x {per} reads of the config-2 stream per step (one shard per thread, counts merged by addition)"
    real = None if args.no_real_reference else real_reference(keys, names, spec, args.real_ref_reads, threads)
    emit({
        "impl": "reference", "metric": "M reads/s", "value": v, "unit": "M reads/s", "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": dt * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "u8", "data": "synthetic",
        "config": {"workload": WORKLOAD},
        "sample_reads_per_step": threads * per,
        "cpu_baseline": {"value": v, "unit": "M reads/s", "cores": threads, "kind": "port", "sample": sample},
        "cpu_baseline_reference": real,
        "e2e": {"value": v, "unit": "M reads/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    })


# ------------------------------------------------------------------------------------------------------------
class _DevArr:
    def __init__(self, ptr, n):
        self.__cuda_array_interface__ = {"shape": (n,), "typestr": "<i8", "data": (ptr, False), "version": 2}


def oracle_threads():
    return max(1, min(os.cpu_count() or 1, 32))


def oracle_count_parallel(O, cfg, keys, host, rec):
    """oracle.count of a stream of fixed-size records on all host threads (records are independent); sums counts and stats"""
    from concurrent.futures import ThreadPoolExecutor
    n = host.size // rec
    T = max(1, min(oracle_threads(), n // 1000 or 1))
    cuts = [(n * t // T) * rec for t in range(T + 1)]
    with ThreadPoolExecutor(T) as ex:
        res = list(ex.map(lambda ab: O.count(cfg, keys, host[ab[0]:ab[1]]), zip(cuts[:-1], cuts[1:])))
    counts = np.zeros(len(keys), dtype=np.uint64)
    stats = {k: 0 for k in O.STAT_NAMES}
    for c, s in res:
        counts += c
        for k in stats:
            stats[k] += s[k]
    return counts, stats


def oracle_ec_parallel(O, cfg, host, rec):
    from concurrent.futures import ThreadPoolExecutor
    n = host.size // rec
    T = max(1, min(oracle_threads(), n // 1000 or 1))
    cuts = [(n * t // T) * rec for t in range(T + 1)]
    with ThreadPoolExecutor(T) as ex:
        res = list(ex.map(lambda ab: O.extract_count(cfg, host[ab[0]:ab[1]]), zip(cuts[:-1], cuts[1:])))
    merged, stats = {}, {k: 0 for k in O.STAT_NAMES}
    for d, s in res:
        for k, v in d.items():
            merged[k] = merged.get(k, 0) + v
        for k in stats:
            stats[k] += s[k]
    return merged, stats


class Workload:
    """one BASELINE shape: library + generator spec + engine parameters + sizes"""

    def __init__(self, name, label, params, keys, guides, spec, *, reads, scaling, chunk_reads, parity_reads, n_samples=1):
        self.name, self.label, self.params, self.keys, self.guides, self.spec = name, label, params, keys, guides, spec
        self.reads, self.scaling, self.chunk_reads, self.parity_reads, self.n_samples = reads, scaling, chunk_reads, parity_reads, n_samples
        self.rec = 2 * spec["read_len"] + 18
        self.ec = "EC" in str(params.get("mode", "C")).upper()


def build_workloads(args):
    synth = importlib.import_module("2fast2q_b200.synth")
    S = args.scale
    W = {}

    def n(x, lo=200_000):
        return max(lo, int(x * S))
    want = set(args.configs.split(","))
    if want & {"north_star", "config3", "all"}:
        names100k, keys100k = synth.make_library(3, 100_000, 20)
    if want & {"north_star", "all"}:
        spec = dict(synth.default_spec(2), seed=12)
        W["north_star"] = Workload("north_star", "north-star shape: synthetic 50bp reads vs 100000-guide library, --st 0 --l 20 --m 1 --ph 30",
                                   dict(mode="C", miss=1, phred=30, length=20, start="0"), keys100k, keys100k, spec,
                                   reads=n(50_000_000), scaling="weak", chunk_reads=n(50_000_000), parity_reads=n(1_048_576, 100_000))
    if want & {"config3", "all"}:
        spec = synth.default_spec(3)
        W["config3"] = Workload("config3", "config3: synthetic 1e9 x 75bp reads vs 100000-guide library, --st 0 --l 20 --m 2 --ph 30",
                                dict(mode="C", miss=2, phred=30, length=20, start="0"), keys100k, keys100k, spec,
                                reads=n(1_000_000_000), scaling="strong", chunk_reads=n(25_000_000), parity_reads=n(1_048_576, 100_000))
    if want & {"config4", "all"}:
        spec = synth.shape_spec("4")
        pool = synth.random_kmers(4, n(1_000_000, 10_000), 20)
        W["config4"] = Workload("config4", "config4: Extract+Count Bar-seq, synthetic 500M x 75bp reads, --mo EC --us GTTCAGAGTTCT --ds CTGAATAGGCCA "
                                "--msu 1 --msd 1 --ph 30, 1M-barcode pool",
                                dict(mode="EC", phred=30, upstream=synth.BARSEQ_US.decode(), downstream=synth.BARSEQ_DS.decode(),
                                     miss_search_up=1, miss_search_down=1), None, pool, spec,
                                reads=n(500_000_000), scaling="strong", chunk_reads=n(25_000_000), parity_reads=n(1_048_576, 100_000))
    if want & {"config5a", "config5b", "all"}:
        dn, dkeys, xs, ys = synth.dual_keys(10_000)
    for tag, params in (("config5a", dict(mode="C", miss=1, phred=30, length=20, start="0,30")),
                        ("config5b", dict(mode="C", miss=1, phred=30, upstream="ACCGGT,GGATCC", downstream="TTGACA,CAATTG"))):
        if want & {tag, "all"}:
            spec = synth.shape_spec(tag[-2:])
            flags = "--st 0,30 --l 20" if tag == "config5a" else "--us ACCGGT,GGATCC --ds TTGACA,CAATTG"
            W[tag] = Workload(tag, f"{tag}: 48 samples x 1.5M x 75bp dual-feature reads vs 10000 X:Y keys + singles (30000 keys), {flags} --m 1 --ph 30",
                              params, dkeys, xs + ys, spec, reads=n(1_500_000, 50_000), scaling="strong (48 samples over the GPUs)",
                              chunk_reads=n(1_500_000, 50_000), parity_reads=n(1_048_576, 50_000), n_samples=48)
    return W


def run_workload(w, env):
    """resident + end-to-end timing and parity of one workload; returns the dict that goes under other_configs[w.name]"""
    import torch
    import torch.distributed as dist
    lib, multi, host_mod = env["lib"], env["multi"], env["host"]
    rank, world, dev, stream, local_rank = env["rank"], env["world"], env["dev"], env["stream"], env["local_rank"]
    synth = importlib.import_module("2fast2q_b200.synth")
    rec = w.rec
    cfg = lib.make_config(**w.params)
    eng = lib.Engine(cfg, local_rank, stream.cuda_stream, time_kernels=1)
    if w.keys is not None:
        eng.set_library(w.keys)
    n_keys = len(w.keys) if w.keys is not None else 0
    if world > 1:
        eng.comm_share(env["comm"])                                          # the rank's NCCL communicator (libf2q's own C-ABI collectives)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    def merge_counts():
        if world > 1:
            eng.allreduce_counts()                                           # f2q_allreduce_counts: ncclAllReduce(sum, uint64) on the engine's stream

    def merge_ec():
        """Extract+Count: every rank's key table becomes the merged table (f2q_ec_merge: all-gather + device merge)"""
        if world > 1:
            eng.ec_merge()

    # ---- this rank's reads ----
    if w.n_samples > 1:
        my_samples = list(range(rank, w.n_samples, world))                    # samples round-robin over the GPUs
        my_reads = len(my_samples) * w.reads
        total_reads = w.n_samples * w.reads
    elif w.scaling == "strong":
        first, my_reads = multi.rank_read_range(w.reads, rank, world)
        total_reads = w.reads
    else:
        first, my_reads = rank * w.reads, w.reads
        total_reads = world * w.reads
    if w.n_samples > 1:
        first = 0
    chunk = min(w.chunk_reads, max(my_reads, 1)) if w.n_samples == 1 else w.reads
    buf_reads = max(chunk, w.parity_reads) if w.n_samples == 1 else max(len(my_samples) * w.reads, w.parity_reads)
    data = torch.empty(max(buf_reads, 1) * rec, dtype=torch.uint8, device=dev)
    dptr = data.data_ptr()
    eng.synth(dptr, w.guides, 0, 1, **w.spec)                                # uploads the guide table once

    def gen(first_read, n_reads, at=0):
        eng.synth(dptr + at, w.guides, first_read, n_reads, reuse_guides=True, **w.spec)

    # ---- parity: the first parity_reads of rank 0's stream ----
    parity = {"reads": w.parity_reads}
    P = w.parity_reads
    gen(0, P)
    eng.begin()
    eng.submit_device(dptr, P * rec, True)
    got_c, got_s = eng.end()
    got_ec = eng.ec_items() if w.ec else None
    hostbytes = eng.d2h(dptr, P * rec)
    if rank == 0:
        from oracle import oracle as O
        ocfg = O.make_config(**w.params)
        t0 = time.perf_counter()
        if w.ec:
            want_ec, want_s = oracle_ec_parallel(O, ocfg, hostbytes, rec)
            assert got_s == want_s, (w.name, got_s, want_s)
            assert got_ec == want_ec, (w.name, "Extract+Count tables differ", len(got_ec), len(want_ec))
        else:
            want_c, want_s = oracle_count_parallel(O, ocfg, w.keys, hostbytes, rec)
            assert got_s == want_s, (w.name, got_s, want_s)
            assert np.array_equal(got_c, want_c), (w.name, "counts differ", int((got_c != want_c).sum()))
        parity.update(ok=True, oracle_s=round(time.perf_counter() - t0, 2), stats=got_s,
                      checker=f"oracle/f2q_oracle.c on {oracle_threads()} host threads, bit-exact counts + stats")
    if world > 1:
        # --fs style: the slice cut at record boundaries into shards, rank r parses shards r, r+N, ... through f2q_submit
        blocks = (hostbytes[o:o + (4 << 20)].tobytes() for o in range(0, hostbytes.size, 4 << 20))
        shards = host_mod.record_aligned_shards(blocks, shard_bytes=8 << 20)
        eng.begin()
        for shard, _final in multi.rank_shards(shards, rank, world):
            eng.submit(shard, False)
        eng.submit(b"", True)
        if w.ec:
            merge_counts()                                                   # the five statistics
            _c, st_all = eng.end()
            merge_ec()
            merged = eng.ec_items()
            if rank == 0:
                assert st_all == want_s, (w.name, "sharded stats differ")
                assert merged == want_ec, (w.name, "sharded Extract+Count tables differ")
        else:
            merge_counts()
            sc, ss = eng.end()
            if rank == 0:
                assert ss == want_s and np.array_equal(sc, want_c), (w.name, "sharded counts differ")
        parity["multi_gpu_shards_ok"] = True
        parity["multi_gpu_shards"] = f"record-aligned 8 MiB shards of the slice round-robin over {world} ranks via f2q_submit, merged over NCCL"

    # ---- resident timing ----
    chunks = []
    if w.n_samples == 1:
        o = 0
        while o < my_reads:
            m = min(chunk, my_reads - o)
            chunks.append((first + o, m))
            o += m
        resident_once = len(chunks) == 1
        if resident_once:
            gen(*chunks[0])
    else:
        for k, s in enumerate(my_samples):
            gen(s * w.reads, w.reads, at=k * w.reads * rec)                   # every sample owns its own read range
        resident_once = True
    pin_res = [lib.PinnedBuffer(8 * (n_keys + 6)) for _ in range(max(1, len(my_samples) if w.n_samples > 1 else 1))]
    ec_stats = {}

    def resident_pass(limit=None):
        """returns device ms of the pass (synth of per-chunk generated workloads excluded)"""
        ms = 0.0
        if w.n_samples > 1:
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(stream)
            for k in range(len(my_samples)):
                eng.begin()
                eng.submit_device(dptr + k * w.reads * rec, w.reads * rec, True)
                eng.end_async(pin_res[k])
            e1.record(stream)
            eng.sync()
            return e0.elapsed_time(e1)
        use = chunks if limit is None else chunks[:limit]
        evs = []
        eng.begin()
        for k, (f, m) in enumerate(use):
            if not resident_once:
                gen(f, m)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(stream)
            last = k == len(use) - 1
            eng.submit_device(dptr, m * rec, last)
            if last and not w.ec:
                merge_counts()
                eng.end_async(pin_res[0])
            e1.record(stream)
            evs.append((e0, e1))
        if w.ec:
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(stream)
            merge_counts()
            ec_stats.update(eng.end()[1])
            merge_ec()
            e1.record(stream)
            evs.append((e0, e1))
        eng.sync()
        return sum(a.elapsed_time(b) for a, b in evs)

    for _ in range(3):                                                        # warm-up
        resident_pass(limit=min(2, len(chunks)) if w.n_samples == 1 else None)
    barrier()
    n_pass = env["args"].steps
    l0 = eng.launches
    t_w0 = time.perf_counter()
    ms_res = sum(resident_pass() for _ in range(n_pass)) / n_pass
    env["windows"].append((t_w0, time.perf_counter()))
    launches = (eng.launches - l0) // n_pass
    kt = eng.kernel_times()
    if not w.ec:
        c_k, s_k = eng.read_async_result(pin_res[-1] if w.n_samples > 1 else pin_res[0])
        exp_reads = w.reads if w.n_samples > 1 else total_reads
        assert s_k["reads"] == exp_reads, (w.name, s_k, exp_reads)
    dump = env["dump"]
    if dump and w.ec:
        dump.save_table(w.name + "_table", eng.ec_items())
        dump.save_stats(w.name + "_stats", ec_stats)
    elif dump and w.n_samples > 1:
        res = [eng.read_async_result(b) for b in pin_res]                   # this rank's samples
        dump.save(w.name + "_counts", [c for c, _ in res])
        dump.save_stats(w.name + "_stats", [s for _, s in res])
    elif dump:
        dump.save(w.name + "_counts", c_k)
        dump.save_stats(w.name + "_stats", s_k)
    t = torch.tensor([ms_res], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_res = float(t.item())

    # ---- end to end: pinned host memory -> f2q_submit (H2D inside the timed region) -> counts on the host ----
    e2e = None
    if not env["args"].no_e2e and my_reads:
        if w.n_samples > 1:
            pin = lib.PinnedBuffer(len(my_samples) * w.reads * rec, local_rank)
            eng._ck(eng.L.f2q_memcpy_d2h(eng.h, pin.ptr, dptr, pin.nbytes))
        else:
            if not resident_once:
                gen(*chunks[0])
            pin = lib.PinnedBuffer(chunks[0][1] * rec, local_rank)
            eng._ck(eng.L.f2q_memcpy_d2h(eng.h, pin.ptr, dptr, pin.nbytes))

        def e2e_pass(limit=None):
            if w.n_samples > 1:
                for k in range(len(my_samples)):
                    eng.begin()
                    eng.submit_ptr(pin.ptr.value + k * w.reads * rec, w.reads * rec, True)
                    eng.end()
                return len(my_samples) * w.reads
            use = chunks if limit is None else chunks[:limit]
            eng.begin()
            done = 0
            for k, (f, m) in enumerate(use):
                eng.submit_ptr(pin.ptr.value, min(m, chunks[0][1]) * rec, k == len(use) - 1)
                done += min(m, chunks[0][1])
            merge_counts()
            eng.end()
            if w.ec:
                merge_ec()
            return done

        e2e_pass(limit=2 if w.n_samples == 1 else None)
        barrier()
        f0, f1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        tw = time.perf_counter()
        f0.record(stream)
        for _ in range(n_pass):
            done = e2e_pass()
        f1.record(stream)
        barrier()
        env["windows"].append((tw, time.perf_counter()))
        wall = (time.perf_counter() - tw) * 1e3 / n_pass
        ms2 = f0.elapsed_time(f1) / n_pass
        t = torch.tensor([ms2, wall, float(done)], dtype=torch.float64, device=dev)
        if world > 1:
            tm = t.clone()
            dist.all_reduce(tm, op=dist.ReduceOp.MAX)
            ts = t.clone()
            dist.all_reduce(ts, op=dist.ReduceOp.SUM)
            ms2, wall, done_all = float(tm[0]), float(tm[1]), float(ts[2])
        else:
            done_all = float(done)
        e2e = {"value": done_all / (ms2 / 1e3) / 1e6, "unit": "M reads/s", "ms_per_step": ms2, "wall_ms_per_step": wall,
               "h2d_bytes_per_step": int(done * rec), "d2h_bytes_per_step": (n_keys + 5) * 8 * max(1, len(my_samples) if w.n_samples > 1 else 1),
               "h2d_gbs_per_gpu": done * rec / (ms2 / 1e3) / 1e9,
               "note": ("one pinned chunk of %d reads re-submitted per chunk of the stream" % chunks[0][1]) if (w.n_samples == 1 and len(chunks) > 1) else
                       "every byte of the step copied from pinned host memory"}
        pin.free()
    for b in pin_res:
        b.free()
    eng.close()
    del data
    torch.cuda.empty_cache()

    if rank != 0:
        return None
    peak, peak_src = measured_peak()
    per_gpu_bytes = my_reads * rec
    tile_ms, tile_n = kt["tile"]
    scale_k = 1                                                              # (kernel times accumulate over the samples of a pass)
    tile_total = tile_ms * scale_k
    return {
        "workload": w.label, "value": total_reads / (ms_res / 1e3) / 1e6, "unit": "M reads/s", "ms_per_step": ms_res,
        "scaling": w.scaling, "reads_per_step": total_reads, "reads_per_gpu": my_reads, "bytes_per_read": rec,
        "chunks_per_gpu": len(chunks) if w.n_samples == 1 else len(my_samples), "gpu_launches_per_step": launches,
        "kernel_ms_per_step": {"tile": tile_total, "resolve": kt["resolve"][0] * scale_k, "generic": kt["generic"][0] * scale_k,
                               "verify_commit_fallback": kt["aux"][0] * scale_k},
        "roofline": {"bound": "hbm", "unit": "GB/s", "peak": peak, "peak_source": peak_src,
                     "achieved": per_gpu_bytes / (tile_total / 1e3) / 1e9 if tile_total > 0 else None,
                     "frac": per_gpu_bytes / (tile_total / 1e3) / 1e9 / peak if tile_total > 0 else None,
                     "whole_step_frac": per_gpu_bytes / (ms_res / 1e3) / 1e9 / peak,
                     "kernel": "the fused streaming kernel(s) over the chunk (kernel class 'tile' of f2q_kernel_times)",
                     "algorithmic_bytes_per_step_per_gpu": per_gpu_bytes},
        "e2e": e2e, "parity": parity,
    }


def run_gpu(args, rank, local_rank, world):
    import torch
    import torch.distributed as dist
    f2q = importlib.import_module("2fast2q_b200")
    lib = f2q._lib
    multi = importlib.import_module("2fast2q_b200.multi")
    host_mod = importlib.import_module("2fast2q_b200.fast2q")
    lib.load()                                                     # raises if the CUDA library is missing
    torch.cuda.set_device(local_rank)
    try:
        gpu_uuid = str(torch.cuda.get_device_properties(local_rank).uuid)
    except Exception:
        gpu_uuid = None
    placement = numa_bind(gpu_uuid, local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    dev = torch.device("cuda", local_rank)
    stream = torch.cuda.Stream(device=dev)
    want = set(args.configs.split(","))
    comm_eng = None
    if world > 1:
        # one NCCL communicator per rank for libf2q's own collectives (f2q_comm_*); the 128-byte id travels over torch.distributed
        comm_eng = lib.Engine(lib.make_config(), local_rank, stream.cuda_stream)
        box = [lib.comm_unique_id() if rank == 0 else None]
        dist.broadcast_object_list(box, src=0)
        comm_eng.comm_init_rank(box[0], world, rank)
    clocks = ClockSampler(local_rank, gpu_uuid)
    windows = []
    dump = OutputDump(args.dump_outputs) if args.dump_outputs and rank == 0 else None
    out = None

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    if want & {"headline", "all"}:
        (names, keys), spec = library()
        n_reads = args.reads
        nbytes = n_reads * REC
        cfg = lib.make_config(mode="C", miss=1, phred=30, length=FEAT_LEN, start="0")
        opts = {"time_kernels": 1}
        if args.tile_threads:
            opts["tile_threads"] = args.tile_threads
        eng = lib.Engine(cfg, local_rank, stream.cuda_stream, **opts)
        eng.set_library(keys)
        data = torch.empty(nbytes, dtype=torch.uint8, device=dev)
        eng.synth(data.data_ptr(), keys, rank * n_reads, n_reads, **spec)      # every rank owns its own contiguous read range
        if world > 1:
            eng.comm_share(comm_eng)

        def merge():
            if world > 1:
                eng.allreduce_counts()                   # f2q_allreduce_counts: ncclAllReduce(sum, uint64) of [counts | stats] over NVLink

        def step_resident():
            eng.begin()
            eng.submit_device(data.data_ptr(), nbytes, True)
            merge()
            return eng.end()

        # ---- resident leg ----
        for _ in range(args.warmup):
            counts, stats = step_resident()
        assert stats["reads"] == n_reads * world, stats
        tile_ms = []
        if rank == 0 and not os.environ.get("F2Q_BENCH_NO_CLOCKS"):
            clocks.start()
        barrier()
        l0 = eng.launches
        # the K timed passes run back to back: each one ends with f2q_end_sample_async, i.e. its [counts | stats] vector is
        # copied into its own pinned host buffer, stream-ordered, and checked after the timed region (no host round trip
        # between passes; the end-to-end leg below does the blocking read every step)
        res_bufs = [lib.PinnedBuffer(8 * (len(keys) + 6)) for _ in range(args.steps)]
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        w_res0 = time.perf_counter()
        e0.record(stream)
        for k in range(args.steps):
            eng.begin()
            eng.submit_device(data.data_ptr(), nbytes, True)
            merge()
            eng.end_async(res_bufs[k])
        e1.record(stream)
        barrier()
        eng.sync()
        windows.append((w_res0, time.perf_counter()))
        tile_ms.append(eng.kernel_times()["tile"])
        for b in res_bufs:
            c_k, s_k = eng.read_async_result(b)
            assert s_k == stats and np.array_equal(c_k, counts), "a timed pass returned different counts"
            b.free()
        if dump:
            dump.save("headline_counts", c_k)
            dump.save_stats("headline_stats", s_k)
        launches = eng.launches - l0
        ms = e0.elapsed_time(e1) / args.steps
        t = torch.tensor([ms], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms_res = float(t.item())
        ktimes = eng.kernel_times()
        spec_counts = eng.spec_counts()

        # ---- end-to-end leg: host (pinned) buffers through f2q_submit ----
        e2e = None
        if not args.no_e2e:
            pin = lib.PinnedBuffer(nbytes, local_rank, write_combined=args.pinned == "wc")      # near this rank's GPU (f2q_host_alloc_near)
            eng._ck(eng.L.f2q_memcpy_d2h(eng.h, pin.ptr, data.data_ptr(), nbytes))

            def step_e2e():
                eng.begin()
                eng.submit_ptr(pin.ptr.value, nbytes, True)
                merge()
                return eng.end()

            for _ in range(max(1, min(args.warmup, 3))):
                c2, s2 = step_e2e()
            assert s2 == stats and np.array_equal(c2, counts)
            # the ingest roofline: a plain pinned -> device copy of the same bytes on the same link (best of 2)
            pcie = 0.0
            for _ in range(2):
                torch.cuda.synchronize(dev)
                tp = time.perf_counter()
                eng.h2d(data.data_ptr(), pin.array)
                pcie = max(pcie, nbytes / (time.perf_counter() - tp) / 1e9)
            barrier()
            f0, f1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            t0 = time.perf_counter()
            f0.record(stream)
            for _ in range(args.steps):
                c2, s2 = step_e2e()
            f1.record(stream)
            barrier()
            windows.append((t0, time.perf_counter()))
            wall = (time.perf_counter() - t0) / args.steps * 1e3
            ms2 = max(f0.elapsed_time(f1) / args.steps, 0.0)
            if dump:
                dump.save("headline_e2e_counts", c2)
                dump.save_stats("headline_e2e_stats", s2)
            t = torch.tensor([ms2, wall], dtype=torch.float64, device=dev)
            if world > 1:
                dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms2, wall = float(t[0].item()), float(t[1].item())
            e2e = {"value": world * n_reads / (ms2 / 1e3) / 1e6, "unit": "M reads/s", "h2d_bytes_per_step": nbytes,
                   "d2h_bytes_per_step": (len(keys) + 5) * 8, "ms_per_step": ms2, "wall_ms_per_step": wall,
                   "h2d_gbs_per_gpu": nbytes / (ms2 / 1e3) / 1e9, "pcie_copy_gbs_measured": pcie,
                   "pinned_numa_node": pin.numa_node, "pinned_kind": args.pinned,
                   "pcie_frac": (nbytes / (ms2 / 1e3) / 1e9) / pcie if pcie else None}
            pin.free()

        if rank == 0:
            peak, peak_src = measured_peak()
            tm = [m for m, n in tile_ms if n]
            tile_avg = sum(tm) / max(1, sum(n for m, n in tile_ms if n))            # ms per tile-kernel launch
            achieved = n_reads * REC / (tile_avg / 1e3) / 1e9 if tile_avg > 0 else None
            traffic = committed_traffic()
            out = {
                "metric": "M reads/s", "value": world * n_reads / (ms_res / 1e3) / 1e6, "unit": "M reads/s", "n_gpus": world,
                "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_res, "higher_is_better": True, "scaling": "weak",
                "vs_baseline": None, "dtype": "u8", "data": "synthetic",
                "config": {"workload": WORKLOAD,
                           "reads_per_gpu": n_reads, "bytes_per_read": REC, "input_bytes_per_gpu": nbytes,
                           "l2": "inputs (%.1f GB/GPU) are far larger than the 126 MB L2; no flush needed" % (nbytes / 1e9),
                           "parallelism": f"reads sharded by contiguous range over {world} GPU(s); counts merged by f2q_allreduce_counts (ncclAllReduce, uint64 sum)",
                           "host_placement": placement, "host_topology": host_topology()},
                "e2e": e2e,
                "gpu_launches": launches,
                "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s",
                             "frac": (achieved / peak) if achieved else None,
                             "traffic": traffic["dram_bytes_per_read"] * n_reads if traffic else None,
                             "kernel": "k_spec<POLICY_FAST1, CH=7, W=16> (speculative streaming kernel, csrc/spec.cuh)",
                             "kernel_ms_per_launch": tile_avg, "peak_source": peak_src,
                             "algorithmic_bytes_per_launch": n_reads * REC,
                             "other_kernels_ms_per_step": {"resolve": ktimes["resolve"][0] / args.steps, "generic": ktimes["generic"][0] / args.steps,
                                                           "verify_commit_fallback": ktimes["aux"][0] / args.steps},
                             "host_gap_ms_per_step": ms_res - (tile_avg + (ktimes["resolve"][0] + ktimes["generic"][0] + ktimes["aux"][0]) / args.steps),
                             "traffic_note": traffic.get("note") if traffic else "no committed ncu --set full capture yet"},
                "speculation": {"chunks_committed": spec_counts[0], "chunks_parsed_by_exact_kernel": spec_counts[1]},
                "stats": stats,
            }
            if not args.no_cpu:
                out["cpu_baseline"], out["parity"] = cpu_baseline_and_parity(eng, data.data_ptr(), args.cpu_reads, keys)
        eng.close()
        del data
        torch.cuda.empty_cache()
    elif rank == 0:
        if not os.environ.get("F2Q_BENCH_NO_CLOCKS"):
            clocks.start()
        out = {"metric": "M reads/s", "value": None, "unit": "M reads/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
               "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u8", "data": "synthetic",
               "config": {"workload": "headline skipped (--configs)"}}

    # ---- the other BASELINE shapes ----
    others = {}
    if want - {"headline"}:
        env = dict(lib=lib, multi=multi, host=host_mod, rank=rank, world=world, dev=dev, stream=stream, local_rank=local_rank,
                   args=args, windows=windows, comm=comm_eng, dump=dump)
        for name, w in build_workloads(args).items():
            t0 = time.perf_counter()
            r = run_workload(w, env)
            if rank == 0:
                r["bench_wall_s"] = round(time.perf_counter() - t0, 1)
                others[name] = r
                log(name, "%.1f M reads/s resident, e2e %s, %.1f s" % (r["value"], ("%.1f" % r["e2e"]["value"]) if r["e2e"] else "-", r["bench_wall_s"]))
    if rank == 0:
        out["other_configs"] = others
        out["clocks"] = clocks.stop(windows)
        emit(out)
    if comm_eng is not None:
        comm_eng.close()
    if world > 1:
        dist.destroy_process_group()


def cpu_baseline_and_parity(eng, dptr, n, keys):
    """oracle port on the first n reads of rank 0's stream, one core (the reported CPU baseline) — and the parity check of
    the benchmarked workload itself: the GPU's counts of those n reads must equal the oracle's"""
    from oracle import oracle as O
    host = eng.d2h(dptr, n * REC)
    cfg = O.make_config(miss=1, phred=30, length=FEAT_LEN, start="0")
    O.lib()
    t0 = time.perf_counter()
    want_c, want_s = O.count(cfg, keys, host)
    dt = time.perf_counter() - t0
    eng.begin()
    eng.submit_device(dptr, n * REC, True)
    got_c, got_s = eng.end()
    assert got_s == want_s, ("headline parity: stats differ", got_s, want_s)
    assert np.array_equal(got_c, want_c), ("headline parity: counts differ", int((got_c != want_c).sum()))
    base = {"value": n / dt / 1e6, "unit": "M reads/s", "cores": 1, "kind": "port",
            "sample": f"first {n} reads of the same synthetic stream, oracle/f2q_oracle.c single thread, {dt:.1f} s"}
    return base, {"reads": n, "ok": True, "stats": got_s, "checker": "oracle/f2q_oracle.c, bit-exact counts + stats of the first reads of the benchmarked stream"}


def host_topology():
    """what the box shows about host memory placement (a VM usually shows ONE node, whatever the hardware below it has)"""
    import glob
    nodes = sorted(glob.glob("/sys/devices/system/node/node[0-9]*"))
    gpus = {}
    for d in glob.glob("/sys/bus/pci/devices/*"):
        try:
            if open(os.path.join(d, "class")).read().startswith("0x0302"):
                gpus[os.path.basename(d)] = int(open(os.path.join(d, "numa_node")).read())
        except (OSError, ValueError):
            pass
    return {"numa_nodes_visible": len(nodes), "gpu_numa_node": gpus, "cpus": os.cpu_count(),
            "cpus_allowed": len(os.sched_getaffinity(0))}


def numa_bind(gpu_uuid, gpu_index):
    """run this rank (and first-touch its pinned buffers) on the CPUs nearest to its GPU, when the container allows it"""
    try:
        import pynvml as nv
        nv.nvmlInit()
        try:
            h = nv.nvmlDeviceGetHandleByUUID(f"GPU-{gpu_uuid}".encode()) if gpu_uuid else nv.nvmlDeviceGetHandleByIndex(gpu_index)
        except Exception:
            h = nv.nvmlDeviceGetHandleByIndex(gpu_index)
        allowed = os.sched_getaffinity(0)
        words = nv.nvmlDeviceGetCpuAffinity(h, (max(allowed) // 64) + 1)
        ideal = {64 * w + b for w, x in enumerate(words) for b in range(64) if (int(x) >> b) & 1}
        both = allowed & ideal
        if both and both != allowed:
            os.sched_setaffinity(0, both)
            return f"bound to {len(both)} of {len(allowed)} allowed CPUs near the GPU"
        return "not bound (all allowed CPUs are equally near, or none is)"
    except Exception as e:                                        # noqa: BLE001 — placement is an optimisation only
        return f"not bound ({type(e).__name__})"


def main():
    # anything a library prints on stdout (NCCL's version banner) must not precede the ONE JSON line: fd 1 -> stderr,
    # the line itself goes to the saved descriptor
    global _JSON_OUT
    sys.stdout.flush()
    _JSON_OUT = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="f2q")
    ap.add_argument("--reads", type=int, default=100_000_000, help="reads per GPU of the headline (configs[1] = 100 M)")
    ap.add_argument("--configs", default="all", help="comma list of headline,north_star,config3,config4,config5a,config5b (default all)")
    ap.add_argument("--scale", type=float, default=1.0, help="size factor of the other_configs workloads (development runs)")
    ap.add_argument("--cpu-reads", type=int, default=6_000_000)
    ap.add_argument("--ref-reads-per-thread", type=int, default=400_000)
    ap.add_argument("--real-ref-reads", type=int, default=1_600_000)
    ap.add_argument("--no-real-reference", action="store_true")
    ap.add_argument("--tile-threads", type=int, default=0)
    ap.add_argument("--pinned", default="default", choices=["default", "wc"], help="pinned host memory of the end-to-end leg: default | write-combined")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write what the last timed step of each leg returned as DIR/<name>.npy")
    args = ap.parse_args()
    args.warmup = max(args.warmup, 3) if args.impl != "reference" else args.warmup
    rank, local_rank, world = env_int("RANK", 0), env_int("LOCAL_RANK", 0), env_int("WORLD_SIZE", 1)
    if args.impl == "reference":
        run_reference(args, rank, world)
    else:
        run_gpu(args, rank, local_rank, world)


if __name__ == "__main__":
    main()
