"""
Scaling of one file over several contexts (f2q_submit_file_sharded): file -> counts, host clock from the submit to the end of
f2q_end_sample, with a parity check of every run against the one-context result.

    python tools/shard_probe.py [--gb 4] [--dir /dev/shm] [--reps 2] [--out shard_probe.json]

Inputs (seeded, written to --dir and removed afterwards): a plain FASTQ file of config-2 reads (2 000 guides, m = 1) of at
least --gb GB, generated on the GPU, and the same file as bgzip.  Reported per input: GB/s of FASTQ text and M reads/s for
n = 1, 2, ... contexts with one context per visible GPU, and n = 2 and 4 contexts sharing GPU 0; plus the GPU name and power
limit, read in the same run.
"""
import argparse
import importlib
import json
import os
import struct
import subprocess
import sys
import time
import zlib
from concurrent.futures import ThreadPoolExecutor

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
lib = importlib.import_module("2fast2q_b200._lib")
synth = importlib.import_module("2fast2q_b200.synth")


def bgzf_block(chunk, level=1):
    c = zlib.compressobj(level, zlib.DEFLATED, -15)
    cd = c.compress(chunk) + c.flush()
    return (b"\x1f\x8b\x08\x04\x00\x00\x00\x00\x00\xff\x06\x00BC\x02\x00" + struct.pack("<H", 18 + len(cd) + 8 - 1) + cd
            + struct.pack("<II", zlib.crc32(chunk) & 0xFFFFFFFF, len(chunk)))


def make_inputs(d, gb, keys, spec):
    rec = 2 * spec["read_len"] + 18
    n_reads = int(gb * 1e9) // rec + 1
    plain, bgz = os.path.join(d, "shard_probe.fastq"), os.path.join(d, "shard_probe.fastq.gz")
    per = (1 << 30) // rec
    pool = ThreadPoolExecutor(max(2, os.cpu_count() or 2))
    with lib.Engine(lib.make_config(miss=1), 0) as e, open(plain, "wb") as fp, open(bgz, "wb") as fz:
        dptr = e.device_alloc(per * rec)
        for first in range(0, n_reads, per):
            n = min(per, n_reads - first)
            e.synth(dptr, keys, first, n, **spec)
            text = e.d2h(dptr, n * rec).tobytes()
            fp.write(text)
            for blk in pool.map(bgzf_block, [text[o:o + 65280] for o in range(0, len(text), 65280)]):
                fz.write(blk)
        fz.write(bgzf_block(b""))
        e.device_free(dptr)
    pool.shutdown()
    return plain, bgz, n_reads, n_reads * rec


def run(keys, path, gz, devices, reps):
    cfg = lib.make_config(miss=1)
    engines = [lib.Engine(cfg, d, memo_entries=1 << 20) for d in devices]
    try:
        for e in engines:
            e.set_library(keys)
        times, out = [], None
        for _ in range(reps + 1):                                   # (the first pass allocates rings and staging: warm-up)
            for e in engines:
                e.begin()
            t0 = time.perf_counter()
            lib.submit_file_sharded(engines, path, gz, threads=16)
            counts, stats = engines[0].end()
            times.append(time.perf_counter() - t0)
            shards, fb = engines[0].info("shards"), engines[0].info("shard_fallback")
            for e in engines[1:]:
                e.end()
            out = (counts, stats, shards, fb)
        return times[1:], out
    finally:
        for e in engines:
            e.close()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gb", type=float, default=4.0)
    ap.add_argument("--dir", default="/dev/shm")
    ap.add_argument("--reps", type=int, default=2)
    ap.add_argument("--out", default="shard_probe.json", help="where the JSON report goes")
    a = ap.parse_args()
    n_dev = lib.device_count()
    assert n_dev >= 1, "no B200 visible"
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=index,name,power.limit", "--format=csv,noheader"], capture_output=True, text=True).stdout.strip()
    spec = synth.default_spec(2)
    names, keys = synth.make_library(2, 2000, 20)
    st = os.statvfs(a.dir)
    if st.f_bavail * st.f_frsize < 2.2 * a.gb * 1e9:
        raise SystemExit(f"{a.dir} has no room for {2.2 * a.gb:.1f} GB of inputs: pass --dir")
    t0 = time.perf_counter()
    plain, bgz, n_reads, text_bytes = make_inputs(a.dir, a.gb, keys, spec)
    report = dict(gpus=gpu.splitlines(), visible_gpus=n_dev, reads=n_reads, text_bytes=text_bytes, plain_bytes=os.path.getsize(plain),
                  bgzip_bytes=os.path.getsize(bgz), input_seconds=round(time.perf_counter() - t0, 1), runs=[])
    try:
        layouts = [("one per GPU", list(range(n))) for n in range(1, n_dev + 1)] + [("GPU 0 shared", [0] * n) for n in (2, 4)]
        for fmt, path, gz in (("plain", plain, False), ("bgzip", bgz, True)):
            ref = None
            for kind, devices in layouts:
                times, (counts, stats, shards, fb) = run(keys, path, gz, devices, a.reps)
                if ref is None:
                    ref = (counts, stats)
                parity = bool(np.array_equal(counts, ref[0]) and stats == ref[1])
                best = min(times)
                row = dict(input=fmt, layout=kind, contexts=len(devices), shards=shards, fallback=fb, seconds=[round(t, 3) for t in times],
                           text_GBps=round(text_bytes / best / 1e9, 2), Mreads_per_s=round(n_reads / best / 1e6, 1), parity_with_n1=parity)
                report["runs"].append(row)
                print(json.dumps(row), flush=True)
        report["not_measured"] = f"more than {n_dev} GPU(s)"
    finally:
        for p in (plain, bgz):
            if os.path.exists(p):
                os.remove(p)
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(report, f, indent=1)
    print(json.dumps(dict(gpus=report["gpus"], reads=n_reads, text_bytes=text_bytes)))


if __name__ == "__main__":
    main()
