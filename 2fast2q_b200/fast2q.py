"""
Host-side mirror of the reference's interface for the read -> feature -> count path (2FAST2Q v2.8.1,
fast2q/fast2q.py).  Same function names, argument meaning, outputs and error behaviour as the reference, so
that `python -m 2fast2q_b200 -c ...` is a drop-in for `2fast2q -c ...`; the work between "bytes of FASTQ" and
"count vector + 5 statistics" is done by libf2q.so (CUDA, sm_100a) through ctypes (_lib.py).

    reference (fast2q.py)                      here
    -------------------------------------------------------------------------------------------
    Features :21-44                            Features
    colourful_errors :46-67                    colourful_errors (no colours)
    path_finder / path_parser :69-123          same names
    features_loader :125-186                   features_loader
    reads_counter :514-582  (boundary)         reads_counter  -> Engine (f2q_begin_sample/f2q_submit/f2q_end_sample)
    fastq_parser :306-409, sequence_tinder,    CUDA kernels behind the C-ABI (csrc/)
      border_finder, features_all_vs_all,
      mismatch_search_handler
    seq2bin :584-599                           seq2bin (host, numpy)
    border_finder / sequence_tinder (public    border_finder / sequence_tinder -> f2q_border_finder /
      helpers, README.md:259-298)                f2q_sequence_tinder (device)
    aligner :752-801, csv_writer :803-809      aligner, csv_writer
    initializer :1082-1169                     initializer
    input_parser :1171-1314                    input_parser (+ --gpus, an addition)
    compiling :1316-1384, run_stats :1386-1412 compiling, run_stats (csv half; the PNG plots are out of scope)
    aligner_mp_dispenser :1619-1655,           aligner_mp_dispenser: files over GPUs (feeder threads), or one file
      single_file_reads_binner :411-512          cut at record boundaries into shards over all GPUs
    file_sizer_split :1657-1689, main :1691    same names

There is no CPU implementation of the path here: without libf2q.so or without a B200-class device every
counting call raises.
"""
from __future__ import annotations

import argparse
import csv
import datetime
import glob
import gzip
import os
import queue
import io
import sys
import threading
import time
import zlib
from dataclasses import dataclass
from pathlib import Path

import numpy as np

from . import _lib

version = "2.8.1"            # the reference version whose command-line surface and outputs are reproduced

STAT_KEYS = _lib.STAT_NAMES  # reads, perfect_counter, imperfect_counter, non_aligned_counter, quality_failed


@dataclass
class Features:
    """value type of the library dict keyed by sequence (fast2q.py:21-44)"""
    name: str
    counts: int


def colourful_errors(warning_type, error):
    """timestamped console message (fast2q.py:46-67, without the colours)"""
    print(f" {datetime.datetime.now().strftime('%c')} [{warning_type}] {error}", flush=True)


# ------------------------------------------------------------------------------------------------------------
# file discovery (fast2q.py:69-123)
# ------------------------------------------------------------------------------------------------------------
def path_finder(folder_path, extension):
    found = []
    for pattern in extension:
        for filename in glob.glob(os.path.join(folder_path, pattern)):
            found.append([filename, os.path.getsize(filename)])
    return found


def path_parser(folder_path, extension):
    """sequencing files: [path, size] pairs sorted by size; '*reads.csv': paths sorted by name"""
    found = path_finder(folder_path, extension)
    if extension != ['*reads.csv']:
        ordered = sorted(found, key=lambda e: e[-1])
        if not ordered:
            colourful_errors("FATAL", f"Check the path to the {extension} files folder. No files of this type found.\n")
            sys.exit()
        return ordered
    return [p[0] for p in sorted(found)]


# ------------------------------------------------------------------------------------------------------------
# features .csv loader (fast2q.py:125-186)
# ------------------------------------------------------------------------------------------------------------
def features_loader(guides):
    """features .csv -> dict[sequence] = Features(name, 0).

    Semantics kept from the reference: the file is parsed three times (',', ';', tab) into the SAME dict; a line
    without a second column ends that separator's pass (everything loaded before it stays); the sequence is
    column 2 upper-cased with blanks removed, the name is column 1 untouched; the first name wins a shared
    sequence; a repeated name only warns."""
    colourful_errors("INFO", "Loading Features")
    if not os.path.isfile(guides):
        colourful_errors("FATAL", f"Check the path to the features file.\nNo .csv file found in the following path: {guides}\n")
        sys.exit()

    features = {}
    for separator in (",", ";", "\t"):
        names = set()
        with open(guides) as handle:
            for line in handle:
                cols = line.rstrip().split(separator)
                if len(cols) < 2:
                    break                                   # IndexError in the reference: this pass is over
                name, sequence = cols[0], cols[1].upper().replace(" ", "")
                if name in names:
                    colourful_errors("WARNING", f"The name {name} seems to appear at least twice. This MIGHT result in unexpected "
                                     "behaviour. Please have only unique name entries in your features.csv file.")
                if sequence not in features:
                    features[sequence] = Features(name, 0)
                    names.add(name)
                else:
                    colourful_errors("WARNING", f"{features[sequence].name} and {name} share the same sequence. Only "
                                     f"{features[sequence].name} will be considered valid. {name} will be ignored.")
    if not features:
        colourful_errors("FATAL", "The given .csv file doesn't seem to be comma, semicolon, or tab separated. Please double "
                         "check that the file's column separation\n")
        sys.exit()
    colourful_errors("INFO", f"{len(features)} different features were provided.")
    return features


# ------------------------------------------------------------------------------------------------------------
# public helpers (README.md:259-298, tests/test_mainfunctions.py)
# ------------------------------------------------------------------------------------------------------------
def seq2bin(sequence):
    """str -> int8 array of its UTF-8 bytes (fast2q.py:584-599)"""
    return np.array(bytearray(sequence, "utf8"), dtype=np.int8)


def _as_bytes(x):
    if isinstance(x, np.ndarray):
        return x.astype(np.int8).tobytes()
    if isinstance(x, str):
        return x.encode()
    return bytes(x)


def border_finder(seq, read, mismatch, start_place=0):
    """first index >= start_place where `seq` occurs in `read` with <= mismatch mismatches, else None
    (fast2q.py:628-658); evaluated by the device kernel behind f2q_border_finder"""
    return _lib.border_finder_device(_as_bytes(seq), _as_bytes(read), int(mismatch), int(start_place))


def sequence_tinder(read_bin, qual, param, i=0):
    """(start, end) of the feature between / next to the search sequences, or (None, None) (fast2q.py:215-285);
    evaluated by the device kernel behind f2q_sequence_tinder.  `param` as in the reference: upstream/downstream
    (str or None), upstream_bin/downstream_bin (lists), miss_search_up/down, quality_set_up/down, length."""
    up = [_as_bytes(b) for b in param.get("upstream_bin", [])] if param.get("upstream") is not None else None
    down = [_as_bytes(b) for b in param.get("downstream_bin", [])] if param.get("downstream") is not None else None
    cfg = _lib.Config()
    cfg.length = int(param.get("length", 20))
    cfg.miss_up, cfg.miss_down = int(param.get("miss_search_up", 0)), int(param.get("miss_search_down", 0))
    cfg.has_up, cfg.has_down = int(up is not None), int(down is not None)
    cfg.n_iter = max(len(up or []), len(down or []), 1)
    for dst, dlen, items in ((cfg.up, cfg.up_len, up or []), (cfg.down, cfg.down_len, down or [])):
        for k, u in enumerate(items):
            dlen[k] = len(u)
            for j, b in enumerate(u):
                dst[k][j] = b
    return _lib.sequence_tinder_device(cfg, _as_bytes(read_bin), _as_bytes(qual), i,
                                       set_up=param.get("quality_set_up", set()), set_down=param.get("quality_set_down", set()))


# ------------------------------------------------------------------------------------------------------------
# uncompressed byte stream of one sequencing file (replaces `for line in current`, fast2q.py:566-578)
# ------------------------------------------------------------------------------------------------------------
CHUNK_BYTES = 32 << 20
SPLIT_NATIVE_SINGLE_GPU = True      # File-Split mode streams each file through the native ingest of ONE GPU instead of sharding it in Python


class TruncatedGzip(Exception):
    """the gzip stream ended before its end-of-stream marker (the reference's EOFError, fast2q.py:405-407)"""


def _bgzf_block_size(hdr):
    """total size of the BGZF block that starts with these (>= 18) bytes, or None when this is not a BGZF member
    (gzip member with FEXTRA whose first subfield is 'B','C' of length 2 holding BSIZE-1: SAM spec §4.1)"""
    if len(hdr) < 18 or hdr[:4] != b"\x1f\x8b\x08\x04" or hdr[12:16] != b"BC\x02\x00" or (hdr[10] | hdr[11] << 8) < 6:
        return None
    return (hdr[16] | hdr[17] << 8) + 1


_inflate_pool = None
_inflate_pool_lock = threading.Lock()
_BGZF_EOF = bytes.fromhex("1f8b08040000000000ff0600424302001b0003000000000000000000")


def _input_kind(files):
    """'gzip' when any file is an ordinary gzip stream (host zlib), else 'bgzf' / 'plain' (the context's own readers)"""
    kind = "plain"
    for raw in files:
        if not raw.endswith(".gz"):
            continue
        try:
            with open(raw, "rb") as f:
                head = f.read(18)
                f.seek(0, os.SEEK_END)
                size = f.tell()
                tail = b""
                if size >= 28:
                    f.seek(size - 28)
                    tail = f.read(28)
        except OSError:
            return "gzip"
        if _bgzf_block_size(head) and tail == _BGZF_EOF:
            kind = "bgzf"
        else:
            return "gzip"
    return kind


_INFLATE_WORKERS = max(2, min(32, os.cpu_count() or 2))


def _shared_inflate_pool():
    """one pool of inflate workers for the whole process (zlib releases the GIL): feeder threads of several files share it"""
    global _inflate_pool
    with _inflate_pool_lock:
        if _inflate_pool is None:
            from concurrent.futures import ThreadPoolExecutor
            _inflate_pool = ThreadPoolExecutor(_INFLATE_WORKERS, thread_name_prefix="f2q-inflate")
        return _inflate_pool


def _inflate_serial(f, want, pending=b""):
    """the generic path: one zlib stream at a time, multi-member files and zero padding between members included"""
    d = zlib.decompressobj(31)
    fresh = True                                            # at a member boundary, nothing consumed yet
    while True:
        if not pending:
            pending = f.read(4 << 20)
            if not pending:
                if fresh:
                    return
                raise TruncatedGzip(getattr(f, "name", "gzip stream"))
        if fresh:
            pending = pending.lstrip(b"\x00")               # padding between members is skipped (gzip module behaviour)
            if not pending:
                continue
            fresh = False
        out = d.decompress(pending, want)
        pending = d.unconsumed_tail
        if out:
            yield out
        if d.eof:
            pending = d.unused_data
            d = zlib.decompressobj(31)
            fresh = True


def _inflate_group(blob, sizes):
    """a run of whole BGZF blocks (their sizes in order) -> their uncompressed bytes"""
    mv, out, pos = memoryview(blob), [], 0
    for n in sizes:
        out.append(zlib.decompress(mv[pos:pos + n], 31))
        pos += n
    return b"".join(out)


def _inflate_blocks(path, want=None, parallel=True):
    """yields the uncompressed bytes of a (multi-member) gzip file in pieces of <= want bytes.  zlib releases the GIL, so
    several feeder threads inflate in parallel; a BGZF file (bgzip: independent blocks of <= 64 KiB that carry their own
    size) is additionally inflated block-parallel on the shared pool, in order, with a bounded number of groups in
    flight (SURVEY.md §8f rank 1: host zlib on ONE stream is the end-to-end bound of a single-file run).
    Raises TruncatedGzip after the last decodable piece."""
    want = want or CHUNK_BYTES
    group_bytes = 4 << 20                                   # compressed bytes per task (<= ~16 MiB uncompressed <= want)
    with open(path, "rb") as f:
        head = f.read(18)
        if not (parallel and _bgzf_block_size(head)):
            yield from _inflate_serial(f, want, head)
            return
        pool = _shared_inflate_pool()
        depth = 2 * _INFLATE_WORKERS
        inflight = []                                       # futures, in file order
        buf = head
        eof = False
        while True:
            # cut whole blocks off the front of buf into one group
            group_end, pos, fallback, sizes = 0, 0, False, []
            while pos + 18 <= len(buf) and group_end < group_bytes:
                n = _bgzf_block_size(buf[pos:pos + 18])
                if n is None:
                    fallback = True                         # not BGZF from here on (a foreign member was appended): serial
                    break
                if pos + n > len(buf):
                    break
                pos += n
                group_end = pos
                sizes.append(n)
            if group_end:
                inflight.append(pool.submit(_inflate_group, buf[:group_end], sizes))
                buf = buf[group_end:]
            while inflight and (len(inflight) >= depth or eof or fallback or inflight[0].done()):
                out = inflight.pop(0).result()
                for o in range(0, len(out), want):
                    yield out[o:o + want]
            if fallback or (eof and not group_end):
                break
            if not group_end or len(buf) < 18:
                more = f.read(group_bytes)
                if not more:
                    eof = True
                buf += more
        if buf:
            # what is left is a partial block (truncated file) or a non-BGZF continuation: the serial reader finishes it
            yield from _inflate_serial(f, want, buf)


def _raw_blocks(path, want=None):
    want = want or CHUNK_BYTES
    with open(path, "rb", buffering=0) as f:
        while True:
            b = f.read(want)
            if not b:
                return
            yield b


class _PinnedRing:
    """a few page-locked buffers a feeder cycles through (f2q_host_alloc_near: on the NUMA node of the GPU they feed);
    allocated on first use — the file mode streams through libf2q's own ring (f2q_submit_file) and never needs them"""

    def __init__(self, n=3, nbytes=None, device=None):
        self.nbytes = nbytes or CHUNK_BYTES
        self.n, self.device = n, device
        self.bufs = []
        self.k = 0

    def next(self):
        if not self.bufs:
            self.bufs = [_lib.PinnedBuffer(self.nbytes, self.device) for _ in range(self.n)]
        b = self.bufs[self.k % len(self.bufs)]
        self.k += 1
        return b

    def __len__(self):
        return self.n

    def free(self):
        for b in self.bufs:
            b.free()
        self.bufs = []


def _stream_file(engine, ring, raw, limit_lines=None):
    """feeds one file through the engine; returns False when the gzip stream was truncated.
    The work is native (f2q_submit_file): the file is read, or inflated with zlib — bgzip files block-parallel on host
    threads — straight into page-locked ring buffers near the GPU; no byte passes through a Python object.  While a gzip
    stream is open only whole lines are submitted, so a truncated stream ends exactly like the reference's line iterator:
    every complete line before the break is parsed, the partial one is dropped (fast2q.py:405-407)."""
    gz = os.path.splitext(raw)[1] == ".gz"
    try:
        complete, _ = engine.submit_file(raw, gz, limit_lines or 0, _INFLATE_WORKERS)
    except _lib.F2QError as e:
        if e.code == -1 and "corrupted gzip" in str(e):
            raise zlib.error(str(e)) from None
        if e.code == -1 and "cannot open" in str(e):
            raise OSError(str(e)) from None
        raise
    return complete


# ------------------------------------------------------------------------------------------------------------
# engines: one libf2q context per (thread, device, configuration, library)
# ------------------------------------------------------------------------------------------------------------
_tls = threading.local()


def _config_of(param):
    try:
        return _lib.make_config(mode=param["Running Mode"], miss=param["miss"], phred=param["phred"], length=param["length"],
                                start=param["start"], upstream=param["upstream"], downstream=param["downstream"],
                                miss_search_up=param["miss_search_up"], miss_search_down=param["miss_search_down"],
                                qual_up=param["qual_up"], qual_down=param["qual_down"])
    except ValueError as e:
        colourful_errors("FATAL", str(e))                   # fast2q.py:553-556
        sys.exit()


def _engine_for(param, features, device, slot=0):
    """cached per thread: creating a context and uploading a 100k-guide library once per file would dominate small files.
    `slot` keeps several engines of one thread apart (split_file_native: one per shard, several may share a device)"""
    cfg = _config_of(param)
    keys = list(features.keys()) if param["Running Mode"] == "C" else None
    sig = (device, bytes(cfg), None if keys is None else hash(tuple(keys)), slot)
    cache = getattr(_tls, "engines", None)
    if cache is None:
        cache = _tls.engines = {}
    if sig not in cache:
        for old_sig in [k for k in cache if k[-1] == slot]:
            old = cache.pop(old_sig)
            old[0].close(); old[1].free()
        # the device memo of resolved non-exact keys (the reference's passed_reads / failed_reads): real screens repeat them
        eng = _lib.Engine(cfg, device, memo_entries=1 << 20) if keys is not None else _lib.Engine(cfg, device)
        if keys is not None:
            eng.set_library(keys)
        cache[sig] = (eng, _PinnedRing(device=device))
    return cache[sig]


def release_engines():
    cache = getattr(_tls, "engines", None)
    if cache:
        t0 = time.perf_counter()
        for eng, ring in cache.values():
            eng.close(); ring.free()
        cache.clear()
        if os.environ.get("F2Q_CLI_TIMING"):
            print(f" [timing] engines of this thread released in {time.perf_counter() - t0:.3f} s", flush=True)


def _derive_positions(param):
    """the parameter derivation reads_counter performs on `param` (fast2q.py:536-558), kept for callers that look at it"""
    if param["upstream"] is None and param["downstream"] is None:
        param["start_positioning"] = [int(n) for n in str(param["start"]).split(",")]
        param["end_positioning"] = [n + int(param["length"]) for n in param["start_positioning"]]
        param["search_iterations"] = len(param["end_positioning"])
    else:
        n_up = n_down = 0
        if param["upstream"] is not None:
            param["upstream_bin"] = [seq2bin(n.upper()) for n in param["upstream"].split(",")]
            n_up = len(param["upstream_bin"])
        if param["downstream"] is not None:
            param["downstream_bin"] = [seq2bin(n.upper()) for n in param["downstream"].split(",")]
            n_down = len(param["downstream_bin"])
        if param["upstream"] is not None and param["downstream"] is not None and n_up != n_down:
            colourful_errors("FATAL", "Up and Downstream sequences must be submitted in concurrent pairs, separated by ,.\n "
                             f"You submitted {n_down} downstream sequences and {n_up} upstream sequences.")
            sys.exit()
        param["search_iterations"] = max(n_up, n_down)


def _features_from(param, features, counts, engine):
    """per-sample result dict in the reference's shape: Counter -> every library entry (zeros included) in library
    order; Extract+Count -> every key seen (fast2q.py:365-367, 382-387)"""
    if param["Running Mode"] == "C":
        return {seq: Features(f.name, int(c)) for (seq, f), c in zip(features.items(), counts)}
    out = {}
    for key, c in engine.ec_items().items():
        s = key.decode("latin-1")
        out[s] = Features(s, c)
    return out


def _count_file(raw, features, param, preprocess=False):
    """one file through the engine of this thread: (counts, stats, engine), or None when the file cannot be opened as gzip"""
    _derive_positions(param)
    device = int(param.get("device", 0))
    t_a = time.perf_counter()
    engine, ring = _engine_for(param, features, device)
    t_b = time.perf_counter()
    engine.begin()
    try:
        complete = _stream_file(engine, ring, raw, limit_lines=40000 if preprocess else None)
        if os.environ.get("F2Q_CLI_TIMING"):
            engine.sync()
            print(f" [timing] {os.path.basename(raw)}: engine {t_b - t_a:.3f} s, stream {time.perf_counter() - t_b:.3f} s", flush=True)
    except (zlib.error, gzip.BadGzipFile, EOFError) as e:     # (other I/O errors surface, as in the reference: fast2q.py:580)
        try:
            engine.end()
        except _lib.F2QError:
            pass
        colourful_errors("WARNING", f"{raw} is an incomplete or corrupted gzip file. ({e})")
        return None
    except BaseException:
        try:
            engine.end()                                     # leave the cached engine reusable
        except _lib.F2QError:
            pass
        raise
    try:
        counts, stats = engine.end()
    except _lib.F2QError as e:
        # a bgzip block inflated on the device that failed its size or CRC-32 check: reported when the sample ends
        if e.code == -1 and "corrupted gzip" in str(e):
            colourful_errors("WARNING", f"{raw} is an incomplete or corrupted gzip file. ({e})")
            return None
        raise
    if not complete:
        colourful_errors("WARNING", f"{raw} is an incomplete or corrupted gzip file. Only partial processing might have occurred.")
    return counts, stats, engine


def reads_counter(i, raw, features, param, reads_stats, preprocess=False):
    """THE drop-in boundary (fast2q.py:514-582): counts the reads of one FASTQ(.gz) file.

    Returns (features, reads_stats, local_read_stats) like the reference — `features` holds this sample's counts,
    `local_read_stats` the five counters — or None when the file cannot be opened as gzip at all.  A gzip stream
    that breaks off mid-way gives a warning and the counts of everything before the break (fast2q.py:405-407).
    `reads_stats` (the reference's memo of non-exact reads) is passed through untouched: the device resolves
    every non-exact key directly, and the memo never changes a count.  preprocess=True parses only the first
    10 000 reads (fast2q.py:398-400)."""
    got = _count_file(raw, features, param, preprocess)
    if got is None:
        return None
    counts, stats, engine = got
    return _features_from(param, features, counts, engine), reads_stats, stats


# ------------------------------------------------------------------------------------------------------------
# per-sample output (fast2q.py:752-809)
# ------------------------------------------------------------------------------------------------------------
def csv_writer(path, outfile):
    with open(path, "w", newline='') as output:
        csv.writer(output).writerows(outfile)                # "\r\n" line ends, minimal quoting — as the reference


def sample_name(raw):
    """x.fastq.gz -> x ; x.fq.gz -> x.fq ; x.fastq -> x   (fast2q.py:779-783)"""
    name = Path(raw).stem
    if ".fastq" in name:
        name = Path(name).stem
    return name


def _timing_text(seconds):
    if seconds > 3600:
        return str(round(seconds / 3600, 2)) + " hours"
    if seconds > 60:
        return str(round(seconds / 60, 2)) + " minutes"
    return str(round(seconds, 2)) + " seconds"


def write_sample(raw, features, local_read_stats, param, seconds):
    """<sample>_reads.csv: statistics sentence, '#Feature,Reads', one row per feature sorted numerically by name
    when every name is an integer, else alphabetically (fast2q.py:768-799)"""
    rows = [[f.name, f.counts] for f in features.values()]
    timing = _timing_text(seconds)
    name = sample_name(raw)
    sentence = _statistics_sentence(raw, local_read_stats, seconds)
    if not param['Progress bar']:
        colourful_errors("INFO", f"Sample {name} was processed in {timing}")
    try:
        rows.sort(key=lambda r: int(r[0]))
    except ValueError:
        rows.sort(key=lambda r: r[0])
    rows.insert(0, ["#Feature", "Reads"])
    rows.insert(0, [sentence])
    csv_writer(os.path.join(param["directory"], name + "_reads.csv"), rows)


_order_cache = {}
_order_lock = threading.Lock()


def _library_order(features):
    """row order and csv-quoted names of a Counter library, computed once per run: numerically by name when every name is
    an integer, else alphabetically; equal names keep library order (fast2q.py:786-791, a stable sort)"""
    key = id(features)
    with _order_lock:
        hit = _order_cache.get(key)
        if hit is not None and hit[0] == len(features):
            return hit[1], hit[2]
        names = [f.name for f in features.values()]
        try:
            order = sorted(range(len(names)), key=lambda k: int(names[k]))
        except ValueError:
            order = sorted(range(len(names)), key=lambda k: names[k])
        buf = io.StringIO()
        w = csv.writer(buf)
        quoted = []
        for k in order:                                      # the csv module decides the quoting, as in csv_writer
            buf.seek(0); buf.truncate()
            w.writerow([names[k]])
            quoted.append(buf.getvalue()[:-2])
        order = np.asarray(order, dtype=np.int64)
        _order_cache.clear()
        _order_cache[key] = (len(features), order, quoted)
        return order, quoted


def _statistics_sentence(raw, s, seconds):
    return (f'#script ran in {_timing_text(seconds)} for file {sample_name(raw)}. {s["perfect_counter"] + s["imperfect_counter"]} reads out of '
            f'{s["reads"]} were aligned. {s["perfect_counter"]} were perfectly aligned. {s["imperfect_counter"]} were '
            f'aligned with mismatch. {s["non_aligned_counter"]} passed quality filtering but were not aligned. '
            f'{s["quality_failed"]} did not pass quality filtering.')


def _write_sample_counts(raw, features, counts, local_read_stats, param, seconds):
    """write_sample for a Counter sample straight from the count vector: the same bytes, without 30 000 objects per sample"""
    order, quoted = _library_order(features)
    name = sample_name(raw)
    if not param['Progress bar']:
        colourful_errors("INFO", f"Sample {name} was processed in {_timing_text(seconds)}")
    head = io.StringIO()
    w = csv.writer(head)
    w.writerow([_statistics_sentence(raw, local_read_stats, seconds)])
    w.writerow(["#Feature", "Reads"])
    vals = np.asarray(counts)[order].tolist()
    body = "".join([f"{q},{v}\r\n" for q, v in zip(quoted, vals)])
    with open(os.path.join(param["directory"], name + "_reads.csv"), "w", newline='') as output:
        output.write(head.getvalue())
        output.write(body)


def aligner(i, raw, features, param, reads_stats):
    """per-sample driver: count, time, write <sample>_reads.csv (fast2q.py:752-801)"""
    tempo = time.perf_counter()
    got = _count_file(raw, features, param)
    if got is None:
        return reads_stats
    counts, local_read_stats, engine = got
    if param["Running Mode"] == "C":
        _write_sample_counts(raw, features, counts, local_read_stats, param, time.perf_counter() - tempo)
    else:
        write_sample(raw, _features_from(param, features, counts, engine), local_read_stats, param, time.perf_counter() - tempo)
    return reads_stats


# ------------------------------------------------------------------------------------------------------------
# parameters (fast2q.py:1082-1314)
# ------------------------------------------------------------------------------------------------------------
def cpu_counter(param):
    """host feeder threads: --cp, else cores-2 (>=3 cores) / 1 (fast2q.py:1543-1570)"""
    available = os.cpu_count() or 1
    if type(param["cpu"]) is not int:
        cpu = available
        if cpu >= 3:
            cpu -= 2
        if cpu == 2:
            cpu -= 1
        return cpu
    return min(param["cpu"], available)


def initializer(cmd):
    """banner-less equivalent of fast2q.py:1082-1169: Phred clamps, fail sets, output directory, thread count"""
    if cmd is None:
        colourful_errors("FATAL", "the graphical front end is not part of this build; run with -c (see -h)")
        sys.exit()
    param = cmd
    print(f"\n 2FAST2Q (B200 engine)  Version: {version}")
    if param["test_mode"]:
        colourful_errors("WARNING", "Running test mode!\n")
    param["version"] = version
    quality_list = "".join(chr(q + 33) for q in range(94))
    for key in ("phred", "qual_up", "qual_down"):
        if int(param[key]) <= 0:
            param[key] = 1                                   # fast2q.py:1118-1125
    param["quality_set"] = set(quality_list[:int(param['phred']) - 1])
    param["quality_set_up"] = set(quality_list[:int(param['qual_up']) - 1])
    param["quality_set_down"] = set(quality_list[:int(param['qual_down']) - 1])
    current_time = datetime.datetime.now().strftime('%Y_%m_%d_%H_%M_%S')
    param["directory"] = os.path.join(param['out'], f"2FAST2Q_output_{current_time}")

    print("\n -- Parameters -- ")
    if param['Running Mode'] == 'C':
        print("\n Mode: Align and count")
        print(f" Allowed mismatches per alignement: {param['miss']}")
    else:
        print("\n Mode: Extract and count")
    print(f" Minimal Phred Score per bp >= {param['phred']}")
    if param['upstream'] is not None:
        print(f" Upstream search sequence: {param['upstream']}")
        print(f" Mismatches allowed in the upstream search sequence: {param['miss_search_up']}")
        print(f" Minimal Phred-score in the upstream search sequence: {param['qual_up']}")
    if param['downstream'] is not None:
        print(f" Downstream search sequence: {param['downstream']}")
        print(f" Mismatches allowed in the downstream search sequence: {param['miss_search_down']}")
        print(f" Minimal Phred-score in the downstream search sequence: {param['qual_down']}")
    if param['upstream'] is None or param['downstream'] is None:
        print(f" Finding features with the folowing length: {param['length']}bp")
    if param['upstream'] is None and param['downstream'] is None:
        print(f" Read alignment start position: {param['start']}")
    print(f" All data will be saved into {param['directory']}")
    print("\n ---- ")
    param["cpu_given"] = type(param["cpu"]) is int
    param["cpu"] = cpu_counter(param)
    return param


def input_parser(argv=None):
    """the reference's command line (fast2q.py:1171-1314): same flags, defaults and `used_cmd` string.
    --gpus is an addition (number of GPUs to use, default all)."""
    parser = argparse.ArgumentParser(prog="2fast2q")
    parser.add_argument("-c", nargs='?', const=True, help="cmd line mode.")
    parser.add_argument("-t", nargs='?', const=True, help="Runs in test mode with example data.")
    parser.add_argument("-v", nargs='?', const=True, help="Prints the current version.")
    parser.add_argument("--s", help="The full path to the directory with the sequencing files.")
    parser.add_argument("--g", help="The full path to the .csv file with the features.")
    parser.add_argument("--o", help="The full path to the output directory")
    parser.add_argument("--fn", nargs='?', const="compiled", help="Output compiled file name (default: compiled)")
    parser.add_argument("--pb", nargs='?', const=False, help="Progress bars (presence disables them, as in the reference)")
    parser.add_argument("--m", help="Allowed mismatches per feature (default 1); ignored in Extract + Count mode.")
    parser.add_argument("--ph", help="Minimal Phred-score (default 30).")
    parser.add_argument("--st", help="Feature start position(s) in the read (default 0); ignored with search sequences.")
    parser.add_argument("--l", help="Feature length in bp (default 20); unused with two search sequences.")
    parser.add_argument("--us", help="Upstream search sequence(s).")
    parser.add_argument("--ds", help="Downstream search sequence(s).")
    parser.add_argument("--msu", help="Mismatches allowed in the upstream search sequence (default 0).")
    parser.add_argument("--msd", help="Mismatches allowed in the downstream search sequence (default 0).")
    parser.add_argument("--qsu", help="Minimal Phred-score in the upstream search sequence (default 30)")
    parser.add_argument("--qsd", help="Minimal Phred-score in the downstream search sequence (default 30)")
    parser.add_argument("--mo", help="Running Mode (default C) [Counter (C) / Extractor + Counter (EC)].")
    parser.add_argument("--cp", help="Number of host threads that read / inflate files (the reference's cpu count).")
    parser.add_argument("--fs", nargs='?', const=False, help="File Split mode: one file at a time, sharded over all GPUs.")
    parser.add_argument("--k", nargs='?', const=False, help="Keeps the per-sample _reads.csv files.")
    parser.add_argument("--gpus", help="Number of GPUs to use (default: all visible B200s).")
    args = parser.parse_args(argv)

    if args.v is not None:
        print(f"\nVersion: {version}\n")
        sys.exit()
    if args.c is None:
        return None

    p = {"cmd": True, "big_file_split": False}
    p['used_cmd'] = " ".join(f"--{k}" if isinstance(v, bool) and v else f"--{k} {v}" for k, v in vars(args).items() if v is not None)
    p['Running Mode'] = "EC" if args.mo is not None and "EC" in args.mo.upper() else "C"
    if args.t is None:
        p["test_mode"] = False
        paths = [[args.s, 'seq_files'], [args.g, 'feature'], [args.o, 'out']]
    else:
        p["test_mode"] = True
        from . import testdata                               # surrogate of the reference's bundled example (see testdata.py)
        paths = [[testdata.ensure_example(), 'seq_files'], [testdata.GUIDES, 'feature'], [os.getcwd(), 'out']]
    p['out_file_name'] = args.fn if args.fn is not None else "compiled"
    p['length'] = int(args.l) if args.l is not None else 20
    p['Progress bar'] = args.pb is None
    p['start'] = args.st if args.st is not None else "0"
    p['phred'] = int(args.ph) if args.ph is not None else 30
    p['miss'] = int(args.m) if args.m is not None else 1
    p['upstream'] = args.us
    p['downstream'] = args.ds
    p['miss_search_up'] = int(args.msu) if args.msu is not None else 0
    p['miss_search_down'] = int(args.msd) if args.msd is not None else 0
    p['qual_up'] = int(args.qsu) if args.qsu is not None else 30
    p['qual_down'] = int(args.qsd) if args.qsd is not None else 30
    p['delete'] = args.k is None
    p['cpu'] = int(args.cp) if args.cp is not None else False
    p['big_file_split'] = args.fs is not None
    p['gpus'] = int(args.gpus) if args.gpus is not None else None
    for value, key in paths:
        if value is None:
            p[key] = os.getcwd()
            if key == 'feature' and p['Running Mode'] != "EC":
                found = path_finder(os.getcwd(), ["*.csv"])
                if len(found) > 1:
                    colourful_errors("FATAL", "There is more than one .csv in the current directory. If not directly indicating a "
                                     "path for the features .csv, please have only 1 .csv file in the directory.\n")
                    sys.exit()
                if len(found) == 1:
                    p[key] = found[0][0]
        else:
            p[key] = value
    return p


def file_sizer_split(param):
    """lists the sequencing files (smallest first); a single file switches File-Split mode on (fast2q.py:1657-1689)"""
    if param["test_mode"]:
        param["sequencing_files"] = {"len_files": 1, "preprocess_files": [param["seq_files"]], "files": [param["seq_files"]]}
        return param
    files = path_parser(param["seq_files"], ["*.gz", "*.fastq"])
    if len(files) == 1:
        param['big_file_split'] = True
    names = [f[0] for f in files]
    param["sequencing_files"] = {"len_files": len(names), "preprocess_files": names[:param["cpu"]], "files": names}
    return param


# ------------------------------------------------------------------------------------------------------------
# orchestration: files over GPUs, or one file sharded over GPUs
# ------------------------------------------------------------------------------------------------------------
def gpu_count(param):
    n = _lib.device_count()
    if n < 1:
        raise _lib.F2QError(-7, "no B200-class (sm_100) device is visible; this build has no CPU path")
    want = param.get("gpus")
    return max(1, min(n, want)) if want else n


def record_aligned_shards(blocks, shard_bytes=None):
    """cuts an uncompressed byte stream into shards that end at record boundaries (every 4th '\\n' counted from byte 0),
    so that shards are independent FASTQ streams: the counts of a file are the sum of the counts of its shards
    (what single_file_reads_binner + merge_feature_dicts compute with 400 000-line chunks, fast2q.py:411-512).
    Yields (bytes, is_final); the final shard carries the unterminated / left-over lines."""
    shard_bytes = shard_bytes or CHUNK_BYTES
    pend, size = [], 0
    for block in blocks:
        pend.append(block)
        size += len(block)
        if size < shard_bytes:
            continue
        buf = pend[0] if len(pend) == 1 else b"".join(pend)
        extra = buf.count(b"\n") & 3                         # newlines behind the last record boundary
        pos = len(buf)
        for _ in range(extra + 1):                           # walk back to the newline that ends the last whole record
            pos = buf.rfind(b"\n", 0, pos)
            if pos < 0:
                break
        if pos < 0:                                          # fewer than 4 newlines: not even one record yet
            pend, size = [buf], len(buf)
            continue
        yield buf[:pos + 1], False
        rest = buf[pos + 1:]
        pend, size = ([rest], len(rest)) if rest else ([], 0)
    yield b"".join(pend), True


def _merge_sample(param, features, results):
    """sum of per-GPU results of one sample: merge_feature_dicts + the stats additions (fast2q.py:439-445, 487-495)"""
    stats = {k: 0 for k in STAT_KEYS}
    merged = {}
    for feats, st in results:
        for k in STAT_KEYS:
            stats[k] += st[k]
        for key, f in feats.items():
            if key in merged:
                merged[key].counts += f.counts
            else:
                merged[key] = Features(f.name, f.counts)
    if param["Running Mode"] == "C":                         # library order
        merged = {seq: merged.get(seq, Features(f.name, 0)) for seq, f in features.items()}
    return merged, stats


def split_file_counter(raw, features, param, n_gpus):
    """File-Split mode on GPUs: one reader cuts the file into record-aligned shards, every GPU parses every n-th shard
    as its own stream, results are added.  Returns (features, local_read_stats, complete)."""
    _derive_positions(param)
    gz = os.path.splitext(raw)[1] == ".gz"
    qs = [queue.Queue(maxsize=3) for _ in range(n_gpus)]
    results = [None] * n_gpus
    errors = []

    def worker(g):
        drained = False
        try:
            engine, ring = _engine_for(param, features, g)
            engine.begin()
            n = 0
            while True:
                item = qs[g].get()
                if item is None:
                    drained = True
                    break
                for o in range(0, max(len(item), 1), ring.nbytes):
                    piece = item[o:o + ring.nbytes]
                    buf = ring.next()
                    if n >= len(ring):
                        engine.sync_copies()
                    buf.array[:len(piece)] = np.frombuffer(piece, dtype=np.uint8)
                    engine.submit_ptr(buf.ptr.value, len(piece), False)
                    n += 1
            engine.submit_ptr(0, 0, True)
            counts, stats = engine.end()
            results[g] = (_features_from(param, features, counts, engine), stats)
        except BaseException as e:                           # noqa: BLE001 — reported by the caller
            errors.append(e)
            while not drained and qs[g].get() is not None:
                pass
        finally:
            release_engines()

    threads = [threading.Thread(target=worker, args=(g,), daemon=True) for g in range(n_gpus)]
    for t in threads:
        t.start()
    complete = True
    g = 0

    def whole_lines(blocks):
        nonlocal complete
        tail = b""
        try:
            for b in blocks:
                cut = b.rfind(b"\n") + 1
                if cut == 0:
                    tail += b
                    continue
                yield tail + b[:cut] if tail else b[:cut]
                tail = b[cut:]
        except TruncatedGzip:
            complete = False
            tail = b""
        if tail:
            yield tail

    try:
        for shard, final in record_aligned_shards(whole_lines(_inflate_blocks(raw) if gz else _raw_blocks(raw))):
            qs[g % n_gpus].put(shard)
            g += 1
    finally:
        for q in qs:
            q.put(None)
        for t in threads:
            t.join()
    if errors:
        raise errors[0]
    merged, stats = _merge_sample(param, features, [r for r in results if r is not None])
    return merged, stats, complete


def split_file_native(raw, features, param, devices):
    """File-Split mode on several GPUs: one plain or bgzip file as ONE sample, parsed by one cached engine per entry of
    `devices` (entries may repeat a device).  Each engine reads and parses its own byte range of the file natively
    (f2q_submit_file_sharded); the first one ends with the whole sample.  Writes <sample>_reads.csv as aligner does."""
    tempo = time.perf_counter()
    _derive_positions(param)
    engines = [_engine_for(param, features, int(d), slot=k)[0] for k, d in enumerate(devices)]
    gz = os.path.splitext(raw)[1] == ".gz"

    def end_all():
        for e in engines:
            try:
                e.end()
            except _lib.F2QError:
                pass

    for e in engines:
        e.begin()
    try:
        complete, _ = _lib.submit_file_sharded(engines, raw, gz, threads=_INFLATE_WORKERS)
    except _lib.F2QError as e:
        end_all()
        if e.code == -1 and "corrupted gzip" in str(e):
            colourful_errors("WARNING", f"{raw} is an incomplete or corrupted gzip file. ({e})")
            return
        if e.code == -1 and "cannot open" in str(e):
            raise OSError(str(e)) from None
        raise
    except BaseException:
        end_all()
        raise
    try:
        counts, local_read_stats = engines[0].end()
    except _lib.F2QError as e:
        end_all()
        if e.code == -1 and "corrupted gzip" in str(e):     # (a bgzip block of some range failed its size or CRC-32 check)
            colourful_errors("WARNING", f"{raw} is an incomplete or corrupted gzip file. ({e})")
            return
        raise
    for e in engines[1:]:
        e.end()                                              # (closed and empty: leaves the cached engine reusable)
    if not complete:
        colourful_errors("WARNING", f"{raw} is an incomplete or corrupted gzip file. Only partial processing might have occurred.")
    if param["Running Mode"] == "C":
        _write_sample_counts(raw, features, counts, local_read_stats, param, time.perf_counter() - tempo)
    else:
        write_sample(raw, _features_from(param, features, counts, engines[0]), local_read_stats, param, time.perf_counter() - tempo)


def aligner_mp_dispenser(features, param, start=0):
    """processes every sample (fast2q.py:1619-1655).  File mode: `cpu` feeder threads take files from a queue, thread k
    drives GPU k mod n_gpus through its own context (samples are independent: no collective).  File-Split mode
    (--fs, or a single file): one file at a time, sharded over all GPUs."""
    os.makedirs(param["directory"], exist_ok=True)
    reads_stats = {"failed_reads": set(), "passed_reads": {}}
    files = param['sequencing_files']['files']
    n_gpus = gpu_count(param)
    colourful_errors("INFO", f"Processing {param['sequencing_files']['len_files']} files on {n_gpus} GPU(s). Please hold.")

    if param['big_file_split']:
        for raw in files:
            tempo = time.perf_counter()
            if SPLIT_NATIVE_SINGLE_GPU:
                # The native ingest (parallel reads / BGZF-parallel inflate into pinned memory) feeds ONE context faster than
                # the Python reader below can cut shards for eight (measured: 2.4 GB/s against 0.26 GB/s on a 5.9 GB file).
                # With several GPUs a plain or bgzip file is cut natively instead: every GPU reads and parses its own byte
                # range (split_file_native).  Ordinary gzip is one deflate stream with nowhere to cut: one GPU.  Counts are the same
                try:
                    if n_gpus > 1 and _input_kind([raw]) != "gzip":
                        split_file_native(raw, features, dict(param, device=0), list(range(n_gpus)))
                    else:
                        aligner(0, raw, features, dict(param, device=0), reads_stats)
                finally:
                    release_engines()
                continue
            try:
                merged, stats, complete = split_file_counter(raw, features, param, n_gpus)
            except (zlib.error, gzip.BadGzipFile, EOFError) as e:
                colourful_errors("WARNING", f"{raw} is an incomplete or corrupted gzip file. ({e})")
                continue
            if not complete:
                colourful_errors("WARNING", f"{raw} is an incomplete or corrupted gzip file. Only partial processing might have occurred.")
            write_sample(raw, merged, stats, param, time.perf_counter() - tempo)
        return

    work = queue.Queue()
    for i, raw in sorted(enumerate(files), key=lambda e: -os.path.getsize(e[1])):     # largest first balances the GPUs
        work.put((i, raw))
    errors = []

    def feeder(k):
        p = dict(param, device=k % n_gpus)
        try:
            while True:
                try:
                    i, raw = work.get_nowait()
                except queue.Empty:
                    return
                aligner(i, raw, features, p, reads_stats)
        except BaseException as e:                           # noqa: BLE001
            errors.append(e)
        finally:
            release_engines()

    # feeder threads = contexts on the GPUs.  Ordinary gzip is inflated by zlib on the feeder's host thread, one stream per
    # file: every core gets a file.  Plain and bgzip files are read by the context's own reader threads and (bgzip) inflated
    # on the GPU at tens of GB/s: two contexts per GPU (one streams while the other writes its sample) — sixteen of them on
    # one GPU spend seconds allocating their staging buffers one after the other (measured: 19 s against 6 s for 48 files)
    if param.get("cpu_given") or _input_kind(files) == "gzip":
        n_threads = max(int(param["cpu"]), n_gpus)
    else:
        n_threads = 2 * n_gpus
    n_threads = max(1, min(len(files), n_threads))
    threads = [threading.Thread(target=feeder, args=(k,), daemon=True) for k in range(n_threads)]
    for t in threads:
        t.start()
    for t in threads:
        t.join()
    if errors:
        raise errors[0]


# ------------------------------------------------------------------------------------------------------------
# compiled.csv / compiled_stats.csv (fast2q.py:1316-1412)
# ------------------------------------------------------------------------------------------------------------
def compiling(param):
    """merges the per-sample csv files (sorted by path) into <fn>.csv and <fn>_stats.csv; rows appear in first-seen
    order, samples a feature is missing from get 0, rows whose name contains '#' are skipped — as the reference"""
    ordered_csv = path_parser(param["directory"], ['*reads.csv'])
    headers = [f"#2FAST2Q version: {param['version']}",
               f"#Mismatch: {param['miss']}",
               f"#Phred Score: {param['phred']}",
               f"#Feature Length: {param['length']}",
               f"#Feature start position in the read: {param['start']}",
               f"#Running mode: {param['Running Mode']}",
               f"#Upstream search sequence: {param['upstream']}",
               f"#Downstream search sequence: {param['downstream']}",
               f"#Mismatches in the upstream search sequence: {param['miss_search_up']}",
               f"#Mismatches in the downstream search sequence: {param['miss_search_down']}",
               f"#Minimal Phred-score in the upstream search sequence: {param['qual_up']}",
               f"#Minimal Phred-score in the downstream search sequence: {param['qual_down']}"]
    if "used_cmd" in param:
        headers.insert(1, f"#cmd used: {param['used_cmd']}")
    sentences = []
    compiled = {}
    head = ["#Feature"]
    for i, file in enumerate(ordered_csv):
        stem = Path(os.path.splitext(file)[0]).stem
        head.append(stem[:-len("_reads")])
        with open(file) as current:
            for line in current:
                cols = line.rstrip().split(",")
                if "#" not in cols[0]:
                    if cols[0] in compiled:
                        compiled[cols[0]] = compiled[cols[0]] + [int(cols[1])]
                    else:
                        compiled[cols[0]] = [0] * i + [int(cols[1])]
                elif "#Feature" not in cols[0]:
                    sentences.append(cols[0][1:])
        for entry in compiled:                               # features this sample did not list
            if len(compiled[entry]) < i + 1:
                compiled[entry] = compiled[entry] + [0] * (i + 1 - len(compiled[entry]))

    table = run_stats(headers, sentences, param)
    final = [[feature] + compiled[feature] for feature in compiled]
    final.insert(0, head)
    csv_writer(os.path.join(param["directory"], f"{param['out_file_name']}.csv"), final)
    # the four summary plots of the output folder (fast2q.py:1414-1527), drawn by plots.py
    try:
        from . import plots
        if plots.write_all(table, head, compiled, os.path.join(param["directory"], param["out_file_name"])) is None:
            colourful_errors("WARNING", "Pillow is not installed: the four summary plots were not drawn (the .csv files are complete).")
    except Exception as e:                                   # noqa: BLE001  (a picture never fails a run whose counts are written)
        colourful_errors("WARNING", f"The summary plots could not be drawn ({type(e).__name__}: {e}).")
    if param["delete"]:
        for file in ordered_csv:
            os.remove(file)
    colourful_errors("INFO", "Analysis successfully completed")
    print("\n If you find 2FAST2Q useful, please consider citing:\n Bravo AM, Typas A, Veening J. 2022. \n 2FAST2Q: a general-purpose "
          "sequence search and counting program for FASTQ files. PeerJ 10:e14041\n DOI: 10.7717/peerj.14041\n")
    if param["test_mode"]:
        colourful_errors("WARNING", "Test successful. 2FAST2Q is working as intended!\n")


def run_stats(headers, sentences, param):
    """<fn>_stats.csv: the parameter lines, a header row, then per sample the fields of its statistics sentence taken by
    whitespace-token position exactly as the reference does (fast2q.py:1392-1412).  Returns the table (the four PNG
    plots are drawn from it by plots.py)."""
    table = [[h] for h in headers]
    table.append(["#Sample name", "Running Time", "Running Time unit", "Total number of reads in sample",
                  "Total number of reads that were aligned", "Number of reads that were aligned without mismatches",
                  "Number of reads that were aligned with mismatches",
                  "Number of reads that passed quality filtering but were not aligned",
                  "Number of reads that did not pass quality filtering."])
    for run in sentences:
        if "script ran" in run:
            t = run.split()
            table.append([t[7][:-1], t[3], t[4], t[12], t[8], t[15], t[19], t[24], t[32]])
        else:
            table.insert(0, [run])
    csv_writer(os.path.join(param["directory"], f"{param['out_file_name']}_stats.csv"), table)
    return table


def main(argv=None):
    t0 = time.perf_counter()
    param = file_sizer_split(initializer(input_parser(argv)))
    features = {}
    if param['Running Mode'] == 'C':
        features = features_loader(param["feature"])
    t1 = time.perf_counter()
    aligner_mp_dispenser(features, param)
    t2 = time.perf_counter()
    compiling(param)
    if os.environ.get("F2Q_CLI_TIMING"):
        print(f" [timing] parameters + features {t1 - t0:.2f} s, samples {t2 - t1:.2f} s, compiling {time.perf_counter() - t2:.2f} s", flush=True)


if __name__ == "__main__":
    main()
