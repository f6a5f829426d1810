"""
-m gpu: the bgzip inflate on the device, byte for byte against zlib, and the CRC-32 check behind it.

Kernel cases go through Engine.inflate_blocks (f2q_inflate_blocks: the launch f2q_submit_file uses, kernel choice included)
on every variant: lock-step lanes with the automatic, 8+6 and 9+7 lookup tables, and the free-running threads.  Payloads
(FASTQ of configs 2 and 4, one byte, random bytes, runs, periods 2-12, text, exactly 65 280 and 65 536 bytes) are compressed
at levels 0/1/6/9, with every zlib strategy and with flushes in the middle, and laid out so that every warp mixes kinds, at
every source / destination alignment, contiguous or with canary gaps, and in the largest case behind 1 GiB of input and 2 GiB
of output.  Streams that zlib decodes to the right length with wrong bytes, wrong CRC / isize fields, truncated and garbage
payloads must set ERR_INFLATE while the other 31 lanes of their warp still produce zlib's bytes.

File cases go through submit_file / submit_file_sharded on every path (device lanes / threads, host block-parallel, host
serial): a silently corrupted block is refused wherever it is, empty blocks are checked like the others, and a batch limit
(65 536 blocks, or the output buffer) ends only the batch, never the device path.
"""
import functools
import gzip
import importlib
import random
import struct
import zlib

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

f2q = importlib.import_module("2fast2q_b200")
lib = f2q._lib
synth = importlib.import_module("2fast2q_b200.synth")
fq = importlib.import_module("2fast2q_b200.fast2q")

ERR_INFLATE = 16
KERNEL_VARIANTS = [dict(gpu_inflate=1, gpu_inflate_bits=b) for b in (0, 8, 9)] + [dict(gpu_inflate=2, gpu_inflate_bits=0)]
FILE_VARIANTS = [(dict(v), 6) for v in KERNEL_VARIANTS] + [(dict(gpu_inflate=0), 1), (dict(gpu_inflate=0), 6)]
CANARY = 0xA5
BGZF_EOF = bytes.fromhex("1f8b08040000000000ff0600424302001b0003000000000000000000")


def _vid(v):
    return "-".join(f"{k}{x}" for k, x in v.items())


# ---- payloads and compressors ------------------------------------------------------------------------------------------
def _deflate(data, level=6, strategy=zlib.Z_DEFAULT_STRATEGY):
    c = zlib.compressobj(level, zlib.DEFLATED, -15, 9, strategy)
    return c.compress(data) + c.flush()


def _flushed(data):
    """several deflate blocks in one member: a sync flush (an empty stored block) and a full flush in the middle"""
    c = zlib.compressobj(6, zlib.DEFLATED, -15)
    a, b = len(data) // 3, 2 * len(data) // 3
    return c.compress(data[:a]) + c.flush(zlib.Z_SYNC_FLUSH) + c.compress(data[a:b]) + c.flush(zlib.Z_FULL_FLUSH) + c.compress(data[b:]) + c.flush()


COMPRESSORS = [("l0", lambda d: _deflate(d, 0)), ("l1", lambda d: _deflate(d, 1)), ("l6", lambda d: _deflate(d, 6)),
               ("l9", lambda d: _deflate(d, 9)), ("filtered", lambda d: _deflate(d, 6, zlib.Z_FILTERED)),
               ("huffman", lambda d: _deflate(d, 6, zlib.Z_HUFFMAN_ONLY)), ("rle", lambda d: _deflate(d, 6, zlib.Z_RLE)),
               ("fixed", lambda d: _deflate(d, 6, zlib.Z_FIXED)), ("flush", _flushed)]


@functools.lru_cache(maxsize=None)
def payloads():
    rnd = random.Random(41)
    spec = synth.default_spec(2)
    _, keys = synth.make_library(2, 300, 20)
    fq2 = synth.fixed_reads(keys, 0, 700, **spec).tobytes()
    fq4 = synth.barseq_reads(4, 400)
    out = [("fastq2", fq2[:60001]), ("fastq4", fq4[:50003]), ("one_byte", b"G"), ("random", rnd.randbytes(30000)),
           ("runs", b"A" * 20000 + b"C" * 774 + b"\n" * 259)]                              # distance 1, length 258
    for p in range(2, 13):
        out.append((f"period{p}", (rnd.randbytes(p) * (24000 // p + 1))[:24000 + p]))   # distance p < 8, 8-11 and 12
    out += [("text", (b"the quick brown fox jumps over the lazy dog\n" * 1000)[:43210]),
            ("exact65280", fq2[:65280]), ("exact65536", fq2[:65536])]                   # (level 0: two stored blocks)
    assert len(fq2) >= 65536
    return out


@functools.lru_cache(maxsize=None)
def cases():
    """every payload under every compressor: (name, data, compressed)"""
    out = []
    for pn, data in payloads():
        for cn, fn in COMPRESSORS:
            comp = fn(data)
            assert zlib.decompress(comp, -15) == data
            out.append((f"{pn}/{cn}", data, comp))
    return out


# ---- one launch of Engine.inflate_blocks -------------------------------------------------------------------------------
class Block:
    """one block of a launch: the payload and the trailer fields; want = the bytes zlib gives (None: the block is bad)"""

    def __init__(self, comp, isize, crc, want):
        self.comp, self.isize, self.crc, self.want = comp, isize, crc, want


def good(case):
    _, data, comp = case
    return Block(comp, len(data), zlib.crc32(data), data)


def run_blocks(eng, blocks, canary=True, far=0):
    """places the blocks (src alignment b % 4, one copy of a payload per alignment; dst contiguous, or behind 64-byte canary
    gaps at alignment b % 8; the last `far` blocks at src just under 1 GiB and dst above 2^31), inflates them, and returns
    (error bits, the blocks whose output differs from zlib's, canaries intact)"""
    n, near = len(blocks), len(blocks) - far
    table = np.zeros((n, 5), dtype=np.uint32)
    placed = [{}, {}]                                              # (payload, alignment) -> src, near / far
    pos = [0, (1 << 30) - 4096 - sum(len(B.comp) + 4 for B in blocks[near:]) if far else 0]
    base = list(pos)
    src = []
    for b, B in enumerate(blocks):
        side = int(b >= near)
        key = (id(B.comp), b % 4)
        if key not in placed[side]:
            s = (pos[side] + 3) // 4 * 4 + b % 4
            placed[side][key] = (s, B.comp)
            pos[side] = s + len(B.comp)
        src.append(placed[side][key][0])
    assert not far or pos[0] < base[1]
    dst, out_len = [], 0
    for b, B in enumerate(blocks):
        if b == near and far:
            out_len = max(out_len, (1 << 31) + 4096) + 3
        if canary:
            out_len = (out_len + 64 + 7) // 8 * 8 + b % 8
        dst.append(out_len)
        out_len += B.isize
        table[b] = (src[b], len(B.comp), dst[b], B.isize, B.crc & 0xFFFFFFFF)
    comp_size, out_size = max(pos) + 65536, out_len + 64 + 65536
    if far:
        comp_size, out_size = max(comp_size, (1 << 30) + 65536), max(out_size, 3 << 30)
    d_comp = eng.device_alloc(comp_size)
    d_out = eng.device_alloc(out_size)
    try:
        for side in (0, 1):
            if placed[side]:
                buf = bytearray(b"\x5c" * (pos[side] - base[side]))
                for s, c in placed[side].values():
                    buf[s - base[side]:s - base[side] + len(c)] = c
                eng.h2d(d_comp + base[side], bytes(buf))
        segs = [(lo, hi) for lo, hi in ((0, near), (near, n)) if lo < hi]
        bounds = []
        for lo, hi in segs:
            s0 = (dst[lo] - 64) // 8 * 8 if canary else dst[lo]
            s1 = dst[hi - 1] + blocks[hi - 1].isize + (64 if canary else 0)
            if canary:
                eng.h2d(d_out + s0, np.full(s1 - s0, CANARY, dtype=np.uint8))
            bounds.append((s0, s1, lo, hi))
        err = eng.inflate_blocks(d_comp, table, d_out)
        wrong, canary_ok = [], True
        for s0, s1, lo, hi in bounds:
            got = eng.d2h(d_out + s0, s1 - s0)
            gap = np.ones(s1 - s0, dtype=bool) if canary else None
            for b in range(lo, hi):
                B, o = blocks[b], dst[b] - s0
                if B.want is not None and not np.array_equal(got[o:o + B.isize], np.frombuffer(B.want, dtype=np.uint8)):
                    wrong.append(b)
                if canary:
                    gap[o:o + B.isize] = False                     # (a bad block's own bytes are not specified)
            if canary:
                canary_ok = canary_ok and bool(np.all(got[gap] == CANARY))
            del got
        return err, wrong, canary_ok
    finally:
        eng.device_free(d_comp)
        eng.device_free(d_out)


def mixed(n, K=None):
    """n blocks, lane i of warp w taking case (7 i + w) mod K: every warp mixes kinds"""
    cs = cases()
    K = K or len(cs)
    return [good(cs[(7 * (b % 32) + b // 32) % K]) for b in range(n)]


@pytest.fixture(scope="module", params=KERNEL_VARIANTS, ids=_vid)
def engine(request):
    e = lib.Engine(lib.make_config(miss=1), 0, None, **request.param)
    yield e
    e.close()


@pytest.mark.parametrize("n", [1, 31, 32, 33, len(cases())])
@pytest.mark.parametrize("canary", [True, False], ids=["canary", "contiguous"])
def test_blocks_equal_zlib(engine, n, canary):
    blocks = mixed(n)
    err, wrong, canary_ok = run_blocks(engine, blocks, canary)
    names = [cases()[(7 * (b % 32) + b // 32) % len(cases())][0] for b in wrong[:5]]
    assert err == 0 and not wrong and canary_ok, (err, names, canary_ok)


def test_every_case_in_every_lane(engine):
    """each case once in each of the 32 lanes (at every src / dst alignment on the way)"""
    cs = cases()
    blocks = [good(cs[(b + b // 32) % len(cs)]) for b in range(32 * len(cs))]
    err, wrong, canary_ok = run_blocks(engine, blocks, True)
    assert err == 0 and not wrong and canary_ok, (err, [cs[(b + b // 32) % len(cs)][0] for b in wrong[:5]])


def test_65536_blocks_far_offsets(engine):
    """a full batch: the automatic pick takes the 8+6 tables; the last 64 blocks at src just under 1 GiB and dst above 2^31"""
    blocks = mixed(65536)
    err, wrong, _ = run_blocks(engine, blocks, canary=False, far=64)
    assert err == 0 and not wrong, (err, wrong[:5])


# ---- corrupted blocks --------------------------------------------------------------------------------------------------
@functools.lru_cache(maxsize=None)
def silent_flips():
    """single-bit flips that zlib decodes to the right length with wrong bytes (the CRC is all that can see them)"""
    rnd = random.Random(43)
    out = []
    for name in ("fastq2/l6", "fastq2/l1", "fastq4/l9", "text/fixed", "fastq2/flush", "period5/huffman"):
        _, data, comp = next(c for c in cases() if c[0] == name)
        for _ in range(2000):
            bad = bytearray(comp)
            bad[rnd.randrange(len(bad))] ^= 1 << rnd.randrange(8)
            d = zlib.decompressobj(-15)
            try:
                got = d.decompress(bytes(bad))
            except zlib.error:
                continue
            if d.eof and len(got) == len(data) and got != data:
                out.append((name, Block(bytes(bad), len(data), zlib.crc32(data), None)))
                break
    assert len(out) >= 4
    return out


def bad_blocks():
    cs = {c[0]: c for c in cases()}
    _, data, comp = cs["fastq2/l6"]
    crc = zlib.crc32(data)
    out = list(silent_flips())
    out += [("wrong_crc", Block(comp, len(data), crc ^ 0x00010000, None)),
            ("isize+1", Block(comp, len(data) + 1, crc, None)),
            ("isize-1", Block(comp, len(data) - 1, crc, None)),
            ("truncated", Block(comp[:len(comp) * 2 // 3], len(data), crc, None)),
            ("garbage", Block(random.Random(44).randbytes(len(comp)), len(data), crc, None)),
            ("empty_wrong_crc", Block(b"\x03\x00", 0, 1, None)),
            ("empty_with_bytes", Block(_deflate(b"A"), 0, 0, None))]
    _, d1, c1 = cs["one_byte/l6"]
    out.append(("one_byte_wrong_crc", Block(c1, 1, zlib.crc32(d1) ^ 1, None)))
    return out


@pytest.mark.parametrize("lane", [0, 13, 31])
def test_corrupted_block_sets_the_error_and_spares_its_warp(engine, lane):
    for name, bad in bad_blocks():
        blocks = mixed(32)
        blocks[lane] = bad
        err, wrong, canary_ok = run_blocks(engine, blocks, True)
        assert err & ERR_INFLATE, (name, lane)
        assert not wrong and canary_ok, (name, lane, wrong)


def test_empty_blocks_are_checked(engine):
    """isize 0: a valid empty stream with CRC 0 passes, next to other blocks"""
    blocks = mixed(32)
    blocks[5] = Block(b"\x03\x00", 0, 0, b"")
    blocks[6] = Block(_deflate(b""), 0, 0, b"")
    err, wrong, canary_ok = run_blocks(engine, blocks, True)
    assert err == 0 and not wrong and canary_ok


# ---- files -------------------------------------------------------------------------------------------------------------
def member(comp, isize, crc):
    """one BGZF block around a raw deflate payload"""
    return (b"\x1f\x8b\x08\x04\x00\x00\x00\x00\x00\xff\x06\x00BC\x02\x00" + struct.pack("<H", 18 + len(comp) + 8 - 1) + comp
            + struct.pack("<II", crc & 0xFFFFFFFF, isize))


def bgzf_blocks(data, bs=65280, level=6):
    return [(data[o:o + bs], _deflate(data[o:o + bs], level)) for o in range(0, len(data), bs)]


def silent(data, comp, seed):
    """a payload that zlib decodes to len(data) bytes other than data"""
    rnd = random.Random(seed)
    for _ in range(3000):
        bad = bytearray(comp)
        bad[rnd.randrange(len(bad))] ^= 1 << rnd.randrange(8)
        d = zlib.decompressobj(-15)
        try:
            got = d.decompress(bytes(bad))
        except zlib.error:
            continue
        if d.eof and len(got) == len(data) and got != data:
            return bytes(bad)
    i = data.index(b"\n") + 1                                     # (no flip found: the same length, one base changed)
    alt = data[:i] + (b"C" if data[i:i + 1] != b"C" else b"G") + data[i + 1:]
    return _deflate(alt)


def build_file(blocks, bad=None, seed=0):
    """blocks [(data, comp)] -> a bgzip file; bad = index of a block whose payload is silently corrupted"""
    parts = []
    for k, (d, c) in enumerate(blocks):
        parts.append(member(silent(d, c, seed) if k == bad else c, len(d), zlib.crc32(d)))
    return b"".join(parts) + BGZF_EOF


@pytest.fixture(scope="module")
def world(oracle):
    spec = synth.default_spec(2)
    _, keys = synth.make_library(2, 400, 20)
    body = synth.fixed_reads(keys, 0, 20_000, **spec).tobytes()           # 37 blocks
    ocfg = oracle.make_config(miss=1)
    want = oracle.count(ocfg, keys, body)
    engines = {}

    def eng(opts, slot=0):
        k = (tuple(sorted(opts.items())), slot)
        if k not in engines:
            e = lib.Engine(lib.make_config(miss=1), 0, None, **opts)
            e.set_library(keys)
            engines[k] = e
        return engines[k]

    class W:
        pass
    w = W()
    w.keys, w.body, w.want, w.ocfg, w.eng, w.oracle = keys, body, want, ocfg, eng, oracle
    yield w
    for e in engines.values():
        e.close()


def run_file(e, path, threads):
    e.begin()
    try:
        e.submit_file(str(path), True, 0, threads)
    except lib.F2QError:
        try:
            e.end()
        except lib.F2QError:
            pass
        raise
    return e.end()


def run_sharded(engines, path, cuts):
    for e in engines:
        e.begin()
    try:
        lib.submit_file_sharded(engines, str(path), True, cuts=cuts, threads=8)
    except lib.F2QError:
        for e in engines:
            try:
                e.end()
            except lib.F2QError:
                pass
        raise
    out = engines[0].end()
    for e in engines[1:]:
        e.end()
    return out


def even_cuts(size, n):
    return [size * k // n for k in range(1, n)]


def test_silently_corrupted_block_is_refused_on_every_path(world, tmp_path):
    blocks = bgzf_blocks(world.body)
    assert len(blocks) == 37
    g = tmp_path / "bad.fastq.gz"
    for bad in (None, 0, 18, 36):
        g.write_bytes(build_file(blocks, bad, seed=bad or 0))
        if bad is not None:
            with pytest.raises(gzip.BadGzipFile):
                gzip.decompress(g.read_bytes())                         # (what the reference's reader does with it)
        for opts, threads in FILE_VARIANTS:
            e = world.eng(opts)
            if bad is None:
                c, s = run_file(e, g, threads)
                assert s == world.want[1] and np.array_equal(c, world.want[0]), opts
                continue
            with pytest.raises(lib.F2QError) as err:
                run_file(e, g, threads)
            assert "corrupted gzip" in str(err.value), (bad, opts, threads)
        for n in (2, 4):
            es = [world.eng({"gpu_inflate": 1}, slot=k) for k in range(n)]
            if bad is None:
                c, s = run_sharded(es, g, even_cuts(g.stat().st_size, n))
                assert s == world.want[1] and np.array_equal(c, world.want[0])
                assert es[0].info("shards") == n and es[0].info("shard_fallback") == 0
                continue
            with pytest.raises(lib.F2QError) as err:
                run_sharded(es, g, even_cuts(g.stat().st_size, n))
            assert "corrupted gzip" in str(err.value), (bad, n)


def test_empty_blocks_mid_file(world, tmp_path):
    """an empty block in the middle is inflated and checked like any other: valid -> accepted; invalid payload or a non-zero
    CRC -> refused, as gzip.open refuses it"""
    blocks = bgzf_blocks(world.body)
    members = [member(c, len(d), zlib.crc32(d)) for d, c in blocks]
    g = tmp_path / "e.fastq.gz"
    for name, empty, ok in (("valid", member(b"\x03\x00", 0, 0), True), ("valid_l9", member(_deflate(b"", 9), 0, 0), True),
                            ("bad_payload", member(b"\xff\xff", 0, 0), False), ("bad_crc", member(b"\x03\x00", 0, 0x1234), False),
                            ("has_bytes", member(_deflate(b"ACGT\n"), 0, 0), False)):
        g.write_bytes(b"".join(members[:20]) + empty + b"".join(members[20:]) + BGZF_EOF)
        try:
            ref_ok = gzip.decompress(g.read_bytes()) == world.body
        except (gzip.BadGzipFile, zlib.error, EOFError):
            ref_ok = False
        assert ref_ok == ok, name
        for opts, threads in FILE_VARIANTS:
            e = world.eng(opts)
            if ok:
                c, s = run_file(e, g, threads)
                assert s == world.want[1] and np.array_equal(c, world.want[0]), (name, opts)
                if opts["gpu_inflate"]:
                    assert e.info("gz_blocks") == len(blocks), (name, opts)
            else:
                with pytest.raises(lib.F2QError) as err:
                    run_file(e, g, threads)
                assert "corrupted gzip" in str(err.value), (name, opts, threads)


@pytest.fixture(scope="module")
def tiny_file(world, tmp_path_factory):
    """100 000 blocks of 2 records each (~16 MB): more blocks than one batch takes, in a single ring piece"""
    spec = synth.default_spec(2)
    rec = 2 * spec["read_len"] + 18
    text = synth.fixed_reads(world.keys, 0, 200_000, **spec).tobytes()
    parts = []
    for o in range(0, len(text), 2 * rec):
        d = text[o:o + 2 * rec]
        parts.append(member(_deflate(d, 1), len(d), zlib.crc32(d)))
    p = tmp_path_factory.mktemp("tiny") / "tiny.fastq.gz"
    p.write_bytes(b"".join(parts) + BGZF_EOF)
    return p, len(parts), world.oracle.count(world.ocfg, world.keys, text), text


@pytest.fixture(scope="module")
def dense_file(world, tmp_path_factory):
    """21 000 blocks of 553 records drawn from 16 distinct ones (20 kinds of block, ~1.9 KB each at level 6): ~1.4 GB of text
    in ~40 MB, so more than one ring piece, and more text than two batches' output buffers take, so that a batch fills up
    after the whole file has been read.  Each block holds whole records, so the oracle's
    counts are the sums over the blocks"""
    spec = synth.default_spec(2)
    rec = 2 * spec["read_len"] + 18
    recs = synth.fixed_reads(world.keys, 0, 16, **spec).tobytes()
    recs = [recs[k * rec:(k + 1) * rec] for k in range(16)]
    rnd = random.Random(45)
    kinds = []
    squeeze = [fn for name, fn in COMPRESSORS if name in ("l6", "filtered")] * 10
    for k in range(20):
        d = b"".join(rnd.choice(recs) for _ in range(553))
        c, s = world.oracle.count(world.ocfg, world.keys, d)
        kinds.append((member(squeeze[k](d), len(d), zlib.crc32(d)), np.asarray(c, dtype=np.int64), s))
    n = 21_000
    seq = [rnd.randrange(20) for _ in range(n)]
    p = tmp_path_factory.mktemp("dense") / "dense.fastq.gz"
    with open(p, "wb") as f:
        for k in seq:
            f.write(kinds[k][0])
        f.write(BGZF_EOF)
    counts = sum(kinds[k][1] for k in seq)
    stats = {k: sum(kinds[j][2][k] for j in seq) for k in kinds[0][2]}
    return p, n, (counts, stats)


def _check_batches(world, path, n_blocks, want, min_batches):
    e = world.eng({"gpu_inflate": 1})
    c, s = run_file(e, path, 8)
    assert s == want[1] and np.array_equal(np.asarray(c, dtype=np.int64), np.asarray(want[0], dtype=np.int64))
    assert e.info("gz_blocks") == n_blocks                    # every block on the device: no hand-over to the host reader
    assert e.info("gz_batches") >= min_batches
    size = path.stat().st_size
    for n in (2, 4):
        es = [world.eng({"gpu_inflate": 1}, slot=k) for k in range(n)]
        c, s = run_sharded(es, path, even_cuts(size, n))
        assert es[0].info("shards") == n and es[0].info("shard_fallback") == 0, n
        assert s == want[1] and np.array_equal(np.asarray(c, dtype=np.int64), np.asarray(want[0], dtype=np.int64)), n
        assert sum(x.info("gz_blocks") for x in es) == n_blocks, n


def test_batch_full_of_blocks_stays_on_the_device(world, tiny_file):
    p, n_blocks, want, _ = tiny_file
    _check_batches(world, p, n_blocks, want, 2)


def test_batch_full_of_text_stays_on_the_device(world, dense_file):
    p, n_blocks, want = dense_file
    _check_batches(world, p, n_blocks, want, 3)


def test_corrupted_block_in_a_later_batch(world, tiny_file, tmp_path):
    """the bad block behind the first 65 536: in the second batch of the device path"""
    p, n_blocks, _, text = tiny_file
    raw = bytearray(p.read_bytes())
    # walk to block 80 000 and corrupt it silently (its CRC no longer matches what it inflates to)
    off = 0
    for _ in range(80_000):
        off += (raw[off + 16] | raw[off + 17] << 8) + 1
    bs = (raw[off + 16] | raw[off + 17] << 8) + 1
    d = text[80_000 * 236:80_001 * 236]
    comp = bytes(raw[off + 18:off + bs - 8])
    assert zlib.decompress(comp, -15) == d
    bad = silent(d, comp, 46)
    g = tmp_path / "late.fastq.gz"
    g.write_bytes(bytes(raw[:off]) + member(bad, len(d), zlib.crc32(d)) + bytes(raw[off + bs:]))
    for opts, threads in FILE_VARIANTS:
        with pytest.raises(lib.F2QError) as err:
            run_file(world.eng(opts), g, threads)
        assert "corrupted gzip" in str(err.value), opts
    for n in (2, 4):
        es = [world.eng({"gpu_inflate": 1}, slot=k) for k in range(n)]
        with pytest.raises(lib.F2QError) as err:
            run_sharded(es, g, even_cuts(g.stat().st_size, n))
        assert "corrupted gzip" in str(err.value), n


def test_cli_skips_a_silently_corrupted_bgzip_sample_like_a_corrupted_gzip_one(world, tmp_path, capsys):
    """one folder with a good and a silently corrupted bgzip file, one with the same good file and an ordinary gzip file whose
    CRC does not match: the same warning and the same outputs (the bad sample skipped)"""
    import glob
    import os
    blocks = bgzf_blocks(world.body[:1_180_000])
    good_file = build_file(blocks)
    bad_bgzf = build_file(blocks, bad=9, seed=9)
    plain = gzip.compress(world.body[:1_180_000], mtime=0)
    bad_gz = plain[:-8] + struct.pack("<I", (zlib.crc32(world.body[:1_180_000]) ^ 0x10) & 0xFFFFFFFF) + plain[-4:]
    libtxt = "\n".join(f"g{i},{k.decode()}" for i, k in enumerate(world.keys)) + "\n"
    results = {}
    for kind, bad in (("bgzf", bad_bgzf), ("gzip", bad_gz)):
        root = tmp_path / kind
        (root / "in").mkdir(parents=True)
        (root / "out").mkdir()
        (root / "in" / "good.fastq.gz").write_bytes(good_file)
        (root / "in" / "bad.fastq.gz").write_bytes(bad)
        (root / "library.csv").write_text(libtxt)
        capsys.readouterr()
        fq.main(["-c", "--s", str(root / "in"), "--o", str(root / "out"), "--g", str(root / "library.csv"), "--m", "1", "--pb", "--k", "--cp", "2"])
        printed = capsys.readouterr()
        assert "bad.fastq.gz is an incomplete or corrupted gzip file" in printed.out + printed.err, kind
        d = glob.glob(str(root / "out" / "2FAST2Q_output_*"))
        assert len(d) == 1
        results[kind] = {f: open(os.path.join(d[0], f), newline="").read() for f in sorted(os.listdir(d[0])) if not f.endswith(".png")}
    assert sorted(results["bgzf"]) == sorted(results["gzip"])
    assert "good_reads.csv" in results["bgzf"] and "bad_reads.csv" not in results["bgzf"]
    assert results["bgzf"]["compiled.csv"] == results["gzip"]["compiled.csv"]
