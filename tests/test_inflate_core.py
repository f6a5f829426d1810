"""
CPU: the DEFLATE decoder the GPU inflate kernel runs per BGZF block (2fast2q_b200/csrc/inflate_core.h, compiled here with g++)
against zlib: stored, fixed-Huffman and dynamic-Huffman blocks, every compression level, FASTQ text, random bytes, long
matches, empty input, and corrupted / truncated streams (which must be refused, never mis-decoded silently).
"""
import ctypes as C
import importlib
import random
import zlib

import numpy as np
import pytest

import hostcheck

synth = importlib.import_module("2fast2q_b200.synth")
DECODERS = ("hc_inflate_raw", "hc_inflate_lane", "hc_inflate_lane8")   # free-running; lock-step with 9+7 / 8+6 table index bits


def infl(comp: bytes, out_len: int, fn="hc_inflate_raw"):
    H = hostcheck.lib()
    f = getattr(H, fn)
    f.argtypes = [C.c_char_p, C.c_uint32, C.c_char_p, C.c_uint32]
    out = C.create_string_buffer(max(out_len, 1) + 16)
    rc = f(comp + b"\xAA" * 16, len(comp), out, out_len)              # (readable slack behind the stream, as in the staging buffer)
    return rc, out.raw[:out_len]


def raw_deflate(data, level=6, strategy=zlib.Z_DEFAULT_STRATEGY):
    c = zlib.compressobj(level, zlib.DEFLATED, -15, 9, strategy)
    return c.compress(data) + c.flush()


def payloads():
    rnd = random.Random(3)
    spec = synth.default_spec(3)
    _, keys = synth.make_library(3, 300, 20)
    fastq = synth.fixed_reads(keys, 0, 380, **spec).tobytes()          # ~64 KB of FASTQ text: one BGZF block's worth
    yield "fastq", fastq
    yield "fastq_short", fastq[:777]
    yield "empty", b""
    yield "one_byte", b"A"
    yield "random", bytes(rnd.randrange(256) for _ in range(30000))
    yield "runs", b"A" * 40000 + b"CG" * 10000 + b"\n" * 300
    yield "text", (b"the quick brown fox jumps over the lazy dog\n" * 1400)[:65280]


@pytest.mark.parametrize("name,data", list(payloads()), ids=[n for n, _ in payloads()])
def test_decoder_equals_zlib(name, data):
    for level in (0, 1, 4, 6, 9):
        for strategy in (zlib.Z_DEFAULT_STRATEGY, zlib.Z_FIXED, zlib.Z_HUFFMAN_ONLY, zlib.Z_RLE):
            comp = raw_deflate(data, level, strategy)
            for fn in DECODERS:
                rc, out = infl(comp, len(data), fn)
                assert rc == 0 and out == data, (name, level, strategy, fn)


def test_corrupted_and_truncated_streams_are_refused():
    data = next(d for n, d in payloads() if n == "fastq")
    comp = raw_deflate(data, 6)
    for fn in DECODERS:
        assert infl(comp, len(data), fn)[0] == 0
        assert infl(comp, len(data) - 1, fn)[0] != 0         # produces more than the trailer promised
        assert infl(comp, len(data) + 1, fn)[0] != 0         # produces less
        for cut in (0, 1, 10, len(comp) // 2, len(comp) - 1):
            assert infl(comp[:cut], len(data), fn)[0] != 0, (fn, cut)
    rnd = random.Random(9)
    bad = 0
    for _ in range(200):
        b = bytearray(comp)
        p = rnd.randrange(len(b))
        b[p] ^= 1 << rnd.randrange(8)
        rc, out = infl(bytes(b), len(data))
        for fn in DECODERS[1:]:
            rc2, out2 = infl(bytes(b), len(data), fn)
            assert (rc == 0) == (rc2 == 0) and (rc != 0 or out == out2), fn  # all decoders accept / refuse the same streams
        if rc != 0 or out != data:
            bad += 1
        assert rc != 0 or len(out) == len(data)
    assert bad > 150                                         # (a flipped bit may leave a valid stream of the same length; that is what the CRC is for)


def test_corrupted_streams_read_no_further_than_the_slack():
    """the lock-step decoder may read 16 bytes behind its input (the staging buffer's slack), never more, whatever the stream
    asks for: a truncated stream whose output is far from complete, garbage, and streams of empty blocks"""
    H = hostcheck.lib()
    H.hc_inflate_lane_guarded.argtypes = [C.c_char_p, C.c_uint32, C.c_uint32]
    data = next(d for n, d in payloads() if n == "fastq")
    rnd = random.Random(12)
    streams = [(raw_deflate(data, 6), len(data)), (raw_deflate(data, 1, zlib.Z_HUFFMAN_ONLY), len(data))]
    for comp, n in list(streams):
        for cut in (1, 2, 5, 17, 100, len(comp) // 3):
            streams.append((comp[:cut], n))
    streams += [(bytes(rnd.randrange(256) for _ in range(k)), 65536) for k in (1, 3, 8, 64, 500)]
    streams += [(b"\x00\x00\x00\xff\xff" * 7, 65536), (b"\x02\x00" * 9, 100), (b"\x00" * 13, 65536)]
    for k, (comp, n) in enumerate(streams):
        rc = H.hc_inflate_lane_guarded(comp, len(comp), n)
        assert rc != 99, (k, len(comp))                              # a load behind the slack
        assert rc != 0 or k < 2, k
    assert H.hc_inflate_lane_guarded(streams[0][0], len(streams[0][0]), len(data)) == 0


def _crc_fns():
    H = hostcheck.lib()
    H.hc_crc32.restype = H.hc_crc32_lanes.restype = H.hc_crc32_shift.restype = C.c_uint32
    H.hc_crc32.argtypes = [C.c_void_p, C.c_uint32]
    H.hc_crc32_lanes.argtypes = [C.c_void_p, C.c_uint32, C.c_uint32]
    H.hc_crc32_shift.argtypes = [C.c_uint32, C.c_uint32]
    return H


def _at(data: bytes, align: int):
    """data at an address with (address mod 8) == align; the buffer stays alive with the returned pointer"""
    buf = C.create_string_buffer(len(data) + 16)
    base = C.addressof(buf)
    off = (align - base) % 8
    C.memmove(base + off, data, len(data))
    return buf, base + off


def test_crc32_equals_zlib_at_every_length_and_alignment():
    """the CRC-32 the device checks every inflated BGZF block with (crc32_update / crc32_lane_part, inflate_core.h): every
    length 0-300 and random lengths up to 65 536, at start addresses 0-7 mod 8, in one pass and as a warp of 32 lanes
    (and of 1, 3 and 7 lanes, so that slices of every length and position occur)"""
    H = _crc_fns()
    rnd = random.Random(21)
    blob = bytes(rnd.randrange(256) for _ in range(65536 + 8))
    lengths = list(range(301)) + [rnd.randrange(301, 65537) for _ in range(60)] + [65280, 65535, 65536]
    for n in lengths:
        data = blob[n % 7:n % 7 + n]
        want = zlib.crc32(data) & 0xFFFFFFFF
        for align in range(8):
            keep, p = _at(data, align)
            assert H.hc_crc32(p, n) == want, (n, align)
            assert H.hc_crc32_lanes(p, n, 32) == want, (n, align)
        for lanes in (1, 3, 7):
            keep, p = _at(data, n % 8)
            assert H.hc_crc32_lanes(p, n, lanes) == want, (n, lanes)
    # a wrong byte anywhere changes the lanes' CRC
    data = bytearray(blob[:65280])
    keep, p = _at(bytes(data), 3)
    good = H.hc_crc32_lanes(p, len(data), 32)
    for pos in (0, 1, 2039, 2040, 2041, 32639, 65279):
        bad = bytearray(data)
        bad[pos] ^= 1 << rnd.randrange(8)
        keep, p = _at(bytes(bad), 3)
        assert H.hc_crc32_lanes(p, len(bad), 32) != good, pos


def test_crc32_combine_at_random_split_points():
    """crc(A || B) = shift(crc(A), |B|) xor crc(B), the operator that joins the lanes' slices"""
    H = _crc_fns()
    rnd = random.Random(22)
    blob = bytes(rnd.randrange(256) for _ in range(70000))
    for _ in range(300):
        n = rnd.choice((rnd.randrange(0, 64), rnd.randrange(0, 65537)))
        k = rnd.randrange(0, n + 1)
        a, b = blob[:k], blob[k:n]
        want = zlib.crc32(a + b) & 0xFFFFFFFF
        assert H.hc_crc32_shift(zlib.crc32(a), len(b)) ^ (zlib.crc32(b) & 0xFFFFFFFF) == want, (n, k)
    assert H.hc_crc32_shift(0x12345678, 0) == 0x12345678
    assert H.hc_crc32_shift(0, 1000) == 0
