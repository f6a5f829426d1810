"""
CPU: the bit-parallel extraction code the CUDA kernels run for delimiter / multi-feature configurations
(2fast2q_b200/csrc/flex_core.h, compiled here with g++ through tests/native/hostcheck.cpp) against the oracle's key builder
(oracle f2qo_build_key, pinned to the reference): same key — or the same "every iteration flagged" — for every read.
"""
import ctypes as C
import importlib

import pytest

import hostcheck

synth = importlib.import_module("2fast2q_b200.synth")
lib = importlib.import_module("2fast2q_b200._lib")


def flex_key(cfg, pw, read, qual, extra=0):
    """extra: how much longer the longest line of the (imagined) warp is than this read's lines"""
    H = hostcheck.lib()
    H.hc_flex_key.argtypes = [C.c_void_p, C.c_int, C.c_char_p, C.c_int, C.c_char_p, C.c_int, C.c_int, C.c_char_p, C.POINTER(C.c_int)]
    out = C.create_string_buffer(256)
    n = C.c_int()
    rc = H.hc_flex_key(C.byref(cfg), pw, read, len(read), qual, len(qual), extra, out, C.byref(n))
    return rc, (out.raw[:n.value] if rc >= 0 else None)


CONFIGS = [
    dict(mode="EC", upstream="GTTCAGAGTTCT", downstream="CTGAATAGGCCA", miss_search_up=1, miss_search_down=1),
    dict(mode="EC", upstream="GTTCAGAGTTCT", downstream="CTGAATAGGCCA", miss_search_up=0, miss_search_down=2),
    dict(mode="EC", upstream="GTTCAGAGTTCT", miss_search_up=1, length=20),
    dict(mode="EC", downstream="CTGAATAGGCCA", miss_search_down=1, length=20),
    dict(mode="EC", downstream="CTGAATAGGCCA", miss_search_down=3, length=31, qual_down=20, phred=25),
    dict(mode="C", upstream="ACCGGT,GGATCC", downstream="TTGACA,CAATTG"),
    dict(mode="C", upstream="ACCGGT,GGATCC", downstream="TTGACA,CAATTG", miss_search_up=1, qual_up=35, phred=10),
    dict(mode="C", start="0,30", length=20),
    dict(mode="C", start="5", length=32),
    dict(mode="C", start="-25,3", length=12),
    dict(mode="EC", upstream="A", downstream="C", phred=0),
    dict(mode="EC", upstream="ACGTACGTACGTACGTACGTACGTACGTACGT", miss_search_up=3, length=5),
]


def fuzz_reads(seed, n, cfg_kw):
    """reads built around the configuration's search sequences, with every nuisance the reference tolerates"""
    r = synth.SM64(seed)
    ups = (cfg_kw.get("upstream") or "").split(",")
    downs = (cfg_kw.get("downstream") or "").split(",")
    for _ in range(n):
        s = bytearray(r.dna(r.below(9)))
        for i in range(max(len(ups), len(downs))):
            u = ups[i % len(ups)].encode() if ups[0] else b""
            d = downs[i % len(downs)].encode() if downs[0] else b""
            if u and r.below(100) < 25:
                u = synth.mutate(r, u, 1 + r.below(3))
            if d and r.below(100) < 25:
                d = synth.mutate(r, d, 1 + r.below(3))
            if r.below(100) < 7:
                u = b""
            if r.below(100) < 7:
                d = b""
            s += u + r.dna(r.choice([0, 1, 5, 19, 20, 21, 30, 33])) + d + r.dna(r.below(6))
        if not s or r.below(100) < 5:
            s = bytearray(r.dna(r.below(96)))
        s = bytes(s)[:96]
        t = r.below(100)
        if t < 10 and s:
            a = r.below(len(s)); b = a + r.below(len(s) - a + 1)
            s = s[:a] + s[a:b].lower() + s[b:]
        elif t < 20 and s:
            p = r.below(len(s))
            s = s[:p] + bytes([r.choice([ord("N"), ord("n"), ord("E"), ord("U"), ord(":"), 0x80, 0xC1, ord("@"), ord("V"), ord("D")])]) + s[p + 1:]
        q = bytearray(63 + r.below(11) for _ in range(len(s)))
        for _ in range(r.choice([0, 0, 0, 1, 1, 2, 6])):
            if q:
                q[r.below(len(q))] = r.choice([33, 34, 47, 52, 53, 54, 57, 58, 61, 62, 63, 64, 66, 67, 125, 126, 200])
        q = bytes(q)
        t = r.below(100)
        if t < 6:
            q = q[: r.below(len(q) + 1)]
        elif t < 10:
            q = (q + bytes(63 + r.below(11) for _ in range(1 + r.below(8))))[:96]
        yield s, q


@pytest.mark.parametrize("k", range(len(CONFIGS)))
def test_flex_extraction_equals_oracle_key(k, oracle):
    kw = CONFIGS[k]
    cfg = lib.make_config(**kw)
    ocfg = oracle.make_config(**kw)
    H = hostcheck.lib()
    H.hc_flex_eligible.argtypes = [C.c_void_p]
    assert H.hc_flex_eligible(C.byref(cfg)) == 1
    n_keys = n_fail = 0
    for s, q in fuzz_reads(1000 + k, 4000, kw):
        want = oracle.build_key(ocfg, s, q)
        for pw, extra in ((3, 0), (5, 0), (3, 13), (5, 40)):
            rc, got = flex_key(cfg, pw, s, q, extra)
            if rc == -2:                                # a piece longer than 32 symbols: the kernels hand the read to the generic code
                assert want is not None and max(len(p) for p in want.split(b":")) > 32 or len(want) > 32, (kw, s, q, want)
                continue
            assert rc != -3
            if want is None:
                assert rc == -1, (kw, s, q, got)
                n_fail += 1
            else:
                assert rc >= 0 and got == want, (kw, pw, extra, s, q, got, want)
                n_keys += 1
    assert n_keys > 100 and n_fail > 20, (n_keys, n_fail)


def test_ineligible_configurations_are_refused():
    H = hostcheck.lib()
    H.hc_flex_eligible.argtypes = [C.c_void_p]
    for kw in (dict(upstream="ACGN"), dict(upstream="ACGT", miss_search_up=4), dict(start="0,1,2"), dict(upstream="A" * 33),
               dict(start="0", length=33)):
        assert H.hc_flex_eligible(C.byref(lib.make_config(**kw))) == 0, kw


# the 160-position planes of flex_B (PW = 5): flex_pieces (flex_core.h) loads 8 * (4 PW - 2) = 144 positions when the warp's
# longest line allows it and all 160 otherwise (PW = 3: 80 / 96).  Reads of 81..160 positions, pieces of 29..33 symbols
# around the 32-symbol piece limit (FLEX_MAX_PIECE), each read also run as if the warp's longest line sat on either side of
# the 80/81 and 144/145 group boundaries
LONG_CONFIGS = [
    dict(mode="EC", upstream="GTTCAGAGTTCT", downstream="CTGAATAGGCCA", miss_search_up=1, miss_search_down=1),
    dict(mode="EC", upstream="GTTCAGAGTTCT", downstream="CTGAATAGGCCA", miss_search_up=3, miss_search_down=2),
    dict(mode="EC", upstream="ACGTTGCAACGTTGCAACGTTGCAACGTTGCA", miss_search_up=3, length=31),
    dict(mode="EC", downstream="G", miss_search_down=0, length=32),
    dict(mode="C", upstream="ACCGGT,GGATCC", downstream="TTGACA,CAATTG", miss_search_up=1, miss_search_down=1),
]
LONG_LENGTHS = [81, 82, 95, 96, 97, 120, 143, 144, 145, 146, 159, 160]


def long_reads(seed, n, kw):
    r = synth.SM64(seed)
    ups = (kw.get("upstream") or "").split(",")
    downs = (kw.get("downstream") or "").split(",")
    for _ in range(n):
        target = r.choice(LONG_LENGTHS) if r.below(2) else 81 + r.below(80)
        s = bytearray(r.dna(r.below(40)))
        for i in range(max(len(ups), len(downs))):
            u = ups[i % len(ups)].encode() if ups[0] else b""
            d = downs[i % len(downs)].encode() if downs[0] else b""
            if u and r.below(100) < 30:
                u = synth.mutate(r, u, 1 + r.below(4))
            if d and r.below(100) < 30:
                d = synth.mutate(r, d, 1 + r.below(3))
            s += u + r.dna(29 + r.below(5)) + d
        s = bytes(s + r.dna(max(0, target - len(s))))[:target]
        t = r.below(100)
        if t < 8:
            p = r.below(len(s))
            s = s[:p] + r.choice([b"N", b"n", b"a", b"\xc1"] + ([b":"] if len(ups) == len(downs) == 1 else [])) + s[p + 1:]
        q = bytearray(63 + r.below(11) for _ in range(len(s)))
        if r.below(100) < 15:
            q[r.below(len(q))] = r.choice([33, 40, 52, 61])
        q = bytes(q)
        t = r.below(100)
        if t < 6:
            q = q[: r.below(len(q) + 1)]
        elif t < 12:
            q = (q + bytes(63 + r.below(11) for _ in range(1 + r.below(20))))[:160]     # quality line longer than the sequence line
        yield s, q


@pytest.mark.parametrize("k", range(len(LONG_CONFIGS)))
def test_flex_extraction_of_reads_longer_than_96_positions(k, oracle):
    kw = LONG_CONFIGS[k]
    cfg = lib.make_config(**kw)
    ocfg = oracle.make_config(**kw)
    n_keys = n_long_piece = 0
    sides = set()
    for s, q in long_reads(2000 + k, 2500, kw):
        want = oracle.build_key(ocfg, s, q)
        m = max(len(s), len(q))
        # the warp's longest line: this read's own, and either side of the group boundaries it can still reach
        for maxlen in sorted({m} | {b for b in (80, 81, 144, 145, 160) if b >= m}):
            sides.add(maxlen <= 144)                            # narrow plane load (flex_pieces: maxlen <= 8 * (4 PW - 2))
            rc, got = flex_key(cfg, 5, s, q, maxlen - m)
            assert rc != -3, (kw, s, q)
            if rc == -2:
                assert want is not None, (kw, s, q)
                pieces = want.split(b":") if cfg.n_iter > 1 else [want]     # (a single piece may hold a ':' of the read)
                assert max(len(p) for p in pieces) > 32, (kw, s, q, want)
                n_long_piece += 1
                continue
            if want is None:
                assert rc == -1, (kw, s, q, got)
            else:
                assert rc >= 0 and got == want, (kw, maxlen, s, q, got, want)
                n_keys += 1
    assert n_keys > 500, n_keys
    assert sides == {True, False}
    if kw.get("upstream") and kw.get("downstream"):
        assert n_long_piece > 10, n_long_piece                  # 33-symbol pieces reached the generic hand-over
