"""
-m gpu: both sides of every size threshold on which the device path changes shape.  f2q_set_library (csrc/f2q_api.cu)
picks the lookup table (probing / compact / two-choice cuckoo / cuckoo with the Hamming-1 neighbours) and the seed plan of
the resolver; decide_policy / decide_ch pick the per-read code of the streaming kernel (fast1 / flex_S / flex_B / generic);
the flex code hands single reads to the byte-wise generic kernel.  Each of them packs keys into its own bit budget, and a
wrong count from any of them is silent, so every case here is compared with the oracle (pinned to the reference) bit for
bit, and proves through Engine.info (f2q_get_info) which side of its threshold it landed on.

Every case runs three ways: the default path (the speculation must commit every chunk), odd host chunks, and a queue of 16
entries when a resolver is involved.  Inputs come from the seeded synth.SM64; nothing is read from disk.
"""
import importlib
import math

import pytest

pytestmark = pytest.mark.gpu

synth = importlib.import_module("2fast2q_b200.synth")
INFO = ("policy", "table", "hist", "seed_parts", "flex_table", "generic_reads")


@pytest.fixture(scope="module")
def gu():
    import gpu_util
    assert gpu_util.lib.device_count() >= 1, "no B200 visible"
    return gpu_util


# ---------------------------------------------------------------------------------------------------------------------
# inputs
# ---------------------------------------------------------------------------------------------------------------------
def fastq(recs):
    return b"".join(h + b"\n" + s + b"\n+\n" + q + b"\n" for h, s, q in recs)


def library(r, n, length, n_close=True):
    """n distinct ACGT keys of `length` symbols (length may be a list to draw from).  keys[1] is at distance 1 from
    keys[0], keys[2] at distance 2 (their shared and self-colliding Hamming-1 neighbours); returns (keys, pairs)"""
    lengths = length if isinstance(length, (list, tuple)) else [length]
    keys, seen, pairs = [], set(), []
    L0 = lengths[0]
    if n_close and n >= 2 and L0 >= 2:
        a = r.dna(L0)
        b = synth.mutate(r, a, 1)
        keys += [a, b]
        pairs.append((a, b))
        if n >= 3:
            c = synth.mutate(r, a, 2)
            if c not in (a, b):
                keys.append(c)
                pairs.append((a, c))
        seen.update(keys)
    while len(keys) < n:
        k = r.dna(r.choice(lengths))
        if k not in seen:
            seen.add(k)
            keys.append(k)
    return keys, pairs


def tie(r, pair):
    """a window at distance 1 from both keys of the pair (a shared neighbour for distance 1, the midpoint for distance 2)"""
    a, b = pair
    diff = [i for i in range(len(a)) if a[i] != b[i]]
    w = bytearray(a)
    if len(diff) == 1:
        p = diff[0]
        w[p] = [c for c in b"ACGT" if c not in (a[p], b[p])][r.below(2)]
    else:
        p = diff[r.below(len(diff))]
        w[p] = b[p]
    return bytes(w)


def variant(r, g, pairs):
    """the window content of one read built around library key g"""
    k = r.below(100)
    if k < 35:
        return g
    if k < 50:
        return synth.mutate(r, g, 1)
    if k < 58:
        return synth.mutate(r, g, 2)
    if k < 63:
        return synth.mutate(r, g, 3)
    if k < 70 and g:
        p = r.below(len(g))
        return g[:p] + b"N" + g[p + 1:]
    if k < 76 and g:
        a = r.below(len(g)); b = a + 1 + r.below(len(g) - a)
        return g[:a] + g[a:b].lower() + g[b:]
    if k < 88 and pairs:
        return tie(r, r.choice(pairs))
    return r.dna(len(g))


def window_reads(seed, keys, pairs, n, *, length, start=0, tail=12):
    """Counter reads with one fixed window [start, start + length): exact keys, 1-3 mismatches, N and lower case inside the
    window, shared / tied neighbours, lines that end inside the window; keys shorter than the window also as the whole
    (short) line"""
    r = synth.SM64(seed)
    recs = []
    for i in range(n):
        g = r.choice(keys)
        w = variant(r, g, pairs)
        s = r.dna(start) + w
        k = r.below(10)
        if k == 0:
            s = s[:start + r.below(length + 1)]                       # the line ends inside the window
        elif len(w) >= length or k < 5:
            s += r.dna(max(0, length - len(w)) + r.below(tail))
        # (17-byte headers: records of a 4-symbol window stay long enough for the speculation, whose tiles keep at most
        # SPEC_CAP newlines and leave denser ones to the exact kernel)
        recs.append((b"@sample:%08d:1" % i, s, synth.qual_line(r, len(s), 0.05)))
    return fastq(recs)


def run_engine(gu, params, keys, data, chunk=None, **opts):
    cfg = gu.lib.make_config(**params)
    with gu.lib.Engine(cfg, 0, None, **opts) as e:
        if keys is not None:
            e.set_library(keys)
        counts, stats = e.run(data, chunk)
        got = e.ec_items() if keys is None else [int(x) for x in counts]
        info = {k: e.info(k) for k in INFO}
        info["spec"] = e.spec_counts()
    return got, stats, info


def check(gu, oracle, params, keys, data, *, resolver=True, more=(), engine_opts=None):
    """oracle == the default path (committed by the speculation) == odd host chunks (== a 16-entry queue); returns the
    Engine.info of each run, the default one first"""
    ocfg = oracle.make_config(**params)
    if keys is None:
        want, want_s = oracle.extract_count(ocfg, data)
    else:
        c, want_s = oracle.count(ocfg, keys, data)
        want = [int(x) for x in c]
    eo = engine_opts or {}
    runs = [(None, dict(eo)), (len(data) // 3 + 7, dict(eo))]
    if resolver:
        runs.append((None, dict(eo, queue_entries=16)))
    runs += [(None, dict(eo, **m)) for m in more]
    infos = []
    for chunk, opts in runs:
        got, stats, info = run_engine(gu, params, keys, data, chunk, **opts)
        tag = (chunk, opts, info)
        assert stats == want_s, tag
        assert got == want, tag
        infos.append(info)
    committed, fell_back = infos[0]["spec"]
    if keys is not None or infos[0]["policy"] != "generic":         # (Extract+Count speculates on the flex policies only)
        assert committed >= 1 and fell_back == 0, infos[0]
    return infos


# ---------------------------------------------------------------------------------------------------------------------
# fast1: window length (decide_policy) and the lookup-table forms of f2q_set_library
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("length,policy", [(32, "fast1"), (33, "generic")])
def test_fast1_window_length_limit(gu, oracle, length, policy):
    """decide_policy (f2q_api.cu:258): fast1 takes Counter mode with one fixed window of 0..32 symbols; a 33-symbol window has no packed
    form (and is no flex window either: flex_prepare caps it at FLEX_MAX_PIECE) and runs the byte-wise generic code.
    A 32-symbol library fills all 64 key bits: never compact (c_len < 32), always the probing table"""
    r = synth.SM64(100 + length)
    keys, pairs = library(r, 300, length)
    data = window_reads(1 + length, keys, pairs, 3000, length=length, start=3)
    params = dict(miss=2, length=length, start="3")
    info = check(gu, oracle, params, keys, data)[0]
    assert info["policy"] == policy
    if length == 32:
        assert info["table"] == "probing" and info["generic_reads"] == 0


# (L, n, table): compact needs n < 2^(64 - 2L) - 1 for L > 16 (f2q_api.cu:986, `compact = c_len >= 1 && c_len < 32 &&
# (idx_bits >= 32 || n_keys < (1 << idx_bits) - 1)`); the cuckoo form needs 2n + 1 < 2^(32 - hshift) - 2 with
# hshift = max(2L, 32) - 32 (`fits`, f2q_api.cu:1015), and holds the Hamming-1 neighbours when m >= 1 and
# n (3L + 1) <= 2^20 (f2q_api.cu:1021); a neighbour shared by two keys is stored as the tie marker (f2q_api.cu:1034)
TABLE_CASES = [
    (31, 2, "compact"), (31, 3, "probing"),
    (30, 6, "cuckoo+neighbours"), (30, 7, "compact"), (30, 14, "compact"), (30, 15, "probing"),
    (29, 30, "cuckoo+neighbours"), (29, 31, "compact"), (29, 62, "compact"), (29, 63, "probing"),
    (28, 126, "cuckoo+neighbours"), (28, 127, "compact"), (28, 254, "compact"), (28, 255, "probing"),
    (24, 32766, "cuckoo"), (24, 32767, "compact"),
    (20, 17189, "cuckoo+neighbours"), (20, 17190, "cuckoo"),
]


@pytest.mark.parametrize("L,n,table", TABLE_CASES, ids=[f"L{L}-n{n}-{t}" for L, n, t in TABLE_CASES])
def test_lookup_table_forms(gu, oracle, L, n, table):
    """each side of the compact / cuckoo / neighbour limits, m = 1 (the neighbours decide 1-mismatch reads in the
    streaming kernel, the queue and the seed resolver take the rest)"""
    r = synth.SM64(L * 100_003 + n)
    keys, pairs = library(r, n, L)
    n_reads = 3000 if n > 5000 else 4000
    data = window_reads(L + n, keys, pairs, n_reads, length=L, start=2)
    info = check(gu, oracle, dict(miss=1, length=L, start="2"), keys, data)[0]
    assert info["policy"] == "fast1"
    assert info["table"] == table
    assert info["generic_reads"] == 0


def test_no_neighbours_without_mismatches(gu, oracle):
    """m = 0: the cuckoo table holds the keys only (the neighbour entries need m >= 1)"""
    r = synth.SM64(7)
    keys, pairs = library(r, 500, 20)
    data = window_reads(8, keys, pairs, 3000, length=20)
    info = check(gu, oracle, dict(miss=0), keys, data, resolver=False)[0]
    assert info["table"] == "cuckoo"


@pytest.mark.parametrize("n_packable,n_nkeys,table", [(126, 0, "cuckoo+neighbours"), (126, 2, "compact"), (252, 2, "compact"), (252, 3, "probing")])
def test_keys_outside_the_packed_table_count_toward_its_limits(gu, oracle, n_packable, n_nkeys, table):
    """the table limits count every library key (n_keys, f2q_api.cu:986 / 1015), the non-packable ones too: 126 packable 28-symbol keys build the
    cuckoo table, two 27-byte keys with an N in front of them leave 128 > 126 and the compact table.  The N-keys come
    FIRST, so the packable keys carry feature indices up to 127 / 254: a limit computed from the packable keys alone would
    let those overflow the 8 value bits of the slot.  (The N-keys are one byte shorter than the window, so the generic
    queue takes only reads whose line ends one symbol early.)"""
    r = synth.SM64(28_000 + n_packable + n_nkeys)
    packable, pairs = library(r, n_packable, 28)
    nkeys = [r.dna(5) + b"N" + r.dna(21) for _ in range(n_nkeys)]
    keys = nkeys + packable
    data = window_reads(n_packable + n_nkeys, keys, pairs, 5000, length=28, start=1)
    info = check(gu, oracle, dict(miss=1, length=28, start="1"), keys, data)[0]
    assert info["table"] == table


@pytest.mark.parametrize("with_n_keys", [False, True])
def test_generic_length_sends_every_read_of_that_length_to_the_generic_queue(gu, oracle, with_n_keys):
    """generic_len_mask (f2q_api.cu:970): a key length with non-packable library keys (N, other bytes) is decided by the byte-wise generic
    code for every read of that window length; a pure ACGT library sends nothing there"""
    r = synth.SM64(2020 + with_n_keys)
    keys, pairs = library(r, 800, [20, 19, 21])
    if with_n_keys:
        keys += [r.dna(7) + b"N" + r.dna(12) for _ in range(5)] + [r.dna(19) + b"R"]
    data = window_reads(33 + with_n_keys, keys, pairs, 4000, length=20)
    info = check(gu, oracle, dict(miss=2), keys, data)[0]
    assert info["policy"] == "fast1"
    assert (info["generic_reads"] > 0) == with_n_keys, info


@pytest.mark.parametrize("n", [8192, 8193])
def test_shared_memory_histogram_limit(gu, oracle, n):
    """HIST_MAX_KEYS = 8192 (f2q_api.cu:268): the exact kernel counts into a per-CTA shared-memory histogram up to that many features and
    into global atomics above (launch_tile); run once more with the speculation off so that the exact kernel parses"""
    r = synth.SM64(8000 + n)
    keys, pairs = library(r, n, 20)
    data = window_reads(n, keys, pairs, 4000, length=20)
    infos = check(gu, oracle, dict(miss=1), keys, data, more=[dict(spec=0)])
    assert bool(infos[-1]["hist"] & 2) == (n <= 8192), infos[-1]


# ---------------------------------------------------------------------------------------------------------------------
# the seed plan of the resolver (f2q_set_library: P segments, seeds = every choice of K = P - m of them)
# ---------------------------------------------------------------------------------------------------------------------
def expected_seed_parts(keys, m, forced):
    """restates the plan choice of f2q_set_library (f2q_api.cu:1098): P in m+1..8 with C(P, m) <= 32 seeds and K * ceil(maxlen / P) <= 16
    symbols per seed, the cheapest by the fitted cost; 0 = the classic m + 1 one-segment seeds"""
    fl = [len(k) for k in keys if all(c in b"ACGT" for c in k) and len(k) <= 32]
    maxlen, meanlen = max(fl), float(sum(fl)) / len(fl)

    def n_choose(n, k):
        x = 1.0
        for i in range(k):
            x = x * (n - i) / (i + 1)
        return x

    best, parts = -1.0, 0
    for P in range(m + 1, 9):
        K = P - m
        seeds = n_choose(P, m)
        if seeds > 32 or K * ((maxlen + P - 1) // P) > 16:
            continue
        if forced and forced != P:
            continue
        cost = seeds * (1.5 + K + len(fl) / math.pow(4.0, K * meanlen / P))
        if best < 0 or cost < best:
            best, parts = cost, P
    return parts if best >= 0 else 0


SEED_CASES = [(L, m) for L in (4, 8, 28, 32) for m in (1, 2, 3)] + [("mixed", 2), ("mixed", 3)]


@pytest.mark.parametrize("L,m", SEED_CASES, ids=[f"L{L}-m{m}" for L, m in SEED_CASES])
def test_seed_plans(gu, oracle, L, m):
    """every seed plan P = 2..8 and the automatic one, at key lengths 4 / 8 / 28 / 32 and in a library of 3..12-symbol
    keys (segments of a key shorter than P are empty); plans that do not fit fall back to the classic seeds"""
    r = synth.SM64(31 * m + (L if L != "mixed" else 99))
    if L == "mixed":
        keys, pairs = library(r, 200, [12, 3, 5, 7, 8, 10, 11])
        length = 12
    else:
        keys, pairs = library(r, 60 if L == 4 else 300, L)
        length = L
    data = window_reads(5 * m + length, keys, pairs, 2500, length=length, tail=20)
    params = dict(miss=m, length=length)
    sides = set()
    for P in [0] + list(range(2, 9)):
        info = check(gu, oracle, params, keys, data, engine_opts=dict(seed_parts=P))[0]
        want = expected_seed_parts(keys, m, P)
        assert info["seed_parts"] == want, (P, info)
        sides.add(want > 0)
    assert sides == {True, False} or m == 1                   # (m = 1 fits every P at these lengths)


# ---------------------------------------------------------------------------------------------------------------------
# flex: record length sniff (decide_ch), the plane limits of flex_read_warp / flex_pieces
# ---------------------------------------------------------------------------------------------------------------------
US, DS = b"ACCGGT", b"TTGACA"
FLEX_PARAMS = dict(mode="C", miss=1, upstream=US.decode(), downstream=DS.decode(), miss_search_up=1, miss_search_down=1)


def flex_reads(seed, keys, pairs, lengths, *, n=3000, head=None, first_lengths=None, header_len=None, qual_extra=0):
    """Counter reads with the feature between US and DS (search sequences sometimes one mismatch off) padded to a length
    drawn from `lengths`.  first_lengths / header_len: the first records (the record length is sniffed from two);
    qual_extra: the first qual_extra records have a quality line 1-3 symbols longer than the sequence line.  (They lie in
    the first range of the streaming kernel, which starts at a record start; the line phase of a later range is guessed
    from records whose two lines have one length.)"""
    r = synth.SM64(seed)
    recs = []
    for i in range(n):
        R = first_lengths[i] if first_lengths and i < len(first_lengths) else r.choice(lengths)
        g = r.choice(keys)
        w = variant(r, g, pairs)
        u = synth.mutate(r, US, 1) if r.below(10) == 0 else US
        d = synth.mutate(r, DS, 1) if r.below(10) == 0 else DS
        s = r.dna(r.below(max(1, R - len(w) - 12 + 1))) + u + w + d
        s = (s + r.dna(max(0, R - len(s))))[:R]
        q = synth.qual_line(r, len(s), 0.05)
        if i < qual_extra:
            q += bytes(63 + r.below(11) for _ in range(1 + r.below(3)))
        H = header_len if (header_len and i < 2) else 3 + r.below(30)
        h = (b"@" + b"%d" % i + b"x" * 64)[:H]
        recs.append((h, s, q))
    return fastq(recs)


# (name, read lengths, first two read lengths, header length of the first two records, quality longer (%), k of the
#  search sequences, policy, generic_reads > 0).  decide_ch (f2q_api.cu:402): record length = (bytes of the first 8 lines) / 2, flex_B above
# 2 * 96 + 24 = 216; a record of a 96-bp read is 197 bytes + its header.  flex_read_warp (flex.cuh:134): r or q > 32 * PW
# -> generic.  flex_pieces (flex_core.h:472) loads 8 * (4 PW - 2) positions when the warp's longest line allows it.
SNIFF_CASES = [
    ("96bp-header19-flex_S", [96], None, 19, 0, 1, "flex_S", False),
    ("96bp-header20-flex_B", [96], None, 20, 0, 1, "flex_B", False),
    ("97bp-under-flex_S", [95, 96, 97], [95, 95], 5, 0, 1, "flex_S", True),
    ("quality-97-under-flex_S", [90, 96], [96] * 30, 5, 30, 1, "flex_S", True),
    ("short-first-then-long", [100, 120], [60, 60], 10, 0, 1, "flex_S", True),
    ("long-first-then-short", [50, 75, 100, 160], [160, 160], 10, 0, 1, "flex_B", False),
    ("160bp-under-flex_B", [150, 160], [160, 160], 10, 0, 1, "flex_B", False),
    ("161bp-under-flex_B", [159, 160, 161], [160, 160], 10, 0, 1, "flex_B", True),
    ("quality-161-under-flex_B", [150, 160], [160] * 30, 10, 30, 1, "flex_B", True),
    ("narrow-planes-80-81-flex_S", [70, 78, 79, 80, 81], None, None, 0, 1, "flex_S", False),
    ("narrow-planes-144-145-flex_B", [136, 143, 144, 145], None, None, 0, 1, "flex_B", False),
    ("k2-short-reads-flex_B", [60, 80, 81, 96], None, None, 0, 2, "flex_B", False),
]


@pytest.mark.parametrize("case", SNIFF_CASES, ids=[c[0] for c in SNIFF_CASES])
def test_flex_record_sniff_and_plane_limits(gu, oracle, case):
    name, lengths, first, hdr, qx, k, policy, to_generic = case
    r = synth.SM64(len(name))
    keys, pairs = library(r, 400, [20, 19, 21])
    data = flex_reads(sum(name.encode()), keys, pairs, lengths, first_lengths=first, header_len=hdr, qual_extra=qx)
    params = dict(FLEX_PARAMS, miss_search_up=k)
    info = check(gu, oracle, params, keys, data)[0]
    assert info["policy"] == policy and info["flex_table"] == 1, info
    assert (info["generic_reads"] > 0) == to_generic, info


# two windows (two search sequence pairs): key = piece1 ':' piece2
US2, DS2 = (b"ACCGGT", b"GGATCC"), (b"TTGACA", b"CAATTG")
TWO_PARAMS = dict(mode="C", miss=2, upstream="ACCGGT,GGATCC", downstream="TTGACA,CAATTG")


MOTIFS = US2 + DS2


def clean(piece):
    """no search sequence inside a piece (it would move the piece boundaries the read was built with)"""
    return not any(m in piece.upper() for m in MOTIFS)


def clean_dna(r, n):
    while True:
        d = r.dna(n)
        if clean(d):
            return d


def two_piece_reads(seed, shapes_and_keys, n=3000):
    """reads whose two pieces come from (key, read-piece transform) pairs"""
    r = synth.SM64(seed)
    recs = []
    for i in range(n):
        p1, p2 = r.choice(shapes_and_keys)(r)
        s = r.dna(r.below(6)) + US2[0] + p1 + DS2[0] + r.dna(r.below(4)) + US2[1] + p2 + DS2[1] + r.dna(r.below(6))
        recs.append((b"@t%d" % i, s, synth.qual_line(r, len(s), 0.03)))
    return fastq(recs)


def pieces_of(keys):
    """pieces of a library key, one of them (same length) varied"""
    def make(r):
        a, _, b = r.choice(keys).partition(b":")
        if r.below(2):
            v = variant(r, a, [])
            a = v if clean(v) else a
        else:
            v = variant(r, b, [])
            b = v if clean(v) else b
        return a, b
    return make


@pytest.mark.parametrize("case", ["fits", "mixed-shapes", "one-symbol-keys", "piece33-library-lacks", "piece33-library-has-34",
                                  "41-symbols-library-lacks", "41-symbols-library-has"])
def test_flex_key_shapes(gu, oracle, case):
    """FLEX_MAX_PIECE (32) / FX_MAX_SYMBOLS (40) / fx_len_sig (flex.cuh:178, f2q_api.cu:1208 / 1220): a key the flex code cannot pack is
    not aligned when the library has no key of its byte length, and goes to the generic code when it has one; a byte length
    shared by keys of different shapes (FX_SIG_MIXED), or with keys of fewer symbols than the m + 1 seed segments, sends
    its non-exact reads to the generic code.  A library key the flex table cannot hold makes the whole library generic."""
    r = synth.SM64(sum(case.encode()))
    base = [clean_dna(r, 10) + b":" + clean_dna(r, 12) for _ in range(200)]   # one shape per byte length
    base = list(dict.fromkeys(base))
    keys, sources, flex, to_generic = list(base), [], True, False
    if case == "mixed-shapes":
        # AAAA:CCCCC next to AAAAA:CCCC; reads of the second shape one piece boundary off a key of the first (distance 2)
        k45 = [clean_dna(r, 4) + b":" + clean_dna(r, 5) for _ in range(30)]
        k54 = [clean_dna(r, 5) + b":" + clean_dna(r, 4) for _ in range(30)]
        keys += list(dict.fromkeys(k45 + k54))
        sources.append(lambda rr: (lambda k: (k[:4] + clean_dna(rr, 1), k[6:]))(rr.choice(k45)))
        to_generic = True
    elif case == "one-symbol-keys":
        keys = [r.dna(20) for _ in range(200)] + [b"A", b"C"]
        keys = list(dict.fromkeys(keys))
        p = dict(FLEX_PARAMS, miss=1)
        data = flex_reads(5, keys, [], [40, 60], n=3000)
        info = check(gu, oracle, p, keys, data)[0]
        assert info["policy"] == "flex_S" and info["generic_reads"] > 0, info
        return
    elif case.startswith("piece33"):
        sources.append(lambda rr: (clean_dna(rr, 33), b""))                  # (33, 0): 34 bytes
        if case.endswith("has-34"):
            keys.append(clean_dna(r, 17) + b":" + clean_dna(r, 16))
            to_generic = True
    elif case.startswith("41-symbols"):
        sources.append(lambda rr: (clean_dna(rr, 20), clean_dna(rr, 21)))    # 41 symbols, 42 bytes
        sources.append(lambda rr: (clean_dna(rr, 20), clean_dna(rr, 20)))    # 40 symbols
        keys.append(clean_dna(r, 20) + b":" + clean_dna(r, 20))
        if case.endswith("has"):
            keys.append(clean_dna(r, 20) + b":" + clean_dna(r, 21))
            flex = False
    keys = list(dict.fromkeys(keys))
    make = pieces_of(keys)
    data = two_piece_reads(len(case), [make, make, make] + sources)
    info = check(gu, oracle, TWO_PARAMS, keys, data)[0]
    if not flex:
        assert info["flex_table"] == 0 and info["policy"] == "generic", info
        return
    assert info["flex_table"] == 1 and info["policy"] == "flex_S", info
    assert (info["generic_reads"] > 0) == to_generic, info


# ---------------------------------------------------------------------------------------------------------------------
# Extract+Count: the packed key table (EC_PK_MAX_LEN = 29 symbols, flex.cuh) and flex_prepare's limits
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("lengths,to_generic", [((0, 20, 28, 29), False), ((30,), True), ((32,), True), ((33,), True)],
                         ids=["0-28-29", "30", "32", "33"])
def test_extract_count_packed_key_length(gu, oracle, lengths, to_generic):
    """EC_PK_MAX_LEN (flex.cuh:94 / 185): single ACGT pieces of up to 29 symbols go through the insert log into the packed table; longer ones (and pieces
    longer than 32) to the byte arena through the generic code"""
    r = synth.SM64(sum(lengths) + 1)
    pool = {L: [r.dna(L) for _ in range(50)] for L in lengths}
    recs = []
    for i in range(4000):
        k = r.choice(pool[r.choice(lengths)])
        if k and r.below(10) == 0:
            k = synth.mutate(r, k, 1)
        # (nothing in front of US: an earlier chance match of US would lengthen the piece)
        s = (synth.mutate(r, US, 1) if r.below(8) == 0 else US) + k + DS + r.dna(r.below(10))
        recs.append((b"@e%d" % i, s, synth.qual_line(r, len(s), 0.05)))
    data = fastq(recs)
    info = check(gu, oracle, dict(mode="EC", upstream=US.decode(), downstream=DS.decode(), miss_search_up=1, miss_search_down=1),
                 None, data, resolver=False)[0]
    assert info["policy"] == "flex_S"
    assert (info["generic_reads"] > 0) == to_generic, info


FLEX_PREPARE_CASES = [
    ("us32", dict(upstream="ACGTTGCAACGTTGCAACGTTGCAACGTTGCA", length=20), "flex_S"),
    ("us33", dict(upstream="ACGTTGCAACGTTGCAACGTTGCAACGTTGCAT", length=20), "generic"),
    ("k3", dict(upstream="GTTCAGAGTTCT", downstream="CTGAATAGGCCA", miss_search_up=3), "flex_B"),
    ("k4", dict(upstream="GTTCAGAGTTCT", downstream="CTGAATAGGCCA", miss_search_up=4), "generic"),
    ("2-iterations", dict(upstream="ACCGGT,GGATCC", downstream="TTGACA,CAATTG"), "flex_S"),
    ("3-iterations", dict(upstream="ACCGGT,GGATCC,AAGCTT", downstream="TTGACA,CAATTG,GTCGAC"), "generic"),
]


@pytest.mark.parametrize("name,kw,policy", FLEX_PREPARE_CASES, ids=[c[0] for c in FLEX_PREPARE_CASES])
def test_flex_prepare_limits(gu, oracle, name, kw, policy):
    """flex_prepare (flex_core.h:489 / 493): search sequences of 1..32 ACGT symbols, k <= 3, at most 2 iterations; beyond them the generic policy"""
    r = synth.SM64(len(name) * 7)
    ups = kw["upstream"].encode().split(b",")
    downs = kw["downstream"].encode().split(b",") if "downstream" in kw else [b""] * len(ups)
    recs = []
    for i in range(3000):
        s = r.dna(r.below(6))
        for u, d in zip(ups, downs):
            kk = r.below(4)
            s += (synth.mutate(r, u, kk) if kk < 3 else u) + r.dna(14 + r.below(12)) + d + r.dna(r.below(4))
        recs.append((b"@p%d" % i, s, synth.qual_line(r, len(s), 0.05)))
    params = dict(mode="EC", **kw)
    info = check(gu, oracle, params, None, fastq(recs), resolver=False)[0]
    assert info["policy"] == policy
