"""
-m gpu: one plain or bgzip file as ONE sample on several contexts (f2q_submit_file_sharded).  Every range after the first
guesses its first record start on the device; the guesses are verified against the range before, the bytes around the cuts
are stitched on the first context and the other contexts' results are added into it.  Whatever the cuts and the bytes, the
first context must end with exactly the oracle's results; input the protocol cannot split or verify must be parsed again,
whole, on the first context (shards == 1, shard_fallback == 1).

Every case runs with 2, 3, 4 and 8 contexts on device 0 and, when several GPUs are visible, with one context per GPU.
"""
import gzip
import importlib
import os
import struct
import zlib

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

lib = importlib.import_module("2fast2q_b200._lib")
synth = importlib.import_module("2fast2q_b200.synth")

NS = (2, 3, 4, 8)


def _layouts():
    try:
        n_dev = lib.device_count()
    except ImportError:
        n_dev = 0
    out = [("dev0", n) for n in NS]
    if n_dev > 1:
        out += [("per_gpu", n) for n in NS if n <= n_dev]
    return out


LAYOUTS = _layouts()
LAYOUT_IDS = [f"{k}-{n}" for k, n in LAYOUTS]


def _devices(layout):
    kind, n = layout
    return [0] * n if kind == "dev0" else list(range(n))


def _bgzf(data, bs=65280, level=4, eof=True):
    """a BGZF (bgzip) file of `data`: independent gzip members with a 'BC' extra field holding their size (+ the EOF block)"""
    out = []
    offsets = list(range(0, len(data), bs)) + ([None] if eof else [])
    for o in offsets:
        chunk = b"" if o is None else data[o:o + bs]
        c = zlib.compressobj(level, zlib.DEFLATED, -15)
        cd = c.compress(chunk) + c.flush()
        out.append(b"\x1f\x8b\x08\x04\x00\x00\x00\x00\x00\xff\x06\x00BC\x02\x00" + struct.pack("<H", 18 + len(cd) + 8 - 1) + cd
                   + struct.pack("<II", zlib.crc32(chunk) & 0xFFFFFFFF, len(chunk)))
    return b"".join(out)


class Pool:
    """engines per (configuration, library, devices), reused across samples"""

    def __init__(self):
        self.cache = {}

    def get(self, params, keys, devices, **options):
        sig = (repr(sorted(params.items())), None if keys is None else hash(tuple(keys)), tuple(devices), repr(sorted(options.items())))
        if sig not in self.cache:
            cfg = lib.make_config(**params)
            engines = [lib.Engine(cfg, d, None, **options) for d in devices]
            if keys is not None:
                for e in engines:
                    e.set_library(keys)
            self.cache[sig] = engines
        return self.cache[sig]

    def close(self):
        for engines in self.cache.values():
            for e in engines:
                e.close()
        self.cache.clear()


@pytest.fixture(scope="module")
def pool():
    assert lib.device_count() >= 1, "no B200 visible"
    p = Pool()
    yield p
    p.close()


def run_sharded(pool, params, keys, path, gz, devices, cuts=None, **options):
    """(counts or EC items, stats, complete, shards, fallback); asserts that every other context ends empty"""
    engines = pool.get(params, keys, devices, **options)
    for e in engines:
        e.begin()
    complete, nbytes = lib.submit_file_sharded(engines, str(path), gz, cuts=cuts, threads=8)
    counts, stats = engines[0].end()
    got = engines[0].ec_items() if keys is None else counts
    shards, fallback = engines[0].info("shards"), engines[0].info("shard_fallback")
    for e in engines[1:]:
        c, s = e.end()
        assert not c.any() and not any(s.values())
        if keys is None:
            assert e.ec_items() == {}
    return got, stats, complete, shards, fallback, nbytes


def want_of(oracle, params, keys, data):
    ocfg = oracle.make_config(**params)
    return oracle.extract_count(ocfg, data) if keys is None else oracle.count(ocfg, keys, data)


def same(got, want):
    return got == want if isinstance(want, dict) else np.array_equal(got, want)


def even_cuts(size, n):
    return [size * k // n for k in range(1, n)]


# ---- inputs (seeded) ------------------------------------------------------------------------------------------------
_DATA = {}


def config2():
    if "c2" not in _DATA:
        spec = synth.default_spec(2)
        names, keys = synth.make_library(2, 2000, 20)
        _DATA["c2"] = (dict(miss=1), keys, synth.fixed_reads(keys, 0, 200_000, **spec).tobytes())
    return _DATA["c2"]


def mixed(crlf=False, n=20_000):
    """reads of 40-200 bp with a library guide at offset 0, optionally with CRLF line ends"""
    key = ("mixed", crlf)
    if key not in _DATA:
        r = synth.SM64(4242)
        guides = [r.dna(20) for _ in range(300)]
        nl = b"\r\n" if crlf else b"\n"
        out = []
        for i in range(n):
            g = r.choice(guides)
            if r.below(4) == 0:
                g = synth.mutate(r, g, 1)
            s = g + r.dna(20 + r.below(181))
            out.append(b"@m%d" % i + nl + s + nl + b"+" + nl + synth.qual_line(r, len(s), 0.05) + nl)
        _DATA[key] = (dict(miss=1), guides, b"".join(out))
    return _DATA[key]


def shaped(config, n_reads=150_000):
    if config not in _DATA:
        spec = synth.shape_spec(config)
        if config == "4":
            guides = synth.random_kmers(4, 20_000, 20)
            params = dict(mode="EC", upstream=synth.BARSEQ_US.decode(), downstream=synth.BARSEQ_DS.decode(), miss_search_up=1, miss_search_down=1)
            lines = synth.shaped_reads(guides, 0, n_reads, **spec).tobytes().split(b"\n")
            us = synth.BARSEQ_US
            for i in range(1, len(lines), 4 * 37):                             # an N in every 37th barcode: byte-arena keys
                j = lines[i].find(us)
                if j >= 0 and j + len(us) < len(lines[i]):
                    k = j + len(us)
                    lines[i] = lines[i][:k] + b"N" + lines[i][k + 1:]
            _DATA[config] = (params, None, b"\n".join(lines))
        else:
            names, keys, xs, ys = synth.dual_keys(3000)
            params = dict(mode="C", miss=1, upstream="ACCGGT,GGATCC", downstream="TTGACA,CAATTG")
            _DATA[config] = (params, keys, synth.shaped_reads(xs + ys, 0, n_reads, **spec).tobytes())
    return _DATA[config]


def hostile(kind, n=40_000):
    """FASTQ-shaped bytes that defeat a local record-start guess (the four kinds of test_gpu_spec)"""
    r = synth.SM64(1234)
    guides = [r.dna(20) for _ in range(64)]
    out = []
    for i in range(n):
        g = r.choice(guides)
        if r.below(5) == 0:
            g = synth.mutate(r, g, 1)
        s = g + r.dna(30)
        q = synth.qual_line(r, len(s), 0.05)
        if kind == "at_plus_everywhere":
            out.append(b"@" + s[1:] + b"\n" + b"+" + s[1:] + b"\n+" + q[1:] + b"\n@" + q[1:] + b"\n")
        elif kind == "blank_lines":
            out.append(b"@r%d\n" % i + s + b"\n+\n" + q + b"\n" + (b"\n" if i % 7 == 0 else b""))
        elif kind == "quality_is_header":
            out.append(b"@r%d\n" % i + s + b"\n" + q + b"\n")
        elif kind == "unequal_lengths":
            out.append(b"@r%d\n" % i + s + b"\n+\n" + q[:-3] + b"\n")
        else:
            raise ValueError(kind)
    return dict(miss=1), guides, b"".join(out)


def misaligned_cuts(data, n):
    """n-1 cuts on the newline in front of header lines that are NOT record starts (line index % 4 != 0) and have no blank
    line inside or right behind their two records: the guess there is that header, and it is wrong"""
    starts, line, pos = [], 0, 0
    while True:
        nl = data.find(b"\n", pos)
        if nl < 0:
            break
        line += 1
        if line % 4 != 0 and data[nl + 1:nl + 3] == b"@r":
            i = int(data[nl + 3:data.index(b"\n", nl + 1)])
            if i % 7 != 0 and (i + 1) % 7 != 0:
                starts.append(nl)
        pos = nl + 1
    return [starts[len(starts) * k // n] for k in range(1, n)]


def write(tmp_path, data, name="x.fastq"):
    p = tmp_path / name
    p.write_bytes(data)
    return p


# ---- the config-2 shape, plain and bgzip ----------------------------------------------------------------------------
@pytest.mark.parametrize("fmt", ["plain", "bgzip"])
@pytest.mark.parametrize("layout", LAYOUTS, ids=LAYOUT_IDS)
def test_config2_is_exact_on_every_shard_count(pool, oracle, tmp_path, layout, fmt):
    params, keys, data = config2()
    want_c, want_s = want_of(oracle, params, keys, data)
    blob = data if fmt == "plain" else _bgzf(data)
    p = write(tmp_path, blob, "x.fastq" if fmt == "plain" else "x.fastq.gz")
    n = layout[1]
    got, stats, complete, shards, fallback, nbytes = run_sharded(pool, params, keys, p, fmt == "bgzip", _devices(layout), even_cuts(len(blob), n))
    assert stats == want_s and same(got, want_c)
    assert complete and nbytes == len(data)
    assert (shards, fallback) == (n, 0)


# ---- cuts near one record in every position -------------------------------------------------------------------------
def _positions(data, rec_start):
    """cut offsets around the record at rec_start: its start, just after each of its newlines, inside every line, and on
    the last byte before each newline"""
    nls, pos = [], rec_start
    for _ in range(4):
        pos = data.index(b"\n", pos)
        nls.append(pos)
        pos += 1
    out = {rec_start, rec_start + 1}
    prev = rec_start
    for nl in nls:
        out.update({nl + 1, nl, nl - 1, (prev + nl) // 2})
        prev = nl + 1
    return sorted(out)


@pytest.mark.parametrize("kind", ["lf", "crlf", "mixed_lengths"])
@pytest.mark.parametrize("layout", LAYOUTS, ids=LAYOUT_IDS)
def test_cuts_near_one_record_in_every_position(pool, oracle, tmp_path, layout, kind):
    if kind == "lf":
        params, keys, data = config2()
        data = data[:118 * 30_000]
    else:
        params, keys, data = mixed(crlf=kind == "crlf")
    want_c, want_s = want_of(oracle, params, keys, data)
    p = write(tmp_path, data)
    n = layout[1]
    # the record the first cut moves around sits at about 1/(2n) of the file; the other cuts stay evenly spread behind it
    target = len(data) // (2 * n)
    rec = 0
    while True:
        nxt = rec
        for _ in range(4):
            nxt = data.index(b"\n", nxt) + 1
        if nxt > target:
            break
        rec = nxt
    rest = [len(data) * k // n for k in range(1, n)][1:]
    for x in _positions(data, rec):
        got, stats, complete, shards, fallback, _ = run_sharded(pool, params, keys, p, False, _devices(layout), [x] + rest)
        assert stats == want_s and same(got, want_c), (x - rec)
        assert (shards, fallback) == (n, 0), (x - rec)


# ---- flex workloads -------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("config", ["4", "5b"])
@pytest.mark.parametrize("layout", LAYOUTS, ids=LAYOUT_IDS)
def test_flex_workloads(pool, oracle, tmp_path, layout, config):
    """config 4 (Extract+Count, N barcodes: byte-arena keys exist) and config 5b (Counter, dual delimiters)"""
    params, keys, data = shaped(config)
    want, want_s = want_of(oracle, params, keys, data)
    if keys is None:
        assert any(b"N" in k for k in want)                                   # (the byte-arena table is exercised)
    p = write(tmp_path, data)
    n = layout[1]
    got, stats, complete, shards, fallback, _ = run_sharded(pool, params, keys, p, False, _devices(layout), even_cuts(len(data), n))
    assert stats == want_s and same(got, want)
    assert (shards, fallback) == (n, 0)


# ---- fallbacks ------------------------------------------------------------------------------------------------------
def _fallback_case(name):
    if name == "odd_line_in_front":
        params, keys, data = config2()
        return params, keys, b"@odd\n" + data[:118 * 60_000], "plain"
    if name.startswith("hostile_"):
        params, keys, data = hostile(name[len("hostile_"):])
        return params, keys, data, "plain"
    params, keys, data = config2()
    data = data[:118 * 40_000]
    if name == "shard_smaller_than_a_record":
        return params, keys, data, "plain"
    if name == "bgzip_without_eof_block":
        return params, keys, data, "bgzip_noeof"
    if name == "bgzip_foreign_trailing_member":
        extra = synth.fixed_reads(keys, 40_000, 500, **synth.default_spec(2)).tobytes()
        return params, keys, data + extra, "bgzip_foreign"
    if name == "ordinary_gzip":
        return params, keys, data, "gzip"
    raise ValueError(name)


FALLBACKS = ["odd_line_in_front", "hostile_at_plus_everywhere", "hostile_blank_lines", "hostile_quality_is_header",
             "hostile_unequal_lengths", "shard_smaller_than_a_record", "bgzip_without_eof_block", "bgzip_foreign_trailing_member",
             "ordinary_gzip"]


@pytest.mark.parametrize("name", FALLBACKS)
@pytest.mark.parametrize("layout", LAYOUTS, ids=LAYOUT_IDS)
def test_fallbacks_are_exact(pool, oracle, tmp_path, layout, name):
    params, keys, data, fmt = _fallback_case(name)
    want_c, want_s = want_of(oracle, params, keys, data)
    n = layout[1]
    if fmt == "plain":
        blob = data
        if name == "shard_smaller_than_a_record":
            cuts = even_cuts(len(blob), n - 1) + [len(blob) - 30]            # (the last range: 30 bytes)
        elif name == "hostile_blank_lines":
            cuts = misaligned_cuts(data, n)
        else:
            cuts = even_cuts(len(blob), n)
    elif fmt == "bgzip_noeof":
        blob = _bgzf(data, eof=False)
        cuts = even_cuts(len(blob), n)
    elif fmt == "bgzip_foreign":
        main_part = data[:118 * 40_000]
        blob = _bgzf(main_part)[:-28] + gzip.compress(data[len(main_part):])
        cuts = even_cuts(len(blob), n)
    else:
        blob = gzip.compress(data)
        cuts = even_cuts(len(blob), n)
    p = write(tmp_path, blob, "x.fastq" if fmt == "plain" else "x.fastq.gz")
    got, stats, complete, shards, fallback, _ = run_sharded(pool, params, keys, p, fmt != "plain", _devices(layout), cuts)
    assert stats == want_s and same(got, want_c)
    assert complete
    assert (shards, fallback) == (1, 1)


@pytest.mark.parametrize("layout", LAYOUTS, ids=LAYOUT_IDS)
def test_truncated_gzip_falls_back_like_submit_file(pool, tmp_path, layout):
    params, keys, data = config2()
    blob = gzip.compress(data[:118 * 40_000])
    p = write(tmp_path, blob[:len(blob) * 2 // 3], "x.fastq.gz")
    single = pool.get(params, keys, (0,))
    single[0].begin()
    ok1, nb1 = single[0].submit_file(str(p), True, 0, 8)
    want_c, want_s = single[0].end()
    got, stats, complete, shards, fallback, nbytes = run_sharded(pool, params, keys, p, True, _devices(layout), even_cuts(len(blob), layout[1]))
    assert not ok1 and not complete and nbytes == nb1
    assert stats == want_s and same(got, want_c)
    assert (shards, fallback) == (1, 1)


# ---- edge cases -----------------------------------------------------------------------------------------------------
def _edge(name):
    params, keys, data = config2()
    data = data[:118 * 30_000]
    if name == "empty":
        return params, keys, b""
    if name == "smaller_than_n_shards":
        return params, keys, data[:118 * 3]
    if name == "unterminated_last_line":
        return params, keys, data[:-1]
    if name.startswith("leftover_"):
        k = int(name[-1])
        return params, keys, data + b"".join([b"@left\n", b"ACGTACGTACGTACGTACGTAC\n", b"+\n"][:k])
    if name == "cuts_at_zero_and_end":
        return params, keys, data
    raise ValueError(name)


EDGES = ["empty", "smaller_than_n_shards", "unterminated_last_line", "leftover_1", "leftover_2", "leftover_3", "cuts_at_zero_and_end"]


@pytest.mark.parametrize("fmt", ["plain", "bgzip"])
@pytest.mark.parametrize("name", EDGES)
@pytest.mark.parametrize("layout", LAYOUTS, ids=LAYOUT_IDS)
def test_edge_cases(pool, oracle, tmp_path, layout, name, fmt):
    params, keys, data = _edge(name)
    want_c, want_s = want_of(oracle, params, keys, data)
    blob = data if fmt == "plain" else _bgzf(data)
    p = write(tmp_path, blob, "x.fastq" if fmt == "plain" else "x.fastq.gz")
    n = layout[1]
    if name == "cuts_at_zero_and_end":
        cuts = [0] + even_cuts(len(blob), n - 1)[:n - 3] + [len(blob)] if n > 2 else [0]
        expect = (max(1, n - 2), 0)
    elif name in ("empty", "smaller_than_n_shards"):
        cuts = None                                                            # (even ranges of >= 64 MiB: one range)
        expect = (1, 0)
    else:
        cuts = even_cuts(len(blob), n)
        expect = (n, 0)
    got, stats, complete, shards, fallback, _ = run_sharded(pool, params, keys, p, fmt == "bgzip", _devices(layout), cuts)
    assert stats == want_s and same(got, want_c)
    assert complete
    assert (shards, fallback) == expect


# ---- errors ---------------------------------------------------------------------------------------------------------
def test_errors(pool, tmp_path):
    params, keys, data = config2()
    p = write(tmp_path, data[:118 * 20_000])
    cfg = lib.make_config(**params)
    with lib.Engine(cfg, 0) as a, lib.Engine(cfg, 0) as b, lib.Engine(lib.make_config(miss=2), 0) as other_cfg, lib.Engine(cfg, 0) as other_lib:
        for e in (a, b, other_cfg):
            e.set_library(keys)
        other_lib.set_library(keys[:-1])
        a.begin()
        with pytest.raises(lib.F2QError) as ei:                               # b is not inside a sample
            lib.submit_file_sharded([a, b], str(p), False)
        assert ei.value.code == -4
        b.begin(); other_cfg.begin(); other_lib.begin()
        for engines in ([a, other_cfg], [a, other_lib]):
            with pytest.raises(lib.F2QError) as ei:
                lib.submit_file_sharded(engines, str(p), False)
            assert ei.value.code == -1
        with pytest.raises(lib.F2QError) as ei:
            lib.submit_file_sharded([a, b, a], str(p), False)
        assert ei.value.code == -1
        # the engines are still usable
        lib.submit_file_sharded([a, b], str(p), False, cuts=[os.path.getsize(p) // 2])
        counts, stats = a.end()
        assert stats["reads"] == 20_000
        b.end()


@pytest.mark.parametrize("layout", [l for l in LAYOUTS if l[1] == 4], ids=[i for l, i in zip(LAYOUTS, LAYOUT_IDS) if l[1] == 4])
def test_record_longer_than_carry_bytes_fails_the_sample(pool, tmp_path, layout):
    """a record longer than carry_bytes that shard 2 has to carry into the stitch: ctxs[0]'s sample fails with F2Q_ETOOLONG"""
    params, keys, data = config2()
    data = data[:118 * 40_000]
    q = len(data) // 4
    at = (3 * q - 20_000) // 118 * 118                                         # a record start in range 2 (118-byte records)
    long_seq = b"ACGT" * 2500
    long_rec = b"@long\n" + long_seq + b"\n+\n" + b"I" * len(long_seq) + b"\n"
    data = data[:at] + long_rec + data[at:]
    cut3 = at + len(long_rec) - 100                                           # inside its quality line, near its end
    p = write(tmp_path, data)
    engines = pool.get(params, keys, _devices(layout), carry_bytes=4096)
    for e in engines:
        e.begin()
    lib.submit_file_sharded(engines, str(p), False, cuts=[q, 2 * q, cut3])
    with pytest.raises(lib.F2QError) as ei:
        engines[0].end()
    assert ei.value.code == -6
    for e in engines[1:]:
        e.end()


# ---- command line ---------------------------------------------------------------------------------------------------
def _cli_param(fq, tmp_path, out):
    p = fq.input_parser(["-c", "--s", str(tmp_path), "--g", "x", "--o", str(out), "--pb"])
    return fq.initializer(p)


def test_split_file_native_writes_the_single_gpu_csv(tmp_path):
    """three contexts on device 0 over a file of three 64 MiB ranges write the same <sample>_reads.csv as one context"""
    import cli_golden as CG
    fq = importlib.import_module("2fast2q_b200.fast2q")
    params, keys, data = config2()
    raw = tmp_path / "in" / "big.fastq"
    raw.parent.mkdir()
    raw.write_bytes(data * 9)                                                 # 212 MB
    feats = {k: fq.Features(f"g{i}", 0) for i, k in enumerate(keys)}
    outs = []
    for sharded in (False, True):
        p = _cli_param(fq, tmp_path / "in", tmp_path / ("out%d" % sharded))
        os.makedirs(p["directory"], exist_ok=True)
        try:
            if sharded:
                fq.split_file_native(str(raw), feats, dict(p, device=0), [0, 0, 0])
            else:
                fq.aligner(0, str(raw), feats, dict(p, device=0), {"failed_reads": set(), "passed_reads": {}})
        finally:
            fq.release_engines()
        outs.append(open(os.path.join(p["directory"], "big_reads.csv"), newline="").read())
    assert CG.mask_reads_csv(outs[0]) == CG.mask_reads_csv(outs[1])


def test_cli_file_split_on_two_gpus_equals_one(tmp_path):
    if lib.device_count() < 2:
        pytest.skip("needs two GPUs")
    import glob
    import cli_golden as CG
    fq = importlib.import_module("2fast2q_b200.fast2q")
    c = CG.case("cli_counter")
    got = []
    for g in ("1", "2"):
        root = tmp_path / g
        argv = CG.write_inputs(c, str(root)) + ["--fs", "--gpus", g]
        fq.main(argv)
        d = glob.glob(os.path.join(str(root), "out", "2FAST2Q_output_*"))[0]
        got.append(open(os.path.join(d, "compiled.csv"), newline="").read())
    assert got[0] == got[1]
