"""
ctypes binding of libf2q.so (include/f2q.h) and the `Engine` convenience wrapper.

No CPU fallback exists: if the library is missing or no B200-class device is present, loading / creating an
engine raises — the product path never routes through oracle/ or any host implementation.
"""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "libf2q.so")

ABI_VERSION = 2
MAX_ITER = 8
MAX_DELIM = 64
N_STATS = 5
STAT_NAMES = ("reads", "perfect_counter", "imperfect_counter", "non_aligned_counter", "quality_failed")
MODE_COUNT, MODE_EXTRACT_COUNT = 0, 1
ERRORS = {0: "OK", -1: "EINVAL", -2: "ENOMEM", -3: "ECUDA", -4: "ESTATE", -5: "EUNSUPPORTED", -6: "ETOOLONG",
          -7: "ENODEVICE", -8: "EINTERNAL"}


class F2QError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__(f"libf2q {ERRORS.get(code, code)}: {msg}")
        self.code = code


class Config(C.Structure):
    """struct f2q_config (include/f2q.h)"""
    _fields_ = [
        ("mode", C.c_int32), ("miss", C.c_int32), ("phred", C.c_int32), ("qual_up", C.c_int32),
        ("qual_down", C.c_int32), ("miss_up", C.c_int32), ("miss_down", C.c_int32), ("length", C.c_int32),
        ("n_iter", C.c_int32), ("has_up", C.c_int32), ("has_down", C.c_int32),
        ("starts", C.c_int32 * MAX_ITER), ("up_len", C.c_int32 * MAX_ITER), ("down_len", C.c_int32 * MAX_ITER),
        ("up", (C.c_uint8 * MAX_DELIM) * MAX_ITER), ("down", (C.c_uint8 * MAX_DELIM) * MAX_ITER),
    ]


class SynthSpec(C.Structure):
    """struct f2q_synth_spec (include/f2q.h)"""
    _fields_ = [
        ("seed", C.c_uint64), ("first_read", C.c_uint64), ("n_reads", C.c_uint64), ("read_len", C.c_uint32),
        ("feat_len", C.c_uint32), ("n_guides", C.c_uint32), ("cum_exact", C.c_uint32), ("cum_sub1", C.c_uint32),
        ("cum_sub2", C.c_uint32), ("cum_sub3", C.c_uint32), ("cum_n", C.c_uint32), ("lowq_per_65536", C.c_uint32),
        ("shape", C.c_uint32), ("delim_len", C.c_uint32 * 4), ("delim", (C.c_uint8 * 16) * 4),
    ]


# every symbol include/f2q.h declares: name -> (restype, argtypes)
_VP, _U64P, _I32P = C.c_void_p, C.POINTER(C.c_uint64), C.POINTER(C.c_int32)
SYMBOLS = {
    "f2q_abi_version": (C.c_int, []),
    "f2q_device_count": (C.c_int, []),
    "f2q_create": (C.c_int, [C.POINTER(Config), C.c_int, _VP, C.POINTER(_VP)]),
    "f2q_destroy": (None, [_VP]),
    "f2q_last_error": (C.c_char_p, [_VP]),
    "f2q_set_option": (C.c_int, [_VP, C.c_char_p, C.c_int64]),
    "f2q_set_library": (C.c_int, [_VP, _VP, _VP, C.c_uint32]),
    "f2q_begin_sample": (C.c_int, [_VP]),
    "f2q_submit": (C.c_int, [_VP, _VP, C.c_uint64, C.c_int]),
    "f2q_submit_file_sharded": (C.c_int, [C.POINTER(_VP), C.c_int, C.c_char_p, C.c_int, _U64P, C.c_int, _I32P, _U64P]),
    "f2q_submit_device": (C.c_int, [_VP, _VP, C.c_uint64, C.c_int]),
    "f2q_submit_file": (C.c_int, [_VP, C.c_char_p, C.c_int, C.c_uint64, C.c_int, _I32P, _U64P]),
    "f2q_sync": (C.c_int, [_VP]),
    "f2q_sync_copies": (C.c_int, [_VP]),
    "f2q_end_sample": (C.c_int, [_VP, _VP, _VP]),
    "f2q_end_sample_async": (C.c_int, [_VP, _VP]),
    "f2q_result_device": (C.c_int, [_VP, C.POINTER(_VP), _U64P]),
    "f2q_ec_size": (C.c_int, [_VP, _U64P, _U64P]),
    "f2q_ec_drain": (C.c_int, [_VP, _VP, _VP, _VP]),
    "f2q_comm_load": (C.c_int, [C.c_char_p]),
    "f2q_comm_unique_id": (C.c_int, [_VP]),
    "f2q_comm_init_rank": (C.c_int, [_VP, _VP, C.c_int, C.c_int]),
    "f2q_comm_init": (C.c_int, [C.POINTER(_VP), C.c_int]),
    "f2q_comm_destroy": (C.c_int, [_VP]),
    "f2q_comm_share": (C.c_int, [_VP, _VP]),
    "f2q_allreduce_counts": (C.c_int, [C.POINTER(_VP), C.c_int]),
    "f2q_ec_merge": (C.c_int, [C.POINTER(_VP), C.c_int]),
    "f2q_host_alloc": (C.c_int, [C.POINTER(_VP), C.c_uint64]),
    "f2q_host_alloc_near": (C.c_int, [C.POINTER(_VP), C.c_uint64, C.c_int, C.c_int, _I32P]),
    "f2q_host_free": (C.c_int, [_VP]),
    "f2q_border_finder": (C.c_int, [C.c_int, C.c_char_p, C.c_uint32, C.c_char_p, C.c_uint32, C.c_int32, C.c_int32, _I32P]),
    "f2q_sequence_tinder": (C.c_int, [C.c_int, C.POINTER(Config), C.c_int32, C.c_char_p, C.c_uint32, C.c_char_p, C.c_uint32,
                                      _VP, _VP, _I32P, _I32P, _I32P]),
    "f2q_synth_fastq": (C.c_int, [_VP, C.POINTER(SynthSpec), _VP, _VP]),
    "f2q_inflate_blocks": (C.c_int, [_VP, _VP, _VP, C.c_uint32, _VP, C.POINTER(C.c_uint32)]),
    "f2q_device_alloc": (C.c_int, [_VP, C.POINTER(_VP), C.c_uint64]),
    "f2q_device_free": (C.c_int, [_VP, _VP]),
    "f2q_memcpy_d2h": (C.c_int, [_VP, _VP, _VP, C.c_uint64]),
    "f2q_memcpy_h2d": (C.c_int, [_VP, _VP, _VP, C.c_uint64]),
    "f2q_launch_count": (C.c_uint64, [_VP]),
    "f2q_kernel_times": (C.c_int, [_VP, C.POINTER(C.c_double), _U64P]),
    "f2q_spec_counts": (C.c_int, [_VP, _U64P, _U64P]),
    "f2q_memo_counts": (C.c_int, [_VP, _U64P, _U64P]),
    "f2q_get_info": (C.c_int, [_VP, C.c_char_p, C.POINTER(C.c_int64)]),
}
POLICIES = ("generic", "fast1", "flex_S", "flex_B")          # f2q_get_info "policy"
TABLES = ("probing", "compact", "cuckoo", "cuckoo+neighbours")   # f2q_get_info "table"

_lib = None


def load():
    """dlopen libf2q.so and bind every declared symbol; raises if the CUDA library has not been built."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise ImportError(f"{LIB_PATH} is missing: build it with `python 2fast2q_b200/build.py` "
                              "(nvcc, sm_100a).  There is no CPU fallback.")
        L = C.CDLL(LIB_PATH)
        for name, (res, args) in SYMBOLS.items():
            fn = getattr(L, name)           # AttributeError if the ABI is incomplete
            fn.restype, fn.argtypes = res, args
        if L.f2q_abi_version() != ABI_VERSION:
            raise ImportError("libf2q.so ABI version mismatch")
        _lib = L
    return _lib


def device_count() -> int:
    return load().f2q_device_count()


def make_config(mode="C", miss=1, phred=30, length=20, start="0", upstream=None, downstream=None,
                miss_search_up=0, miss_search_down=0, qual_up=30, qual_down=30) -> Config:
    """hot-path parameters as reads_counter derives them (fast2q.py:538-558).  Raises ValueError where the reference
    prints FATAL and exits (unequal numbers of up/downstream sequences, fast2q.py:553-556)."""
    c = Config()
    c.mode = MODE_EXTRACT_COUNT if "EC" in str(mode).upper() else MODE_COUNT
    c.miss, c.phred, c.length = int(miss), int(phred), int(length)
    c.qual_up, c.qual_down = int(qual_up), int(qual_down)
    c.miss_up, c.miss_down = int(miss_search_up), int(miss_search_down)
    if upstream is None and downstream is None:
        st = [int(n) for n in str(start).split(",")]
        if len(st) > MAX_ITER:
            raise ValueError(f"at most {MAX_ITER} start positions are supported")
        c.n_iter = len(st)
        for i, s in enumerate(st):
            c.starts[i] = s
        return c
    ups = [u.upper().encode() for u in upstream.split(",")] if upstream is not None else []
    downs = [d.upper().encode() for d in downstream.split(",")] if downstream is not None else []
    if upstream is not None and downstream is not None and len(ups) != len(downs):
        raise ValueError("Up and Downstream sequences must be submitted in concurrent pairs, separated by ,.\n You submitted "
                         f"{len(downs)} downstream sequences and {len(ups)} upstream sequences.")
    c.has_up, c.has_down = int(upstream is not None), int(downstream is not None)
    c.n_iter = max(len(ups), len(downs))
    if c.n_iter > MAX_ITER:
        raise ValueError(f"at most {MAX_ITER} search sequence pairs are supported")
    for dst, dlen, items in ((c.up, c.up_len, ups), (c.down, c.down_len, downs)):
        for i, u in enumerate(items):
            if len(u) > MAX_DELIM:
                raise ValueError(f"search sequences longer than {MAX_DELIM} bp are not supported")
            dlen[i] = len(u)
            for j, b in enumerate(u):
                dst[i][j] = b
    return c


def make_synth_spec(n_seqs: int, first_read: int, n_reads: int, *, seed, read_len, feat_len, lowq_per_65536, shape=0, delims=(),
                    cum_exact=0, cum_sub1=0, cum_sub2=0, cum_sub3=0, cum_n=0) -> SynthSpec:
    """struct f2q_synth_spec from the dicts of synth.default_spec / synth.shape_spec; n_seqs = len(guides)"""
    s = SynthSpec()
    s.seed, s.first_read, s.n_reads = seed, first_read, n_reads
    s.read_len, s.feat_len, s.shape = read_len, feat_len, shape
    s.n_guides = n_seqs // 2 if shape >= 2 else n_seqs
    s.cum_exact, s.cum_sub1, s.cum_sub2, s.cum_sub3, s.cum_n = cum_exact, cum_sub1, cum_sub2, cum_sub3, cum_n
    s.lowq_per_65536 = lowq_per_65536
    for k, d in enumerate(delims):
        s.delim_len[k] = len(d)
        for j, ch in enumerate(d):
            s.delim[k][j] = ch
    return s


def pack_keys(keys):
    bs = [k.encode() if isinstance(k, str) else bytes(k) for k in keys]
    off = np.zeros(len(bs) + 1, dtype=np.uint64)
    if bs:
        off[1:] = np.cumsum([len(b) for b in bs], dtype=np.uint64)
    blob = np.frombuffer(b"".join(bs) + b"\0", dtype=np.uint8).copy()
    return blob, off


def nccl_library_path():
    """libnccl.so.2 of the nvidia-nccl wheel beside torch, or None (libf2q then uses F2Q_NCCL_LIB / the default search)"""
    try:
        import importlib.util
        spec = importlib.util.find_spec("nvidia.nccl")
        for base in (spec.submodule_search_locations or []) if spec else []:
            p = os.path.join(base, "lib", "libnccl.so.2")
            if os.path.exists(p):
                return p
    except Exception:
        pass
    return None


def comm_load():
    L = load()
    p = nccl_library_path()
    rc = L.f2q_comm_load(p.encode() if p else None)
    if rc:
        raise F2QError(rc, L.f2q_last_error(None).decode())


def comm_unique_id() -> bytes:
    comm_load()
    buf = (C.c_uint8 * 128)()
    rc = load().f2q_comm_unique_id(buf)
    if rc:
        raise F2QError(rc, load().f2q_last_error(None).decode())
    return bytes(buf)


def comm_init(engines):
    """one process, several engines on distinct devices: one communicator over all of them"""
    comm_load()
    arr = (C.c_void_p * len(engines))(*[e.h for e in engines])
    rc = load().f2q_comm_init(arr, len(engines))
    if rc:
        raise F2QError(rc, load().f2q_last_error(engines[0].h).decode() or load().f2q_last_error(None).decode())


def allreduce_counts(engines):
    arr = (C.c_void_p * len(engines))(*[e.h for e in engines])
    engines[0]._ck(load().f2q_allreduce_counts(arr, len(engines)))


def ec_merge(engines):
    arr = (C.c_void_p * len(engines))(*[e.h for e in engines])
    engines[0]._ck(load().f2q_ec_merge(arr, len(engines)))


def submit_file_sharded(engines, path, is_gzip, cuts=None, threads=8):
    """one plain or bgzip file as one sample parsed by every engine (each inside a freshly begun sample; f2q_submit_file_sharded).
    engines[0] then holds the whole sample (end() / ec_items() on it), the others are closed and empty.  cuts: None (even
    ranges of >= 64 MiB) or len(engines) - 1 file offsets.  Returns (complete, uncompressed bytes) as Engine.submit_file."""
    arr = (C.c_void_p * len(engines))(*[e.h for e in engines])
    cut_arr = (C.c_uint64 * max(1, len(engines) - 1))(*[int(x) for x in cuts]) if cuts is not None else None
    if cuts is not None and len(cuts) != len(engines) - 1:
        raise ValueError("cuts needs one offset fewer than there are engines")
    ok, nb = C.c_int32(1), C.c_uint64(0)
    engines[0]._ck(load().f2q_submit_file_sharded(arr, len(engines), os.fsencode(path), int(bool(is_gzip)), cut_arr, int(threads),
                                                  C.byref(ok), C.byref(nb)))
    return bool(ok.value), int(nb.value)


class PinnedBuffer:
    """page-locked host memory from f2q_host_alloc, exposed as a writable numpy uint8 array / memoryview"""

    def __init__(self, nbytes: int, device: int | None = None, write_combined: bool = False):
        """device: allocate near that GPU (its NUMA node, when the platform shows several; f2q_host_alloc_near)"""
        self.ptr = C.c_void_p()
        self.numa_node = -1
        if device is None and not write_combined:
            rc = load().f2q_host_alloc(C.byref(self.ptr), nbytes)
        else:
            node = C.c_int32(-1)
            rc = load().f2q_host_alloc_near(C.byref(self.ptr), nbytes, device or 0, 1 if write_combined else 0, C.byref(node))
            self.numa_node = node.value
        if rc:
            raise F2QError(rc, load().f2q_last_error(None).decode())
        self.nbytes = nbytes
        self.array = np.ctypeslib.as_array((C.c_uint8 * nbytes).from_address(self.ptr.value))

    def free(self):
        if self.ptr:
            self.array = None
            load().f2q_host_free(self.ptr)
            self.ptr = C.c_void_p()

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass


class Engine:
    """one f2q_ctx: one GPU, one sample in flight"""

    def __init__(self, cfg: Config, device: int = 0, stream: int | None = None, **options):
        self.L = load()
        self.cfg = cfg
        self.device = device
        self.h = C.c_void_p()
        rc = self.L.f2q_create(C.byref(cfg), device, C.c_void_p(stream) if stream else None, C.byref(self.h))
        if rc:
            raise F2QError(rc, self.L.f2q_last_error(None).decode())
        self.n_keys = 0
        for k, v in options.items():
            self.set_option(k, v)

    # -- plumbing
    def _ck(self, rc):
        if rc:
            raise F2QError(rc, self.L.f2q_last_error(self.h).decode())

    def close(self):
        if getattr(self, "h", None):
            self.L.f2q_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    def set_option(self, name: str, value: int):
        self._ck(self.L.f2q_set_option(self.h, name.encode(), int(value)))

    # -- library
    def set_library(self, keys):
        blob, off = pack_keys(keys)
        self._ck(self.L.f2q_set_library(self.h, blob.ctypes.data, off.ctypes.data, len(keys)))
        self.n_keys = len(keys)

    # -- sample
    def begin(self):
        self._ck(self.L.f2q_begin_sample(self.h))

    def submit(self, data, is_last: bool | int = False):
        """data: bytes / bytearray / memoryview / numpy uint8 array in HOST memory"""
        if isinstance(data, np.ndarray):
            a = np.ascontiguousarray(data, dtype=np.uint8)
            self._ck(self.L.f2q_submit(self.h, a.ctypes.data if a.size else None, a.size, int(is_last)))
        else:
            mv = memoryview(data)
            n = mv.nbytes
            if n == 0:
                self._ck(self.L.f2q_submit(self.h, None, 0, int(is_last)))
            else:
                a = np.frombuffer(mv, dtype=np.uint8)
                self._ck(self.L.f2q_submit(self.h, a.ctypes.data, n, int(is_last)))

    def submit_ptr(self, host_ptr: int, nbytes: int, is_last: bool | int = False):
        self._ck(self.L.f2q_submit(self.h, C.c_void_p(host_ptr), nbytes, int(is_last)))

    def submit_file(self, path: str, gzip: bool, limit_lines: int = 0, threads: int = 1):
        """one sequencing file -> the current sample, read / inflated natively into pinned ring buffers (f2q_submit_file).
        Returns (complete, uncompressed bytes); complete is False for a gzip stream that broke off before its end."""
        ok, nb = C.c_int32(1), C.c_uint64(0)
        self._ck(self.L.f2q_submit_file(self.h, os.fsencode(path), int(bool(gzip)), int(limit_lines), int(threads), C.byref(ok), C.byref(nb)))
        return bool(ok.value), int(nb.value)

    def submit_device(self, dptr: int, nbytes: int, is_last: bool | int = False):
        self._ck(self.L.f2q_submit_device(self.h, C.c_void_p(dptr), nbytes, int(is_last)))

    def sync(self):
        self._ck(self.L.f2q_sync(self.h))

    def sync_copies(self):
        """pinned host buffers passed to submit_ptr may be refilled after this returns"""
        self._ck(self.L.f2q_sync_copies(self.h))

    def end(self):
        """returns (counts uint64[n_keys], stats dict)"""
        counts = np.zeros(max(self.n_keys, 1), dtype=np.uint64)
        stats = np.zeros(N_STATS, dtype=np.uint64)
        self._ck(self.L.f2q_end_sample(self.h, counts.ctypes.data, stats.ctypes.data))
        return counts[:self.n_keys], dict(zip(STAT_NAMES, (int(x) for x in stats)))

    def end_async(self, pinned: "PinnedBuffer"):
        """finish the sample without waiting; `pinned` (>= 8 * (n_keys + 6) bytes) holds the result after sync()"""
        assert pinned.nbytes >= 8 * (self.n_keys + 6)
        self._ck(self.L.f2q_end_sample_async(self.h, pinned.ptr))

    def read_async_result(self, pinned: "PinnedBuffer"):
        """(counts, stats) from a buffer filled by end_async — call sync() first"""
        v = np.frombuffer(pinned.array, dtype=np.uint64, count=self.n_keys + 6)
        if int(v[self.n_keys + 5]):
            raise F2QError(-8, f"device-side failure, flags={int(v[self.n_keys + 5]):#x}")
        return v[:self.n_keys].copy(), dict(zip(STAT_NAMES, (int(x) for x in v[self.n_keys:self.n_keys + 5])))

    # -- several GPUs, one process per GPU (f2q_comm_*)
    def comm_init_rank(self, unique_id: bytes, nranks: int, rank: int):
        comm_load()
        buf = (C.c_uint8 * 128).from_buffer_copy(unique_id)
        self._ck(self.L.f2q_comm_init_rank(self.h, buf, nranks, rank))

    def comm_share(self, other: "Engine"):
        """use `other`'s communicator (same device; `other` must stay open while this engine uses it)"""
        self._ck(self.L.f2q_comm_share(self.h, other.h))

    def allreduce_counts(self):
        """sum [counts | stats] over all ranks in place (stream-ordered); then end() / end_async() as usual"""
        allreduce_counts([self])

    def ec_merge(self):
        """Extract+Count: every rank's key table becomes the merged table of all ranks (call after end())"""
        ec_merge([self])

    def result_device(self):
        p, n = C.c_void_p(), C.c_uint64()
        self._ck(self.L.f2q_result_device(self.h, C.byref(p), C.byref(n)))
        return p.value, n.value

    def ec_items(self):
        """Extract+Count: dict key(bytes) -> count (call after end())"""
        n, nb = C.c_uint64(), C.c_uint64()
        self._ck(self.L.f2q_ec_size(self.h, C.byref(n), C.byref(nb)))
        kb = np.zeros(nb.value + 1, dtype=np.uint8)
        ko = np.zeros(n.value + 1, dtype=np.uint64)
        cnt = np.zeros(n.value + 1, dtype=np.uint64)
        self._ck(self.L.f2q_ec_drain(self.h, kb.ctypes.data, ko.ctypes.data, cnt.ctypes.data))
        raw = kb.tobytes()
        return {raw[int(ko[j]):int(ko[j + 1])]: int(cnt[j]) for j in range(n.value)}

    # -- convenience: one whole in-memory stream, optionally cut into chunks
    def run(self, data: bytes, chunk: int | None = None):
        self.begin()
        if chunk is None or chunk >= len(data):
            self.submit(data, True)
        else:
            mv = memoryview(data)
            for o in range(0, len(data), chunk):
                self.submit(mv[o:o + chunk], o + chunk >= len(data))
        return self.end()

    # -- device helpers (bench / tests)
    def device_alloc(self, nbytes: int) -> int:
        p = C.c_void_p()
        self._ck(self.L.f2q_device_alloc(self.h, C.byref(p), nbytes))
        return p.value

    def device_free(self, dptr: int):
        self._ck(self.L.f2q_device_free(self.h, C.c_void_p(dptr)))

    def d2h(self, dptr: int, nbytes: int) -> np.ndarray:
        out = np.empty(nbytes, dtype=np.uint8)
        self._ck(self.L.f2q_memcpy_d2h(self.h, out.ctypes.data, C.c_void_p(dptr), nbytes))
        return out

    def h2d(self, dptr: int, data):
        a = np.ascontiguousarray(np.frombuffer(data, dtype=np.uint8) if not isinstance(data, np.ndarray) else data)
        self._ck(self.L.f2q_memcpy_h2d(self.h, C.c_void_p(dptr), a.ctypes.data, a.size))

    def synth(self, dptr: int, guides, first_read: int, n_reads: int, reuse_guides: bool = False, **spec):
        """K0: write reads [first_read, first_read + n_reads) of the workload `spec` at dptr.  guides: list of equal-length
        byte strings (shapes 2/3: the X's then the Y's).  reuse_guides=True skips the upload (the table of the previous
        call is used) and makes the call asynchronous on the engine's stream."""
        s = make_synth_spec(len(guides), first_read, n_reads, **spec)
        if reuse_guides:
            self._ck(self.L.f2q_synth_fastq(self.h, C.byref(s), None, C.c_void_p(dptr)))
            return
        g = np.frombuffer(b"".join(guides), dtype=np.uint8)
        self._ck(self.L.f2q_synth_fastq(self.h, C.byref(s), g.ctypes.data, C.c_void_p(dptr)))

    def inflate_blocks(self, d_comp: int, blocks, d_out: int) -> int:
        """f2q_inflate_blocks: the bgzip inflate + CRC check of f2q_submit_file on len(blocks) payloads placed by the caller.
        blocks: rows (src, csize, dst, isize, crc) (uint32; device offsets into d_comp / d_out).  Returns the device error
        bits (0: every block inflated to its isize bytes with its CRC)."""
        t = np.ascontiguousarray(np.asarray(blocks, dtype=np.uint32).reshape(-1, 5))
        err = C.c_uint32(0)
        self._ck(self.L.f2q_inflate_blocks(self.h, C.c_void_p(d_comp), t.ctypes.data if t.size else None, t.shape[0],
                                           C.c_void_p(d_out), C.byref(err)))
        return int(err.value)

    @property
    def launches(self) -> int:
        return int(self.L.f2q_launch_count(self.h))

    def spec_counts(self):
        """(chunks committed by the speculative kernel, chunks parsed by the exact kernel) of the last finished sample"""
        a, b = C.c_uint64(), C.c_uint64()
        self._ck(self.L.f2q_spec_counts(self.h, C.byref(a), C.byref(b)))
        return int(a.value), int(b.value)

    def memo_counts(self):
        """(lookups, hits) of the device memo of resolved non-exact keys during the last finished sample"""
        a, b = C.c_uint64(), C.c_uint64()
        self._ck(self.L.f2q_memo_counts(self.h, C.byref(a), C.byref(b)))
        return int(a.value), int(b.value)

    def info(self, name: str):
        """f2q_get_info: which table / policy / plan the context chose.  "policy" and "table" come back as the names of
        POLICIES / TABLES, everything else as an int"""
        v = C.c_int64()
        self._ck(self.L.f2q_get_info(self.h, name.encode(), C.byref(v)))
        if name == "policy":
            return POLICIES[v.value]
        if name == "table":
            return TABLES[v.value]
        return int(v.value)

    def kernel_times(self):
        """{'tile': (ms, launches), 'resolve': ..., 'generic': ..., 'aux': ...} of the last finished sample (option time_kernels)"""
        ms, n = (C.c_double * 4)(), (C.c_uint64 * 4)()
        self._ck(self.L.f2q_kernel_times(self.h, ms, n))
        return {k: (ms[i], int(n[i])) for i, k in enumerate(("tile", "resolve", "generic", "aux"))}


def border_finder_device(seq: bytes, read: bytes, mismatch: int, start_place: int = 0, device: int = 0):
    L = load()
    pos = C.c_int32()
    rc = L.f2q_border_finder(device, seq, len(seq), read, len(read), mismatch, start_place, C.byref(pos))
    if rc:
        raise F2QError(rc, L.f2q_last_error(None).decode())
    return None if pos.value < 0 else pos.value


def byteset_mask(chars):
    m = np.zeros(4, dtype=np.uint64)
    for ch in chars:
        b = ord(ch) if isinstance(ch, str) else int(ch)
        m[b >> 6] |= np.uint64(1) << np.uint64(b & 63)
    return m


def sequence_tinder_device(cfg: Config, read: bytes, qual: bytes, i: int = 0, set_up=None, set_down=None, device: int = 0):
    L = load()
    f, s, e = C.c_int32(), C.c_int32(), C.c_int32()
    mu = byteset_mask(set_up) if set_up is not None else None
    md = byteset_mask(set_down) if set_down is not None else None
    rc = L.f2q_sequence_tinder(device, C.byref(cfg), i, read, len(read), qual, len(qual),
                               mu.ctypes.data if mu is not None else None, md.ctypes.data if md is not None else None,
                               C.byref(f), C.byref(s), C.byref(e))
    if rc:
        raise F2QError(rc, L.f2q_last_error(None).decode())
    return (s.value, e.value) if f.value else (None, None)
