// f2q_dev.cuh — shared device-side definitions of libf2q (sm_100a).
//
// Everything here is integer / byte work; the path is HBM-bound (one pass over the FASTQ bytes), so there is
// no tensor-core code.  Reference semantics cited as fast2q.py:<lines> (2FAST2Q v2.8.1).
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/f2q.h"

namespace f2q {

// ------------------------------------------------------------------------------------------------
// geometry of the tile kernel: see TileGeom<CH, NT> in tile.cuh (NT owned rows of 16*CH bytes + read-ahead rows)
// ------------------------------------------------------------------------------------------------
// device error bits (sticky, reported by f2q_end_sample as F2Q_EINTERNAL / F2Q_ETOOLONG)
constexpr uint32_t ERR_LOOKBACK_TIMEOUT = 1u;
constexpr uint32_t ERR_RECORD_TOO_LONG = 2u;
constexpr uint32_t ERR_QUEUE = 4u;
constexpr uint32_t ERR_EC_FULL = 8u;
constexpr uint32_t ERR_INFLATE = 16u;         // a bgzip block is not valid DEFLATE data of the promised size and CRC-32

// ------------------------------------------------------------------------------------------------
// parameters
// ------------------------------------------------------------------------------------------------
struct DevCfg {
    int32_t mode, miss, length, n_iter, has_up, has_down, miss_up, miss_down;
    int32_t fmax_ph, fmax_up, fmax_down;   // largest failing quality byte (0 = empty fail set): fail iff 33 <= b <= fmax
    int32_t starts[F2Q_MAX_ITER];
    int32_t up_len[F2Q_MAX_ITER], down_len[F2Q_MAX_ITER];
    uint8_t up[F2Q_MAX_ITER][F2Q_MAX_DELIM], down[F2Q_MAX_ITER][F2Q_MAX_DELIM];
};

// one slot of the packed-key hash table: 2-bit packed bases (<= 32), key length, feature index
struct __align__(16) FastSlot {
    uint64_t key;
    uint32_t len;
    uint32_t idx;      // 0xFFFFFFFF = empty
};
constexpr uint32_t SLOT_EMPTY = 0xFFFFFFFFu;

// library tables on the device (replace binary_converter, fast2q.py:188-213)
struct LibTables {
    // packed (ACGT-only, <= 32 symbols, single piece) keys
    const FastSlot* slots;
    uint32_t slot_mask;        // capacity - 1 (power of two)
    uint32_t n_fast;
    // compact 8-byte form of the same table for the fused tile kernel, present when every packed key has ONE length c_len and
    // 2*c_len + bits(index) <= 64:  slot = packed key | feature index << 2*c_len;  ~0 = empty.  Load factor <= 1/4, so a probe
    // sequence is short for every lane of a warp and small libraries stay L1-resident (2 000 guides: 64 KB)
    const uint64_t* cslots;
    uint32_t c_mask;           // capacity - 1
    uint32_t c_len;
    uint32_t c_keybits;        // 2 * c_len
    // the same slots as a two-choice cuckoo table (built when the compact form exists): table 0 at [0, ck_mask], table 1 behind it;
    // a lookup is exactly two independent loads, no probe loop, so all lanes of a warp finish together (spec.cuh)
    const uint64_t* cuckoo;
    uint32_t ck_mask;          // slots per table - 1
    uint32_t ck_shift;         // 32 - log2(slots per table)
    uint32_t ck_hshift;        // bit of the slot's high word where the value starts = max(2 * c_len, 32) - 32
    uint32_t ck_mul[4];        // odd multipliers of the two multiplicative hashes (chosen by the host until the build succeeds)
    uint32_t ck_neighbours;    // 1: the table also holds every Hamming-1 neighbour of every key (value bit 0 = imperfect, CK_AMBIG = tie)
    const uint64_t* fast_keys; // n_fast packed keys grouped by length (for the tile-scan resolver)
    const uint32_t* fast_lens;
    const uint32_t* fast_idx;
    // every key as bytes (generic path)
    const uint8_t* key_bytes;
    const uint64_t* key_off;   // n_keys + 1
    uint32_t n_keys;
    const uint32_t* ghash;     // byte-hash table: key index + 1, 0 = empty
    uint32_t ghash_mask;
    uint32_t n_generic;        // keys that are NOT in the packed table
    uint64_t generic_len_mask; // bit L set: some non-packed key has length L (L < 64); bit 63: some length >= 63
    // pigeonhole seed index over the packed keys (resolver 2)
    const uint4* seed_slots;   // {tag lo, tag hi, start, count}: hash of (len, segment, value) -> range in seed_recs; tag 0 = empty
    uint32_t seed_mask;
    const uint4* seed_recs;    // {packed key lo, hi, feature index, 0} of every (key, segment), grouped by seed slot
    uint32_t seed_parts;       // P: segments a key is cut into (>= miss + 1)
    uint32_t seed_ncombo;      // C(P, miss) seeds per key: every choice of P - miss segments (a key within `miss` mismatches agrees on one of them)
    uint8_t seed_combo[32];    // bit s of entry c: segment s belongs to seed c
    // the same idea over the raw key BYTES of every library entry (generic path: multi-feature 'X:Y' keys, odd alphabets, > 32 symbols)
    const uint4* gseed_slots;  // {tag lo, tag hi, start, count}; tag = 64-bit hash of (key length, segment, segment bytes), 0 = empty
    uint32_t gseed_mask;
    const uint32_t* gseed_items;   // key indices
    uint32_t gseed_parts;      // miss + 1 when the index exists (1 <= miss <= 7), else 0
    // flex table (flex.cuh): EVERY key as <= 2 pieces of <= 32 ACGT symbols, <= 40 symbols in all; nullptr when some key is not
    const uint4* fx_slots;     // {lo.x, lo.y, hi | signature << 16, feature index}; index 0xFFFFFFFF = empty
    uint32_t fx_mask;
    const uint16_t* fx_len_sig;    // [FX_MAX_BYTELEN + 1] by key BYTE length: 0 no key | the one signature | FX_SIG_MIXED
    const uint4* fxs_slots;    // seed index over the flex keys: {tag lo, tag hi, start, count}
    uint32_t fxs_mask;
    const uint4* fxs_recs;     // {lo.x, lo.y, hi, feature index} grouped by seed slot
    uint32_t fxs_parts;        // miss + 1
    // memo of resolved non-exact keys (the device analogue of passed_reads / failed_reads, fast2q.py:724-731, 741, 748):
    // direct-mapped, lossy, 16-byte entries {key lo, key hi, shape, result + 1}; lives as long as the library (across chunks
    // AND samples of the context).  A key's result is a function of key, library and m, so a hit never changes a count
    uint4* memo;
    uint32_t memo_mask;        // entries - 1; memo == nullptr: off
};

// entry of the deferred non-exact key queue (filled by the tile kernel, drained by the resolver kernel)
struct __align__(16) QEntry {
    uint64_t key;      // 2-bit packed, bad positions hold 0
    uint32_t bad;      // bit p set: symbol p is not A/C/G/T
    uint32_t len;
};

// a read the packed path cannot decide (record longer than the tile halo, odd key shape, non-packed library keys):
// location of its sequence and quality lines (absolute device addresses), handled by the generic kernel
struct __align__(8) GEntry {
    uint64_t seq_addr;     // device address of the first byte of the sequence line
    uint64_t qual_addr;
    uint32_t seq_len;
    uint32_t qual_len;
};

// per-sample, per-launch device state
struct DevState {
    // carried partial record
    uint32_t tail_len;
    uint32_t tail_nl;
    // current launch
    uint64_t beg, end;             // byte range of the buffer the tile kernel parses; beg is a record start
    uint32_t is_last;              // the range ends at end-of-stream
    uint32_t stitch_len;           // bytes of the stitched record in the carry buffer (0 = none)
    uint32_t stitch_eof;           // the stitched bytes end the stream
    uint32_t appended;             // the whole chunk was appended to the carry buffer (nothing else to parse)
    unsigned long long last_rec_end;   // atomicMax: offset just behind the last complete record
    uint32_t nl_total;             // newlines in [beg, end) (mod 2^30)
    uint32_t ticket;
    uint32_t error;
    uint32_t q_count, q_cap;       // (unused; the non-exact key queue is segmented per CTA, see TileParams)
    uint32_t g_count, g_cap;       // generic read queue
    uint32_t spec_fail;            // speculative kernel (spec.cuh): some range could not guess its line phase / met an odd tile
    uint32_t spec_ok;              // k_spec_verify: every speculated phase was right, the scratch results are committed
    uint32_t spec_off;             // sticky per sample: a speculation failed, later chunks go straight to the exact kernel
    uint32_t spec_commits, spec_fallbacks;   // chunks of this sample whose speculation held / that the exact kernel parsed
    unsigned long long memo_lookups, memo_hits;
    unsigned long long generic_reads;   // reads the generic read queue took this sample (k_generic_queue, f2q_get_info)
    unsigned long long head_len;   // k_shard_head: bytes before the guessed first record of a shard (its head)
    uint32_t head_nl, head_ok;     // ... newlines in the head (1-4); 1 when exactly one candidate start was accepted
    unsigned long long dbg[8];     // diagnostics (F2Q_DEBUG=1): failed mbarrier tries per wait site, look-back rounds / spins
};

// ------------------------------------------------------------------------------------------------
// small helpers
// ------------------------------------------------------------------------------------------------
__host__ __device__ __forceinline__ uint32_t mix32(uint64_t key, uint32_t len) {
    uint64_t h = (key ^ (0x9E3779B97F4A7C15ull * (uint64_t)(len + 1))) * 0xBF58476D1CE4E5B9ull;
    h ^= h >> 29;
    h *= 0x94D049BB133111EBull;
    return (uint32_t)(h >> 32);
}

// hash of a packed key for the compact table (32-bit multiplies only; the table mask takes the HIGH bits' mix)
__host__ __device__ __forceinline__ uint32_t mix_compact(uint32_t klo, uint32_t khi) {
    uint32_t x = klo ^ (khi * 0x9E3779B1u);
    x *= 0x85EBCA6Bu;
    x ^= x >> 15;
    x *= 0xC2B2AE35u;
    x ^= x >> 13;
    return x;
}

// Python slice bounds seq[a:b] for a sequence of length n (fast2q.py:354-355)
__host__ __device__ __forceinline__ void py_slice(int n, int a, int b, int& lo, int& hi) {
    if (a < 0) { a += n; if (a < 0) a = 0; } else if (a > n) a = n;
    if (b < 0) { b += n; if (b < 0) b = 0; } else if (b > n) b = n;
    if (b < a) b = a;
    lo = a; hi = b;
}

// bytes.rstrip() whitespace set: b" \t\n\r\x0b\x0c" (fast2q.py:326)
__host__ __device__ __forceinline__ bool is_py_space(uint32_t c) { return c == 32u || (c - 9u) <= 4u; }

__host__ __device__ __forceinline__ uint32_t upper8(uint32_t c) { return (c - 97u) <= 25u ? c - 32u : c; }

// 2-bit code of an (upper- or lower-case) base: A=0 C=1 T=2 G=3  ((c >> 1) & 3); valid iff upper8(c) in ACGT
__host__ __device__ __forceinline__ bool base_code(uint32_t c, uint32_t& code) {
    uint32_t u = c & 0xDFu;
    code = (c >> 1) & 3u;
    return u == 'A' || u == 'C' || u == 'G' || u == 'T';
}

#ifdef __CUDACC__
// 16-byte single-copy-atomic accesses (PTX .b128 with memory-model semantics; SASS LDG/STG.E.128.STRONG.GPU): a memo entry is
// read and written as a whole, whoever races
__device__ __forceinline__ void st_b128(uint4* p, uint4 v) {
    asm volatile("{\n\t.reg .b128 q;\n\tmov.b128 q, {%1, %2};\n\tst.relaxed.gpu.global.b128 [%0], q;\n\t}"
                 :: "l"(p), "l"(((uint64_t)v.y << 32) | v.x), "l"(((uint64_t)v.w << 32) | v.z) : "memory");
}
__device__ __forceinline__ uint4 ld_b128(const uint4* p) {
    uint64_t lo, hi;
    asm volatile("{\n\t.reg .b128 q;\n\tld.relaxed.gpu.global.b128 q, [%2];\n\tmov.b128 {%0, %1}, q;\n\t}" : "=l"(lo), "=l"(hi) : "l"(p) : "memory");
    return make_uint4((uint32_t)lo, (uint32_t)(lo >> 32), (uint32_t)hi, (uint32_t)(hi >> 32));
}
__device__ __forceinline__ uint32_t memo_slot(const LibTables& T, uint32_t x, uint32_t y, uint32_t z) {
    uint64_t h = ((((uint64_t)y << 32) | x) ^ ((uint64_t)z * 0x9E3779B97F4A7C15ull)) * 0xD6E8FEB86659FD93ull;
    h ^= h >> 32;
    return (uint32_t)h & T.memo_mask;
}
// stored result + 1 of the key (x, y, z), or 0 when the memo does not hold it
__device__ __forceinline__ uint32_t memo_lookup(const LibTables& T, uint32_t x, uint32_t y, uint32_t z) {
    const uint4 e = ld_b128(T.memo + memo_slot(T, x, y, z));
    return (e.x == x && e.y == y && e.z == z) ? e.w : 0u;
}
__device__ __forceinline__ void memo_store(const LibTables& T, uint32_t x, uint32_t y, uint32_t z, uint32_t result_plus_1) {
    st_b128(T.memo + memo_slot(T, x, y, z), make_uint4(x, y, z, result_plus_1));
}

// swizzled address of the byte at tile offset o (see the tile geometry above)
__device__ __forceinline__ uint32_t swz(uint32_t o) { return o ^ ((o >> 3) & 0x70u); }

// exact per-byte equality flags (0x80 in every byte of w that equals the byte replicated in c4); 3 instructions
__device__ __forceinline__ uint32_t eq_bytes(uint32_t w, uint32_t c4) {
    uint32_t x = (w ^ c4);
    uint32_t t = (x & 0x7F7F7F7Fu) + 0x7F7F7F7Fu;
    return ~(t | x) & 0x80808080u;
}

// 8-byte read-only load that stays where it is written (the compiler may not sink it towards its use): issued early on purpose
__device__ __forceinline__ uint2 ldg_u2_here(const uint2* p) {
    uint2 r;
    asm volatile("ld.global.nc.v2.u32 {%0,%1}, [%2];" : "=r"(r.x), "=r"(r.y) : "l"(p));
    return r;
}

// streaming 16-byte global load (read once, do not keep in L1)
__device__ __forceinline__ uint4 ldg_stream(const uint4* p) {
    uint4 r;
    asm volatile("ld.global.nc.L1::no_allocate.v4.u32 {%0,%1,%2,%3}, [%4];"
                 : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w) : "l"(p));
    return r;
}

__device__ __forceinline__ uint32_t ld_volatile_u32(const uint32_t* p) {
    uint32_t v;
    asm volatile("ld.volatile.global.u32 %0, [%1];" : "=r"(v) : "l"(p));
    return v;
}
__device__ __forceinline__ void st_volatile_u32(uint32_t* p, uint32_t v) {
    asm volatile("st.volatile.global.u32 [%0], %1;" :: "l"(p), "r"(v) : "memory");
}

// probe the packed-key table; returns feature index or SLOT_EMPTY
__device__ __forceinline__ uint32_t fast_lookup(const LibTables& T, uint64_t key, uint32_t len) {
    uint32_t h = mix32(key, len) & T.slot_mask;
    #pragma unroll 1
    for (;;) {
        uint4 raw = __ldg(reinterpret_cast<const uint4*>(T.slots + h));
        uint64_t k = ((uint64_t)raw.y << 32) | raw.x;
        if (raw.w == SLOT_EMPTY) return SLOT_EMPTY;
        if (k == key && raw.z == len) return raw.w;
        h = (h + 1) & T.slot_mask;
    }
}

// probe the compact table (all keys have T.c_len symbols; the caller checked len == T.c_len); feature index or SLOT_EMPTY
__device__ __forceinline__ uint32_t compact_lookup(const LibTables& T, uint32_t klo, uint32_t khi) {
    uint32_t h = mix_compact(klo, khi) & T.c_mask;
    const uint64_t key = ((uint64_t)khi << 32) | klo;
    const uint64_t keymask = T.c_keybits >= 64 ? ~0ull : ((1ull << T.c_keybits) - 1ull);
    #pragma unroll 1
    for (;;) {
        const uint2 raw = __ldg(reinterpret_cast<const uint2*>(T.cslots) + h);
        const uint64_t sl = ((uint64_t)raw.y << 32) | raw.x;
        if ((sl & keymask) == key && sl != ~0ull) return (uint32_t)(sl >> T.c_keybits);
        if (sl == ~0ull) return SLOT_EMPTY;
        h = (h + 1) & T.c_mask;
    }
}
#endif  // __CUDACC__

// the two slots a packed key can live in (host and device must agree).  Multiplicative hashing keeps the TOP bits of
// the products: every key bit reaches them (the table also holds keys that differ from each other in one 2-bit symbol
// only).  Multipliers by value: as kernel parameters they stay constant-bank operands of the multiplies.
__host__ __device__ __forceinline__ void cuckoo_slots(uint32_t m0, uint32_t m1, uint32_t m2, uint32_t m3, uint32_t shift, uint32_t klo, uint32_t khi,
                                                      uint32_t& h1, uint32_t& h2) {
    h1 = (klo * m0 + khi * m1) >> shift;
    h2 = (((klo * m2) ^ (khi * m3)) >> shift) + (1u << (32u - shift));
}

#ifdef __CUDACC__
// two-choice lookup (caller checked len == T.c_len).  Slot layout: low word = key bits 0..31, high word = key bits 32..
// below bit ck_hshift and the VALUE above it (feature index << 1 | imperfect; all ones = empty slot, all ones - 1 = the
// tie marker), so that matching and decoding are 32-bit operations.  Returns the value or CK_NONE.
constexpr uint32_t CK_NONE = 0xFFFFFFFFu;
__host__ __device__ __forceinline__ uint32_t cuckoo_valmax(uint32_t hshift) { return 0xFFFFFFFFu >> hshift; }
__device__ __forceinline__ uint32_t cuckoo_ambig(const LibTables& T) { return cuckoo_valmax(T.ck_hshift) - 1u; }
__device__ __forceinline__ uint32_t cuckoo_match(const LibTables& T, uint2 ra, uint2 rb, uint32_t klo, uint32_t khi) {
    const uint32_t hs = T.ck_hshift, himask = hs ? (0xFFFFFFFFu >> (32u - hs)) : 0u, empty = cuckoo_valmax(hs);
    const uint32_t va = ra.y >> hs, vb = rb.y >> hs;
    uint32_t v = CK_NONE;
    if (ra.x == klo && (ra.y & himask) == khi && va != empty) v = va;
    if (rb.x == klo && (rb.y & himask) == khi && vb != empty) v = vb;
    return v;
}
#endif  // __CUDACC__

}  // namespace f2q
