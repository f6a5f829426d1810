// generic.cuh — the byte-wise device path: complete semantics of fastq_parser's per-read work
// (fast2q.py:332-393) for ANY configuration: multi-feature keys, the three delimiter modes, arbitrary library
// alphabets and key lengths, Extract+Count.  One thread per read, straight from global memory.
// The packed kernels (tile.cuh / resolve.cuh) cover the common shapes at memory speed and hand every read they
// cannot decide exactly to this code, so results never depend on which path ran.
#pragma once

#include "f2q_dev.cuh"
#include "flex_core.h"

namespace f2q {

struct ByteSet { uint64_t w[4]; };
__host__ __device__ __forceinline__ bool in_set(const ByteSet& s, uint32_t b) { return (s.w[b >> 6] >> (b & 63)) & 1ull; }

struct GenericCfg {
    DevCfg c;
    ByteSet set_ph, set_up, set_down;   // fail sets (fast2q.py:1127-1129), or explicit sets for the helper API
    FlexCfg flex;                       // the same configuration prepared for the bit-parallel path (flex_core.h), when eligible
};

// Extract+Count hash of novel keys (fast2q.py:382-387).  slot word: 0 = empty, else ((arena_off << 24) | len) + 1
struct EcTable {
    // packed table (flex.cuh): single-piece keys of <= 29 ACGT symbols, 16-byte slots {tag, count}; everything else lives in
    // the byte-arena table below.  A key is in exactly one of the two (by its content)
    unsigned long long* pk_slots;
    uint64_t pk_mask;              // capacity - 1
    unsigned long long* pk_n;      // distinct keys in the packed table
    unsigned long long* slots;
    unsigned long long* counts;
    uint64_t mask;                 // capacity - 1
    uint8_t* arena;
    unsigned long long* arena_used;
    uint64_t arena_cap;
    unsigned long long* n_keys;
};

struct Outputs {
    unsigned long long* counts;    // [n_keys] feature counts (Counter mode)
    unsigned long long* stats;     // [5]
    uint32_t* error;
};

// The same three blocks in GLOBAL memory, for everything that is not inlined into a kernel's hot loop (g_process_read,
// slow_record, the in-place resolver).  Those take references; a reference to a by-value kernel parameter would make the
// compiler keep a copy of the whole parameter block in local memory and read even hot-path fields from there.
struct SlowArgs {
    LibTables T;
    EcTable E;
    Outputs O;
};

struct Piece { uint32_t off, len; };

// ---- binary_subtract / border_finder (fast2q.py:601-658), byte-wise ---------------------------
__device__ __forceinline__ bool g_within(const uint8_t* a, const uint8_t* b, int n, int mismatch) {
    int miss = 0;
    for (int i = 0; i < n; i++) {
        if (a[i] != b[i]) miss++;
        if (miss > mismatch) return false;
    }
    return true;
}

__device__ __noinline__ int g_border_finder(const uint8_t* seq, int s, const uint8_t* read, int r, int mismatch, int start_place) {
    if (start_place >= 0 && s >= 1) {
        // the ordinary call: only positions with the whole search sequence inside the read can be returned (a shorter tail
        // slice is compared but then cut off by fall_over).  Written for a warp: every position costs the same s byte
        // compares (no data-dependent inner exit), so the lanes of a warp walk their reads in lockstep and only leave at
        // their own first match — the byte-wise early-exit form ran at 2.4 active lanes per instruction.
        const int last = r - s;
        for (int p = start_place; p <= last; p++) {
            int miss = 0;
            #pragma unroll 4
            for (int i = 0; i < s; i++) miss += (seq[i] != read[p + i]) ? 1 : 0;
            if (miss <= mismatch) return p;
        }
        return -1;
    }
    int fall_over = r - s;
    int lo, hi;
    py_slice(r, start_place, r, lo, hi);
    int iters = hi - lo;
    for (int i = 0; i < iters; i++) {
        int a, b;
        py_slice(r, start_place + i, s + start_place + i, a, b);
        int n = (b - a) < s ? (b - a) : s;
        bool ok = g_within(seq, read + a, n, mismatch);
        if (i + start_place > fall_over) return -1;
        if (ok) return i + start_place;
    }
    return -1;
}

__device__ __forceinline__ bool g_slice_fails(const uint8_t* q, int n, int a, int b, const ByteSet& s) {
    int lo, hi;
    py_slice(n, a, b, lo, hi);
    bool fails = false;                                               // (no early exit: the slice length is the same for every lane)
    for (int i = lo; i < hi; i++) fails |= in_set(s, q[i]);
    return fails;
}

// sequence_tinder (fast2q.py:215-285)
__device__ inline bool g_sequence_tinder(const GenericCfg& G, int i, const uint8_t* R, int r, const uint8_t* Q, int q,
                                         int& start_out, int& end_out) {
    const DevCfg& c = G.c;
    if (c.has_up && c.has_down) {
        int ul = c.up_len[i], dl = c.down_len[i];
        int start = g_border_finder(c.up[i], ul, R, r, c.miss_up, 0);
        if (start >= 0) {
            int end = g_border_finder(c.down[i], dl, R, r, c.miss_down, start + ul);
            if (end >= 0) {
                bool bad = g_slice_fails(Q, q, start, start + ul, G.set_up) | g_slice_fails(Q, q, end, end + dl, G.set_down);
                if (!bad) { start_out = start + ul; end_out = end; return true; }
            }
        }
    } else if (c.has_up) {
        int ul = c.up_len[i];
        int start = g_border_finder(c.up[i], ul, R, r, c.miss_up, 0);
        if (start >= 0 && !g_slice_fails(Q, q, start, start + ul, G.set_up)) {
            start_out = start + ul; end_out = start + ul + c.length; return true;
        }
    } else if (c.has_down) {
        int dl = c.down_len[i];
        int end = g_border_finder(c.down[i], dl, R, r, c.miss_down, 0);
        if (end >= 0 && !g_slice_fails(Q, q, end, end + dl, G.set_down)) {
            start_out = end - c.length; end_out = end; return true;
        }
    }
    return false;
}

// key pieces of one read (fast2q.py:332-363); returns the number of pieces, -1 when every iteration was flagged
__device__ inline int g_build_pieces(const GenericCfg& G, const uint8_t* R, int r, const uint8_t* Q, int q, Piece* pc) {
    const DevCfg& c = G.c;
    const bool fixed = !(c.has_up || c.has_down);
    int np = 0;
    bool any = false;
    for (int i = 0; i < c.n_iter; i++) {
        int start, end;
        if (fixed) { start = c.starts[i]; end = c.starts[i] + c.length; }
        else {
            if (!g_sequence_tinder(G, i, R, r, Q, q, start, end)) continue;
            if (end < start) continue;                                   // fast2q.py:343-345
        }
        int slo, shi;
        py_slice(r, start, end, slo, shi);
        if (g_slice_fails(Q, q, start, end, G.set_ph)) continue;          // fast2q.py:357-360
        pc[np].off = (uint32_t)slo; pc[np].len = (uint32_t)(shi - slo);
        np++; any = true;
    }
    return any ? np : -1;
}

// visit the key's symbols in order (upper-cased pieces joined by ':'); f returns false to stop
template <class F>
__device__ __forceinline__ void g_for_each_symbol(const uint8_t* R, const Piece* pc, int np, F f) {
    for (int p = 0; p < np; p++) {
        if (p && !f((uint32_t)':')) return;
        const uint8_t* s = R + pc[p].off;
        for (uint32_t k = 0; k < pc[p].len; k++) if (!f(upper8(s[k]))) return;
    }
}

__host__ __device__ __forceinline__ uint32_t fnv_step(uint32_t h, uint32_t b) { return (h ^ b) * 16777619u; }
constexpr uint32_t FNV_INIT = 2166136261u;
__host__ __device__ __forceinline__ uint32_t fnv_final(uint32_t h) { h ^= h >> 15; h *= 0x2C1B3C6Du; h ^= h >> 12; return h; }

// byte-level pigeonhole seeds (see LibTables::gseed_*): two 32-bit FNV streams make the 64-bit tag of one key segment
constexpr uint32_t GSEED_MAX_PARTS = 8;
__host__ __device__ __forceinline__ void gseed_init(uint32_t len, uint32_t seg, uint32_t& a, uint32_t& b) {
    a = fnv_step(fnv_step(FNV_INIT, len & 0xFFu), seg + 1u);
    b = (0x9E3779B9u ^ (len * 0x85EBCA6Bu)) + seg * 0xC2B2AE35u;
}
__host__ __device__ __forceinline__ void gseed_step(uint32_t sym, uint32_t& a, uint32_t& b) {
    a = fnv_step(a, sym);
    b = (b ^ (sym + 0x7Fu)) * 0x01000193u + 0x9E3779B9u;
}
__host__ __device__ __forceinline__ uint64_t gseed_tag(uint32_t a, uint32_t b) {
    return (1ull << 63) | ((uint64_t)fnv_final(b) << 32) | fnv_final(a);
}
__host__ __device__ __forceinline__ uint32_t gseed_hash(uint64_t tag) {
    uint64_t h = tag * 0x9E3779B97F4A7C15ull;
    return (uint32_t)(h >> 32) ^ (uint32_t)h;
}

__device__ __forceinline__ bool g_key_equals(const uint8_t* R, const Piece* pc, int np, const uint8_t* lib, uint32_t len) {
    uint32_t i = 0; bool eq = true;
    g_for_each_symbol(R, pc, np, [&](uint32_t s) { eq = (lib[i++] == s); return eq; });
    return eq && i == len;
}

// Counter mode for one read key: exact lookup, then min-distance-unique resolution (fast2q.py:365-380, 692-750)
__device__ inline void g_count_key(const GenericCfg& G, const LibTables& T, const Outputs& O, const uint8_t* R, const Piece* pc,
                                   int np, unsigned long long* st /*local stats[5]*/) {
    uint32_t klen = np ? (uint32_t)(np - 1) : 0, h = FNV_INIT;
    for (int p = 0; p < np; p++) klen += pc[p].len;
    g_for_each_symbol(R, pc, np, [&](uint32_t s) { h = fnv_step(h, s); return true; });
    h = fnv_final(h);
    for (uint32_t i = h & T.ghash_mask;; i = (i + 1) & T.ghash_mask) {
        uint32_t e = __ldg(T.ghash + i);
        if (e == 0) break;
        uint64_t o0 = __ldg(T.key_off + (e - 1)), o1 = __ldg(T.key_off + e);
        if ((uint32_t)(o1 - o0) == klen && g_key_equals(R, pc, np, T.key_bytes + o0, klen)) {
            atomicAdd(O.counts + (e - 1), 1ull);
            st[F2Q_STAT_PERFECT]++;
            return;
        }
    }
    const int m = G.c.miss;
    if (m <= 0) { st[F2Q_STAT_NON_ALIGNED]++; return; }
    int best_d = m + 1; uint32_t best_n = 0, best_g = 0;
    const uint32_t parts = T.gseed_parts;
    if (parts && klen >= parts) {
        // pigeonhole: an entry within m mismatches agrees exactly with the key on one of m+1 segments.  Tags of the key's
        // segments in one pass, then per segment: bucket -> candidates -> full distance.  An entry reached through several
        // segments is counted at the first segment it agrees on.  Same answer as the scan below.
        uint32_t ha[GSEED_MAX_PARTS], hb[GSEED_MAX_PARTS], bnd[GSEED_MAX_PARTS + 1];
        for (uint32_t sg = 0; sg <= parts; sg++) bnd[sg] = sg * klen / parts;
        for (uint32_t sg = 0; sg < parts; sg++) gseed_init(klen, sg, ha[sg], hb[sg]);
        { uint32_t i = 0, cs = 0;
          g_for_each_symbol(R, pc, np, [&](uint32_t sym) { while (i >= bnd[cs + 1]) cs++; gseed_step(sym, ha[cs], hb[cs]); i++; return true; }); }
        for (uint32_t sg = 0; sg < parts; sg++) {
            const uint64_t tag = gseed_tag(ha[sg], hb[sg]);
            uint32_t start = 0, count = 0;
            for (uint32_t hh = gseed_hash(tag) & T.gseed_mask;; hh = (hh + 1) & T.gseed_mask) {
                const uint4 raw = __ldg(T.gseed_slots + hh);
                const uint64_t t = ((uint64_t)raw.y << 32) | raw.x;
                if (t == 0) break;
                if (t == tag) { start = raw.z; count = raw.w; break; }
            }
            for (uint32_t c = 0; c < count; c++) {
                const uint32_t g = __ldg(T.gseed_items + start + c);
                const uint64_t o0 = __ldg(T.key_off + g), o1 = __ldg(T.key_off + g + 1);
                if ((uint32_t)(o1 - o0) != klen) continue;
                const uint8_t* lib = T.key_bytes + o0;
                int d = 0; uint32_t i = 0, cs = 0, segbad = 0;
                g_for_each_symbol(R, pc, np, [&](uint32_t sym) {
                    while (i >= bnd[cs + 1]) cs++;
                    const uint32_t ne = lib[i++] != sym;
                    d += (int)ne; segbad |= ne << cs;
                    return d <= m;
                });
                if (d > m) continue;
                const uint32_t agree = ~segbad & ((1u << parts) - 1u);
                if (agree == 0 || (uint32_t)__ffs((int)agree) - 1u != sg) continue;      // a hash collision, or counted at an earlier segment
                if (d < best_d) { best_d = d; best_n = 1; best_g = g; }
                else if (d == best_d) best_n++;
            }
        }
    } else
    for (uint32_t g = 0; g < T.n_keys; g++) {                              // features_all_vs_all, fast2q.py:660-690
        uint64_t o0 = __ldg(T.key_off + g), o1 = __ldg(T.key_off + g + 1);
        if ((uint32_t)(o1 - o0) != klen) continue;
        const uint8_t* lib = T.key_bytes + o0;
        int d = 0; uint32_t i = 0;
        g_for_each_symbol(R, pc, np, [&](uint32_t s) { d += (lib[i++] != s); return d <= best_d; });
        if (d < best_d) { best_d = d; best_n = 1; best_g = g; }
        else if (d == best_d && d <= m) best_n++;
    }
    if (best_d <= m && best_n == 1) { atomicAdd(O.counts + best_g, 1ull); st[F2Q_STAT_IMPERFECT]++; }
    else st[F2Q_STAT_NON_ALIGNED]++;
}

// Extract+Count insert-or-increment of one key (fast2q.py:383-387)
__device__ __forceinline__ void ec_pk_insert(const EcTable& E, const Outputs& O, unsigned long long tag, unsigned long long add);   // flex.cuh

__device__ inline void g_ec_insert(const EcTable& E, const Outputs& O, const uint8_t* R, const Piece* pc, int np) {
    if (np == 1 && pc[0].len <= 29u && E.pk_slots) {
        // a single piece of pure ACGT that fits the packed table must go THERE (the streaming kernel puts it there too)
        uint64_t codes = 0; bool pure = true;
        const uint8_t* s = R + pc[0].off;
        for (uint32_t k = 0; k < pc[0].len; k++) { uint32_t code; pure = pure && base_code(s[k], code); codes |= (uint64_t)code << (2u * k); }
        if (pure) { ec_pk_insert(E, O, ((codes << 6) | pc[0].len) + 1ull, 1ull); return; }
    }
    uint32_t klen = np ? (uint32_t)(np - 1) : 0, h = FNV_INIT;
    for (int p = 0; p < np; p++) klen += pc[p].len;
    g_for_each_symbol(R, pc, np, [&](uint32_t s) { h = fnv_step(h, s); return true; });
    uint64_t i = (uint64_t)fnv_final(h) * 0x9E3779B1ull;       // spread 32-bit hash over large tables
    i = (i ^ (i >> 29)) & E.mask;
    unsigned long long mine = 0;
    for (uint64_t probes = 0; probes <= E.mask; probes++, i = (i + 1) & E.mask) {
        unsigned long long s = *(volatile unsigned long long*)(E.slots + i);
        if (s == 0) {
            if (!mine) {
                unsigned long long off = atomicAdd(E.arena_used, (unsigned long long)klen);
                if (off + klen > E.arena_cap || klen >= (1u << 24)) { atomicOr(O.error, ERR_EC_FULL); return; }
                uint8_t* dst = E.arena + off;
                uint32_t k = 0;
                g_for_each_symbol(R, pc, np, [&](uint32_t sym) { dst[k++] = (uint8_t)sym; return true; });
                __threadfence();
                mine = ((off << 24) | klen) + 1ull;
            }
            s = atomicCAS(E.slots + i, 0ull, mine);
            if (s == 0) { atomicAdd(E.n_keys, 1ull); atomicAdd(E.counts + i, 1ull); return; }
        }
        __threadfence();
        uint32_t slen = (uint32_t)((s - 1) & 0xFFFFFFull);
        if (slen == klen) {
            const uint8_t* a = E.arena + ((s - 1) >> 24);
            uint32_t k = 0; bool eq = true;
            g_for_each_symbol(R, pc, np, [&](uint32_t sym) { eq = (__ldcg(a + k) == (uint8_t)sym); k++; return eq; });
            if (eq) { atomicAdd(E.counts + i, 1ull); return; }
        }
    }
    atomicOr(O.error, ERR_EC_FULL);
}

// everything for one read; R/Q are the rstripped sequence and quality lines.  st = local stats accumulators
__device__ __noinline__ void g_process_read(const GenericCfg& G, const LibTables& T, const EcTable& E, const Outputs& O,
                                            const uint8_t* R, int r, const uint8_t* Q, int q, unsigned long long* st) {
    Piece pc[F2Q_MAX_ITER];
    int np = g_build_pieces(G, R, r, Q, q, pc);
    if (np < 0) { st[F2Q_STAT_QUALITY_FAILED]++; return; }
    if (G.c.mode == F2Q_MODE_COUNT) g_count_key(G, T, O, R, pc, np, st);
    else { g_ec_insert(E, O, R, pc, np); st[F2Q_STAT_PERFECT]++; }
}

__device__ __forceinline__ int g_rstrip(const uint8_t* p, int n) {
    while (n > 0 && is_py_space(p[n - 1])) n--;
    return n;
}

// drains the generic read queue: one thread per entry (and one thread of the launch adds the fill to S->generic_reads)
__global__ void __launch_bounds__(128) k_generic_queue(const GenericCfg* __restrict__ Gp, const SlowArgs* __restrict__ X,
                                                       const GEntry* q, DevState* S) {
    __shared__ GenericCfg G;
    for (uint32_t i = threadIdx.x; i < sizeof(GenericCfg) / 4; i += blockDim.x)
        reinterpret_cast<uint32_t*>(&G)[i] = reinterpret_cast<const uint32_t*>(Gp)[i];
    __syncthreads();
    unsigned long long st[F2Q_N_STATS] = {0, 0, 0, 0, 0};
    uint32_t n = S->g_count < S->g_cap ? S->g_count : S->g_cap;
    if (blockIdx.x == 0 && threadIdx.x == 0) S->generic_reads += n;
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        GEntry e = q[i];
        const uint8_t* R = reinterpret_cast<const uint8_t*>(e.seq_addr);
        const uint8_t* Q = reinterpret_cast<const uint8_t*>(e.qual_addr);
        g_process_read(G, X->T, X->E, X->O, R, g_rstrip(R, (int)e.seq_len), Q, g_rstrip(Q, (int)e.qual_len), st);
    }
    for (int k = 1; k < F2Q_N_STATS; k++) if (st[k]) atomicAdd(X->O.stats + k, st[k]);
}

// ---- single-read helpers behind f2q_border_finder / f2q_sequence_tinder ------------------------
__global__ void k_border_finder(const uint8_t* seq, int s, const uint8_t* read, int r, int mismatch, int start_place, int* out) {
    if (threadIdx.x == 0 && blockIdx.x == 0) *out = g_border_finder(seq, s, read, r, mismatch, start_place);
}

__global__ void k_sequence_tinder(GenericCfg G, int i, const uint8_t* R, int r, const uint8_t* Q, int q, int* out /*found,start,end*/) {
    if (threadIdx.x == 0 && blockIdx.x == 0) {
        int s = 0, e = 0;
        bool f = g_sequence_tinder(G, i, R, r, Q, q, s, e);
        out[0] = f; out[1] = s; out[2] = e;
    }
}

}  // namespace f2q
