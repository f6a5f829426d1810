// inflate_core.h — DEFLATE (RFC 1951) decoder for ONE raw deflate stream per thread: the payload of a BGZF block
// (bgzip writes gzip members of <= 64 KiB that carry their compressed size in an extra field and their uncompressed size in
// their trailer, so the blocks of a file are independent and their output offsets are known before anything is inflated).
//
// SURVEY.md §8(f)-1 / VERDICT r1 task 9: the reference inflates with `gzip.open` on one host thread (fast2q.py:568); here a
// chunk of COMPRESSED bytes crosses PCIe (3-4x fewer bytes than the FASTQ text) and k_inflate_bgzf (stream.cuh) decodes
// thousands of blocks at once, one thread each, straight into the chunk buffer the streaming kernel parses.
//
// The decoder is the canonical-Huffman, bit-serial one (code lengths -> counts + sorted symbols; a symbol is decoded by walking
// the code lengths): small per-thread state (about 1 KB of local memory), no shared tables, and FASTQ text has short codes.
// It is a pure function compiled for the device by nvcc and for the host by g++: tests/native/hostcheck.cpp checks it
// against zlib on the CPU (stored, fixed and dynamic blocks, every compression level), the -m gpu tests against the same
// files through the kernel.  The CRC-32 check of every inflated block (k_bgzf_crc) is at the end of this file.
#pragma once

#include <stdint.h>

#include "synth_gen.h"      // F2Q_HD

namespace f2q {

constexpr int INFL_MAXBITS = 15, INFL_MAXLCODES = 286, INFL_MAXDCODES = 30, INFL_FIXLCODES = 288;

struct InflState {
    const uint8_t* in; uint32_t in_len, in_pos;
    uint64_t bitbuf; uint32_t bitcnt;
    uint8_t* out; uint32_t out_len, out_pos;
    int err;                 // sticky: 1 input exhausted, 2 bad data, 3 output overflow
};

struct InflHuff {
    uint16_t count[INFL_MAXBITS + 1];
    uint16_t symbol[INFL_FIXLCODES];
};
struct InflHuffD {
    uint16_t count[INFL_MAXBITS + 1];
    uint16_t symbol[INFL_MAXDCODES];
};

F2Q_HD void infl_refill(InflState& s) {
    while (s.bitcnt <= 56u && s.in_pos < s.in_len) { s.bitbuf |= (uint64_t)s.in[s.in_pos++] << s.bitcnt; s.bitcnt += 8u; }
}
// n <= 16 bits, LSB first
F2Q_HD uint32_t infl_bits(InflState& s, uint32_t n) {
    if (s.bitcnt < n) { infl_refill(s); if (s.bitcnt < n) { s.err = s.err ? s.err : 1; return 0; } }
    const uint32_t v = (uint32_t)(s.bitbuf & ((1ull << n) - 1ull));
    s.bitbuf >>= n; s.bitcnt -= n;
    return v;
}

// one symbol of a canonical code (count[len] codes of each length, symbols sorted by code)
template <class H>
F2Q_HD int infl_decode(InflState& s, const H& h) {
    if (s.bitcnt < (uint32_t)INFL_MAXBITS) infl_refill(s);
    int code = 0, first = 0, index = 0;
    uint64_t buf = s.bitbuf;
    const uint32_t have = s.bitcnt;
    for (uint32_t len = 1; len <= (uint32_t)INFL_MAXBITS; len++) {
        if (len > have) { s.err = s.err ? s.err : 1; return -1; }
        code |= (int)(buf & 1u); buf >>= 1;
        const int count = h.count[len];
        if (code - count < first) { s.bitbuf = buf; s.bitcnt = have - len; return h.symbol[index + (code - first)]; }
        index += count; first += count; first <<= 1; code <<= 1;
    }
    s.err = s.err ? s.err : 2;
    return -1;
}

// code lengths -> canonical decoding tables; returns 0 complete code, < 0 over-subscribed, > 0 incomplete
template <class H>
F2Q_HD int infl_construct(H& h, const uint8_t* length, int n) {
    for (int len = 0; len <= INFL_MAXBITS; len++) h.count[len] = 0;
    for (int sym = 0; sym < n; sym++) h.count[length[sym]]++;
    if (h.count[0] == n) return 0;
    int left = 1;
    for (int len = 1; len <= INFL_MAXBITS; len++) { left <<= 1; left -= h.count[len]; if (left < 0) return left; }
    uint16_t offs[INFL_MAXBITS + 1];
    offs[1] = 0;
    for (int len = 1; len < INFL_MAXBITS; len++) offs[len + 1] = (uint16_t)(offs[len] + h.count[len]);
    for (int sym = 0; sym < n; sym++) if (length[sym] != 0) h.symbol[offs[length[sym]]++] = (uint16_t)sym;
    return left;
}

F2Q_HD void infl_codes(InflState& s, const InflHuff& lencode, const InflHuffD& distcode) {
    static const uint16_t lens[29] = {3, 4, 5, 6, 7, 8, 9, 10, 11, 13, 15, 17, 19, 23, 27, 31, 35, 43, 51, 59, 67, 83, 99, 115, 131, 163, 195, 227, 258};
    static const uint8_t lext[29] = {0, 0, 0, 0, 0, 0, 0, 0, 1, 1, 1, 1, 2, 2, 2, 2, 3, 3, 3, 3, 4, 4, 4, 4, 5, 5, 5, 5, 0};
    static const uint16_t dists[30] = {1, 2, 3, 4, 5, 7, 9, 13, 17, 25, 33, 49, 65, 97, 129, 193, 257, 385, 513, 769, 1025, 1537, 2049, 3073, 4097, 6145, 8193, 12289, 16385, 24577};
    static const uint8_t dext[30] = {0, 0, 0, 0, 1, 1, 2, 2, 3, 3, 4, 4, 5, 5, 6, 6, 7, 7, 8, 8, 9, 9, 10, 10, 11, 11, 12, 12, 13, 13};
    for (;;) {
        int symbol = infl_decode(s, lencode);
        if (symbol < 0) return;
        if (symbol < 256) {
            if (s.out_pos >= s.out_len) { s.err = s.err ? s.err : 3; return; }
            s.out[s.out_pos++] = (uint8_t)symbol;
        } else if (symbol == 256) return;
        else {
            symbol -= 257;
            if (symbol >= 29) { s.err = s.err ? s.err : 2; return; }
            const uint32_t len = lens[symbol] + infl_bits(s, lext[symbol]);
            const int ds = infl_decode(s, distcode);
            if (ds < 0) return;
            if (ds >= 30) { s.err = s.err ? s.err : 2; return; }
            const uint32_t dist = dists[ds] + infl_bits(s, dext[ds]);
            if (s.err) return;
            if (dist > s.out_pos) { s.err = 2; return; }
            if (s.out_pos + len > s.out_len) { s.err = 3; return; }
            uint8_t* o = s.out + s.out_pos;
            const uint8_t* f = o - dist;
            for (uint32_t k = 0; k < len; k++) o[k] = f[k];
            s.out_pos += len;
        }
    }
}

// inflates one raw deflate stream; returns 0 when exactly out_len bytes were produced and the final block ended, else the error
F2Q_HD int inflate_raw(const uint8_t* in, uint32_t in_len, uint8_t* out, uint32_t out_len) {
    InflState s;
    s.in = in; s.in_len = in_len; s.in_pos = 0; s.bitbuf = 0; s.bitcnt = 0; s.out = out; s.out_len = out_len; s.out_pos = 0; s.err = 0;
    InflHuff lencode;
    InflHuffD distcode;
    uint8_t lengths[INFL_MAXLCODES + INFL_MAXDCODES + 4];
    int last;
    do {
        last = (int)infl_bits(s, 1);
        const uint32_t type = infl_bits(s, 2);
        if (s.err) break;
        if (type == 0) {
            // stored: skip to the byte boundary, LEN / NLEN, raw bytes
            const uint32_t drop = s.bitcnt & 7u;
            s.bitbuf >>= drop; s.bitcnt -= drop;
            const uint32_t len = infl_bits(s, 16), nlen = infl_bits(s, 16);
            if (s.err) break;
            if ((len ^ 0xFFFFu) != nlen) { s.err = 2; break; }
            if (s.out_pos + len > s.out_len) { s.err = 3; break; }
            for (uint32_t k = 0; k < len; k++) {
                const uint32_t b = infl_bits(s, 8);
                if (s.err) break;
                s.out[s.out_pos++] = (uint8_t)b;
            }
        } else if (type == 1) {
            int sym = 0;
            for (; sym < 144; sym++) lengths[sym] = 8;
            for (; sym < 256; sym++) lengths[sym] = 9;
            for (; sym < 280; sym++) lengths[sym] = 7;
            for (; sym < INFL_FIXLCODES; sym++) lengths[sym] = 8;
            infl_construct(lencode, lengths, INFL_FIXLCODES);
            for (sym = 0; sym < INFL_MAXDCODES; sym++) lengths[sym] = 5;
            infl_construct(distcode, lengths, INFL_MAXDCODES);
            infl_codes(s, lencode, distcode);
        } else if (type == 2) {
            static const uint8_t order[19] = {16, 17, 18, 0, 8, 7, 9, 6, 10, 5, 11, 4, 12, 3, 13, 2, 14, 1, 15};
            const int nlen = (int)infl_bits(s, 5) + 257, ndist = (int)infl_bits(s, 5) + 1, ncode = (int)infl_bits(s, 4) + 4;
            if (s.err) break;
            if (nlen > INFL_MAXLCODES || ndist > INFL_MAXDCODES) { s.err = 2; break; }
            int index = 0;
            for (; index < ncode; index++) lengths[order[index]] = (uint8_t)infl_bits(s, 3);
            for (; index < 19; index++) lengths[order[index]] = 0;
            if (s.err) break;
            if (infl_construct(lencode, lengths, 19) != 0) { s.err = 2; break; }
            index = 0;
            while (index < nlen + ndist) {
                int symbol = infl_decode(s, lencode);
                if (symbol < 0) break;
                if (symbol < 16) lengths[index++] = (uint8_t)symbol;
                else {
                    int len = 0, rep;
                    if (symbol == 16) { if (index == 0) { s.err = 2; break; } len = lengths[index - 1]; rep = 3 + (int)infl_bits(s, 2); }
                    else if (symbol == 17) rep = 3 + (int)infl_bits(s, 3);
                    else rep = 11 + (int)infl_bits(s, 7);
                    if (s.err) break;
                    if (index + rep > nlen + ndist) { s.err = 2; break; }
                    while (rep--) lengths[index++] = (uint8_t)len;
                }
            }
            if (s.err) break;
            if (lengths[256] == 0) { s.err = 2; break; }
            int e = infl_construct(lencode, lengths, nlen);
            if (e < 0 || (e > 0 && nlen - lencode.count[0] != 1)) { s.err = 2; break; }
            e = infl_construct(distcode, lengths + nlen, ndist);
            if (e < 0 || (e > 0 && ndist - distcode.count[0] != 1)) { s.err = 2; break; }
            infl_codes(s, lencode, distcode);
        } else s.err = 2;
    } while (!last && !s.err);
    if (!s.err && s.out_pos != s.out_len) s.err = 2;
    return s.err;
}


// ------------------------------------------------------------------------------------------------------------
// The same decoder as a LOCK-STEP state machine, for a warp whose 32 lanes inflate 32 blocks.
// inflate_raw above lets every lane follow its own control flow; measured on the device (ncu: 1.01 active threads per
// warp instruction) the lanes of a warp then run one after the other.  Here every lane executes the SAME loop body; what a
// lane does in an iteration depends on its state: read a block header and build its tables (rare, the only part in which
// lanes wait for each other), decode one literal / length+distance pair through a lookup table and copy up to 8 bytes of the
// match, copy 8 more bytes of a long match, copy up to 4 bytes of a stored block.
//
// What the loop is built around (the kernel runs few warps per SM — shared memory bounds them — so it is the latency of one
// iteration's dependent chain that counts):
//   * the lane's scalars (InflLane) hold no array and never leave registers; the canonical tables (InflTables, local
//     memory) are touched by block headers and by codes longer than the lookup index only;
//   * input arrives in aligned 32-bit words, loaded one refill AHEAD of their use;
//   * a match loads its 8 source bytes as three aligned words (an overlapping match, distance < 8, replicates its period in
//     registers) and stores them ONE ITERATION LATER, behind the next symbol's decode: the decode does not depend on the
//     copied bytes, so the round trip of the loads (the lane's own output, in L2) is off the chain;
//   * length / distance bases and extra-bit counts are computed, not looked up;
//   * a code longer than the lookup index resumes the canonical walk at the first uncovered length, on bit-reversed input.
// lut / dlut: the lane's lookup tables, element i of lane L at lut[i * stride + L] (shared memory on the device: the
// interleaving makes the lanes' random look-ups hit distinct banks); entry = symbol << 4 | code length, 0 = no short code.
// The input must be readable 16 bytes past its end and 3 bytes before its start, the output 3 bytes before its start and
// 16 past its end (aligned word loads; what is read there is never used).
// ------------------------------------------------------------------------------------------------------------
#if defined(__CUDACC__)
#define F2Q_HD_COLD __host__ __device__ __noinline__
#else
#define F2Q_HD_COLD inline
#endif

constexpr int INFL_LUT_BITS = 9, INFL_DLUT_BITS = 7;
enum { INFL_ST_HEADER = 0, INFL_ST_SYMBOL = 1, INFL_ST_COPY = 2, INFL_ST_STORED = 3, INFL_ST_DONE = 4 };

struct InflTables {
    InflHuff lencode;
    InflHuffD distcode;
    int lfirst, lindex, dfirst, dindex;      // the canonical walk's (first, index) behind the lengths the lookup tables cover
};
struct InflLane {
    const uint8_t* in; uint8_t* out;
    uint64_t bitbuf;
    uint32_t ahead;                          // the input word at in_pos, loaded one refill ahead
    uint32_t bitcnt, in_pos, in_len, out_pos, out_len;
    uint32_t state, last, copy_len, copy_dist, err;
    uint32_t pw0, pw1, pw2, pend_sh, pend_dist, pend_o, pend_n;   // a copy's source words, loaded but not yet stored
};

F2Q_HD uint32_t infl_word(const uint8_t* p) { return *reinterpret_cast<const uint32_t*>(p); }   // p is 4-byte aligned
F2Q_HD uint32_t infl_brev(uint32_t v) {
#if defined(__CUDA_ARCH__)
    return __brev(v);
#else
    v = ((v >> 1) & 0x55555555u) | ((v & 0x55555555u) << 1);
    v = ((v >> 2) & 0x33333333u) | ((v & 0x33333333u) << 2);
    v = ((v >> 4) & 0x0F0F0F0Fu) | ((v & 0x0F0F0F0Fu) << 4);
    return (v >> 24) | ((v >> 8) & 0xFF00u) | ((v << 8) & 0xFF0000u) | (v << 24);
#endif
}
// bits [sh, sh + 32) of hi:lo, sh in {0, 8, 16, 24}
F2Q_HD uint32_t infl_fsr(uint32_t lo, uint32_t hi, uint32_t sh) {
#if defined(__CUDA_ARCH__)
    return __funnelshift_r(lo, hi, sh);
#else
    return (uint32_t)((((uint64_t)hi << 32) | lo) >> sh);
#endif
}

// lookup table of a canonical code: every index whose low `len` bits are the (bit-reversed) code of a symbol of length
// len <= bits gets symbol << 4 | len; returns through first / index the state of the canonical walk behind length `bits`
template <class H>
F2Q_HD void infl_build_lut(const H& h, uint16_t* lut, uint32_t stride, int bits, int* first_out, int* index_out) {
    for (uint32_t i = 0; i < (1u << bits); i++) lut[i * stride] = 0;
    uint32_t code = 0, index = 0;
    int first = 0;
    for (int len = 1; len <= bits; len++) {
        const uint32_t cnt = h.count[len];
        for (uint32_t k = 0; k < cnt; k++) {
            const uint32_t sym = h.symbol[index + k], r = infl_brev(code + k) >> (32 - len);
            for (uint32_t hi = 0; hi < (1u << (bits - len)); hi++) lut[(r | (hi << len)) * stride] = (uint16_t)((sym << 4) | (uint32_t)len);
        }
        code = (code + cnt) << 1; index += cnt; first = (first + (int)cnt) << 1;
    }
    *first_out = first; *index_out = (int)index;
}

// 32 more input bits when there is room for them (words behind the stream's end read as what follows it in memory: a valid
// stream never uses them, and the final check refuses a stream that did).  A corrupted stream can ask for bits far behind its
// end (up to 15 bits per output byte, or an endless chain of empty blocks): from 8 bytes behind the end it gets zeros, so that
// no load leaves the 16 bytes of slack the caller provides
F2Q_HD void infl_refill4(InflLane& L) {
    if (L.bitcnt <= 32u) {
        L.bitbuf |= (uint64_t)L.ahead << L.bitcnt; L.bitcnt += 32u; L.in_pos += 4u;
        L.ahead = L.in_pos <= L.in_len + 8u ? infl_word(L.in + L.in_pos) : 0u;
    }
}
F2Q_HD uint32_t infl_take(InflLane& L, uint32_t n) {
    const uint32_t v = (uint32_t)L.bitbuf & ((1u << n) - 1u);          // n <= 16
    L.bitbuf >>= n; L.bitcnt -= n;
    return v;
}
// one symbol; at least 33 bits are buffered
template <int BITS, class H>
F2Q_HD int infl_decode_lut(InflLane& L, const H& h, const uint16_t* lut, uint32_t stride, int first, int index) {
    const uint32_t e = lut[((uint32_t)L.bitbuf & ((1u << BITS) - 1u)) * stride];
    if (e & 15u) { L.bitbuf >>= (e & 15u); L.bitcnt -= (e & 15u); return (int)(e >> 4); }
    // a code longer than the table's index: the canonical walk, from the first length the table does not cover
    const uint32_t rev = infl_brev((uint32_t)L.bitbuf);                // the first bit of the code on top
#pragma unroll
    for (int len = BITS + 1; len <= INFL_MAXBITS; len++) {
        const int c = (int)(rev >> (32 - len)), count = h.count[len];
        if (c - count < first) { L.bitbuf >>= len; L.bitcnt -= (uint32_t)len; return h.symbol[index + (c - first)]; }
        index += count; first = (first + count) << 1;
    }
    L.err = L.err ? L.err : 2u;
    return -1;
}

// block header of one lane (the divergent part): stored -> INFL_ST_STORED; fixed / dynamic -> tables + INFL_ST_SYMBOL
template <int LB, int DB>
F2Q_HD_COLD void infl_header(InflLane& L, InflTables& T, uint16_t* lut, uint16_t* dlut, uint32_t stride) {
    uint8_t lengths[INFL_MAXLCODES + INFL_MAXDCODES + 4];
    infl_refill4(L);
    L.last = infl_take(L, 1);
    const uint32_t type = infl_take(L, 2);
    if (type == 0) {
        const uint32_t drop = L.bitcnt & 7u;
        L.bitbuf >>= drop; L.bitcnt -= drop;
        infl_refill4(L);
        const uint32_t len = infl_take(L, 16), nlen = infl_take(L, 16);
        if ((len ^ 0xFFFFu) != nlen) { L.err = 2; return; }
        if (L.out_pos + len > L.out_len) { L.err = 3; return; }
        L.copy_len = len; L.state = len ? INFL_ST_STORED : (L.last ? INFL_ST_DONE : INFL_ST_HEADER);
        return;
    }
    if (type == 1) {
        int sym = 0;
        for (; sym < 144; sym++) lengths[sym] = 8;
        for (; sym < 256; sym++) lengths[sym] = 9;
        for (; sym < 280; sym++) lengths[sym] = 7;
        for (; sym < INFL_FIXLCODES; sym++) lengths[sym] = 8;
        infl_construct(T.lencode, lengths, INFL_FIXLCODES);
        for (sym = 0; sym < INFL_MAXDCODES; sym++) lengths[sym] = 5;
        infl_construct(T.distcode, lengths, INFL_MAXDCODES);
    } else if (type == 2) {
        static const uint8_t order[19] = {16, 17, 18, 0, 8, 7, 9, 6, 10, 5, 11, 4, 12, 3, 13, 2, 14, 1, 15};
        infl_refill4(L);
        const int nlen = (int)infl_take(L, 5) + 257, ndist = (int)infl_take(L, 5) + 1, ncode = (int)infl_take(L, 4) + 4;
        if (nlen > INFL_MAXLCODES || ndist > INFL_MAXDCODES) { L.err = 2; return; }
        int index = 0;
        for (; index < ncode; index++) { infl_refill4(L); lengths[order[index]] = (uint8_t)infl_take(L, 3); }
        for (; index < 19; index++) lengths[order[index]] = 0;
        if (infl_construct(T.lencode, lengths, 19) != 0) { L.err = 2; return; }
        index = 0;
        while (index < nlen + ndist) {
            infl_refill4(L);
            // (the code-length code has at most 19 symbols of <= 7 bits: the bit-serial walk, on buffered bits)
            int code = 0, first = 0, idx2 = 0, symbol = -1;
            for (uint32_t len = 1; len <= 7u; len++) {
                code |= (int)(L.bitbuf & 1u); L.bitbuf >>= 1; L.bitcnt -= 1;
                const int count = T.lencode.count[len];
                if (code - count < first) { symbol = T.lencode.symbol[idx2 + (code - first)]; break; }
                idx2 += count; first += count; first <<= 1; code <<= 1;
            }
            if (symbol < 0) { L.err = 2; return; }
            if (symbol < 16) lengths[index++] = (uint8_t)symbol;
            else {
                int len = 0, rep;
                if (symbol == 16) { if (index == 0) { L.err = 2; return; } len = lengths[index - 1]; rep = 3 + (int)infl_take(L, 2); }
                else if (symbol == 17) rep = 3 + (int)infl_take(L, 3);
                else rep = 11 + (int)infl_take(L, 7);
                if (index + rep > nlen + ndist) { L.err = 2; return; }
                while (rep--) lengths[index++] = (uint8_t)len;
            }
        }
        if (lengths[256] == 0) { L.err = 2; return; }
        int e = infl_construct(T.lencode, lengths, nlen);
        if (e < 0 || (e > 0 && nlen - T.lencode.count[0] != 1)) { L.err = 2; return; }
        e = infl_construct(T.distcode, lengths + nlen, ndist);
        if (e < 0 || (e > 0 && ndist - T.distcode.count[0] != 1)) { L.err = 2; return; }
    } else { L.err = 2; return; }
    infl_build_lut(T.lencode, lut, stride, LB, &T.lfirst, &T.lindex);
    infl_build_lut(T.distcode, dlut, stride, DB, &T.dfirst, &T.dindex);
    L.state = INFL_ST_SYMBOL;
}

F2Q_HD void infl_lane_init(InflLane& L, const uint8_t* in, uint32_t in_len, uint8_t* out, uint32_t out_len) {
    L.in = in; L.in_len = in_len; L.out = out; L.out_len = out_len; L.out_pos = 0; L.err = 0;
    L.bitbuf = 0; L.bitcnt = 0; L.in_pos = 0; L.ahead = 0;
    L.state = in_len ? INFL_ST_HEADER : INFL_ST_DONE; L.last = 0; L.copy_len = 0; L.copy_dist = 0;
    L.pw0 = L.pw1 = L.pw2 = 0; L.pend_sh = 0; L.pend_dist = 8; L.pend_o = 0; L.pend_n = 0;
    if (!in_len && out_len) L.err = 2;
    if (in_len) {
        // the bytes up to the first aligned word, then aligned words only
        const uint32_t mis = (uint32_t)(reinterpret_cast<uintptr_t>(in) & 3u);
        L.bitbuf = infl_word(in - mis) >> (8u * mis); L.bitcnt = 32u - 8u * mis; L.in_pos = 4u - mis;
        L.ahead = infl_word(in + L.in_pos);
    }
}

// the 8 bytes a copy loaded one iteration ago -> the output
F2Q_HD void infl_flush(InflLane& L) {
    if (L.pend_n) {
        uint64_t v = (uint64_t)infl_fsr(L.pw0, L.pw1, L.pend_sh) | ((uint64_t)infl_fsr(L.pw1, L.pw2, L.pend_sh) << 32);
        if (L.pend_dist < 8u) {
            // the source overlaps what this copy writes: its first `dist` bytes are the period
            const uint32_t period = 8u * L.pend_dist;
            v &= (1ull << period) - 1ull;
            v |= v << period;
            if (2u * period < 64u) v |= v << (2u * period);
            if (4u * period < 64u) v |= v << (4u * period);
        }
        uint8_t* o = L.out + L.pend_o;
#pragma unroll
        for (uint32_t k = 0; k < 8u; k++) if (k < L.pend_n) o[k] = (uint8_t)(v >> (8u * k));
        L.pend_n = 0;
    }
}

// one iteration of the state machine for one lane; the caller loops while any lane is not INFL_ST_DONE and calls
// infl_flush behind the loop.  Three phases, so that the loads of a copy have a whole decode to arrive in:
//   A  decode (registers, the lookup tables and the input only)   B  store what the copy of the LAST iteration loaded
//   C  store this iteration's literal, or load (not yet store) the next 8 bytes of a match
template <int LB = INFL_LUT_BITS, int DB = INFL_DLUT_BITS>
F2Q_HD void infl_step(InflLane& L, InflTables& T, uint16_t* lut, uint16_t* dlut, uint32_t stride) {
    int lit = -1;
    if (L.state == INFL_ST_HEADER) {
        InflLane t = L;                                                // (the copy's address escapes, the lane's registers do not)
        infl_header<LB, DB>(t, T, lut, dlut, stride);
        L = t;
        if (L.err) L.state = INFL_ST_DONE;
    } else if (L.state == INFL_ST_SYMBOL) {
        infl_refill4(L);
        const int symbol = infl_decode_lut<LB>(L, T.lencode, lut, stride, T.lfirst, T.lindex);
        if (symbol < 256) {
            if (symbol < 0) L.state = INFL_ST_DONE;
            else if (L.out_pos >= L.out_len) { L.err = 3; L.state = INFL_ST_DONE; }
            else lit = symbol;
        } else if (symbol == 256) L.state = L.last ? INFL_ST_DONE : INFL_ST_HEADER;
        else {
            // length 3..258: symbols 257..264 are 3..10, 265..284 carry (sym - 261) / 4 extra bits, 285 is 258
            const uint32_t sym = (uint32_t)symbol - 257u;
            const uint32_t lx = (sym < 8u || sym == 28u) ? 0u : (sym - 4u) >> 2;
            const uint32_t lbase = sym < 8u ? 3u + sym : sym == 28u ? 258u : 3u + ((4u + (sym & 3u)) << lx);
            const uint32_t len = lbase + infl_take(L, lx);
            infl_refill4(L);
            const int ds = infl_decode_lut<DB>(L, T.distcode, dlut, stride, T.dfirst, T.dindex);
            // distance 1..32768: codes 0..3 are 1..4, the others carry (code - 2) / 2 extra bits
            const uint32_t d = (uint32_t)ds, dx = d < 4u ? 0u : (d - 2u) >> 1;
            const uint32_t dbase = d < 4u ? 1u + d : 1u + ((2u + (d & 1u)) << (dx & 15u));
            const uint32_t dist = dbase + infl_take(L, dx & 15u);
            if (sym >= 29u || ds < 0 || ds >= 30) { L.err = L.err ? L.err : 2u; L.state = INFL_ST_DONE; }
            else if (dist > L.out_pos) { L.err = 2; L.state = INFL_ST_DONE; }
            else if (L.out_pos + len > L.out_len) { L.err = 3; L.state = INFL_ST_DONE; }
            else { L.copy_len = len; L.copy_dist = dist; L.state = INFL_ST_COPY; }
        }
    }
    infl_flush(L);
    if (lit >= 0) L.out[L.out_pos++] = (uint8_t)lit;
    else if (L.state == INFL_ST_COPY) {
        // up to 8 bytes of the match (a lane that has just decoded it starts the copy in the same iteration): the three
        // aligned words that hold them are loaded now and stored by the next iteration's flush
        const uint32_t n = L.copy_len < 8u ? L.copy_len : 8u;
        const uint8_t* f = L.out + L.out_pos - L.copy_dist;
        const uint32_t a = (uint32_t)(reinterpret_cast<uintptr_t>(f) & 3u);
        L.pw0 = infl_word(f - a); L.pw1 = infl_word(f - a + 4); L.pw2 = infl_word(f - a + 8);
        L.pend_sh = 8u * a; L.pend_dist = L.copy_dist; L.pend_o = L.out_pos; L.pend_n = n;
        L.out_pos += n; L.copy_len -= n;
        if (!L.copy_len) L.state = INFL_ST_SYMBOL;
    } else if (L.state == INFL_ST_STORED) {
        // the bit buffer holds whole bytes here
        const uint32_t n = L.copy_len < 4u ? L.copy_len : 4u;
        infl_refill4(L);
        for (uint32_t k = 0; k < n; k++) L.out[L.out_pos++] = (uint8_t)infl_take(L, 8);
        L.copy_len -= n;
        if (!L.copy_len) L.state = L.last ? INFL_ST_DONE : INFL_ST_HEADER;
    }
}

// end of a lane: everything produced, and not a bit taken from behind the stream's end
F2Q_HD int infl_lane_result(const InflLane& L) {
    if (L.err) return (int)L.err;
    if (L.out_pos != L.out_len) return 2;
    if ((uint64_t)L.in_pos * 8u - L.bitcnt > (uint64_t)L.in_len * 8u) return 1;
    return 0;
}


// ------------------------------------------------------------------------------------------------------------
// CRC-32 of gzip (RFC 1952: reflected, polynomial 0xEDB88320, register preset and final value inverted): the trailer of
// every BGZF block carries the CRC of its uncompressed bytes, and a corrupted Huffman stream usually still decodes to the
// promised length, with wrong bytes.  The 32 lanes of a warp check one block: lane j hashes a contiguous slice with
// slicing-by-4 tables, and the slices are joined by linearity,
//     crc(A || B) = crc(A) * x^(8|B|) mod P  xor  crc(B),
// so crc(block) = xor over lanes of crc(slice_j) * x^(8 * bytes behind slice_j) mod P.
// ------------------------------------------------------------------------------------------------------------
constexpr uint32_t CRC32_POLY = 0xEDB88320u;

// entry i of the slicing-by-4 tables (4 x 256 words): table k, byte b = b followed by k zero bytes through the register
F2Q_HD uint32_t crc32_table_entry(uint32_t i) {
    uint32_t c = i & 255u;
    const uint32_t rounds = 8u * ((i >> 8) + 1u);
    for (uint32_t r = 0; r < rounds; r++) c = (c & 1u) ? (c >> 1) ^ CRC32_POLY : c >> 1;
    return c;
}

// the register after n bytes at p (no inversion: crc32 = ~crc32_update(~0, ...)); aligned 32-bit words where it can
F2Q_HD uint32_t crc32_update(uint32_t c, const uint8_t* p, uint32_t n, const uint32_t* tab) {
    uint32_t i = 0;
    for (; i < n && (reinterpret_cast<uintptr_t>(p + i) & 3u); i++) c = tab[(c ^ p[i]) & 255u] ^ (c >> 8);
    for (; i + 4u <= n; i += 4u) {
        c ^= infl_word(p + i);
        c = tab[768u + (c & 255u)] ^ tab[512u + ((c >> 8) & 255u)] ^ tab[256u + ((c >> 16) & 255u)] ^ tab[c >> 24];
    }
    for (; i < n; i++) c = tab[(c ^ p[i]) & 255u] ^ (c >> 8);
    return c;
}

// a * b mod P (bit 31 is x^0, as in the reflected register)
F2Q_HD uint32_t crc32_mulmod(uint32_t a, uint32_t b) {
    uint32_t p = 0;
    for (int k = 0; k < 32; k++) {
        if (a & (0x80000000u >> k)) p ^= b;
        b = (b & 1u) ? (b >> 1) ^ CRC32_POLY : b >> 1;
    }
    return p;
}

// crc * x^(8n) mod P: the CRC of a prefix moved in front of n more bytes
F2Q_HD uint32_t crc32_shift(uint32_t crc, uint32_t n) {
    uint32_t sq = 1u << 23, p = 1u << 31;                              // x^8, 1
    for (; n; n >>= 1) {
        if (n & 1u) p = crc32_mulmod(sq, p);
        sq = crc32_mulmod(sq, sq);
    }
    return crc32_mulmod(p, crc);
}

// lane `lane` of `lanes` (one CRC check of an n-byte block): the CRC of its slice, shifted over the bytes behind the slice.
// The xor of all lanes' values is the block's CRC.  Slices are a multiple of 4 bytes long (word loads from the second on).
F2Q_HD uint32_t crc32_lane_part(const uint8_t* p, uint32_t n, uint32_t lane, uint32_t lanes, const uint32_t* tab) {
    const uint32_t s = ((n + lanes - 1u) / lanes + 3u) & ~3u;
    const uint32_t beg = lane * s < n ? lane * s : n, end = beg + s < n ? beg + s : n;
    if (beg == end) return 0u;
    return crc32_shift(~crc32_update(~0u, p + beg, end - beg, tab), n - end);
}

}  // namespace f2q
