// hostcheck.cpp — TEST INFRASTRUCTURE ONLY: compiles the host-callable halves of the device headers with g++ so that
// CPU tests (no GPU in the build container) can check them against the numpy restatement / the oracle bit for bit.
// Nothing here is part of the product path; libf2q.so never links it.
#include <stdint.h>
#include <string.h>

#include "../../2fast2q_b200/csrc/synth_gen.h"

extern "C" {

__attribute__((visibility("default")))
void hc_synth(const f2q_synth_spec* sp, const uint8_t* guides, uint64_t first, uint64_t n, uint8_t* out) {
    const uint64_t rec = 2ull * sp->read_len + 18;
    for (uint64_t k = 0; k < n; k++) f2q::synth_record(*sp, guides, first + k, out + k * rec);
}

}

// ---- flex_core.h: bit-parallel key extraction of one read, against oracle f2qo_build_key -----------------------------
#include <vector>

#include "../../2fast2q_b200/csrc/flex_core.h"

namespace {
template <int PW, int K>
int flex_key_t(const f2q::FlexCfg& C, const uint8_t* read, int r, const uint8_t* qual, int q, int extra, uint8_t* out, int* out_len) {
    // the lines sit at odd offsets of padded buffers, as they do inside a tile
    std::vector<uint8_t> sb(32 * PW + 64, '\n'), qb(32 * PW + 64, '\n');
    const uint32_t so = 5, qo = 11;
    memcpy(sb.data() + so, read, r); memcpy(qb.data() + qo, qual, q);
    f2q::FlexPiece pc[f2q::FLEX_ITER];
    const uint32_t maxlen = (uint32_t)((r > q ? r : q) + extra);       // (a warp's longest line may be longer than this one)
    const int np = f2q::flex_pieces<PW, K>(C, sb.data(), so, (uint32_t)r, qb.data(), qo, (uint32_t)q, maxlen > 32u * PW ? 32u * PW : maxlen, pc);
    if (np < 0) return np < -2 ? -2 : np;
    int n = 0;
    for (int p = 0; p < np; p++) {
        if (p) out[n++] = ':';
        for (uint32_t i = 0; i < pc[p].len; i++) {
            uint8_t c = read[pc[p].off + i];
            if ((pc[p].notok >> i) & 1u) { if (c >= 'a' && c <= 'z') c -= 32; }      // the caller's look at the raw byte
            else c = (uint8_t)("ACTG"[(pc[p].codes >> (2 * i)) & 3u]);                 // decoded from the packed codes
            out[n++] = c;
        }
    }
    *out_len = n;
    return np;
}
}  // namespace

extern "C" {

// returns 1 when the configuration is eligible for the bit-parallel path, else 0
__attribute__((visibility("default")))
int hc_flex_eligible(const f2q_config* cfg) {
    f2q::FlexCfg C;
    return f2q::flex_prepare(*cfg, C) ? 1 : 0;
}

// key of one read through flex_pieces: returns np >= 0 (key in out), -1 all iterations flagged, -2 generic path needed,
// -3 not eligible / read too long for pw planes
__attribute__((visibility("default")))
int hc_flex_key(const f2q_config* cfg, int pw, const uint8_t* read, int r, const uint8_t* qual, int q, int extra, uint8_t* out, int* out_len) {
    f2q::FlexCfg C;
    if (!f2q::flex_prepare(*cfg, C)) return -3;
    if (r > 32 * pw || q > 32 * pw) return -3;
    const int K = C.max_k <= 1 ? 1 : 3;                              // the two instances the kernels have
#define F2Q_HC_CASE(PWV, KV) if (pw == PWV && K == KV) return flex_key_t<PWV, KV>(C, read, r, qual, q, extra, out, out_len);
    F2Q_HC_CASE(3, 1) F2Q_HC_CASE(3, 3) F2Q_HC_CASE(5, 1) F2Q_HC_CASE(5, 3)
#undef F2Q_HC_CASE
    return -3;
}

}

// ---- inflate_core.h: the per-block DEFLATE decoder of k_inflate_bgzf, against zlib --------------------------------------
#include "../../2fast2q_b200/csrc/inflate_core.h"

// (the lock-step decoder reads aligned words around its buffers: the copies here carry the margins its contract asks for)
template <int LB, int DB>
static int inflate_lane(const uint8_t* in, uint32_t in_len, uint8_t* out, uint32_t out_len, uint64_t* stats = nullptr) {
    static thread_local uint16_t lut[1 << LB], dlut[1 << DB];
    std::vector<uint8_t> ibuf((size_t)in_len + 64, 0xAA), obuf((size_t)out_len + 64, 0x55);
    for (int mis = 0; mis < (stats ? 1 : 4); mis++) {                  // every alignment of the input and of the output
        uint8_t* ip = ibuf.data() + 16 + mis;
        uint8_t* op = obuf.data() + 16 + ((mis * 3) & 3);
        memcpy(ip, in, in_len);
        f2q::InflLane L;
        f2q::InflTables T;
        f2q::infl_lane_init(L, ip, in_len, op, out_len);
        for (uint64_t it = 0; L.state != f2q::INFL_ST_DONE; it++) {
            if (it > (1ull << 28)) return 9;
            if (stats) stats[L.state]++;
            f2q::infl_step<LB, DB>(L, T, lut, dlut, 1);
        }
        f2q::infl_flush(L);
        const int rc = f2q::infl_lane_result(L);
        if (mis == 0) { memcpy(out, op, out_len); if (rc) return rc; }
        else if (rc || memcmp(out, op, out_len) != 0) return 8;        // an alignment that decodes differently
    }
    return 0;
}

extern "C" {
__attribute__((visibility("default")))
int hc_inflate_raw(const uint8_t* in, uint32_t in_len, uint8_t* out, uint32_t out_len) { return f2q::inflate_raw(in, in_len, out, out_len); }

// the lock-step state machine, one lane; `in` must be readable 8 bytes past in_len (as in the kernel's staging buffer)
__attribute__((visibility("default")))
int hc_inflate_lane(const uint8_t* in, uint32_t in_len, uint8_t* out, uint32_t out_len) { return inflate_lane<9, 7>(in, in_len, out, out_len); }
// (the small tables: more codes take the bit-serial path)
__attribute__((visibility("default")))
int hc_inflate_lane8(const uint8_t* in, uint32_t in_len, uint8_t* out, uint32_t out_len) { return inflate_lane<8, 6>(in, in_len, out, out_len); }
}

// ---- how far behind its input the lock-step decoder reads ----------------------------------------------------------------
// The input ends 16 bytes before an inaccessible page (the slack inflate_core.h asks for); a load behind that is caught
// (SIGSEGV -> siglongjmp) and reported as 99 instead of ending the process.
#include <setjmp.h>
#include <signal.h>
#include <sys/mman.h>
#include <unistd.h>

static sigjmp_buf g_guard_jmp;
static void guard_handler(int) { siglongjmp(g_guard_jmp, 1); }

extern "C" __attribute__((visibility("default")))
int hc_inflate_lane_guarded(const uint8_t* in, uint32_t in_len, uint32_t out_len) {
    const size_t page = (size_t)sysconf(_SC_PAGESIZE), span = ((size_t)in_len + 16 + page - 1) / page * page;
    uint8_t* m = static_cast<uint8_t*>(mmap(nullptr, span + page, PROT_READ | PROT_WRITE, MAP_PRIVATE | MAP_ANONYMOUS, -1, 0));
    if (m == MAP_FAILED) return -1;
    mprotect(m + span, page, PROT_NONE);
    uint8_t* ip = m + span - 16 - in_len;                              // (alignment: whatever in_len gives)
    memcpy(ip, in, in_len);
    memset(ip + in_len, 0x5c, 16);
    std::vector<uint8_t> obuf((size_t)out_len + 64, 0);
    static thread_local uint16_t lut[1 << 9], dlut[1 << 7];
    struct sigaction sa, old;
    memset(&sa, 0, sizeof(sa)); sa.sa_handler = guard_handler; sigemptyset(&sa.sa_mask);
    sigaction(SIGSEGV, &sa, &old);
    volatile int rc = 99;
    if (sigsetjmp(g_guard_jmp, 1) == 0) {
        f2q::InflLane L;
        f2q::InflTables T;
        f2q::infl_lane_init(L, ip, in_len, obuf.data() + 16, out_len);
        for (uint64_t it = 0; L.state != f2q::INFL_ST_DONE && it < (1ull << 26); it++) f2q::infl_step<9, 7>(L, T, lut, dlut, 1);
        f2q::infl_flush(L);
        rc = L.state == f2q::INFL_ST_DONE ? f2q::infl_lane_result(L) : 9;
    }
    sigaction(SIGSEGV, &old, nullptr);
    munmap(m, span + page);
    return rc;
}

// ---- the CRC-32 check of k_bgzf_crc, against zlib.crc32 ----------------------------------------------------------------
static const uint32_t* crc_tables() {
    static uint32_t tab[1024];
    static bool ready = false;
    if (!ready) { for (uint32_t i = 0; i < 1024; i++) tab[i] = f2q::crc32_table_entry(i); ready = true; }
    return tab;
}
extern "C" {
// the CRC of p[0, n) in one pass
__attribute__((visibility("default")))
uint32_t hc_crc32(const uint8_t* p, uint32_t n) { return ~f2q::crc32_update(~0u, p, n, crc_tables()); }
// the CRC of p[0, n) as one warp of k_bgzf_crc computes it: the xor of `lanes` slice values
__attribute__((visibility("default")))
uint32_t hc_crc32_lanes(const uint8_t* p, uint32_t n, uint32_t lanes) {
    uint32_t v = 0;
    for (uint32_t j = 0; j < lanes; j++) v ^= f2q::crc32_lane_part(p, n, j, lanes, crc_tables());
    return v;
}
// crc * x^(8n) mod P
__attribute__((visibility("default")))
uint32_t hc_crc32_shift(uint32_t crc, uint32_t n) { return f2q::crc32_shift(crc, n); }
}

// developer statistics: iterations of the lock-step machine by state (HEADER, SYMBOL, COPY, STORED)
extern "C" __attribute__((visibility("default")))
int hc_inflate_lane_stats(const uint8_t* in, uint32_t in_len, uint8_t* out, uint32_t out_len, uint64_t* stats) {
    return inflate_lane<9, 7>(in, in_len, out, out_len, stats);
}
