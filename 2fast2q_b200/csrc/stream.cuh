// stream.cuh — chunk boundary handling, entirely on the device and stream-ordered (no host round trip):
//   k_prepare  before the tile kernel: completes the partial record carried from the previous chunk with the head
//              of the new chunk ("stitch") and sets the record-aligned start of the range the tile kernel parses
//   k_carry    after the tile kernel: saves the new partial tail record
// Records are "every 4 lines from byte 0" (fast2q.py:324-328), so a chunk cut anywhere needs exactly this much
// state: the bytes of the unfinished record (their newline count mod 4 is the line phase).
#pragma once

#include "f2q_dev.cuh"
#include "inflate_core.h"
#include "synth_gen.h"

namespace f2q {

constexpr int PREP_THREADS = 256;

// chunk = user bytes at buf[delta, delta+n); carry = ctx buffer of carry_cap bytes
// small per-chunk arrays that must be zero before the chunk's kernels run: cleared here instead of by one memset each (a
// sample of a few hundred MB is parsed in ~0.2 ms; every stream operation saved is a few percent of it)
struct PrepClear {
    uint8_t* status_stitch; uint32_t n_status_stitch;
    uint8_t* spec_rec; uint32_t n_spec_rec;
    uint32_t* seg_count; uint32_t n_segs;
};

__global__ void __launch_bounds__(PREP_THREADS) k_prepare(DevState* S, const uint8_t* __restrict__ buf, uint64_t delta, uint64_t n,
                                                          uint32_t is_last, uint8_t* __restrict__ carry, uint64_t carry_cap,
                                                          uint32_t* tickets, uint32_t q_cap, uint32_t g_cap, PrepClear Z) {
    __shared__ uint64_t s_h;          // bytes of the chunk head that complete the carried record
    __shared__ uint32_t s_found, s_cnt;
    const uint32_t tid = threadIdx.x;
    for (uint32_t i = tid; i < Z.n_status_stitch; i += PREP_THREADS) Z.status_stitch[i] = 0;
    for (uint32_t i = tid; i < Z.n_spec_rec; i += PREP_THREADS) Z.spec_rec[i] = 0;
    for (uint32_t i = tid; i < Z.n_segs; i += PREP_THREADS) Z.seg_count[i] = 0;
    const uint32_t tl = S->tail_len, tnl = S->tail_nl;
    __syncthreads();
    if (tid == 0) {
        S->q_count = 0; S->g_count = 0; S->q_cap = q_cap; S->g_cap = g_cap;
        S->last_rec_end = 0; S->nl_total = 0; S->stitch_len = 0; S->stitch_eof = 0; S->appended = 0;
        S->is_last = is_last; S->end = delta + n; S->beg = delta; S->spec_fail = 0; S->spec_ok = 0;
        tickets[0] = 0; tickets[1] = 0; tickets[2] = 0;
        s_found = 0; s_cnt = 0; s_h = 0;
    }
    __syncthreads();
    if (tl == 0) return;

    // find the (4 - tnl)-th newline of the chunk, one warp, 32 x 16 bytes per step
    const uint32_t need = 4 - tnl;
    if (tid < 32) {
        uint32_t seen = 0; uint64_t pos = 0; bool found = false; uint64_t h = 0;
        while (pos < n && !found) {
            const uint64_t a = pos + (uint64_t)tid * 16;
            uint32_t mask = 0;
            for (int b = 0; b < 16; b++) if (a + b < n && buf[delta + a + b] == '\n') mask |= 1u << b;
            const uint32_t c = __popc(mask);
            uint32_t incl = c;
            for (int d = 1; d < 32; d <<= 1) { uint32_t y = __shfl_up_sync(0xffffffffu, incl, d); if (tid >= (uint32_t)d) incl += y; }
            const uint32_t before = seen + incl - c;
            const bool mine = (before < need) && (before + c >= need);
            const uint32_t who = __ballot_sync(0xffffffffu, mine);
            if (who) {
                if (mine) {
                    uint32_t k = need - before;            // the k-th set bit of mask
                    uint32_t m = mask;
                    while (--k) m &= m - 1;
                    h = a + (__ffs(m) - 1) + 1;
                }
                h = __shfl_sync(0xffffffffu, h, __ffs(who) - 1);
                found = true;
            } else {
                seen += __shfl_sync(0xffffffffu, incl, 31);
                pos += 512;
            }
        }
        if (tid == 0) { s_found = found; s_h = h; s_cnt = seen; }
    }
    __syncthreads();
    const bool found = s_found != 0;
    const uint64_t h = found ? s_h : n;                     // bytes of the chunk that go behind the carried tail
    if ((uint64_t)tl + h > carry_cap) {
        if (tid == 0) { atomicOr(&S->error, ERR_RECORD_TOO_LONG); S->tail_len = 0; S->tail_nl = 0; S->beg = S->end; S->appended = 1; }
        return;
    }
    for (uint64_t i = tid; i < h; i += PREP_THREADS) carry[tl + i] = buf[delta + i];
    if (tid == 0) {
        if (found) {
            S->stitch_len = (uint32_t)(tl + h); S->stitch_eof = 0;
            S->beg = delta + h; S->tail_len = 0; S->tail_nl = 0;
        } else {
            // the chunk did not finish the record: keep accumulating; at end of stream parse what we have
            S->tail_len = (uint32_t)(tl + n); S->tail_nl = tnl + s_cnt;
            S->beg = S->end; S->appended = 1;
            if (is_last) { S->stitch_len = (uint32_t)(tl + n); S->stitch_eof = 1; S->tail_len = 0; S->tail_nl = 0; }
        }
    }
}

__global__ void __launch_bounds__(PREP_THREADS) k_carry(DevState* S, const uint8_t* __restrict__ buf, uint8_t* __restrict__ carry,
                                                        uint64_t carry_cap) {
    const uint32_t tid = threadIdx.x;
    if (S->appended) return;
    if (S->is_last) { if (tid == 0) { S->tail_len = 0; S->tail_nl = 0; } return; }
    const uint64_t le = S->last_rec_end;
    const uint64_t tb = le > S->beg ? le : S->beg;
    const uint64_t tlen = S->end - tb;
    const uint32_t nl = S->nl_total & 3u;
    __syncthreads();
    if (tlen > carry_cap) { if (tid == 0) { atomicOr(&S->error, ERR_RECORD_TOO_LONG); S->tail_len = 0; S->tail_nl = 0; } return; }
    for (uint64_t i = tid; i < tlen; i += PREP_THREADS) carry[i] = buf[tb + i];
    if (tid == 0) { S->tail_len = (uint32_t)tlen; S->tail_nl = nl; }
}

// ------------------------------------------------------------------------------------------------
// One file on several contexts (f2q_submit_file_sharded): every shard but the first starts at an arbitrary byte offset.
// k_shard_head guesses where its first record starts, from the local record shape alone: the candidates are the bytes
// behind the 1st..4th newline of the shard, and a candidate is accepted when the two records starting there look like
// FASTQ records ('@' header, '+' third line, sequence and quality lines of equal length, the next record starting with '@').
// Exactly one accepted candidate is the guess h; the head [0, h) (1-4 newlines) is saved for the stitch and the shard is
// parsed from h with line phase 0.  The guess is only a guess: the host verifies it against the shard before (DESIGN.md §5).
// ------------------------------------------------------------------------------------------------
constexpr int SHARD_HEAD_NL = 12;              // newlines candidate 4 needs: 4 to reach it + 8 for its two records

__global__ void __launch_bounds__(PREP_THREADS) k_shard_head(DevState* S, const uint8_t* __restrict__ buf, uint64_t n,
                                                             uint8_t* __restrict__ head, uint64_t head_cap) {
    __shared__ uint64_t nlpos[SHARD_HEAD_NL];
    __shared__ uint64_t s_h;
    const uint32_t tid = threadIdx.x;
    if (tid < 32) {
        // the first SHARD_HEAD_NL newlines, one warp, 32 x 16 bytes per step (as k_prepare)
        uint32_t seen = 0;
        for (uint64_t pos = 0; pos < n && seen < (uint32_t)SHARD_HEAD_NL; pos += 512) {
            const uint64_t a = pos + (uint64_t)tid * 16;
            uint32_t mask = 0;
            for (int b = 0; b < 16; b++) if (a + b < n && buf[a + b] == '\n') mask |= 1u << b;
            const uint32_t c = __popc(mask);
            uint32_t incl = c;
            for (int d = 1; d < 32; d <<= 1) { uint32_t y = __shfl_up_sync(0xffffffffu, incl, d); if (tid >= (uint32_t)d) incl += y; }
            uint32_t r = seen + incl - c;
            for (uint32_t m = mask; m && r < (uint32_t)SHARD_HEAD_NL; m &= m - 1) nlpos[r++] = a + (uint64_t)(__ffs(m) - 1);
            seen += __shfl_sync(0xffffffffu, incl, 31);
        }
        __syncwarp();
        if (tid == 0) {
            uint32_t accepted = 0, nl = 0; uint64_t h = 0;
            if (seen >= (uint32_t)SHARD_HEAD_NL) {
                for (uint32_t i = 1; i <= 4; i++) {
                    const uint64_t* L = nlpos + i - 1;          // L[0] ends the line before the candidate, L[1..8] its 8 lines
                    bool ok = true;
                    for (int r = 0; r < 2 && ok; r++) {
                        const uint64_t* q = L + 4 * r;
                        ok = buf[q[0] + 1] == '@' && buf[q[2] + 1] == '+' && q[2] - q[1] == q[4] - q[3];
                    }
                    ok = ok && L[8] + 1 < n && buf[L[8] + 1] == '@';
                    if (ok) { accepted++; nl = i; h = L[0] + 1; }
                }
            }
            const bool good = accepted == 1 && h <= head_cap;
            S->head_ok = good ? 1u : 0u; S->head_nl = good ? nl : 0u; S->head_len = good ? h : 0ull;
            s_h = good ? h : 0ull;
        }
    }
    __syncthreads();
    const uint64_t h = s_h;
    for (uint64_t i = tid; i < h; i += PREP_THREADS) head[i] = buf[i];
}

// the result of another shard's context (copied next to this one: peer copy or same-device copy) is added to this context's
// result vector; its error words are ORed into this context's, so that a failure in any shard fails the whole sample
__global__ void __launch_bounds__(256) k_shard_sum(unsigned long long* __restrict__ result, const unsigned long long* __restrict__ other, uint64_t n_words,
                                                   uint32_t* error, DevState* S, const uint32_t* __restrict__ other_errors) {
    for (uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x; i < n_words; i += (uint64_t)gridDim.x * blockDim.x) result[i] += other[i];
    if (blockIdx.x == 0 && threadIdx.x == 0) {
        if (other_errors[0]) atomicOr(error, other_errors[0]);
        if (other_errors[1]) atomicOr(&S->error, other_errors[1]);
    }
}

// ------------------------------------------------------------------------------------------------
// GPU inflate of bgzip (BGZF) input: one thread per block (inflate_core.h).  The blocks of a chunk are independent, their
// compressed sizes come from the headers and their output offsets from the trailers, so thousands decode at once straight
// into the buffer the streaming kernel parses; only the COMPRESSED bytes cross PCIe.
// ------------------------------------------------------------------------------------------------
struct BgzfBlock { uint32_t src, csize, dst, isize; };
constexpr int INFLATE_THREADS = 64;

// (first form: every lane follows its own control flow through inflate_raw — measured 1.01 active threads per warp instruction,
// 0.65 GB/s; kept as the cross-check of the lock-step form below, option "gpu_inflate" = 2)
__global__ void __launch_bounds__(INFLATE_THREADS) k_inflate_bgzf(const uint8_t* __restrict__ comp, const BgzfBlock* __restrict__ blk, uint32_t n,
                                                                  uint8_t* __restrict__ out, uint32_t* error) {
    for (uint32_t b = blockIdx.x * blockDim.x + threadIdx.x; b < n; b += gridDim.x * blockDim.x) {
        const BgzfBlock B = blk[b];
        if (inflate_raw(comp + B.src, B.csize, out + B.dst, B.isize) != 0) atomicOr(error, ERR_INFLATE);
    }
}

// lock-step form: the 32 lanes of a warp inflate 32 blocks through the state machine of inflate_core.h — every lane runs the
// same loop body, so the warp stays converged; the lanes' lookup tables live in shared memory, interleaved by lane (entry i
// of lane L at [i * 32 + L]: the lanes' random look-ups fall into distinct banks).  Shared memory bounds the lanes per SM
// (1280 B per lane with 9 + 7 index bits, 640 B with 8 + 6), and the kernel is latency-bound: the smaller tables win when
// the batch has enough blocks to fill the extra warps
constexpr int INFLATE_LANES = 32;                                   // one warp per CTA: the CTA is the unit shared memory is handed out in
template <int LB, int DB>
constexpr size_t inflate_smem() { return ((size_t)(1 << LB) + (size_t)(1 << DB)) * INFLATE_LANES * sizeof(uint16_t); }
template <int LB, int DB>
__global__ void __launch_bounds__(INFLATE_LANES) k_inflate_bgzf_lanes(const uint8_t* __restrict__ comp, const BgzfBlock* __restrict__ blk, uint32_t n,
                                                                      uint8_t* __restrict__ out, uint32_t* error) {
    extern __shared__ __align__(16) uint16_t infl_sm[];
    uint16_t* const lut = infl_sm + threadIdx.x;
    uint16_t* const dlut = infl_sm + ((size_t)INFLATE_LANES << LB) + threadIdx.x;
    const uint32_t b = blockIdx.x * INFLATE_LANES + threadIdx.x;
    InflLane L;
    InflTables T;
    if (b < n) { const BgzfBlock B = blk[b]; infl_lane_init(L, comp + B.src, B.csize, out + B.dst, B.isize); }
    else { infl_lane_init(L, comp, 0, out, 0); }
    while (__any_sync(0xffffffffu, L.state != INFL_ST_DONE)) infl_step<LB, DB>(L, T, lut, dlut, INFLATE_LANES);
    infl_flush(L);
    if (b < n && infl_lane_result(L) != 0) atomicOr(error, ERR_INFLATE);
}

// start of a sample: result vector, scratch vector, error word and the stream state in ONE launch
__global__ void __launch_bounds__(256) k_begin(unsigned long long* __restrict__ result, unsigned long long* __restrict__ scratch, uint64_t n_words,
                                               uint32_t* error, DevState* S) {
    for (uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x; i < n_words; i += (uint64_t)gridDim.x * blockDim.x) {
        result[i] = 0;
        if (scratch) scratch[i] = 0;
    }
    if (blockIdx.x == 0) {
        for (uint32_t i = threadIdx.x; i < sizeof(DevState) / 4; i += blockDim.x) reinterpret_cast<uint32_t*>(S)[i] = 0;
        if (threadIdx.x == 0) *error = 0;
    }
}

// ------------------------------------------------------------------------------------------------
// K0: synthetic FASTQ generator (bench / tests).  One thread per read; the record itself is written by synth_record
// (synth_gen.h), bit-identical to 2fast2q_b200/synth.py.
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) k_synth(f2q_synth_spec sp, const uint8_t* __restrict__ guides, uint8_t* __restrict__ out) {
    const uint64_t rec = 2ull * sp.read_len + 18;
    for (uint64_t k = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x; k < sp.n_reads; k += (uint64_t)gridDim.x * blockDim.x)
        synth_record(sp, guides, sp.first_read + k, out + k * rec);
}

}  // namespace f2q
