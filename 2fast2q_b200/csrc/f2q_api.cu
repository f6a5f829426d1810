// f2q_api.cu — C-ABI of libf2q.so (include/f2q.h): contexts, library tables, streaming submits.
// Host code only orchestrates: every byte of FASTQ is parsed by the kernels in tile.cuh / generic.cuh /
// resolve.cuh.  There is no CPU implementation of the path in this library.
#include <cuda_runtime.h>

#include <algorithm>
#include <atomic>
#include <cstdio>
#include <cstdlib>
#include <chrono>
#include <cstring>
#include <deque>
#include <dlfcn.h>
#include <zlib.h>
#include <thread>
#include <cerrno>
#include <sys/mman.h>
#include <sys/stat.h>
#include <sys/syscall.h>
#include <unistd.h>
#include <cctype>
#include <map>
#include <mutex>
#include <string>
#include <unordered_set>
#include <vector>

#include "f2q_dev.cuh"
#include "generic.cuh"
#include "resolve.cuh"
#include "stream.cuh"
#include "tile.cuh"
#include "spec.cuh"

using namespace f2q;

#define F2Q_EXPORT extern "C" __attribute__((visibility("default")))

namespace {

// message of the last failing call that had no context (f2q_create, the helpers): per THREAD, so that feeder threads creating
// engines concurrently never read a string another thread is replacing
thread_local std::string g_create_err;

struct DevBuf {
    void* p = nullptr; size_t n = 0;
    void release() { if (p) cudaFree(p); p = nullptr; n = 0; }
};

// page-locked ring of f2q_submit_file: the file is read / inflated straight into these, the copy engine drains them
struct FileRing {
    static constexpr int N = 3;
    uint8_t* buf[N] = {nullptr, nullptr, nullptr};
    cudaEvent_t done[N] = {nullptr, nullptr, nullptr};
    bool used[N] = {false, false, false};
    size_t bytes = 0;
    int next = 0;
};

}  // namespace

struct f2q_ctx {
    int device = 0;
    cudaStream_t stream = nullptr, copy_stream = nullptr;
    bool own_stream = false;
    int sm_count = 0;
    f2q_config cfg{};
    GenericCfg hG{};
    GenericCfg* dG = nullptr;
    int policy = POLICY_GENERIC;
    int resolver = 0;                 // 0 auto, 1 probe, 2 seed, 3 scan
    // library
    bool lib_set = false;
    uint32_t n_keys = 0;
    LibTables T{};
    std::vector<DevBuf> lib_bufs;
    // results: [counts n_keys | stats 5]
    DevBuf result;
    uint32_t* d_error = nullptr;
    DevState* dS = nullptr;
    uint32_t* d_tickets = nullptr;
    // streaming
    uint64_t carry_cap = 4ull << 20;
    DevBuf carry, status, status_stitch, queue, gqueue, seg_count;
    uint32_t q_cap = 0, g_cap = 0;     // q_cap = total queue entries (n_segs * seg_cap)
    uint32_t seg_cap = 0, n_segs = 0;
    int force_ch = 0, force_halo = 0;
    bool no_flex = false, force_generic = false, flex_big = false;   // options "flex" = 0 / "force_generic"; flex_big: reads longer than 96 (sniffed)
    size_t rec_bytes = 0;              // record length sniffed from the head of the sample (0 = unknown)
    int halo_rows = 6;
    int ch = 7;                        // row chunks of the tile kernel (row = 16*ch bytes), picked per sample from the record length
    bool ch_decided = false;           // per sample for host submits (sniffed from the host bytes: free); a context fed with
    bool ch_from_device = false;       // DEVICE chunks sniffs once (one 4 KiB D2H + sync) and keeps the geometry for later samples
    int64_t opt_queue_entries = 0;
    // staging for host submits
    uint64_t stage_bytes = 64ull << 20;
    int stage_slots = 3;
    std::vector<uint8_t*> d_stage;
    std::vector<cudaEvent_t> ev_copied, ev_free;
    int next_slot = 0;
    // EC
    EcTable E{};
    DevBuf ec_slots, ec_counts, ec_arena, ec_meta;   // meta (32 bytes): [arena_used, n_keys of the arena table, n_keys of the packed table, -]
    uint64_t ec_cap = 0;
    DevBuf ec_pk, ec_compact; uint64_t ec_pk_cap = 0, ec_pk_min = 0;   // packed key table: 16-byte slots; its compacted (tag, count) pairs
    static constexpr int EC_RING = 16;
    struct EcPend { cudaEvent_t ev; unsigned long long* host; uint64_t bound_pk, bound_keys, bound_bytes; };
    std::deque<EcPend> ec_pend;                      // chunks whose fill counters the host has not seen yet, oldest first
    std::vector<cudaEvent_t> ec_events;
    unsigned long long* ec_meta_host = nullptr;      // pinned ring of EC_RING x 4 words
    uint64_t ec_ring_next = 0;
    unsigned long long ec_known[4] = {0, 0, 0, 0};   // newest counters seen: arena bytes, arena keys, packed keys, spec_off
    int flex_warps = 16;                             // option "flex_warps": warps per CTA of the streaming kernel's flex policies
    // GPU inflate of bgzip input (option "gpu_inflate"): two compressed staging buffers, two output buffers, block tables
    bool gpu_inflate = true;                         // bgzip input is inflated on the device (DESIGN.md §5 has the measurements)
    int gpu_inflate_mode = 1;                        // 1 lock-step lanes | 2 free-running threads (cross-check)
    bool gz_attr = false;
    int opt_seed_parts = 0;                          // 0 auto | segments of the seed plan (developer / test option)
    int gpu_inflate_bits = 0;                        // 0 auto | 8 | 9: index bits of the literal/length lookup table (developer option)
    DevBuf gz_comp[2], gz_out[2], gz_tab[2];
    BgzfBlock* gz_tab_host[2] = {nullptr, nullptr};
    cudaEvent_t gz_copied[2] = {nullptr, nullptr}, gz_free[2] = {nullptr, nullptr};
    uint64_t gz_blocks = 0;                          // blocks inflated on the device by the last f2q_submit_file
    FileRing* file_ring = nullptr;                   // page-locked ring of f2q_submit_file (allocated on first use)
    // multi-GPU (NCCL): the communicator this context is a rank of
    void* comm = nullptr; int comm_rank = 0, comm_size = 1; bool comm_owner = false;
    bool ec_merged = false;                          // f2q_ec_merge ran for this sample: the packed table holds every rank's keys,
    std::vector<uint8_t> ec_extra_keys; std::vector<uint64_t> ec_extra_off, ec_extra_cnt;   // ... and these the merged byte-arena keys
    int seed_group = 1;                              // lanes per key of the fast1 seed resolver (auto)
    int64_t memo_entries = -1;                       // option "memo_entries": -1 / 0 off, else a power of two
    DevBuf memo;
    uint64_t memo_counts[2] = {0, 0};                // last finished sample: memo lookups / hits
    int fx_group = 1, fx_group_opt = 0;              // lanes per key of the flex resolver (auto from the seed index / option)
    size_t q_entry = 0;                              // bytes per entry the queue buffer was sized for
    int64_t opt_generic_entries = 0;
    std::vector<uint64_t> ec_drain_off, ec_drain_cnt; std::vector<uint8_t> ec_drain_keys; bool ec_drained = false;
    // one file on several contexts (f2q_submit_file_sharded)
    uint64_t lib_hash = 0;                           // FNV-1a of the library keys: the contexts of one sharded file must agree
    bool shard_head_pending = false;                 // the next device chunk starts mid-file: k_shard_head runs on it first
    bool shard_noguess = false;                      // ... and found no unique record start
    const std::atomic<bool>* shard_abort = nullptr;  // another shard of the same call gave up: stop parsing
    DevBuf shard_head;                               // the head bytes k_shard_head saved (<= carry_bytes)
    int last_shards = 1, last_shard_fallback = 0;    // f2q_get_info "shards" / "shard_fallback"
    // state
    bool in_sample = false, closed = false;
    int sample_failed = F2Q_OK;        // a submit of this sample failed: every later submit / end of the sample reports it again
    int sticky = F2Q_OK;
    std::string err;
    uint64_t launches = 0;
    int tile_blocks[2][8][2] = {{{0}}};
    // speculative streaming kernel (spec.cuh)
    bool debug_waits = false;          // option "debug_waits": the exact kernel counts the cycles spent in each of its waits
    int spec = 1;                      // 0: always the exact look-back kernel
    int spec_warps = 16;               // warps per CTA (one CTA per SM): 12 or 16
    int spec_range_tiles = 0;          // 0 auto | tiles per range
    int spec_ready[4][8][4] = {{{0}}}; // function attributes set for (policy, ch, warps / 4 - 3)
    DevBuf spec_rec, spec_scratch;
    DevBuf synth_guides; size_t synth_guide_bytes = 0;   // guide table of the last f2q_synth_fastq call (K0, bench / tests)
    // [0] tables + result outputs, [1] tables + scratch outputs, in device memory (SlowArgs, generic.cuh); re-uploaded when they change
    DevBuf slow_args;
    SlowArgs slow_host[2];
    bool slow_valid = false;
    bool async_pending = false;        // f2q_end_sample_async results not yet waited for (kernel timings are collected by f2q_sync)
    uint64_t spec_counts[2] = {0, 0};  // last finished sample: chunks committed by the speculation / parsed by the exact kernel
    int hist_used = 0;                 // this sample: launched with the shared-memory histogram, bit 0 the streaming kernel, bit 1 the exact kernel
    int nt = 256;                      // threads (= owned rows) per tile-kernel CTA: 256 for the packed policy (measured 35 % faster),
    bool nt_user = false;              // 128 for the generic per-read code, unless option "tile_threads" says otherwise
    // optional per-kernel timing (option "time_kernels"): event pairs around the tile / resolver / generic launches
    bool time_kernels = false;
    struct Timed { cudaEvent_t a, b; int kind; };
    std::vector<Timed> timed;
    std::vector<cudaEvent_t> event_pool;
    double kernel_ms[4] = {0, 0, 0, 0};
    uint64_t kernel_launches[4] = {0, 0, 0, 0};
};

namespace {

int fail(f2q_ctx* c, int code, const std::string& msg) {
    if (c) { c->err = msg; if (code == F2Q_ECUDA) c->sticky = code; }
    else g_create_err = msg;
    return code;
}

#define CU(ctx, call)                                                                                      \
    do {                                                                                                   \
        cudaError_t e__ = (call);                                                                          \
        if (e__ != cudaSuccess)                                                                            \
            return fail(ctx, F2Q_ECUDA, std::string(#call) + ": " + cudaGetErrorString(e__));              \
    } while (0)

int dev_alloc(f2q_ctx* c, DevBuf& b, size_t n) {
    if (b.n >= n && b.p) return F2Q_OK;
    b.release();
    cudaError_t e = cudaMalloc(&b.p, n ? n : 16);
    if (e != cudaSuccess) return fail(c, e == cudaErrorMemoryAllocation ? F2Q_ENOMEM : F2Q_ECUDA, std::string("cudaMalloc: ") + cudaGetErrorString(e));
    b.n = n ? n : 16;
    return F2Q_OK;
}

// largest failing byte of the fail set built at fast2q.py:1112-1129 (0 = empty set)
int fail_max(int ph) {
    if (ph <= 0) ph = 1;
    int n = std::min(ph - 1, 94);
    return n == 0 ? 0 : 33 + n - 1;
}

ByteSet fail_set(int ph) {
    ByteSet s{{0, 0, 0, 0}};
    int fm = fail_max(ph);
    for (int b = 33; b <= fm; b++) s.w[b >> 6] |= 1ull << (b & 63);
    return s;
}

int make_generic_cfg(const f2q_config* cfg, GenericCfg& G, std::string& why) {
    if (cfg->n_iter < 1 || cfg->n_iter > F2Q_MAX_ITER) { why = "n_iter out of range"; return F2Q_EINVAL; }
    if (cfg->mode != F2Q_MODE_COUNT && cfg->mode != F2Q_MODE_EXTRACT_COUNT) { why = "unknown mode"; return F2Q_EINVAL; }
    memset(&G, 0, sizeof(G));
    DevCfg& d = G.c;
    d.mode = cfg->mode; d.miss = cfg->miss; d.length = cfg->length; d.n_iter = cfg->n_iter;
    d.has_up = cfg->has_up != 0; d.has_down = cfg->has_down != 0; d.miss_up = cfg->miss_up; d.miss_down = cfg->miss_down;
    d.fmax_ph = fail_max(cfg->phred); d.fmax_up = fail_max(cfg->qual_up); d.fmax_down = fail_max(cfg->qual_down);
    for (int i = 0; i < F2Q_MAX_ITER; i++) {
        d.starts[i] = cfg->starts[i];
        d.up_len[i] = cfg->up_len[i]; d.down_len[i] = cfg->down_len[i];
        if (d.up_len[i] < 0 || d.up_len[i] > F2Q_MAX_DELIM || d.down_len[i] < 0 || d.down_len[i] > F2Q_MAX_DELIM) {
            why = "search sequence length out of range"; return F2Q_EINVAL;
        }
        memcpy(d.up[i], cfg->up[i], F2Q_MAX_DELIM); memcpy(d.down[i], cfg->down[i], F2Q_MAX_DELIM);
    }
    G.set_ph = fail_set(cfg->phred); G.set_up = fail_set(cfg->qual_up); G.set_down = fail_set(cfg->qual_down);
    flex_prepare(*cfg, G.flex);                                        // (eligible = 0 when the bit-parallel path cannot run it)
    return F2Q_OK;
}

bool packable(const uint8_t* k, size_t n, uint64_t& key) {
    if (n > 32) return false;
    key = 0;
    for (size_t i = 0; i < n; i++) {
        uint8_t ch = k[i];
        if (ch != 'A' && ch != 'C' && ch != 'G' && ch != 'T') return false;
        key |= (uint64_t)((ch >> 1) & 3) << (2 * i);
    }
    return true;
}

template <class Tv>
int upload(f2q_ctx* c, const std::vector<Tv>& v, const Tv** out) {
    c->lib_bufs.emplace_back();
    DevBuf& b = c->lib_bufs.back();
    int rc = dev_alloc(c, b, std::max<size_t>(v.size(), 1) * sizeof(Tv));
    if (rc) return rc;
    if (!v.empty()) CU(c, cudaMemcpy(b.p, v.data(), v.size() * sizeof(Tv), cudaMemcpyHostToDevice));
    *out = reinterpret_cast<const Tv*>(b.p);
    return F2Q_OK;
}

uint32_t pow2_at_least(uint64_t n) { uint64_t p = 16; while (p < n) p <<= 1; return (uint32_t)p; }

// per-read code of the streaming kernel: fast1 (one fixed window, Counter) | flex (bit-parallel search sequences / several
// windows; Counter needs every library key in the flex table, Extract+Count has its packed key table) | byte-wise generic.
// The exact look-back kernel (stitched records, fallback) runs fast1 or the generic code: results never depend on the path.
void decide_policy(f2q_ctx* c) {
    const f2q_config& g = c->cfg;
    c->policy = POLICY_GENERIC;
    if (g.mode == F2Q_MODE_COUNT && !g.has_up && !g.has_down && g.n_iter == 1 && g.length >= 0 && g.length <= 32) c->policy = POLICY_FAST1;
    else if (c->hG.flex.eligible && !c->no_flex && (g.mode == F2Q_MODE_EXTRACT_COUNT || c->T.fx_slots))
        c->policy = (c->hG.flex.max_k > 1 || c->flex_big) ? POLICY_FLEX_B : POLICY_FLEX_S;
    if (c->force_generic) c->policy = POLICY_GENERIC;
    if (!c->nt_user) c->nt = c->policy == POLICY_FAST1 ? 256 : 128;
}
bool is_flex(const f2q_ctx* c) { return policy_is_flex(c->policy); }
int tile_policy(const f2q_ctx* c) { return c->policy == POLICY_FAST1 ? POLICY_FAST1 : POLICY_GENERIC; }

constexpr uint64_t EC_SUBCHUNK_BYTES = 1ull << 30;
constexpr uint32_t HIST_MAX_KEYS = 8192;     // shared-memory histogram up to this many features (32 KB of u32)

// persistent grid of the tile kernel for (policy, ch, nt): SM count x resident CTAs per SM
template <int POLICY, int CH, int NT>
int tile_grid(f2q_ctx* c, unsigned* grid) {
    const bool hist = (POLICY == POLICY_FAST1) && c->n_keys > 0 && c->n_keys <= HIST_MAX_KEYS;
    const size_t smem = tile_smem_bytes<CH, NT>(hist ? c->n_keys : 0);
    int& blocks_per_sm = c->tile_blocks[POLICY][CH][NT == 256];
    if (blocks_per_sm == 0) {
        CU(c, cudaFuncSetAttribute(k_tile<POLICY, CH, NT>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(tile_smem_bytes<CH, NT>(HIST_MAX_KEYS))));
        CU(c, cudaFuncSetAttribute(k_tile<POLICY, CH, NT>, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared));
        CU(c, cudaOccupancyMaxActiveBlocksPerMultiprocessor(&blocks_per_sm, k_tile<POLICY, CH, NT>, NT + TILE_CTRL_THREADS, smem));
        if (blocks_per_sm < 1) return fail(c, F2Q_EINTERNAL, "tile kernel does not fit on an SM");
        // leave the rest of the 228 KB to L1: the lookup table of a small library then stays L1-resident
        cudaFuncAttributes fa;
        CU(c, cudaFuncGetAttributes(&fa, k_tile<POLICY, CH, NT>));
        const size_t need = (size_t)blocks_per_sm * (smem + fa.sharedSizeBytes + 1024);
        const int pct = (int)std::min<size_t>(100, (need * 100 + 233472 - 1) / 233472);
        CU(c, cudaFuncSetAttribute(k_tile<POLICY, CH, NT>, cudaFuncAttributePreferredSharedMemoryCarveout, pct));
    }
    *grid = (unsigned)c->sm_count * (unsigned)blocks_per_sm;
    return F2Q_OK;
}

template <int POLICY, int CH, int NT>
int launch_tile(f2q_ctx* c, const TileParams& P, Outputs O, uint64_t n_tiles_upper) {
    const bool hist = (POLICY == POLICY_FAST1) && c->n_keys > 0 && c->n_keys <= HIST_MAX_KEYS;
    TileParams p = P; p.hist_smem = hist;
    if (hist) c->hist_used |= 2;
    const size_t smem = tile_smem_bytes<CH, NT>(hist ? c->n_keys : 0);
    unsigned grid = 0;
    int rc = tile_grid<POLICY, CH, NT>(c, &grid); if (rc) return rc;
    if (p.seg_cap == 0) grid = (unsigned)std::max<uint64_t>(1, std::min<uint64_t>(grid, n_tiles_upper));   // main launches keep one segment per CTA
    k_tile<POLICY, CH, NT><<<grid, NT + TILE_CTRL_THREADS, smem, c->stream>>>(p, c->dG, c->T, c->E, O, reinterpret_cast<const SlowArgs*>(c->slow_args.p));
    c->launches++;
    CU(c, cudaGetLastError());
    return F2Q_OK;
}

#define F2Q_DISPATCH(FN, ...)                                                                                     \
    do {                                                                                                          \
        const bool f = tile_policy(c) == POLICY_FAST1;                                                            \
        if (c->nt == 256) {                                                                                       \
            switch (c->ch) {                                                                                      \
                case 3: return f ? FN<POLICY_FAST1, 3, 256>(__VA_ARGS__) : FN<POLICY_GENERIC, 3, 256>(__VA_ARGS__); \
                case 5: return f ? FN<POLICY_FAST1, 5, 256>(__VA_ARGS__) : FN<POLICY_GENERIC, 5, 256>(__VA_ARGS__); \
                default: return f ? FN<POLICY_FAST1, 7, 256>(__VA_ARGS__) : FN<POLICY_GENERIC, 7, 256>(__VA_ARGS__); \
            }                                                                                                     \
        }                                                                                                         \
        switch (c->ch) {                                                                                          \
            case 3: return f ? FN<POLICY_FAST1, 3, 128>(__VA_ARGS__) : FN<POLICY_GENERIC, 3, 128>(__VA_ARGS__);   \
            case 5: return f ? FN<POLICY_FAST1, 5, 128>(__VA_ARGS__) : FN<POLICY_GENERIC, 5, 128>(__VA_ARGS__);   \
            default: return f ? FN<POLICY_FAST1, 7, 128>(__VA_ARGS__) : FN<POLICY_GENERIC, 7, 128>(__VA_ARGS__);  \
        }                                                                                                         \
    } while (0)

int tile_grid_dyn(f2q_ctx* c, unsigned* grid) { F2Q_DISPATCH(tile_grid, c, grid); }
int launch_tile_dyn(f2q_ctx* c, const TileParams& P, Outputs O, uint64_t n_tiles_upper) { F2Q_DISPATCH(launch_tile, c, P, O, n_tiles_upper); }

// ---- speculative streaming kernel: one CTA of W warps per SM ----
constexpr size_t SM_SMEM_BYTES = 233472, SPEC_SMEM_MARGIN = 4096;     // 228 KB per SM; static shared + the per-CTA reservation

template <int POLICY, int CH, int W>
int launch_spec(f2q_ctx* c, const SpecParams& P, Outputs O) {
    SpecParams p = P;
    constexpr bool FLEX = policy_is_flex(POLICY);
    // (flex: the read-ahead rows shrink until the stages fit; reads reaching further finish through the generic queue)
    uint32_t H = p.halo_rows;
    while (FLEX && H > 2 && spec_smem_bytes<POLICY, CH, W>(H, 0) + sizeof(GenericCfg) + SPEC_SMEM_MARGIN > SM_SMEM_BYTES) H--;
    p.halo_rows = H;
    const size_t base_smem = spec_smem_bytes<POLICY, CH, W>(H, 0);
    const bool hist = (POLICY == POLICY_FAST1 || (FLEX && c->cfg.mode == F2Q_MODE_COUNT)) && c->n_keys > 0 &&
                      base_smem + (size_t)c->n_keys * 4 + sizeof(GenericCfg) + SPEC_SMEM_MARGIN <= SM_SMEM_BYTES;
    p.hist_smem = hist;
    const size_t smem = spec_smem_bytes<POLICY, CH, W>(H, hist ? c->n_keys : 0);
    if (smem + sizeof(GenericCfg) + SPEC_SMEM_MARGIN > SM_SMEM_BYTES) return 1;        // does not fit with W warps: the caller retries with fewer
    int& ready = c->spec_ready[POLICY][CH][W / 4 - 3];
    if (!ready) {
        CU(c, cudaFuncSetAttribute(k_spec<POLICY, CH, W>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(SM_SMEM_BYTES - sizeof(GenericCfg) - SPEC_SMEM_MARGIN)));
        ready = 1;
    }
    if (hist) c->hist_used |= 1;
    k_spec<POLICY, CH, W><<<(unsigned)c->sm_count, W * 32, smem, c->stream>>>(p, c->dG, c->T, c->E, O, reinterpret_cast<const SlowArgs*>(c->slow_args.p) + 1, c->hG.flex);
    c->launches++;
    CU(c, cudaGetLastError());
    return F2Q_OK;
}

int launch_spec_dyn(f2q_ctx* c, const SpecParams& P, Outputs O) {
    int rc12;
    if (is_flex(c)) {
        // 16 warps per CTA (128 registers per thread; measured 5-10 % faster than 12 warps with 168), 12 when the stages do not fit
        const int ch = c->ch == 3 ? 5 : c->ch;
        int rc16 = 1;
        if (c->policy == POLICY_FLEX_S) {
            if (c->flex_warps == 16) rc16 = ch == 5 ? launch_spec<POLICY_FLEX_S, 5, 16>(c, P, O) : launch_spec<POLICY_FLEX_S, 7, 16>(c, P, O);
            if (rc16 != 1) return rc16;
            rc12 = ch == 5 ? launch_spec<POLICY_FLEX_S, 5, 12>(c, P, O) : launch_spec<POLICY_FLEX_S, 7, 12>(c, P, O);
        } else rc12 = ch == 5 ? launch_spec<POLICY_FLEX_B, 5, 12>(c, P, O) : launch_spec<POLICY_FLEX_B, 7, 12>(c, P, O);
        return rc12 == 1 ? fail(c, F2Q_EINTERNAL, "speculative kernel does not fit on an SM") : rc12;
    }
    const bool f = c->policy == POLICY_FAST1;
#define F2Q_SPEC_CASE(CHV)                                                                                         \
    case CHV:                                                                                                      \
        if (c->spec_warps >= 16) {                                                                                 \
            const int rc16 = f ? launch_spec<POLICY_FAST1, CHV, 16>(c, P, O) : launch_spec<POLICY_GENERIC, CHV, 16>(c, P, O); \
            if (rc16 != 1) return rc16;                                                                            \
        }                                                                                                          \
        rc12 = f ? launch_spec<POLICY_FAST1, CHV, 12>(c, P, O) : launch_spec<POLICY_GENERIC, CHV, 12>(c, P, O);      \
        return rc12 == 1 ? fail(c, F2Q_EINTERNAL, "speculative kernel does not fit on an SM") : rc12;
    if (f && c->spec_warps > 16) {
        // 20 / 24 warps with a two-stage ring (the fast1 policy only)
        int rcw = 1;
        if (c->spec_warps == 24) rcw = c->ch == 3 ? launch_spec<POLICY_FAST1, 3, 24>(c, P, O) : c->ch == 5 ? launch_spec<POLICY_FAST1, 5, 24>(c, P, O) : launch_spec<POLICY_FAST1, 7, 24>(c, P, O);
        if (rcw == 1) rcw = c->ch == 3 ? launch_spec<POLICY_FAST1, 3, 20>(c, P, O) : c->ch == 5 ? launch_spec<POLICY_FAST1, 5, 20>(c, P, O) : launch_spec<POLICY_FAST1, 7, 20>(c, P, O);
        if (rcw != 1) return rcw;
    }
    switch (c->ch) {
        F2Q_SPEC_CASE(3)
        F2Q_SPEC_CASE(5)
        default:
        F2Q_SPEC_CASE(7)
    }
#undef F2Q_SPEC_CASE
}

// record length of ordinary FASTQ from the first bytes of a sample -> row size of the tile kernel (16*ch just below it)
void decide_ch(f2q_ctx* c, const uint8_t* head, size_t n) {
    size_t nl = 0, pos = 0;
    for (size_t i = 0; i < n && nl < 8; i++) if (head[i] == '\n') { nl++; pos = i + 1; }
    c->ch = 7;
    size_t rec = 0;
    if (nl == 8) { rec = pos / 2; c->ch = rec >= 112 ? 7 : rec >= 80 ? 5 : 3; }
    c->rec_bytes = rec;
    const bool big = rec > 2 * 96 + 24;                                // reads longer than the 96-position planes
    if (big != c->flex_big) { c->flex_big = big; decide_policy(c); }
    if (c->force_ch) c->ch = c->force_ch;
    // read-ahead rows at the end of each tile: one and a half records' worth (reads that need more finish in global memory)
    const int S = 16 * c->ch, halo_max = c->nt / 2;
    c->halo_rows = rec ? (int)std::min<size_t>(halo_max, std::max<size_t>(2, (rec + rec / 2 + S - 1) / S + 1)) : std::min(halo_max, (1024 + S - 1) / S + 1);
    if (c->force_halo) c->halo_rows = std::min(halo_max, c->force_halo);
    c->ch_decided = true;
}

cudaEvent_t timing_begin(f2q_ctx* c) {
    if (!c->time_kernels) return nullptr;
    cudaEvent_t e;
    if (!c->event_pool.empty()) { e = c->event_pool.back(); c->event_pool.pop_back(); }
    else if (cudaEventCreate(&e) != cudaSuccess) return nullptr;
    cudaEventRecord(e, c->stream);
    return e;
}
void timing_end(f2q_ctx* c, cudaEvent_t a, int kind) {
    if (!a) return;
    cudaEvent_t e;
    if (!c->event_pool.empty()) { e = c->event_pool.back(); c->event_pool.pop_back(); }
    else if (cudaEventCreate(&e) != cudaSuccess) { c->event_pool.push_back(a); return; }
    cudaEventRecord(e, c->stream);
    c->timed.push_back({a, e, kind});
}
void timing_collect(f2q_ctx* c) {
    for (int k = 0; k < 4; k++) { c->kernel_ms[k] = 0; c->kernel_launches[k] = 0; }
    for (auto& t : c->timed) {
        float ms = 0;
        if (cudaEventElapsedTime(&ms, t.a, t.b) == cudaSuccess) { c->kernel_ms[t.kind] += ms; c->kernel_launches[t.kind]++; }
        c->event_pool.push_back(t.a); c->event_pool.push_back(t.b);
    }
    c->timed.clear();
    cudaGetLastError();
}

Outputs outputs_of(f2q_ctx* c) {
    Outputs O;
    O.counts = reinterpret_cast<unsigned long long*>(c->result.p);
    O.stats = O.counts + c->n_keys;
    O.error = c->d_error;
    return O;
}

// ---- Extract+Count tables: sized WITHOUT a host round trip per chunk ----------------------------------------------
// Two device tables (generic.cuh: EcTable): the packed table (single ACGT pieces of <= 29 symbols, 16-byte slots) and the
// byte-arena table (everything else).  The host never waits for the device to learn how full they are: after every chunk
// the fill counters are copied, stream-ordered, into a pinned slot; before a chunk the host adds to the newest counters it
// has SEEN an upper bound of what every chunk still in flight (and the new one) can insert.  Only when that bound does not
// fit does it wait — first for older chunks' counters (the device still has work queued), and, when nothing is in
// flight and it still does not fit, for a stream sync and a rehash ON THE DEVICE into a table twice the size.
void ec_bind(f2q_ctx* c) {
    c->E.pk_slots = reinterpret_cast<unsigned long long*>(c->ec_pk.p);
    c->E.pk_mask = c->ec_pk_cap ? c->ec_pk_cap - 1 : 0;
    c->E.slots = reinterpret_cast<unsigned long long*>(c->ec_slots.p);
    c->E.counts = reinterpret_cast<unsigned long long*>(c->ec_counts.p);
    c->E.mask = c->ec_cap ? c->ec_cap - 1 : 0;
    c->E.arena = reinterpret_cast<uint8_t*>(c->ec_arena.p);
    c->E.arena_cap = c->ec_arena.n;
    c->E.arena_used = reinterpret_cast<unsigned long long*>(c->ec_meta.p);
    c->E.n_keys = c->E.arena_used + 1;
    c->E.pk_n = c->E.arena_used + 2;
}

void ec_fold_done(f2q_ctx* c, bool wait_oldest) {
    while (!c->ec_pend.empty()) {
        f2q_ctx::EcPend& p = c->ec_pend.front();
        if (!p.ev) { c->ec_pend.pop_front(); continue; }               // (a chunk that failed before its counters were queued)
        if (wait_oldest) { cudaEventSynchronize(p.ev); wait_oldest = false; }
        else if (cudaEventQuery(p.ev) != cudaSuccess) { cudaGetLastError(); break; }
        for (int k = 0; k < 3; k++) c->ec_known[k] = p.host[k];
        c->ec_known[3] = p.host[3] & 0xFFFFFFFFull;
        c->ec_events.push_back(p.ev);
        c->ec_pend.pop_front();
    }
}

int ec_reserve(f2q_ctx* c, uint64_t bound_pk, uint64_t bound_keys, uint64_t bound_bytes) {
    int rc;
    if (!c->ec_meta.p) {
        if ((rc = dev_alloc(c, c->ec_meta, 32))) return rc;
        CU(c, cudaMemsetAsync(c->ec_meta.p, 0, 32, c->stream));
        CU(c, cudaHostAlloc(reinterpret_cast<void**>(&c->ec_meta_host), 4 * 8 * f2q_ctx::EC_RING, cudaHostAllocDefault));
        memset(c->ec_meta_host, 0, 4 * 8 * f2q_ctx::EC_RING);
    }
    for (;;) {
        ec_fold_done(c, false);
        uint64_t pk = c->ec_known[2] + bound_pk, keys = c->ec_known[1] + bound_keys, bytes = c->ec_known[0] + bound_bytes;
        for (auto& p : c->ec_pend) { pk += p.bound_pk; keys += p.bound_keys; bytes += p.bound_bytes; }
        const bool fits = 2 * pk + 1024 <= c->ec_pk_cap && 2 * keys + 1024 <= c->ec_cap && bytes + 1024 <= c->ec_arena.n;
        if (fits && (int)c->ec_pend.size() < f2q_ctx::EC_RING - 1) break;
        if (!c->ec_pend.empty()) { ec_fold_done(c, true); continue; }        // wait for the OLDEST chunk's counters only
        // nothing in flight: the counters are exact.  Grow what does not fit (geometric, so this is rare)
        CU(c, cudaStreamSynchronize(c->stream));
        if (2 * pk + 1024 > c->ec_pk_cap) {
            uint64_t cap = std::max<uint64_t>(1 << 16, c->ec_pk_min);
            while (cap < 4 * pk + 2048) cap <<= 1;
            DevBuf nb;
            cudaError_t e = cudaMalloc(&nb.p, cap * 16);
            if (e != cudaSuccess) { cudaGetLastError(); return fail(c, F2Q_ENOMEM, "Extract+Count packed key table: out of device memory (" + std::to_string(cap * 16) + " bytes)"); }
            nb.n = cap * 16;
            CU(c, cudaMemsetAsync(nb.p, 0, cap * 16, c->stream));
            const uint64_t old_cap = c->ec_pk_cap;
            DevBuf old = c->ec_pk;
            c->ec_pk = nb; c->ec_pk_cap = cap;
            ec_bind(c);
            if (old_cap && c->ec_known[2]) {
                k_ec_rehash<<<(unsigned)std::min<uint64_t>((old_cap + 255) / 256, (uint64_t)c->sm_count * 32), 256, 0, c->stream>>>(
                    reinterpret_cast<const unsigned long long*>(old.p), old_cap, c->E, outputs_of(c));
                c->launches++;
                CU(c, cudaStreamSynchronize(c->stream));
            }
            old.release();
        }
        if (bytes + 1024 > c->ec_arena.n) {
            DevBuf nb;
            const size_t sz = std::max<size_t>(bytes + 1024, c->ec_arena.n * 2);
            cudaError_t e = cudaMalloc(&nb.p, sz);
            if (e != cudaSuccess) { cudaGetLastError(); return fail(c, F2Q_ENOMEM, "Extract+Count key arena: out of device memory"); }
            nb.n = sz;
            if (c->ec_arena.p && c->ec_known[0]) CU(c, cudaMemcpy(nb.p, c->ec_arena.p, c->ec_known[0], cudaMemcpyDeviceToDevice));
            c->ec_arena.release(); c->ec_arena = nb;
        }
        if (2 * keys + 1024 > c->ec_cap) {
            uint64_t cap = 1 << 14; while (cap < 4 * keys + 2048) cap <<= 1;
            // the byte-arena table holds the rare keys (other symbols than ACGT, long or multi-piece keys): it is small, and
            // its growth rehashes through the host
            std::vector<unsigned long long> hs, hc;
            std::vector<uint8_t> ar;
            const uint64_t old = c->ec_cap, used = c->ec_known[0];
            if (old && c->ec_known[1]) {
                hs.resize(old); hc.resize(old); ar.resize(used + 1);
                CU(c, cudaMemcpy(hs.data(), c->ec_slots.p, old * 8, cudaMemcpyDeviceToHost));
                CU(c, cudaMemcpy(hc.data(), c->ec_counts.p, old * 8, cudaMemcpyDeviceToHost));
                if (used) CU(c, cudaMemcpy(ar.data(), c->ec_arena.p, used, cudaMemcpyDeviceToHost));
            }
            c->ec_slots.release(); c->ec_counts.release();
            if ((rc = dev_alloc(c, c->ec_slots, cap * 8))) return rc;
            if ((rc = dev_alloc(c, c->ec_counts, cap * 8))) return rc;
            if (hs.empty()) {
                CU(c, cudaMemsetAsync(c->ec_slots.p, 0, cap * 8, c->stream));
                CU(c, cudaMemsetAsync(c->ec_counts.p, 0, cap * 8, c->stream));
            } else {
                std::vector<unsigned long long> ns(cap, 0), nc(cap, 0);
                for (uint64_t i = 0; i < old; i++) {
                    if (!hs[i]) continue;
                    const uint64_t off = (hs[i] - 1) >> 24, len = (hs[i] - 1) & 0xFFFFFF;
                    uint32_t h = FNV_INIT;
                    for (uint64_t k = 0; k < len; k++) h = fnv_step(h, ar[off + k]);
                    uint64_t j = (uint64_t)fnv_final(h) * 0x9E3779B1ull; j = (j ^ (j >> 29)) & (cap - 1);
                    while (ns[j]) j = (j + 1) & (cap - 1);
                    ns[j] = hs[i]; nc[j] = hc[i];
                }
                CU(c, cudaMemcpy(c->ec_slots.p, ns.data(), cap * 8, cudaMemcpyHostToDevice));
                CU(c, cudaMemcpy(c->ec_counts.p, nc.data(), cap * 8, cudaMemcpyHostToDevice));
            }
            c->ec_cap = cap;
        }
        ec_bind(c);
    }
    ec_bind(c);
    // this chunk's bound stays pending until its counters have been seen (ec_after_chunk records the copy)
    f2q_ctx::EcPend p{};
    p.bound_pk = bound_pk; p.bound_keys = bound_keys; p.bound_bytes = bound_bytes; p.ev = nullptr; p.host = nullptr;
    c->ec_pend.push_back(p);
    return F2Q_OK;
}

// after the chunk's kernels: copy the fill counters (and the sticky "speculation is off" flag) to the chunk's pinned slot
int ec_after_chunk(f2q_ctx* c) {
    f2q_ctx::EcPend& p = c->ec_pend.back();
    p.host = c->ec_meta_host + 4 * (c->ec_ring_next++ % f2q_ctx::EC_RING);
    if (!c->ec_events.empty()) { p.ev = c->ec_events.back(); c->ec_events.pop_back(); }
    else CU(c, cudaEventCreateWithFlags(&p.ev, cudaEventDisableTiming));
    CU(c, cudaMemcpyAsync(p.host, c->ec_meta.p, 24, cudaMemcpyDeviceToHost, c->stream));
    CU(c, cudaMemcpyAsync(p.host + 3, &c->dS->spec_off, 4, cudaMemcpyDeviceToHost, c->stream));
    CU(c, cudaEventRecord(p.ev, c->stream));
    return F2Q_OK;
}

// enqueue everything for one chunk that already sits in device memory at dptr[0, n)
int process_device_chunk(f2q_ctx* c, const uint8_t* dptr, uint64_t n, int is_last) {
    int rc;
    if (c->shard_abort && c->shard_abort->load()) return fail(c, F2Q_EINVAL, "another shard of this file found no record start");
    if (c->shard_head_pending && n) {
        // first chunk of a shard that starts mid-file: guess its first record start (one round trip per shard), keep the
        // head for the stitch and parse from the guess with line phase 0
        c->shard_head_pending = false;
        if ((rc = dev_alloc(c, c->shard_head, c->carry_cap + 256))) return rc;
        k_shard_head<<<1, PREP_THREADS, 0, c->stream>>>(c->dS, dptr, n, reinterpret_cast<uint8_t*>(c->shard_head.p), c->carry_cap);
        c->launches++;
        CU(c, cudaGetLastError());
        unsigned long long h = 0; uint32_t ok = 0;
        CU(c, cudaMemcpyAsync(&h, &c->dS->head_len, 8, cudaMemcpyDeviceToHost, c->stream));
        CU(c, cudaMemcpyAsync(&ok, &c->dS->head_ok, 4, cudaMemcpyDeviceToHost, c->stream));
        CU(c, cudaStreamSynchronize(c->stream));
        if (!ok) { c->shard_noguess = true; return fail(c, F2Q_EINVAL, "no unique record start at the head of a shard"); }
        dptr += h; n -= h;                                              // (n > h: the guess needs two whole records behind it)
    }
    const uint64_t addr = reinterpret_cast<uint64_t>(dptr);
    const uint64_t delta = n ? (addr & 127ull) : 0;
    const uint8_t* base = n ? reinterpret_cast<const uint8_t*>(addr - delta) : reinterpret_cast<const uint8_t*>(c->carry.p);
    if (!c->ch_decided) {
        // device chunks: sniff the record length (4 KiB of the first chunk) to size the tile rows — ONCE per context, so that
        // back-to-back samples have no host round trip (the geometry only affects speed, never results)
        uint8_t head[4096];
        const size_t hn = (size_t)std::min<uint64_t>(n, sizeof(head));
        if (hn) { CU(c, cudaMemcpyAsync(head, dptr, hn, cudaMemcpyDeviceToHost, c->stream)); CU(c, cudaStreamSynchronize(c->stream)); }
        decide_ch(c, head, hn);
        c->ch_from_device = hn != 0;
    }
    const bool flex = is_flex(c), ec = c->cfg.mode == F2Q_MODE_EXTRACT_COUNT;
    const uint64_t own_bytes = (uint64_t)(c->nt - c->halo_rows) * 16 * c->ch;
    const uint64_t n_tiles = (delta + n) / own_bytes + 2;
    const uint64_t stitch_tiles = c->carry_cap / (64 * 16 * 3) + 2;
    if ((rc = dev_alloc(c, c->status, n_tiles + 64))) return rc;
    unsigned grid = 0;
    if ((rc = tile_grid_dyn(c, &grid))) return rc;
    // the speculative streaming kernel runs first: Counter mode always (its results can be dropped), Extract+Count on the
    // flex path (its inserts go through a log that is committed only when the speculation verified)
    const bool spec_seen_off = ec && c->ec_known[3] != 0;                      // (the device told us: this sample fell back to the exact kernel)
    const bool use_spec = c->spec && n && (!ec || flex) && !spec_seen_off;
    const int spec_ch = flex && c->ch == 3 ? 5 : c->ch;
    const uint64_t spec_own = 512ull * spec_ch;
    uint64_t spec_range_tiles = 0, n_spec_rec = 0;
    if (flex) grid = (unsigned)c->sm_count;                            // (the exact kernel runs the generic code: no queue segments of its own)
    if (use_spec) {
        grid = std::max<unsigned>(grid, (unsigned)c->sm_count);        // one queue segment per CTA of either kernel
        const uint64_t tiles = (delta + n) / spec_own + 1, streams = (uint64_t)c->sm_count * (flex ? c->flex_warps : c->spec_warps);
        spec_range_tiles = c->spec_range_tiles > 0 ? (uint64_t)c->spec_range_tiles : std::min<uint64_t>(64, std::max<uint64_t>(8, tiles / (streams * 4)));
        const uint64_t n_rec = (delta + n) / (spec_range_tiles * spec_own) + 2;
        if ((rc = dev_alloc(c, c->spec_rec, n_rec))) return rc;
        n_spec_rec = n_rec;
    }
    // queues sized for the chunk.  fast1: one entry per 64 bytes covers every non-exact read of ordinary FASTQ; flex Counter
    // the same; flex Extract+Count: the insert log takes EVERY read's key (1.5 x the reads the sniffed record length
    // predicts).  Anything beyond a queue's capacity is handled in place or by the generic queue, so capacity never changes results
    const size_t entry = flex ? (ec ? 8 : sizeof(FlexQ)) : sizeof(QEntry);
    uint64_t want_q = c->opt_queue_entries > 0 ? (uint64_t)c->opt_queue_entries : std::max<uint64_t>(1 << 16, n / 64 + 1024);
    if (flex && ec && c->opt_queue_entries <= 0) want_q = std::max<uint64_t>(1 << 16, (c->rec_bytes ? 3 * n / (2 * c->rec_bytes) : n / 48) + 4096);
    want_q = std::min<uint64_t>(want_q, 0x7FFFFFFFull);
    if (c->policy == POLICY_GENERIC) want_q = grid;
    if (flex) want_q = ((want_q + FX_BLOCK - 1) / FX_BLOCK + (c->opt_queue_entries > 0 ? 0 : (uint64_t)c->sm_count * 16)) * FX_BLOCK;   // + one open block per warp
    if (want_q > c->q_cap || grid != c->n_segs || entry != c->q_entry) {
        want_q = std::max<uint64_t>(want_q, c->q_cap);
        if ((rc = dev_alloc(c, c->queue, want_q * entry))) return rc;
        if ((rc = dev_alloc(c, c->seg_count, (size_t)grid * 4))) return rc;
        c->q_cap = (uint32_t)want_q; c->n_segs = grid; c->seg_cap = (uint32_t)(want_q / grid); c->q_entry = entry;
    }
    uint64_t want_g = c->policy == POLICY_GENERIC ? 16 : std::max<uint64_t>(1 << 14, want_q / 8);
    if (c->opt_generic_entries > 0) want_g = (uint64_t)c->opt_generic_entries;
    if (want_g > c->g_cap || c->opt_generic_entries > 0) { if ((rc = dev_alloc(c, c->gqueue, want_g * sizeof(GEntry)))) return rc; c->g_cap = (uint32_t)want_g; }
    if (ec) {
        const uint64_t worst = (n + c->carry_cap) / 4 + 16, worst_bytes = (uint64_t)c->cfg.n_iter * (n + c->carry_cap) + 64;
        if (use_spec) {
            // the streaming kernel can insert at most its log + its generic queue; the stitched record adds one
            const uint64_t gq = (uint64_t)c->g_cap + 4;
            rc = ec_reserve(c, (uint64_t)c->q_cap + gq, gq, std::min<uint64_t>(worst_bytes, gq * 1024ull * (uint64_t)c->cfg.n_iter));
        } else if (n == 0) rc = ec_reserve(c, 4, 4, (uint64_t)c->cfg.n_iter * c->carry_cap + 64);     // only the carried last record is left
        else rc = ec_reserve(c, worst, worst, worst_bytes);             // exact kernel: every record could be 4 bytes and every key new
        if (rc) return rc;
    }

    // (zeroing: the big look-back status array only when the exact kernel really parses the chunk — behind a speculation
    // k_spec_verify clears it on failure; the small per-chunk arrays inside k_prepare)
    if (!use_spec) CU(c, cudaMemsetAsync(c->status.p, 0, n_tiles + 64, c->stream));
    PrepClear Z{reinterpret_cast<uint8_t*>(c->status_stitch.p), (uint32_t)(stitch_tiles + 64), reinterpret_cast<uint8_t*>(c->spec_rec.p), (uint32_t)n_spec_rec,
                reinterpret_cast<uint32_t*>(c->seg_count.p), c->n_segs};
    k_prepare<<<1, PREP_THREADS, 0, c->stream>>>(c->dS, base, delta, n, is_last ? 1u : 0u, reinterpret_cast<uint8_t*>(c->carry.p),
                                                 c->carry_cap, c->d_tickets, c->q_cap, c->g_cap, Z);
    c->launches++;
    Outputs O = outputs_of(c);
    {
        // the global-memory copy of the tables and outputs that the non-inlined device functions read
        SlowArgs now[2];
        memset(now, 0, sizeof(now));
        now[0].T = c->T; now[0].E = c->E; now[0].O = O;
        now[1] = now[0];
        if (c->spec_scratch.p) { now[1].O.counts = reinterpret_cast<unsigned long long*>(c->spec_scratch.p); now[1].O.stats = now[1].O.counts + c->n_keys; }
        if ((rc = dev_alloc(c, c->slow_args, sizeof(now)))) return rc;
        if (!c->slow_valid || memcmp(now, c->slow_host, sizeof(now)) != 0) {
            memcpy(c->slow_host, now, sizeof(now));
            CU(c, cudaMemcpyAsync(c->slow_args.p, c->slow_host, sizeof(now), cudaMemcpyHostToDevice, c->stream));
            c->slow_valid = true;
        }
    }
    TileParams P{};
    P.S = c->dS; P.queue = reinterpret_cast<QEntry*>(c->queue.p); P.gqueue = reinterpret_cast<GEntry*>(c->gqueue.p);
    P.halo_rows = (uint32_t)c->halo_rows;
    P.debug = c->debug_waits ? 1u : 0u;
    P.seg_count = reinterpret_cast<uint32_t*>(c->seg_count.p);
    // 1. the chunk itself: speculative streaming kernel -> verify -> commit or drop; then the exact kernel, which returns at
    //    once when the speculation held
    if (use_spec) {
        SpecParams Q{};
        Q.buf = base; Q.S = c->dS; Q.ticket = c->d_tickets + 2; Q.rec = reinterpret_cast<uint8_t*>(c->spec_rec.p);
        Q.range_bytes = spec_range_tiles * spec_own;
        Q.queue = P.queue; Q.seg_count = P.seg_count; Q.seg_cap = flex ? c->q_cap : c->policy != POLICY_GENERIC ? c->seg_cap : 0; Q.gqueue = P.gqueue;
        Q.halo_rows = (uint32_t)std::min<int>(c->halo_rows, (int)SPEC_MAX_HALO);
        Outputs O2 = O;
        O2.counts = reinterpret_cast<unsigned long long*>(c->spec_scratch.p); O2.stats = O2.counts + c->n_keys;
        cudaEvent_t t0 = timing_begin(c);
        rc = launch_spec_dyn(c, Q, O2);
        timing_end(c, t0, 0);
        if (rc) return rc;
        cudaEvent_t t3 = timing_begin(c);
        k_spec_verify<<<1, SPEC_VERIFY_THREADS, 0, c->stream>>>(c->dS, Q.rec, Q.range_bytes, (uint32_t)spec_own, P.seg_count, c->n_segs,
                                                                reinterpret_cast<uint8_t*>(c->status.p), n_tiles + 64);
        const uint64_t nres = (uint64_t)c->n_keys + 5;
        k_spec_merge<<<(unsigned)std::min<uint64_t>((nres + 255) / 256, (uint64_t)c->sm_count * 8), 256, 0, c->stream>>>(c->dS, O2.counts, O.counts, nres);
        c->launches += 2;
        timing_end(c, t3, 3);
        if (flex && ec) {
            // the verified chunk's insert log -> the packed key table
            cudaEvent_t t4 = timing_begin(c);
            k_ec_commit<<<(unsigned)c->sm_count * 16, 256, 0, c->stream>>>(c->dS, c->E, O, reinterpret_cast<const unsigned long long*>(c->queue.p), c->q_cap);
            c->launches++;
            timing_end(c, t4, 1);
        }
    }
    if (n) {
        P.buf = base; P.status = reinterpret_cast<uint8_t*>(c->status.p); P.ticket = c->d_tickets + 1; P.stitch = 0;
        P.seg_cap = c->policy == POLICY_FAST1 ? c->seg_cap : 0;
        P.skip_if_spec_ok = use_spec ? 1u : 0u;
        cudaEvent_t t0 = timing_begin(c);
        rc = launch_tile_dyn(c, P, O, n_tiles);
        timing_end(c, t0, use_spec ? 3 : 0);
        if (rc) return rc;
        P.skip_if_spec_ok = 0;
    }
    // 2. the record stitched from the carried tail and the head of this chunk (lives in the carry buffer)
    P.buf = reinterpret_cast<const uint8_t*>(c->carry.p); P.status = reinterpret_cast<uint8_t*>(c->status_stitch.p);
    P.ticket = c->d_tickets; P.stitch = 1; P.seg_cap = 0;
    if ((rc = launch_tile_dyn(c, P, O, 4))) return rc;
    // 3. deferred work
    if (c->policy == POLICY_FAST1) {
        if (c->cfg.miss > 0) {
            int res = c->resolver ? c->resolver : 2;          // auto: the pigeonhole seed index is the cheapest exact method
            if (res == 1 && c->cfg.miss != 1) res = 2;
            if (res == 2 && c->cfg.miss > 32) res = 3;
            cudaEvent_t t1 = timing_begin(c);
            if (res == 1) k_resolve_probe<<<c->n_segs, 256, 0, c->stream>>>(c->T, P.queue, P.seg_count, c->seg_cap, c->n_segs, O.counts, O.stats);
            else if (res == 2) {
                // pigeonhole seed index; lanes per key from the mean bucket size (option "resolve_group"); the memo sits in front
                const int G = c->fx_group_opt ? c->fx_group_opt : c->seed_group;
                unsigned long long* ms = &c->dS->memo_lookups;
                const dim3 rg(c->n_segs, 8);
                const bool classic = c->T.seed_ncombo == 0;              // (one-segment seeds for many mismatches: the thread kernel only)
                if (classic) k_resolve_seed<<<rg, 256, 0, c->stream>>>(c->T, c->cfg.miss, P.queue, P.seg_count, c->seg_cap, c->n_segs, O.counts, O.stats);
                else if (G == 32) k_resolve_seed_g<32><<<rg, 256, 0, c->stream>>>(c->T, c->cfg.miss, P.queue, P.seg_count, c->seg_cap, c->n_segs, O.counts, O.stats, ms);
                else if (G == 8) k_resolve_seed_g<8><<<rg, 256, 0, c->stream>>>(c->T, c->cfg.miss, P.queue, P.seg_count, c->seg_cap, c->n_segs, O.counts, O.stats, ms);
                else if (c->T.memo) k_resolve_seed_g<1><<<rg, 256, 0, c->stream>>>(c->T, c->cfg.miss, P.queue, P.seg_count, c->seg_cap, c->n_segs, O.counts, O.stats, ms);
                else k_resolve_seed<<<rg, 256, 0, c->stream>>>(c->T, c->cfg.miss, P.queue, P.seg_count, c->seg_cap, c->n_segs, O.counts, O.stats);
            }
            else k_resolve_scan<<<c->n_segs, SCAN_THREADS, 0, c->stream>>>(c->T, c->cfg.miss, P.queue, P.seg_count, c->seg_cap, c->n_segs, O.counts, O.stats);
            timing_end(c, t1, 1);
            c->launches++;
        }
    } else if (flex && !ec && c->cfg.miss > 0 && use_spec) {
        // (a chunk the exact kernel re-parsed has empty segments: k_spec_verify zeroed them)
        cudaEvent_t t1 = timing_begin(c);
        const FlexQ* fq = reinterpret_cast<const FlexQ*>(c->queue.p);
        const int G = c->fx_group_opt ? c->fx_group_opt : c->fx_group;
        const unsigned rg = (unsigned)c->sm_count * 8;
        if (G == 32) k_resolve_flex<32><<<rg, 256, 0, c->stream>>>(c->T, c->cfg.miss, c->dS, fq, c->q_cap, O.counts, O.stats, &c->dS->memo_lookups);
        else if (G == 8) k_resolve_flex<8><<<rg, 256, 0, c->stream>>>(c->T, c->cfg.miss, c->dS, fq, c->q_cap, O.counts, O.stats, &c->dS->memo_lookups);
        else k_resolve_flex<1><<<rg, 256, 0, c->stream>>>(c->T, c->cfg.miss, c->dS, fq, c->q_cap, O.counts, O.stats, &c->dS->memo_lookups);
        timing_end(c, t1, 1);
        c->launches++;
    }
    if (c->policy != POLICY_GENERIC) {
        cudaEvent_t t2 = timing_begin(c);
        k_generic_queue<<<(unsigned)c->sm_count, 128, 0, c->stream>>>(c->dG, reinterpret_cast<const SlowArgs*>(c->slow_args.p), P.gqueue, c->dS);
        timing_end(c, t2, 2);
        c->launches++;
    }
    // 4. carry the new partial record
    k_carry<<<1, PREP_THREADS, 0, c->stream>>>(c->dS, base, reinterpret_cast<uint8_t*>(c->carry.p), c->carry_cap);
    c->launches++;
    CU(c, cudaGetLastError());
    if (ec && (rc = ec_after_chunk(c))) return rc;
    if (is_last) c->closed = true;
    return F2Q_OK;
}

int ensure_staging(f2q_ctx* c) {
    if (!c->d_stage.empty()) return F2Q_OK;
    CU(c, cudaStreamCreateWithFlags(&c->copy_stream, cudaStreamNonBlocking));
    for (int i = 0; i < c->stage_slots; i++) {
        uint8_t* p = nullptr;
        cudaError_t e = cudaMalloc(&p, c->stage_bytes + 256);
        if (e != cudaSuccess) return fail(c, F2Q_ENOMEM, "staging slot: out of device memory");
        c->d_stage.push_back(p);
        cudaEvent_t a, b;
        CU(c, cudaEventCreateWithFlags(&a, cudaEventDisableTiming));
        CU(c, cudaEventCreateWithFlags(&b, cudaEventDisableTiming));
        c->ev_copied.push_back(a); c->ev_free.push_back(b);
    }
    return F2Q_OK;
}

int check_ctx(f2q_ctx* c) {
    if (!c) return F2Q_EINVAL;
    if (c->sticky) return c->sticky;
    cudaError_t e = cudaSetDevice(c->device);
    if (e != cudaSuccess) return fail(c, F2Q_ECUDA, std::string("cudaSetDevice: ") + cudaGetErrorString(e));
    return F2Q_OK;
}

}  // namespace

// ---------------------------------------------------------------------------------------------------
F2Q_EXPORT int f2q_abi_version(void) { return F2Q_ABI_VERSION; }

F2Q_EXPORT int f2q_device_count(void) {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) { cudaGetLastError(); return 0; }
    int ok = 0;
    for (int d = 0; d < n; d++) {
        int major = 0;
        if (cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, d) == cudaSuccess && major == 10) ok++;
    }
    return ok;
}

F2Q_EXPORT const char* f2q_last_error(const f2q_ctx* ctx) {
    if (ctx) return ctx->err.c_str();
    return g_create_err.c_str();
}

F2Q_EXPORT int f2q_create(const f2q_config* cfg, int device, void* stream, f2q_ctx** out) {
    if (!cfg || !out) return fail(nullptr, F2Q_EINVAL, "null argument");
    *out = nullptr;
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) { cudaGetLastError(); return fail(nullptr, F2Q_ENODEVICE, "no CUDA device: libf2q has no CPU path"); }
    if (device < 0 || device >= ndev) return fail(nullptr, F2Q_EINVAL, "device index out of range");
    int major = 0;
    cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, device);
    if (major != 10) return fail(nullptr, F2Q_ENODEVICE, "device is not compute capability 10.x (B200, sm_100a)");
    if (cfg->has_up && cfg->has_down) {
        // counts are checked by the host layer (fast2q.py:553-556); here both lists have n_iter entries
    }
    std::string why;
    GenericCfg G;
    int rc = make_generic_cfg(cfg, G, why);
    if (rc) return fail(nullptr, rc, why);
    f2q_ctx* c = new f2q_ctx();
    c->device = device; c->cfg = *cfg; c->hG = G;
    auto bail = [&](int code, const std::string& m) { fail(nullptr, code, m.empty() ? c->err : m); f2q_destroy(c); return code; };
    if (cudaSetDevice(device) != cudaSuccess) return bail(F2Q_ECUDA, "cudaSetDevice failed");
    cudaDeviceGetAttribute(&c->sm_count, cudaDevAttrMultiProcessorCount, device);
    if (stream) c->stream = reinterpret_cast<cudaStream_t>(stream);
    else { if (cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking) != cudaSuccess) return bail(F2Q_ECUDA, "cudaStreamCreate failed"); c->own_stream = true; }
    if (cudaMalloc(&c->dG, sizeof(GenericCfg)) != cudaSuccess || cudaMalloc(&c->d_error, 4) != cudaSuccess ||
        cudaMalloc(&c->dS, sizeof(DevState)) != cudaSuccess || cudaMalloc(&c->d_tickets, 16) != cudaSuccess)
        return bail(F2Q_ENOMEM, "cudaMalloc failed");
    cudaMemcpy(c->dG, &G, sizeof(G), cudaMemcpyHostToDevice);
    cudaMemset(c->d_error, 0, 4); cudaMemset(c->dS, 0, sizeof(DevState)); cudaMemset(c->d_tickets, 0, 16);
    decide_policy(c);
    if (cfg->mode == F2Q_MODE_EXTRACT_COUNT) {
        // no library in this mode: results are [stats 5]
        if ((rc = dev_alloc(c, c->result, 5 * 8)) || (rc = dev_alloc(c, c->spec_scratch, 5 * 8))) return bail(rc, "");
        cudaMemset(c->spec_scratch.p, 0, 5 * 8);
        std::vector<uint32_t> gh(16, 0); std::vector<uint64_t> ko(1, 0); std::vector<uint8_t> kb(1, 0);
        if ((rc = upload(c, gh, &c->T.ghash)) || (rc = upload(c, ko, &c->T.key_off)) || (rc = upload(c, kb, &c->T.key_bytes))) return bail(rc, "");
        c->T.ghash_mask = 15; c->lib_set = true;
    }
    *out = c;
    return F2Q_OK;
}

F2Q_EXPORT int f2q_comm_destroy(f2q_ctx* c);
F2Q_EXPORT int f2q_host_free(void* ptr);
F2Q_EXPORT int f2q_host_alloc_near(void** ptr, uint64_t nbytes, int device, int flags, int* numa_node);

F2Q_EXPORT void f2q_destroy(f2q_ctx* c) {
    if (!c) return;
    static const bool debug = getenv("F2Q_DEBUG_INGEST") != nullptr;   // developer lap timers
    auto now = [] { return std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now().time_since_epoch()).count(); };
    double t0 = now(), t1, t2, t3, t4;
    cudaSetDevice(c->device);
    if (c->stream) cudaStreamSynchronize(c->stream);
    t1 = now();
    for (auto& b : c->lib_bufs) b.release();
    c->result.release(); c->carry.release(); c->status.release(); c->status_stitch.release(); c->queue.release(); c->gqueue.release();
    c->seg_count.release(); c->spec_rec.release(); c->spec_scratch.release(); c->slow_args.release(); c->synth_guides.release();
    c->ec_slots.release(); c->ec_counts.release(); c->ec_arena.release(); c->ec_meta.release(); c->ec_pk.release(); c->ec_compact.release(); c->memo.release(); c->shard_head.release();
    for (auto& p : c->ec_pend) if (p.ev) cudaEventDestroy(p.ev);
    for (auto e : c->ec_events) cudaEventDestroy(e);
    if (c->ec_meta_host) cudaFreeHost(c->ec_meta_host);
    t2 = now();
    for (int k = 0; k < 2; k++) {
        c->gz_comp[k].release(); c->gz_out[k].release(); c->gz_tab[k].release();
        if (c->gz_tab_host[k]) cudaFreeHost(c->gz_tab_host[k]);
        if (c->gz_copied[k]) cudaEventDestroy(c->gz_copied[k]);
        if (c->gz_free[k]) cudaEventDestroy(c->gz_free[k]);
    }
    t3 = now();
    if (c->file_ring) {
        for (int k = 0; k < FileRing::N; k++) { if (c->file_ring->buf[k]) f2q_host_free(c->file_ring->buf[k]); if (c->file_ring->done[k]) cudaEventDestroy(c->file_ring->done[k]); }
        delete c->file_ring; c->file_ring = nullptr;
    }
    t4 = now();
    f2q_comm_destroy(c);
    for (auto p : c->d_stage) cudaFree(p);
    for (auto e : c->ev_copied) cudaEventDestroy(e);
    for (auto e : c->ev_free) cudaEventDestroy(e);
    for (auto& t : c->timed) { cudaEventDestroy(t.a); cudaEventDestroy(t.b); }
    for (auto e : c->event_pool) cudaEventDestroy(e);
    if (c->dG) cudaFree(c->dG);
    if (c->d_error) cudaFree(c->d_error);
    if (c->dS) cudaFree(c->dS);
    if (c->d_tickets) cudaFree(c->d_tickets);
    if (c->copy_stream) cudaStreamDestroy(c->copy_stream);
    if (c->own_stream && c->stream) cudaStreamDestroy(c->stream);
    cudaGetLastError();
    if (debug) fprintf(stderr, "[f2q destroy] sync %.1f ms, tables %.1f ms, inflate buffers %.1f ms, file ring %.1f ms, staging + rest %.1f ms\n",
                       t1 - t0, t2 - t1, t3 - t2, t4 - t3, now() - t4);
    delete c;
}

F2Q_EXPORT int f2q_set_option(f2q_ctx* c, const char* name, int64_t value) {
    int rc = check_ctx(c); if (rc) return rc;
    if (!name) return fail(c, F2Q_EINVAL, "null option name");
    if (c->in_sample) return fail(c, F2Q_ESTATE, "options must be set before f2q_begin_sample");
    std::string n(name);
    if (n == "carry_bytes") { if (value < 4096 || value > (1ll << 31)) return fail(c, F2Q_EINVAL, "carry_bytes out of range"); c->carry_cap = (uint64_t)value; c->carry.release(); c->status_stitch.release(); }
    else if (n == "stage_bytes") { if (value < 4096 || !c->d_stage.empty()) return fail(c, F2Q_EINVAL, "stage_bytes invalid or staging already allocated"); c->stage_bytes = (uint64_t)value; }
    else if (n == "stage_slots") { if (value < 1 || value > 16 || !c->d_stage.empty()) return fail(c, F2Q_EINVAL, "stage_slots invalid or staging already allocated"); c->stage_slots = (int)value; }
    else if (n == "resolver") { if (value < 0 || value > 3) return fail(c, F2Q_EINVAL, "resolver must be 0..3"); c->resolver = (int)value; }
    else if (n == "queue_entries") { if (value < 0) return fail(c, F2Q_EINVAL, "queue_entries < 0"); c->opt_queue_entries = value; c->q_cap = 0; c->g_cap = 0; c->n_segs = 0; c->queue.release(); c->gqueue.release(); }
    else if (n == "generic_entries") { if (value < 0 || value > (1 << 28)) return fail(c, F2Q_EINVAL, "generic_entries out of range"); c->opt_generic_entries = value; c->g_cap = 0; }
    else if (n == "tile_threads") { if (value != 128 && value != 256) return fail(c, F2Q_EINVAL, "tile_threads must be 128 or 256"); c->nt = (int)value; c->nt_user = true; c->n_segs = 0; }
    else if (n == "halo_rows") { if (value < 0 || value > 128) return fail(c, F2Q_EINVAL, "halo_rows must be 0 (auto) .. 128"); c->force_halo = (int)value; }
    else if (n == "row_chunks") { if (value != 0 && value != 3 && value != 5 && value != 7) return fail(c, F2Q_EINVAL, "row_chunks must be 0 (auto), 3, 5 or 7"); c->force_ch = (int)value; }
    else if (n == "time_kernels") c->time_kernels = value != 0;
    else if (n == "debug_waits") c->debug_waits = value != 0;
    else if (n == "spec") c->spec = value != 0;
    else if (n == "spec_warps") { if (value != 12 && value != 16 && value != 20 && value != 24) return fail(c, F2Q_EINVAL, "spec_warps must be 12, 16, 20 or 24"); c->spec_warps = (int)value; }
    else if (n == "memo_entries") { if (value < -1 || value > (1ll << 28) || (value > 0 && (value & (value - 1)))) return fail(c, F2Q_EINVAL, "memo_entries must be -1 (auto), 0 (off) or a power of two"); c->memo_entries = value; if (c->lib_set) return fail(c, F2Q_ESTATE, "memo_entries must be set before f2q_set_library"); }
    else if (n == "seed_parts") { if (value < 0 || value > SEED_MAX_PARTS) return fail(c, F2Q_EINVAL, "seed_parts must be 0 (auto) .. 8"); if (c->lib_set) return fail(c, F2Q_ESTATE, "seed_parts must be set before f2q_set_library"); c->opt_seed_parts = (int)value; }
    else if (n == "gpu_inflate_bits") { if (value != 0 && value != 8 && value != 9) return fail(c, F2Q_EINVAL, "gpu_inflate_bits must be 0, 8 or 9"); c->gpu_inflate_bits = (int)value; }
    else if (n == "gpu_inflate") { if (value < 0 || value > 2) return fail(c, F2Q_EINVAL, "gpu_inflate must be 0, 1 or 2"); c->gpu_inflate = value != 0; c->gpu_inflate_mode = value == 2 ? 2 : 1; }
    else if (n == "flex_warps") { if (value != 12 && value != 16) return fail(c, F2Q_EINVAL, "flex_warps must be 12 or 16"); c->flex_warps = (int)value; }
    else if (n == "spec_range_tiles") { if (value < 0 || value > (1 << 20)) return fail(c, F2Q_EINVAL, "spec_range_tiles out of range"); c->spec_range_tiles = (int)value; }
    else if (n == "force_generic") { c->force_generic = value != 0; decide_policy(c); c->n_segs = 0; c->q_cap = 0; }
    else if (n == "flex") { c->no_flex = value == 0; decide_policy(c); c->n_segs = 0; c->q_cap = 0; }
    else if (n == "resolve_group") { if (value != 0 && value != 1 && value != 8 && value != 32) return fail(c, F2Q_EINVAL, "resolve_group must be 0 (auto), 1, 8 or 32"); c->fx_group_opt = (int)value; }
    else if (n == "ec_slots") { if (value < 0 || value > (1ll << 34)) return fail(c, F2Q_EINVAL, "ec_slots out of range"); c->ec_pk_min = (uint64_t)value; }
    else return fail(c, F2Q_EINVAL, "unknown option " + n);
    return F2Q_OK;
}

F2Q_EXPORT int f2q_set_library(f2q_ctx* c, const uint8_t* key_bytes, const uint64_t* key_offsets, uint32_t n_keys) {
    int rc = check_ctx(c); if (rc) return rc;
    if (c->cfg.mode != F2Q_MODE_COUNT) return fail(c, F2Q_ESTATE, "Extract+Count mode takes no library (fast2q.py:1700-1702)");
    if (c->in_sample) return fail(c, F2Q_ESTATE, "set_library inside a sample");
    if (n_keys && (!key_bytes || !key_offsets)) return fail(c, F2Q_EINVAL, "null library arrays");
    for (auto& b : c->lib_bufs) b.release();
    c->lib_bufs.clear(); c->T = LibTables{}; c->lib_set = false;
    memset(c->tile_blocks, 0, sizeof(c->tile_blocks));

    std::vector<uint64_t> off(n_keys + 1, 0);
    for (uint32_t i = 0; i <= n_keys && n_keys; i++) off[i] = key_offsets[i] - key_offsets[0];
    const uint8_t* kb = n_keys ? key_bytes + key_offsets[0] : nullptr;
    const uint64_t total = off[n_keys];
    std::vector<uint8_t> bytes(kb, kb + total);
    bytes.push_back(0);

    // uniqueness (the reference's dict has unique keys by construction)
    {
        std::unordered_set<std::string> seen;
        seen.reserve(n_keys * 2);
        for (uint32_t i = 0; i < n_keys; i++)
            if (!seen.emplace(reinterpret_cast<const char*>(bytes.data() + off[i]), off[i + 1] - off[i]).second)
                return fail(c, F2Q_EINVAL, "duplicate library key at index " + std::to_string(i));
    }
    // packed table + arrays
    std::vector<uint64_t> fk; std::vector<uint32_t> fl, fi;
    uint64_t gmask = 0; uint32_t n_generic = 0;
    for (uint32_t i = 0; i < n_keys; i++) {
        uint64_t key; const size_t len = off[i + 1] - off[i];
        if (packable(bytes.data() + off[i], len, key)) { fk.push_back(key); fl.push_back((uint32_t)len); fi.push_back(i); }
        else { n_generic++; gmask |= 1ull << std::min<size_t>(len, 63); }
    }
    const uint32_t cap = pow2_at_least(2 * (uint64_t)fk.size() + 2);
    std::vector<FastSlot> slots(cap, FastSlot{0, 0, SLOT_EMPTY});
    for (size_t k = 0; k < fk.size(); k++) {
        uint32_t h = mix32(fk[k], fl[k]) & (cap - 1);
        while (slots[h].idx != SLOT_EMPTY) h = (h + 1) & (cap - 1);
        slots[h] = FastSlot{fk[k], fl[k], fi[k]};
    }
    // compact 8-byte table for the tile kernel (one key length, index fits above the key bits)
    std::vector<uint64_t> cslots(1, ~0ull);
    uint32_t c_len = 0, c_mask = 0; bool compact = !fk.empty();
    for (size_t k = 0; k < fl.size() && compact; k++) compact = fl[k] == fl[0];
    if (compact) {
        c_len = fl[0];
        const uint32_t idx_bits = 64 - 2 * c_len;
        compact = c_len >= 1 && c_len < 32 && (idx_bits >= 32 || (uint64_t)n_keys < (1ull << idx_bits) - 1);
    }
    if (compact) {
        const uint32_t ccap = pow2_at_least(4 * (uint64_t)fk.size());
        cslots.assign(ccap, ~0ull);
        c_mask = ccap - 1;
        for (size_t k = 0; k < fk.size(); k++) {
            uint32_t h = mix_compact((uint32_t)fk[k], (uint32_t)(fk[k] >> 32)) & c_mask;
            while (cslots[h] != ~0ull) h = (h + 1) & c_mask;
            cslots[h] = fk[k] | ((uint64_t)fi[k] << (2 * c_len));
        }
    }
    // two-choice cuckoo form of the compact table: <= 1/4 full, random-walk insertion, new multipliers until it builds.
    // Slot = packed key | value << 2*c_len, value = feature index << 1 | imperfect.  With m >= 1 the table also holds every
    // Hamming-1 NEIGHBOUR of every key (3*c_len per key): value = the one key at distance 1 (imperfect = 1), or CK_AMBIG
    // when two or more keys are at distance 1 (the reference's unique-hit rule then gives "not aligned" for every m).  A
    // neighbour that is itself a library key keeps its exact entry.  A non-exact read whose window is pure ACGT is thus
    // decided by the same two loads as an exact one; only keys with other symbols, and keys further away when m >= 2, go
    // to the queue and the resolver kernel.
    std::vector<uint64_t> cuckoo;
    uint32_t ck_mask = 0, ck_mul[4] = {0, 0, 0, 0};
    bool ck_neighbours = false;
    uint32_t ck_shift_out = 28, ck_hshift_out = 0;
    if (compact) {
        const uint32_t keybits = 2 * c_len, hshift = (keybits > 32 ? keybits : 32) - 32;   // the value sits in the high word above bit hshift
        const uint64_t kmask = (1ull << keybits) - 1ull;
        const uint64_t valmax = cuckoo_valmax(hshift);                                      // all ones = empty slot
        ck_hshift_out = hshift;
        std::vector<std::pair<uint64_t, uint64_t>> ent;                                    // (packed key, value)
        bool fits = (((uint64_t)n_keys << 1) | 1ull) < valmax - 1ull;
        if (fits) {
            for (size_t k = 0; k < fk.size(); k++) ent.emplace_back(fk[k], (uint64_t)fi[k] << 1);
            // (only while the table stays a few MB: it must live in L2 next to the stream; a 100 000-guide library would need 270 MB,
            // measured slower than the queue + resolver kernel)
            const uint64_t n_nb = (uint64_t)fk.size() * 3ull * c_len;
            if (c->cfg.miss >= 1 && n_nb + fk.size() <= (1ull << 20)) {
                std::vector<std::pair<uint64_t, uint32_t>> nb;
                nb.reserve((size_t)n_nb);
                for (size_t k = 0; k < fk.size(); k++)
                    for (uint32_t pos = 0; pos < c_len; pos++)
                        for (uint64_t d = 1; d < 4; d++) nb.emplace_back(fk[k] ^ (d << (2 * pos)), fi[k]);
                std::sort(nb.begin(), nb.end());
                std::vector<uint64_t> exact(fk);
                std::sort(exact.begin(), exact.end());
                for (size_t i = 0; i < nb.size();) {
                    size_t e = i;
                    while (e < nb.size() && nb[e].first == nb[i].first) e++;
                    if (!std::binary_search(exact.begin(), exact.end(), nb[i].first))
                        ent.emplace_back(nb[i].first, e - i == 1 ? (((uint64_t)nb[i].second << 1) | 1ull) : valmax - 1ull);
                    i = e;
                }
                ck_neighbours = true;
            }
        }
        const uint32_t tcap = pow2_at_least(2 * (uint64_t)ent.size());
        ck_mask = tcap - 1;
        uint32_t ck_shift = 32; while ((1ull << (32 - ck_shift)) < tcap) ck_shift--;
        ck_shift_out = ck_shift;
        uint64_t seed = 0x2FA572ull ^ 0x9E3779B97F4A7C15ull;
        bool built = false;
        for (int attempt = 0; attempt < 64 && !built && fits; attempt++) {
            for (int k = 0; k < 4; k++) { seed = sm_fin(seed + 0x9E3779B97F4A7C15ull * (uint64_t)(attempt * 4 + k + 1)); ck_mul[k] = (uint32_t)(seed >> 16) | 1u; }
            cuckoo.assign(2 * (size_t)tcap, ~0ull);
            built = true;
            for (size_t k = 0; k < ent.size() && built; k++) {
                uint64_t cur = ent[k].first | (ent[k].second << (32 + hshift));
                int kicks = 0;
                uint32_t from = 0xFFFFFFFFu;                            // slot `cur` was evicted from
                for (;; kicks++) {
                    uint32_t h1, h2;
                    cuckoo_slots(ck_mul[0], ck_mul[1], ck_mul[2], ck_mul[3], ck_shift, (uint32_t)(cur & kmask), (uint32_t)((cur & kmask) >> 32), h1, h2);
                    if (cuckoo[h1] == ~0ull) { cuckoo[h1] = cur; break; }
                    if (cuckoo[h2] == ~0ull) { cuckoo[h2] = cur; break; }
                    if (kicks >= 500) { built = false; break; }
                    const uint32_t h = (h1 == from) ? h2 : h1;          // never straight back to where it came from
                    std::swap(cur, cuckoo[h]);
                    from = h;
                }
            }
        }
        if (!built) {
            if (fits) fprintf(stderr, "libf2q: the two-choice lookup table did not build (%zu entries); using the probing table and the resolver kernel\n", ent.size());
            cuckoo.clear(); ck_neighbours = false;
        }
    }
    const uint32_t gcap = pow2_at_least(2 * (uint64_t)n_keys + 2);
    std::vector<uint32_t> gh(gcap, 0);
    for (uint32_t i = 0; i < n_keys; i++) {
        uint32_t h = FNV_INIT;
        for (uint64_t k = off[i]; k < off[i + 1]; k++) h = fnv_step(h, bytes[k]);
        uint32_t j = fnv_final(h) & (gcap - 1);
        while (gh[j]) j = (j + 1) & (gcap - 1);
        gh[j] = i + 1;
    }
    // pigeonhole seed index for <= miss mismatches (resolve.cuh)
    std::vector<uint4> seed_slots(16, make_uint4(0, 0, 0, 0));
    std::vector<uint4> seed_recs;
    // seed plan: P segments, seeds = every choice of K = P - miss of them.  Cost of resolving one key ~ seeds x (probe + expected
    // bucket length); a seed must fit the tag's 32 value bits (<= 16 symbols) for the longest key
    uint32_t parts = (uint32_t)std::max(1, std::min(c->cfg.miss, 32) + 1);
    std::vector<uint8_t> combos;
    if (c->cfg.miss > 0 && !fk.empty()) {
        const uint32_t m = (uint32_t)c->cfg.miss;
        uint32_t maxlen = 0; double meanlen = 0;
        for (uint32_t j = 0; j < fk.size(); j++) { maxlen = std::max(maxlen, (uint32_t)fl[j]); meanlen += fl[j]; }
        meanlen /= (double)fk.size();
        auto n_choose = [](uint32_t n, uint32_t k) { double r = 1; for (uint32_t i = 0; i < k; i++) r = r * (n - i) / (i + 1); return r; };
        double best = -1;
        if (m + 1 <= (uint32_t)SEED_MAX_PARTS)
            for (uint32_t P = m + 1; P <= (uint32_t)SEED_MAX_PARTS; P++) {
                const uint32_t K = P - m;
                const double seeds = n_choose(P, m);
                if (seeds > SEED_MAX_COMBOS || K * ((maxlen + P - 1) / P) > 16) continue;
                if (c->opt_seed_parts && (uint32_t)c->opt_seed_parts != P) continue;
                // (measured at 100 000 guides, m = 1..3, P = m+1 .. m+3: a probe costs about 1.5 + K candidate compares)
                const double cost = seeds * (1.5 + (double)K + (double)fk.size() / std::pow(4.0, (double)K * meanlen / P));
                if (best < 0 || cost < best) { best = cost; parts = P; }
            }
        // (more than SEED_MAX_PARTS - 1 mismatches, or no plan that fits: the classic one-segment seeds, miss + 1 of them, no
        // seed masks — resolve_seed_classic)
        const bool planned = best >= 0;
        if (planned) {
            const uint32_t K = parts - m;
            for (uint32_t mask = 0; mask < (1u << parts); mask++) if ((uint32_t)__builtin_popcount(mask) == K) combos.push_back((uint8_t)mask);
        }
        std::vector<std::pair<uint64_t, uint32_t>> ent;
        ent.reserve(fk.size() * (planned ? combos.size() : parts));
        for (uint32_t j = 0; j < fk.size(); j++) {
            uint32_t sv[33] = {0}, sw[33] = {0};
            for (uint32_t sgm = 0; sgm < parts; sgm++) {
                const uint32_t b0 = sgm * fl[j] / parts, b1 = (sgm + 1) * fl[j] / parts;
                const uint64_t rng = even_range(b0, b1);
                sv[sgm] = (uint32_t)((fk[j] >> (2 * b0)) & ((rng | (rng << 1)) >> (2 * b0)));
                sw[sgm] = 2 * (b1 - b0);
                if (!planned) ent.emplace_back(seed_tag(fl[j], sgm, (fk[j] >> (2 * b0)) & ((rng | (rng << 1)) >> (2 * b0))), j);
            }
            for (uint32_t cb = 0; cb < combos.size(); cb++) ent.emplace_back(seed_tag(fl[j], cb, seed_value(combos[cb], sv, sw)), j);
        }
        std::sort(ent.begin(), ent.end());
        size_t uniq = 0;
        for (size_t i = 0; i < ent.size(); i++) if (i == 0 || ent[i].first != ent[i - 1].first) uniq++;
        const uint32_t scap = pow2_at_least(2 * (uint64_t)uniq + 2);
        seed_slots.assign(scap, make_uint4(0, 0, 0, 0));
        seed_recs.resize(ent.size());
        for (size_t i = 0; i < ent.size();) {
            size_t e = i;
            while (e < ent.size() && ent[e].first == ent[i].first) { const uint32_t j = ent[e].second; seed_recs[e] = make_uint4((uint32_t)fk[j], (uint32_t)(fk[j] >> 32), fi[j], 0u); e++; }
            uint32_t h = seed_hash(ent[i].first) & (scap - 1);
            while (seed_slots[h].x | seed_slots[h].y) h = (h + 1) & (scap - 1);
            seed_slots[h] = make_uint4((uint32_t)ent[i].first, (uint32_t)(ent[i].first >> 32), (uint32_t)i, (uint32_t)(e - i));
            i = e;
        }
    }
    // byte-level seed index over every key (generic path)
    {
        std::vector<uint4> gslots(16, make_uint4(0, 0, 0, 0));
        std::vector<uint32_t> gitems;
        uint32_t gparts = 0;
        if (c->cfg.miss >= 1 && c->cfg.miss + 1 <= (int)GSEED_MAX_PARTS && n_keys) {
            gparts = (uint32_t)c->cfg.miss + 1;
            std::vector<std::pair<uint64_t, uint32_t>> ent;
            ent.reserve((size_t)n_keys * gparts);
            for (uint32_t i = 0; i < n_keys; i++) {
                const uint32_t len = (uint32_t)(off[i + 1] - off[i]);
                if (len < gparts) continue;                            // (such keys are found by the linear scan: the device takes it for klen < parts)
                for (uint32_t sg = 0; sg < gparts; sg++) {
                    uint32_t a, b;
                    gseed_init(len, sg, a, b);
                    for (uint32_t k = sg * len / gparts; k < (sg + 1) * len / gparts; k++) gseed_step(bytes[off[i] + k], a, b);
                    ent.emplace_back(gseed_tag(a, b), i);
                }
            }
            std::sort(ent.begin(), ent.end());
            size_t uniq = 0;
            for (size_t i = 0; i < ent.size(); i++) if (i == 0 || ent[i].first != ent[i - 1].first) uniq++;
            const uint32_t scap = pow2_at_least(2 * (uint64_t)uniq + 2);
            gslots.assign(scap, make_uint4(0, 0, 0, 0));
            gitems.resize(ent.size());
            for (size_t i = 0; i < ent.size();) {
                size_t e = i;
                while (e < ent.size() && ent[e].first == ent[i].first) { gitems[e] = ent[e].second; e++; }
                uint32_t h = gseed_hash(ent[i].first) & (scap - 1);
                while (gslots[h].x | gslots[h].y) h = (h + 1) & (scap - 1);
                gslots[h] = make_uint4((uint32_t)ent[i].first, (uint32_t)(ent[i].first >> 32), (uint32_t)i, (uint32_t)(e - i));
                i = e;
            }
        }
        if ((rc = upload(c, gslots, &c->T.gseed_slots)) || (rc = upload(c, gitems, &c->T.gseed_items))) return rc;
        c->T.gseed_mask = (uint32_t)gslots.size() - 1; c->T.gseed_parts = gparts;
    }
    // flex tables (flex.cuh): every key as <= 2 ACGT pieces -> 80-bit packed key + signature; exact table, the signature of
    // every key BYTE length, and the pigeonhole seed index over the packed symbols for the resolver
    if (c->hG.flex.eligible && !(c->cfg.n_iter == 1 && !c->cfg.has_up && !c->cfg.has_down)) {
        std::vector<FlexKey> fkeys(n_keys);
        bool all = n_keys > 0;
        for (uint32_t i = 0; i < n_keys && all; i++) {
            const uint8_t* k = bytes.data() + off[i];
            const size_t len = off[i + 1] - off[i];
            FlexPiece pc[FLEX_ITER];
            int np = 1; size_t p0 = 0;
            for (int q = 0; q < FLEX_ITER; q++) { pc[q].codes = 0; pc[q].notok = 0; pc[q].len = 0; pc[q].off = 0; }
            for (size_t j = 0; j <= len && all; j++) {
                if (j == len || k[j] == ':') {
                    const size_t pl = j - p0;
                    uint64_t codes = 0;
                    if (pl > (size_t)FLEX_MAX_PIECE || !packable(k + p0, pl, codes)) { all = false; break; }
                    pc[np - 1].codes = codes; pc[np - 1].len = (uint32_t)pl;
                    if (j < len) { if (np == FLEX_ITER) { all = false; break; } np++; p0 = j + 1; }
                }
            }
            if (all) all = fx_assemble(pc, np, fkeys[i]);
        }
        if (all) {
            const uint32_t fcap = pow2_at_least(4 * (uint64_t)n_keys);
            std::vector<uint4> fslots(fcap, make_uint4(0, 0, 0, FX_EMPTY));
            std::vector<uint16_t> len_sig(FX_MAX_BYTELEN + 1, 0);
            for (uint32_t i = 0; i < n_keys; i++) {
                const FlexKey& k = fkeys[i];
                const uint32_t z = k.hi | (k.sig << 16);
                uint32_t h = fx_hash(k.lo, z) & (fcap - 1);
                while (fslots[h].w != FX_EMPTY) h = (h + 1) & (fcap - 1);
                fslots[h] = make_uint4((uint32_t)k.lo, (uint32_t)(k.lo >> 32), z, i);
                uint16_t& ls = len_sig[fx_sig_bytelen(k.sig)];
                ls = ls == 0 ? (uint16_t)k.sig : (ls == (uint16_t)k.sig ? ls : FX_SIG_MIXED);
            }
            // seed index: (signature, segment, segment value) -> keys; shapes with fewer symbols than segments are left to the generic code
            std::vector<uint4> fs_slots(16, make_uint4(0, 0, 0, 0)), fs_recs;
            const uint32_t fparts = (uint32_t)c->cfg.miss + 1;
            if (c->cfg.miss >= 1 && c->cfg.miss <= 15) {
                std::vector<std::pair<uint64_t, uint32_t>> ent;
                ent.reserve((size_t)n_keys * fparts);
                for (uint32_t i = 0; i < n_keys; i++) {
                    const FlexKey& k = fkeys[i];
                    const uint32_t ns = fx_sig_symbols(k.sig);
                    if (ns < fparts || ns > 20 * fparts) { len_sig[fx_sig_bytelen(k.sig)] = FX_SIG_MIXED; continue; }
                    for (uint32_t sg = 0; sg < fparts; sg++)
                        ent.emplace_back(fxs_tag(k.sig, sg, fx_segment(k.lo, k.hi, sg * ns / fparts, (sg + 1) * ns / fparts)), i);
                }
                std::sort(ent.begin(), ent.end());
                size_t uniq = 0;
                for (size_t i = 0; i < ent.size(); i++) if (i == 0 || ent[i].first != ent[i - 1].first) uniq++;
                const uint32_t scap = pow2_at_least(2 * (uint64_t)uniq + 2);
                fs_slots.assign(scap, make_uint4(0, 0, 0, 0));
                fs_recs.resize(ent.size());
                for (size_t i = 0; i < ent.size();) {
                    size_t e = i;
                    while (e < ent.size() && ent[e].first == ent[i].first) {
                        const FlexKey& k = fkeys[ent[e].second];
                        fs_recs[e] = make_uint4((uint32_t)k.lo, (uint32_t)(k.lo >> 32), k.hi, ent[e].second);
                        e++;
                    }
                    uint32_t h = fxs_hash(ent[i].first) & (scap - 1);
                    while (fs_slots[h].x | fs_slots[h].y) h = (h + 1) & (scap - 1);
                    fs_slots[h] = make_uint4((uint32_t)ent[i].first, (uint32_t)(ent[i].first >> 32), (uint32_t)i, (uint32_t)(e - i));
                    i = e;
                }
                // lanes per key of the resolver: from the mean number of candidates a probe returns (weighted by bucket size)
                double w = 0, tot = 0;
                for (size_t i = 0; i < ent.size();) { size_t e = i; while (e < ent.size() && ent[e].first == ent[i].first) e++; w += (double)(e - i) * (double)(e - i); tot += (double)(e - i); i = e; }
                const double mean = tot > 0 ? w / tot : 0;
                (void)mean;
                c->fx_group = 1;                                       // (as for the fast1 resolver: one thread per key)
            }
            if ((rc = upload(c, fslots, &c->T.fx_slots)) || (rc = upload(c, len_sig, &c->T.fx_len_sig)) ||
                (rc = upload(c, fs_slots, &c->T.fxs_slots)) || (rc = upload(c, fs_recs, &c->T.fxs_recs)))
                return rc;
            c->T.fx_mask = fcap - 1; c->T.fxs_mask = (uint32_t)fs_slots.size() - 1; c->T.fxs_parts = fparts;
        }
    }
    {
        // lanes per key of the fast1 seed resolver, from the mean number of candidates a probe returns (weighted by bucket size)
        double w = 0, tot = 0;
        for (const uint4& sl : seed_slots) if (sl.x | sl.y) { w += (double)sl.w * (double)sl.w; tot += (double)sl.w; }
        const double mean = tot > 0 ? w / tot : 0;
        (void)mean;
        c->seed_group = 1;        // measured (config 3: 250 M queued keys, ~36 candidates each): one thread per key 46 ms, 8 / 32 lanes 104 ms — with
                                  // millions of keys in flight the GPU hides the candidate loads' latency itself; lanes per key only add instructions
    }
    {
        // memo of resolved keys: emptied with every new library
        const int64_t want = c->memo_entries < 0 ? 0 : c->memo_entries;     // (off unless asked for: a stream without repeated non-exact keys only pays for it)
        c->memo.release();
        if (want > 0 && c->cfg.miss > 0) {
            if ((rc = dev_alloc(c, c->memo, (size_t)want * 16))) return rc;
            CU(c, cudaMemset(c->memo.p, 0, (size_t)want * 16));
            c->T.memo = reinterpret_cast<uint4*>(c->memo.p); c->T.memo_mask = (uint32_t)want - 1;
        }
    }
    if ((rc = upload(c, seed_slots, &c->T.seed_slots)) || (rc = upload(c, seed_recs, &c->T.seed_recs))) return rc;
    c->T.seed_mask = (uint32_t)seed_slots.size() - 1; c->T.seed_parts = parts;
    c->T.seed_ncombo = (uint32_t)combos.size();
    memset(c->T.seed_combo, 0, sizeof(c->T.seed_combo));
    for (size_t i = 0; i < combos.size(); i++) c->T.seed_combo[i] = combos[i];
    if ((rc = upload(c, slots, &c->T.slots)) || (rc = upload(c, fk, &c->T.fast_keys)) || (rc = upload(c, fl, &c->T.fast_lens)) ||
        (rc = upload(c, fi, &c->T.fast_idx)) || (rc = upload(c, bytes, &c->T.key_bytes)) || (rc = upload(c, off, &c->T.key_off)) ||
        (rc = upload(c, gh, &c->T.ghash)))
        return rc;
    if (compact) {
        if ((rc = upload(c, cslots, &c->T.cslots))) return rc;
        c->T.c_mask = c_mask; c->T.c_len = c_len; c->T.c_keybits = 2 * c_len;
        if (!cuckoo.empty()) {
            if ((rc = upload(c, cuckoo, &c->T.cuckoo))) return rc;
            c->T.ck_mask = ck_mask; for (int k = 0; k < 4; k++) c->T.ck_mul[k] = ck_mul[k];
            c->T.ck_neighbours = ck_neighbours ? 1u : 0u; c->T.ck_shift = ck_shift_out; c->T.ck_hshift = ck_hshift_out;
        }
    }
    c->T.slot_mask = cap - 1; c->T.n_fast = (uint32_t)fk.size(); c->T.n_keys = n_keys; c->T.ghash_mask = gcap - 1;
    c->T.n_generic = n_generic; c->T.generic_len_mask = gmask;
    c->n_keys = n_keys;
    {
        // FNV-1a over every key length and key byte, in library order
        uint64_t lh = 1469598103934665603ull;
        auto mix = [&](uint64_t v, int nb) { for (int b = 0; b < nb; b++) lh = (lh ^ ((v >> (8 * b)) & 0xFF)) * 1099511628211ull; };
        mix(n_keys, 4);
        for (uint32_t i = 0; i < n_keys; i++) { mix(off[i + 1] - off[i], 8); for (uint64_t k = off[i]; k < off[i + 1]; k++) mix(bytes[k], 1); }
        c->lib_hash = lh;
    }
    c->result.release();
    if ((rc = dev_alloc(c, c->result, ((size_t)n_keys + 5) * 8))) return rc;
    c->spec_scratch.release();
    if ((rc = dev_alloc(c, c->spec_scratch, ((size_t)n_keys + 5) * 8))) return rc;
    c->lib_set = true;
    decide_policy(c);                                                  // (the flex policy needs the flex table)
    c->n_segs = 0; c->q_cap = 0;
    return F2Q_OK;
}

F2Q_EXPORT int f2q_begin_sample(f2q_ctx* c) {
    int rc = check_ctx(c); if (rc) return rc;
    if (!c->lib_set) return fail(c, F2Q_ESTATE, "f2q_set_library must be called first in Counter mode");
    if ((rc = dev_alloc(c, c->carry, c->carry_cap + 256))) return rc;
    if ((rc = dev_alloc(c, c->status_stitch, c->carry_cap / (64 * 16 * 3) + 2 + 64))) return rc;
    if (!c->ch_from_device) c->ch_decided = false;
    c->hist_used = 0;
    {
        const uint64_t nw = (uint64_t)c->n_keys + 5;
        k_begin<<<(unsigned)std::min<uint64_t>((nw + 255) / 256, (uint64_t)c->sm_count), 256, 0, c->stream>>>(
            reinterpret_cast<unsigned long long*>(c->result.p), reinterpret_cast<unsigned long long*>(c->spec_scratch.p), nw, c->d_error, c->dS);
        c->launches++;
        CU(c, cudaGetLastError());
    }
    if (c->cfg.mode == F2Q_MODE_EXTRACT_COUNT) {
        while (!c->ec_pend.empty()) { if (c->ec_pend.front().ev) { cudaEventSynchronize(c->ec_pend.front().ev); c->ec_events.push_back(c->ec_pend.front().ev); } c->ec_pend.pop_front(); }
        for (int k = 0; k < 4; k++) c->ec_known[k] = 0;
        if (c->ec_meta.p) CU(c, cudaMemsetAsync(c->ec_meta.p, 0, 32, c->stream));
        if (c->ec_slots.p) { CU(c, cudaMemsetAsync(c->ec_slots.p, 0, c->ec_cap * 8, c->stream)); CU(c, cudaMemsetAsync(c->ec_counts.p, 0, c->ec_cap * 8, c->stream)); }
        if (c->ec_pk.p) CU(c, cudaMemsetAsync(c->ec_pk.p, 0, c->ec_pk_cap * 16, c->stream));
        c->ec_drained = false; c->ec_merged = false;
    }
    c->in_sample = true; c->closed = false; c->sample_failed = F2Q_OK;
    c->last_shards = 1; c->last_shard_fallback = 0;
    c->shard_head_pending = false; c->shard_noguess = false;
    return F2Q_OK;
}

// text already in device memory -> kernels.  Extract+Count: bounded sub-chunks, so that the insert log and the table bounds
// of one launch stay bounded too
static int device_range(f2q_ctx* c, const uint8_t* dptr, uint64_t nbytes, int is_last) {
    const uint64_t sub = c->cfg.mode == F2Q_MODE_EXTRACT_COUNT ? EC_SUBCHUNK_BYTES : ~0ull;
    uint64_t done = 0;
    int rc;
    do {
        const uint64_t len = std::min<uint64_t>(sub, nbytes - done);
        rc = process_device_chunk(c, dptr + done, len, is_last && done + len == nbytes);
        if (rc) { if (!c->sticky) c->sample_failed = rc; return rc; }
        done += len;
    } while (done < nbytes);
    return F2Q_OK;
}

F2Q_EXPORT int f2q_submit_device(f2q_ctx* c, const void* dptr, uint64_t nbytes, int is_last) {
    int rc = check_ctx(c); if (rc) return rc;
    if (!c->in_sample) return fail(c, F2Q_ESTATE, "f2q_submit_device outside a sample");
    if (c->closed) return fail(c, F2Q_ESTATE, "stream already closed with is_last");
    if (nbytes && !dptr) return fail(c, F2Q_EINVAL, "null chunk");
    if (c->sample_failed) return c->sample_failed;
    return device_range(c, reinterpret_cast<const uint8_t*>(dptr), nbytes, is_last);
}

// host chunk -> staging slots -> kernels.  `host_done` (optional) is recorded on the copy stream behind the last copy out of
// host_chunk: the caller may refill the host buffer once it has completed
static int submit_host(f2q_ctx* c, const uint8_t* host_chunk, uint64_t nbytes, int is_last, cudaEvent_t host_done) {
    int rc;
    if ((rc = ensure_staging(c))) return rc;
    // (a shard that starts mid-file sniffs on the device, behind its head)
    if (!c->ch_decided && nbytes && !c->shard_head_pending) { decide_ch(c, host_chunk, (size_t)std::min<uint64_t>(nbytes, 4096)); c->ch_from_device = false; }
    uint64_t done = 0;
    do {
        const uint64_t len = std::min<uint64_t>(c->stage_bytes, nbytes - done);
        const int s = c->next_slot; c->next_slot = (c->next_slot + 1) % c->stage_slots;
        // the copy engine may refill slot s only after the kernels that read it have finished
        CU(c, cudaStreamWaitEvent(c->copy_stream, c->ev_free[s], 0));
        if (len) CU(c, cudaMemcpyAsync(c->d_stage[s], host_chunk + done, len, cudaMemcpyHostToDevice, c->copy_stream));
        CU(c, cudaEventRecord(c->ev_copied[s], c->copy_stream));
        CU(c, cudaStreamWaitEvent(c->stream, c->ev_copied[s], 0));
        done += len;
        if (done == nbytes && host_done) CU(c, cudaEventRecord(host_done, c->copy_stream));
        rc = process_device_chunk(c, c->d_stage[s], len, is_last && done == nbytes);
        CU(c, cudaEventRecord(c->ev_free[s], c->stream));               // (also on failure: kernels already queued may still read the slot)
        if (rc) { if (!c->sticky) c->sample_failed = rc; return rc; }
    } while (done < nbytes);
    return F2Q_OK;
}

F2Q_EXPORT int f2q_submit(f2q_ctx* c, const uint8_t* host_chunk, uint64_t nbytes, int is_last) {
    int rc = check_ctx(c); if (rc) return rc;
    if (!c->in_sample) return fail(c, F2Q_ESTATE, "f2q_submit outside a sample");
    if (c->sample_failed) return c->sample_failed;
    if (c->closed) return fail(c, F2Q_ESTATE, "stream already closed with is_last");
    if (nbytes && !host_chunk) return fail(c, F2Q_EINVAL, "null chunk");
    return submit_host(c, host_chunk, nbytes, is_last, nullptr);
}

// ---- native file ingest ------------------------------------------------------------------------------------------------
// One sequencing file -> the current sample, on host threads and without a copy in between: the file is read (.fastq) or
// inflated (.gz) straight INTO page-locked ring buffers near the GPU, which f2q_submit's copy engine drains.
// Replaces the open / gzip.open + `for line in current` of reads_counter and fastq_parser (fast2q.py:566-578, 324).
//   .fastq   read(2) into the ring, chunks cut anywhere (the device carries the partial record)
//   .gz      zlib inflate into the ring; multi-member files and zero padding between members as Python's gzip module reads
//            them.  Only WHOLE LINES are submitted while the stream is open, so that a stream that breaks off ends exactly
//            like the reference's line iterator: every complete line before the break is parsed, the partial one is dropped
//            and *complete = 0 (the reference's EOFError, fast2q.py:405-407)
//   BGZF     (bgzip: gzip members of <= 64 KiB that carry their compressed size in an extra field and their uncompressed
//            size in their trailer) blocks are independent: `threads` workers inflate a ring buffer's worth of blocks in
//            parallel, each straight to its final offset (SURVEY.md §8f-1: BGZF-aware parallel host inflate)
namespace {

int ring_get(f2q_ctx* c, FileRing& R, uint8_t** out, int* idx) {
    const int k = R.next; R.next = (R.next + 1) % FileRing::N;
    if (R.used[k]) CU(c, cudaEventSynchronize(R.done[k]));              // the copy out of this buffer (N submits ago) has finished
    *out = R.buf[k]; *idx = k;
    return F2Q_OK;
}

int ring_submit(f2q_ctx* c, FileRing& R, int idx, uint64_t n, int last) {
    R.used[idx] = true;
    return submit_host(c, R.buf[idx], n, last, R.done[idx]);
}

// read [off, off + want) of fd into buf with T readers (one reader copies ~3 GB/s out of the page cache, far below what the
// link and the kernels take); returns the contiguous bytes read from `off` (short at the end of the file)
size_t pread_parallel(int fd, uint8_t* buf, size_t want, uint64_t off, int T) {
    if (want == 0) return 0;
    if (T <= 1 || want < ((size_t)1 << 20)) {
        size_t have = 0;
        while (have < want) { const ssize_t g = pread(fd, buf + have, want - have, (off_t)(off + have)); if (g <= 0) break; have += (size_t)g; }
        return have;
    }
    const size_t part = (want / T + 4095) & ~(size_t)4095;
    std::vector<size_t> got(T, 0);
    auto rd = [&](int t) {
        const size_t lo = (size_t)t * part, w = lo < want ? std::min(part, want - lo) : 0;
        size_t have = 0;
        while (have < w) { const ssize_t g = pread(fd, buf + lo + have, w - have, (off_t)(off + lo + have)); if (g <= 0) break; have += (size_t)g; }
        got[t] = have;
    };
    std::vector<std::thread> pool;
    for (int t = 1; t < T; t++) pool.emplace_back(rd, t);
    rd(0);
    for (auto& th : pool) th.join();
    size_t n = 0;
    for (int t = 0; t < T; t++) {                                      // bytes are contiguous up to the first short part
        n += got[t];
        const size_t lo = (size_t)t * part, w = lo < want ? std::min(part, want - lo) : 0;
        if (got[t] < w) break;
    }
    return n;
}

// the page-locked ring lives with the context (allocated on first use), with the staging slots behind it
int ensure_ring(f2q_ctx* c) {
    int rc;
    if (!c->file_ring) c->file_ring = new FileRing();
    FileRing& R = *c->file_ring;
    if (!R.buf[0]) {
        R.bytes = 32u << 20;
        for (int k = 0; k < FileRing::N; k++) {
            void* p = nullptr;
            if ((rc = f2q_host_alloc_near(&p, R.bytes + 65536, c->device, 0, nullptr))) return fail(c, rc, f2q_last_error(nullptr));
            R.buf[k] = static_cast<uint8_t*>(p);
            if (cudaEventCreateWithFlags(&R.done[k], cudaEventDisableTiming) != cudaSuccess) return fail(c, F2Q_ECUDA, "cudaEventCreate failed");
        }
    }
    return ensure_staging(c);
}

const uint8_t* last_newline(const uint8_t* p, size_t n) { return static_cast<const uint8_t*>(memrchr(p, '\n', n)); }

// BGZF block at p (>= 18 bytes available): total block size, or 0 when this is not a BGZF member header
size_t bgzf_block_size(const uint8_t* p, size_t avail) {
    if (avail < 18 || p[0] != 0x1f || p[1] != 0x8b || p[2] != 8 || p[3] != 4) return 0;
    if (p[12] != 'B' || p[13] != 'C' || p[14] != 2 || p[15] != 0 || (unsigned)(p[10] | p[11] << 8) < 6) return 0;
    return (size_t)(p[16] | p[17] << 8) + 1;
}

}  // namespace

namespace {

constexpr size_t GZ_COMP_BYTES = 1u << 30, GZ_OUT_BYTES = 3ull << 30, GZ_MAX_BLOCKS = 1u << 16;
const uint8_t BGZF_EOF[28] = {0x1f, 0x8b, 0x08, 0x04, 0, 0, 0, 0, 0, 0xff, 0x06, 0, 0x42, 0x43, 0x02, 0, 0x1b, 0, 0x03, 0, 0, 0, 0, 0, 0, 0, 0, 0};

// bgzip file -> the sample, inflated ON THE DEVICE: compressed pieces are read into the pinned ring, their block headers and
// trailers are walked on the host (sizes only), the pieces go to a device staging buffer on the copy stream, and one launch
// of k_inflate_bgzf_lanes per batch (<= 1 GiB compressed, <= 3 GiB of output, <= 65 536 blocks: tens of thousands of lanes) writes the FASTQ text straight
// into the buffer process_device_chunk parses.  Two staging / output buffers: the next batch is read and copied while the
// previous one is inflated and parsed.  Stops at the first thing that is not a whole BGZF block (a foreign gzip member, a
// truncated block) and reports the file offset there: the host reader takes over from that offset.  Reads the file bytes
// [begin, end) only (a shard of f2q_submit_file_sharded: whole blocks); `finished` = that range was whole BGZF blocks.
int submit_bgzf_gpu(f2q_ctx* c, FILE* f, FileRing& R, int threads, uint64_t begin, uint64_t end, uint64_t* total, uint64_t* resume_off, bool* finished) {
    int rc;
    const int T = std::max(1, std::min(threads, 8));
    static const bool debug = getenv("F2Q_DEBUG_INGEST") != nullptr;   // developer lap timers: where the host thread spends its time
    double t_read = 0, t_ring = 0, t_free = 0, t_walk = 0;
    auto now = [] { return std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now().time_since_epoch()).count(); };
    const int fd = fileno(f);
    // batches of equal size: the inflate kernel is latency-bound (a launch takes as long as its slowest warp, ~29 ms for 64 KiB
    // blocks, however few blocks it has), so a small last batch costs as much as a full one.  The staging buffers follow the
    // file: a 100 MB sample does not take the 8 GB a 10 GB one is given (many contexts may share the GPU)
    size_t comp_target = GZ_COMP_BYTES;
    if (end > begin) {
        const size_t span = (size_t)(end - begin), usable = GZ_COMP_BYTES - R.bytes - 65536, nbatch = (span + usable - 1) / usable;
        comp_target = std::min(GZ_COMP_BYTES, (span + nbatch - 1) / nbatch + 2 * R.bytes + 65536);
    }
    const size_t out_target = std::min(GZ_OUT_BYTES, std::max<size_t>(6 * comp_target, 8 * R.bytes));
    const double t_alloc0 = now();
    if (c->gz_comp[0].p && (c->gz_comp[0].n < comp_target + 65536 || c->gz_out[0].n < out_target + 65536 + 256))
        CU(c, cudaStreamSynchronize(c->stream));                       // (the buffers grow: nothing may still read the old ones)
    for (int k = 0; k < 2; k++) {
        if ((rc = dev_alloc(c, c->gz_comp[k], comp_target + 65536)) || (rc = dev_alloc(c, c->gz_out[k], out_target + 65536 + 256)) ||
            (rc = dev_alloc(c, c->gz_tab[k], GZ_MAX_BLOCKS * sizeof(BgzfBlock)))) return rc;
        if (!c->gz_tab_host[k]) CU(c, cudaHostAlloc(reinterpret_cast<void**>(&c->gz_tab_host[k]), GZ_MAX_BLOCKS * sizeof(BgzfBlock), cudaHostAllocDefault));
        if (!c->gz_copied[k]) { CU(c, cudaEventCreateWithFlags(&c->gz_copied[k], cudaEventDisableTiming)); CU(c, cudaEventCreateWithFlags(&c->gz_free[k], cudaEventDisableTiming)); }
    }
    const size_t out_cap = c->gz_out[0].n - 65536 - 256;               // (what the buffers hold: at least the targets)
    const double t_alloc = now() - t_alloc0;
    uint64_t off = begin;                                              // file offset of the next unread byte
    std::vector<uint8_t> carry;                                        // the head of a block whose rest is in the next piece
    bool eof = false, stop = false;
    int batch = 0;
    *finished = false;
    c->gz_blocks = 0;
    while (!eof && !stop) {
        const int k = batch & 1;
        // batch k: the copy engine may overwrite its staging buffer only after the previous inflate out of it has finished
        CU(c, cudaStreamWaitEvent(c->copy_stream, c->gz_free[k], 0));
        BgzfBlock* tab = c->gz_tab_host[k];
        // (the host table of batch k-2 was consumed by an H2D copy that completed before gz_free[k] did)
        double t0 = now();
        CU(c, cudaEventSynchronize(c->gz_free[k]));                    // (returns at once for an event that was never recorded)
        t_free += now() - t0;
        uint32_t nb = 0;
        size_t comp_fill = 0, out_fill = 0;
        uint64_t batch_start = off - carry.size();
        while (!eof && !stop && comp_fill + R.bytes + 65536 <= comp_target && out_fill + 4 * R.bytes <= out_cap && nb + 4096 < GZ_MAX_BLOCKS) {
            uint8_t* buf; int idx;
            t0 = now();
            if ((rc = ring_get(c, R, &buf, &idx))) return rc;
            t_ring += now() - t0;
            size_t have = carry.size();
            if (have) memcpy(buf, carry.data(), have);
            carry.clear();
            if (have < R.bytes) {
                t0 = now();
                const size_t want = (size_t)std::min<uint64_t>(R.bytes - have, end - off), g = pread_parallel(fd, buf + have, want, off, T);
                t_read += now() - t0;
                if (g < want || off + g == end) eof = true;
                have += g; off += g;
            }
            t0 = now();
            // whole blocks of this piece
            size_t p = 0;
            while (have - p >= 18) {
                const size_t bs = bgzf_block_size(buf + p, have - p);
                if (!bs) { stop = true; break; }                        // not a BGZF member: the host reader continues from here
                if (bs > have - p) break;
                const uint32_t xlen = (uint32_t)(buf[p + 10] | buf[p + 11] << 8);
                uint32_t isize; memcpy(&isize, buf + p + bs - 4, 4);
                if (bs < 12u + xlen + 8u || isize > 65536u) { stop = true; break; }
                if (out_fill + isize > out_cap || nb >= GZ_MAX_BLOCKS) break;
                if (isize) { tab[nb++] = BgzfBlock{(uint32_t)(comp_fill + p + 12 + xlen), (uint32_t)(bs - 12 - xlen - 8), (uint32_t)out_fill, isize}; out_fill += isize; }
                p += bs;
            }
            t_walk += now() - t0;
            // copy the whole blocks to the device staging buffer; what is left (a partial block) is carried
            if (p) CU(c, cudaMemcpyAsync(reinterpret_cast<uint8_t*>(c->gz_comp[k].p) + comp_fill, buf, p, cudaMemcpyHostToDevice, c->copy_stream));
            R.used[idx] = true;
            CU(c, cudaEventRecord(R.done[idx], c->copy_stream));
            comp_fill += p;
            if (stop) { off = batch_start + comp_fill; carry.clear(); break; }
            if (have > p) {
                if (eof) { stop = true; off = off - (have - p); break; }    // a truncated last block: the host reader delivers its decodable part
                carry.assign(buf + p, buf + have);
            }
            batch_start = off - carry.size() - comp_fill;
        }
        if (stop && !carry.empty()) carry.clear();
        if (nb) {
            CU(c, cudaMemcpyAsync(c->gz_tab[k].p, tab, (size_t)nb * sizeof(BgzfBlock), cudaMemcpyHostToDevice, c->copy_stream));
            CU(c, cudaEventRecord(c->gz_copied[k], c->copy_stream));
            CU(c, cudaStreamWaitEvent(c->stream, c->gz_copied[k], 0));
            // (the output buffer of batch k-2 was parsed by kernels earlier on this same stream)
            if (c->gpu_inflate_mode == 2)
                k_inflate_bgzf<<<(nb + INFLATE_THREADS - 1) / INFLATE_THREADS, INFLATE_THREADS, 0, c->stream>>>(
                    reinterpret_cast<const uint8_t*>(c->gz_comp[k].p), reinterpret_cast<const BgzfBlock*>(c->gz_tab[k].p), nb,
                    reinterpret_cast<uint8_t*>(c->gz_out[k].p), c->d_error);
            else {
                const uint32_t grid = (nb + INFLATE_LANES - 1) / INFLATE_LANES;
                if (!c->gz_attr) {
                    CU(c, cudaFuncSetAttribute(k_inflate_bgzf_lanes<9, 7>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)inflate_smem<9, 7>()));
                    CU(c, cudaFuncSetAttribute(k_inflate_bgzf_lanes<8, 6>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)inflate_smem<8, 6>()));
                    c->gz_attr = true;
                }
                // 9 + 7 index bits: 5 warps per SM; 8 + 6: 11 — the small tables when the batch can fill those warps
                const bool small = c->gpu_inflate_bits ? c->gpu_inflate_bits == 8 : grid > 5u * (uint32_t)c->sm_count;
                if (small)
                    k_inflate_bgzf_lanes<8, 6><<<grid, INFLATE_LANES, inflate_smem<8, 6>(), c->stream>>>(
                        reinterpret_cast<const uint8_t*>(c->gz_comp[k].p), reinterpret_cast<const BgzfBlock*>(c->gz_tab[k].p), nb,
                        reinterpret_cast<uint8_t*>(c->gz_out[k].p), c->d_error);
                else
                    k_inflate_bgzf_lanes<9, 7><<<grid, INFLATE_LANES, inflate_smem<9, 7>(), c->stream>>>(
                        reinterpret_cast<const uint8_t*>(c->gz_comp[k].p), reinterpret_cast<const BgzfBlock*>(c->gz_tab[k].p), nb,
                        reinterpret_cast<uint8_t*>(c->gz_out[k].p), c->d_error);
            }
            c->launches++;
            CU(c, cudaGetLastError());
            CU(c, cudaEventRecord(c->gz_free[k], c->stream));
            c->gz_blocks += nb;
            *total += out_fill;
            if ((rc = device_range(c, reinterpret_cast<const uint8_t*>(c->gz_out[k].p), out_fill, 0))) return rc;
            batch++;
        } else if (!stop && !eof) return fail(c, F2Q_EINTERNAL, "bgzip batch without a block");
    }
    if (debug) fprintf(stderr, "[f2q ingest] bgzf on the device: %d batches, %llu blocks; host thread: buffers %.1f ms, read %.1f ms, ring wait %.1f ms, batch wait %.1f ms, header walk %.1f ms\n",
                       batch, (unsigned long long)c->gz_blocks, t_alloc, t_read, t_ring, t_free, t_walk);
    *resume_off = off;
    *finished = eof && !stop;
    return F2Q_OK;
}

}  // namespace

F2Q_EXPORT int f2q_submit_file(f2q_ctx* c, const char* path, int is_gzip, uint64_t limit_lines, int threads, int* complete, uint64_t* bytes_out) {
    int rc = check_ctx(c); if (rc) return rc;
    if (!c->in_sample) return fail(c, F2Q_ESTATE, "f2q_submit_file outside a sample");
    if (c->sample_failed) return c->sample_failed;
    if (c->closed) return fail(c, F2Q_ESTATE, "stream already closed with is_last");
    if (!path) return fail(c, F2Q_EINVAL, "null path");
    if (complete) *complete = 1;
    if (bytes_out) *bytes_out = 0;
    FILE* f = fopen(path, "rb");
    if (!f) return fail(c, F2Q_EINVAL, std::string("cannot open ") + path + ": " + strerror(errno));
    setvbuf(f, nullptr, _IONBF, 0);
    if ((rc = ensure_ring(c))) { fclose(f); return rc; }
    FileRing& R = *c->file_ring;
    uint64_t total = 0, lines_left = limit_lines;
    bool stop = false;                                                 // preprocess mode: the line limit was reached
    // cut `n` bytes at the line limit; returns the bytes to submit
    auto apply_limit = [&](const uint8_t* p, uint64_t n) -> uint64_t {
        if (!limit_lines) return n;
        const uint8_t* q = p; const uint8_t* e = p + n;
        while (q < e) {
            const uint8_t* nl = static_cast<const uint8_t*>(memchr(q, '\n', (size_t)(e - q)));
            if (!nl) break;
            q = nl + 1;
            if (--lines_left == 0) { stop = true; return (uint64_t)(q - p); }
        }
        return n;
    };
    int idx = 0; uint8_t* buf = nullptr;
    if (!is_gzip) {
        // plain file: `threads` readers pread() the parts of a ring buffer in parallel
        const int fd = fileno(f);
        const int T = std::max(1, std::min(threads, 8));
        uint64_t off = 0;
        for (;;) {
            if ((rc = ring_get(c, R, &buf, &idx))) break;
            const size_t n = pread_parallel(fd, buf, R.bytes, off, T);
            off += n;
            const bool eof = n < R.bytes;
            const uint64_t m = apply_limit(buf, n);
            total += m;
            if ((rc = ring_submit(c, R, idx, m, (eof || stop) ? 1 : 0)) || eof || stop) break;
        }
        fclose(f);
        if (bytes_out) *bytes_out = total;
        return rc;
    }
    // ---- gzip ----
    std::vector<uint8_t> in(8u << 20);
    size_t in_len = fread(in.data(), 1, in.size(), f), in_pos = 0;
    bool in_eof = in_len < in.size();
    auto refill = [&]() {                                              // keep the unread input, append more
        if (in_pos) { memmove(in.data(), in.data() + in_pos, in_len - in_pos); in_len -= in_pos; in_pos = 0; }
        if (!in_eof && in_len < in.size()) { const size_t g = fread(in.data() + in_len, 1, in.size() - in_len, f); if (g < in.size() - in_len) in_eof = true; in_len += g; }
    };
    size_t tail = 0;                                                   // bytes behind the last newline, carried at the start of `buf`
    bool truncated = false, corrupt = false;
    if ((rc = ring_get(c, R, &buf, &idx))) { fclose(f); return rc; }
    size_t fill = 0;                                                   // bytes in buf (the tail included)
    // submit buf[0, cut) (whole lines) and carry the rest into the next ring buffer
    auto flush_lines = [&](bool final_ok) -> int {
        size_t cut = fill;
        if (!final_ok) { const uint8_t* nl = fill ? last_newline(buf, fill) : nullptr; cut = nl ? (size_t)(nl - buf) + 1 : 0; }
        const uint64_t m = apply_limit(buf, cut);
        uint8_t* nb; int nidx;
        int r2 = ring_get(c, R, &nb, &nidx); if (r2) return r2;
        tail = fill - cut;
        if (tail) memcpy(nb, buf + cut, tail);
        total += m;
        if (m || stop) r2 = ring_submit(c, R, idx, m, stop ? 1 : 0);
        buf = nb; idx = nidx; fill = tail;
        return r2;
    };
    bool bgzf = threads > 1 && bgzf_block_size(in.data(), in_len) != 0;
    if (bgzf_block_size(in.data(), in_len) != 0 && c->gpu_inflate && !limit_lines) {
        // a bgzip file that ends with its end-of-file block is inflated on the device; whatever is not a whole BGZF block
        // (a foreign member behind the blocks, a truncated file) is left to the host reader below, from the offset it starts at
        uint8_t tailb[28];
        struct stat sb;
        if (fstat(fileno(f), &sb) == 0 && sb.st_size >= 28 && pread(fileno(f), tailb, 28, sb.st_size - 28) == 28 && memcmp(tailb, BGZF_EOF, 28) == 0) {
            uint64_t resume = 0; bool finished = false;
            if ((rc = submit_bgzf_gpu(c, f, R, threads, 0, (uint64_t)sb.st_size, &total, &resume, &finished))) { fclose(f); return rc; }
            if (finished) {
                fclose(f);
                rc = ring_get(c, R, &buf, &idx);
                if (!rc) rc = ring_submit(c, R, idx, 0, 1);            // close the stream
                if (bytes_out) *bytes_out = total;
                return rc;
            }
            // continue on the host from `resume` (with a ring buffer of our own again: the device path cycled through them)
            if ((rc = ring_get(c, R, &buf, &idx))) { fclose(f); return rc; }
            in_len = 0; in_pos = 0; in_eof = false;
            const ssize_t g = pread(fileno(f), in.data(), in.size(), (off_t)resume);
            in_len = g > 0 ? (size_t)g : 0;
            in_eof = in_len < in.size();
            if (fseek(f, (long)(resume + in_len), SEEK_SET) != 0) { fclose(f); return fail(c, F2Q_EINVAL, "seek failed"); }
            bgzf = threads > 1 && bgzf_block_size(in.data(), in_len) != 0;
        }
    }
    if (bgzf) {
        struct Blk { const uint8_t* src; uint32_t csize, isize; size_t dst; };
        std::vector<Blk> blks;
        bool fell_back = false;
        while (!stop && !rc) {
            // gather whole blocks while they fit into the ring buffer
            blks.clear();
            size_t out = fill;
            for (;;) {
                if (in_len - in_pos < 18 || bgzf_block_size(in.data() + in_pos, in_len - in_pos) > in_len - in_pos) {
                    if (in_eof || !blks.empty()) break;
                    refill();
                    if (in_len - in_pos < 18 && in_eof) break;
                    continue;
                }
                const size_t bs = bgzf_block_size(in.data() + in_pos, in_len - in_pos);
                if (!bs) { fell_back = true; break; }                   // a foreign member: the serial reader takes over
                const uint8_t* p = in.data() + in_pos;
                const uint32_t xlen = (uint32_t)(p[10] | p[11] << 8);
                if (bs < 12u + xlen + 8u) { corrupt = true; break; }
                uint32_t isize; memcpy(&isize, p + bs - 4, 4);
                if (isize > 65536u) { corrupt = true; break; }
                if (out + isize > R.bytes + 65536) break;
                blks.push_back({p + 12 + xlen, (uint32_t)(bs - 12 - xlen - 8), isize, out});
                out += isize; in_pos += bs;
                if (out >= R.bytes) break;
            }
            if (corrupt) break;
            if (blks.empty()) {
                if (fell_back) break;
                if (in_eof) { if (in_len - in_pos) fell_back = true; break; }      // a partial block at the end: the serial reader delivers its decodable part
                continue;
            }
            // inflate them in parallel, each to its final place
            const int T = std::max(1, std::min<int>(threads, (int)blks.size()));
            std::vector<int> bad(T, 0);
            auto work = [&](int t) {
                z_stream z; memset(&z, 0, sizeof(z));
                if (inflateInit2(&z, -15) != Z_OK) { bad[t] = 1; return; }
                for (size_t k = t; k < blks.size(); k += T) {
                    inflateReset(&z);
                    z.next_in = const_cast<Bytef*>(blks[k].src); z.avail_in = blks[k].csize;
                    z.next_out = buf + blks[k].dst; z.avail_out = blks[k].isize;
                    const int zr = inflate(&z, Z_FINISH);
                    if (zr != Z_STREAM_END || z.avail_out != 0) { bad[t] = 1; break; }
                }
                inflateEnd(&z);
            };
            std::vector<std::thread> pool;
            for (int t = 1; t < T; t++) pool.emplace_back(work, t);
            work(0);
            for (auto& th : pool) th.join();
            for (int t = 0; t < T; t++) if (bad[t]) corrupt = true;
            if (corrupt) break;
            fill = out;
            rc = flush_lines(false);
            refill();
        }
        if (fell_back && !corrupt && !rc && !stop) { /* continue below with the serial reader on the remaining input */ }
        else {
            fclose(f);
            if (rc) return rc;
            if (corrupt) { if (complete) *complete = 0; return fail(c, F2Q_EINVAL, std::string(path) + ": corrupted gzip data"); }
            if (!stop) {
                // the last line: complete streams keep an unterminated final line, truncated ones drop it
                if (truncated) { fill = 0; if (complete) *complete = 0; }
                total += fill;
                rc = ring_submit(c, R, idx, fill, 1);
            }
            if (bytes_out) *bytes_out = total;
            return rc;
        }
    }
    {
        z_stream z; memset(&z, 0, sizeof(z));
        if (inflateInit2(&z, 15 + 16) != Z_OK) { fclose(f); return fail(c, F2Q_ENOMEM, "inflateInit2 failed"); }
        bool fresh = true;                                             // at a member boundary, nothing consumed yet
        while (!stop && !rc) {
            if (in_pos == in_len) {
                refill();
                if (in_pos == in_len) { if (!fresh) truncated = true; break; }
            }
            if (fresh) {
                while (in_pos < in_len && in[in_pos] == 0) in_pos++;   // zero padding between members (gzip module behaviour)
                if (in_pos == in_len) continue;
                fresh = false;
            }
            if (fill >= R.bytes) { if ((rc = flush_lines(false))) break; if (fill >= R.bytes) { rc = fail(c, F2Q_ETOOLONG, "a line longer than the ingest buffer"); break; } }
            z.next_in = in.data() + in_pos; z.avail_in = (uInt)std::min<size_t>(in_len - in_pos, 1u << 30);
            z.next_out = buf + fill; z.avail_out = (uInt)(R.bytes - fill);
            const uInt in0 = z.avail_in, out0 = z.avail_out;
            const int zr = inflate(&z, Z_NO_FLUSH);
            in_pos += in0 - z.avail_in; fill += out0 - z.avail_out;
            if (zr == Z_STREAM_END) { inflateReset(&z); fresh = true; }
            else if (zr != Z_OK && zr != Z_BUF_ERROR) { corrupt = true; break; }
            else if (zr == Z_BUF_ERROR && z.avail_in == 0 && in_eof && in_pos == in_len) { truncated = true; break; }
        }
        inflateEnd(&z);
    }
    fclose(f);
    if (rc) return rc;
    if (corrupt) { if (complete) *complete = 0; return fail(c, F2Q_EINVAL, std::string(path) + ": corrupted gzip data"); }
    if (!stop) {
        if (truncated) {
            // every complete line before the break is parsed, the partial one is dropped (fast2q.py:405-407)
            const uint8_t* nl = fill ? last_newline(buf, fill) : nullptr;
            fill = nl ? (size_t)(nl - buf) + 1 : 0;
            if (complete) *complete = 0;
        }
        const uint64_t m = apply_limit(buf, fill);
        total += m;
        rc = ring_submit(c, R, idx, m, 1);
    }
    if (bytes_out) *bytes_out = total;
    return rc;
}

F2Q_EXPORT int f2q_sync(f2q_ctx* c) {
    int rc = check_ctx(c); if (rc) return rc;
    if (c->copy_stream) CU(c, cudaStreamSynchronize(c->copy_stream));
    CU(c, cudaStreamSynchronize(c->stream));
    if (c->async_pending && !c->in_sample) { timing_collect(c); c->async_pending = false; }
    return F2Q_OK;
}

F2Q_EXPORT int f2q_sync_copies(f2q_ctx* c) {
    int rc = check_ctx(c); if (rc) return rc;
    if (c->copy_stream) CU(c, cudaStreamSynchronize(c->copy_stream));
    return F2Q_OK;
}

F2Q_EXPORT int f2q_result_device(f2q_ctx* c, void** dptr, uint64_t* n_words) {
    int rc = check_ctx(c); if (rc) return rc;
    if (!dptr || !n_words) return fail(c, F2Q_EINVAL, "null argument");
    *dptr = c->result.p; *n_words = (uint64_t)c->n_keys + 5;
    return F2Q_OK;
}

F2Q_EXPORT int f2q_end_sample(f2q_ctx* c, uint64_t* counts, uint64_t* stats) {
    int rc = check_ctx(c); if (rc) return rc;
    if (!c->in_sample) return fail(c, F2Q_ESTATE, "f2q_end_sample outside a sample");
    if (!stats) return fail(c, F2Q_EINVAL, "null stats");
    if (!c->closed && (rc = process_device_chunk(c, nullptr, 0, 1))) return rc;     // flush a carried final record
    if ((rc = f2q_sync(c))) return rc;
    c->in_sample = false;
    timing_collect(c);
    uint32_t err = 0;
    CU(c, cudaMemcpy(&err, c->d_error, 4, cudaMemcpyDeviceToHost));
    DevState hs;
    CU(c, cudaMemcpy(&hs, c->dS, sizeof(hs), cudaMemcpyDeviceToHost));
    err |= hs.error;
    c->spec_counts[0] = hs.spec_commits; c->spec_counts[1] = hs.spec_fallbacks;
    c->memo_counts[0] = hs.memo_lookups; c->memo_counts[1] = hs.memo_hits;
    if (c->debug_waits)
        fprintf(stderr, "f2q debug: wait Mcycles  empty(loader) %llu  full(lookback) %llu agg(lookback) %llu  in-lookback %llu | full(consumers) %llu  p0(consumers) %llu | respins %llu | consumer warp Mcycles %llu\n",
                hs.dbg[0] >> 20, hs.dbg[7] >> 20, hs.dbg[1] >> 20, hs.dbg[4] >> 20, hs.dbg[2] >> 20, hs.dbg[3] >> 20, hs.dbg[5], hs.dbg[6] >> 20);
    if (err & ERR_RECORD_TOO_LONG) return fail(c, F2Q_ETOOLONG, "a FASTQ record is longer than carry_bytes; raise it with f2q_set_option");
    if (err & ERR_LOOKBACK_TIMEOUT) return fail(c, F2Q_EINTERNAL, "a device-side wait timed out; this sample's counts are invalid (the context stays usable)");
    if (err & ERR_INFLATE) return fail(c, F2Q_EINVAL, "corrupted gzip data (a bgzip block did not inflate to its promised size on the device)");
    if (err & ERR_EC_FULL) return fail(c, F2Q_EINTERNAL, "an Extract+Count table overflowed (a chunk whose line structure defeated the speculation held more keys than were reserved): rerun with option spec = 0");
    if (err) return fail(c, F2Q_EINTERNAL, "device-side failure, flags=" + std::to_string(err));
    if (counts && c->n_keys) CU(c, cudaMemcpy(counts, c->result.p, (size_t)c->n_keys * 8, cudaMemcpyDeviceToHost));
    CU(c, cudaMemcpy(stats, reinterpret_cast<uint8_t*>(c->result.p) + (size_t)c->n_keys * 8, 5 * 8, cudaMemcpyDeviceToHost));
    return F2Q_OK;
}

F2Q_EXPORT int f2q_end_sample_async(f2q_ctx* c, uint64_t* pinned_out) {
    int rc = check_ctx(c); if (rc) return rc;
    if (!c->in_sample) return fail(c, F2Q_ESTATE, "f2q_end_sample_async outside a sample");
    if (!pinned_out) return fail(c, F2Q_EINVAL, "null output");
    if (c->cfg.mode != F2Q_MODE_COUNT) return fail(c, F2Q_EUNSUPPORTED, "f2q_end_sample_async is for Counter mode (Extract+Count results are drained by f2q_ec_drain)");
    if (!c->closed && (rc = process_device_chunk(c, nullptr, 0, 1))) return rc;     // flush a carried final record
    const size_t n = (size_t)c->n_keys + 5;
    pinned_out[n] = 0;
    CU(c, cudaMemcpyAsync(pinned_out, c->result.p, n * 8, cudaMemcpyDeviceToHost, c->stream));
    CU(c, cudaMemcpyAsync(pinned_out + n, c->d_error, 4, cudaMemcpyDeviceToHost, c->stream));
    CU(c, cudaMemcpyAsync(reinterpret_cast<uint8_t*>(pinned_out + n) + 4, &c->dS->error, 4, cudaMemcpyDeviceToHost, c->stream));
    c->in_sample = false; c->async_pending = true;
    return F2Q_OK;
}

// ---- Extract+Count results ---------------------------------------------------------------------------
// compacts one of the two Extract+Count tables on the device: (tag, count) pairs of its `n` keys land in c->ec_compact behind
// a 16-byte header
static int ec_compact_table(f2q_ctx* c, const unsigned long long* tags, uint32_t ts, const unsigned long long* counts, uint32_t cs, uint64_t cap, uint64_t n) {
    int rc = dev_alloc(c, c->ec_compact, (n + 1) * 16 + 16); if (rc) return rc;
    unsigned long long* d_n = reinterpret_cast<unsigned long long*>(c->ec_compact.p);
    CU(c, cudaMemsetAsync(d_n, 0, 16, c->stream));
    k_ec_compact<<<(unsigned)std::min<uint64_t>((cap + 1023) / 1024, (uint64_t)c->sm_count * 32), 256, 0, c->stream>>>(tags, ts, counts, cs, cap, d_n + 2, d_n);
    c->launches++;
    CU(c, cudaStreamSynchronize(c->stream));
    return F2Q_OK;
}

// number of keys of the packed table and their compacted (tag, count) pairs in c->ec_compact (device)
static int ec_compact_packed(f2q_ctx* c, uint64_t* n_out) {
    *n_out = 0;
    if (!c->ec_pk_cap || !c->ec_meta.p) return F2Q_OK;
    unsigned long long meta[4];
    CU(c, cudaMemcpy(meta, c->ec_meta.p, 32, cudaMemcpyDeviceToHost));
    const uint64_t n = meta[2];
    if (!n) return F2Q_OK;
    const unsigned long long* pk = reinterpret_cast<const unsigned long long*>(c->ec_pk.p);
    int rc = ec_compact_table(c, pk, 2, pk + 1, 2, c->ec_pk_cap, n); if (rc) return rc;
    *n_out = n;
    return F2Q_OK;
}

// the byte-arena table on the host: (slot word, count) pairs of its keys and the arena bytes in use.  The table is sized for
// what a chunk COULD insert (millions of slots), its keys are few: compacted on the device, only they cross the bus.
// NOTE: overwrites c->ec_compact
static int ec_arena_fetch(f2q_ctx* c, std::vector<unsigned long long>& pairs, std::vector<uint8_t>& arena) {
    pairs.clear(); arena.assign(1, 0);
    if (!c->ec_cap || !c->ec_meta.p) return F2Q_OK;
    unsigned long long meta[4];
    CU(c, cudaMemcpy(meta, c->ec_meta.p, 32, cudaMemcpyDeviceToHost));
    if (!meta[1]) return F2Q_OK;
    int rc = ec_compact_table(c, reinterpret_cast<const unsigned long long*>(c->ec_slots.p), 1, reinterpret_cast<const unsigned long long*>(c->ec_counts.p), 1,
                              c->ec_cap, meta[1]);
    if (rc) return rc;
    pairs.resize(2 * meta[1]);
    CU(c, cudaMemcpy(pairs.data(), reinterpret_cast<const uint8_t*>(c->ec_compact.p) + 16, meta[1] * 16, cudaMemcpyDeviceToHost));
    arena.resize(meta[0] + 1);
    if (meta[0]) CU(c, cudaMemcpy(arena.data(), c->ec_arena.p, meta[0], cudaMemcpyDeviceToHost));
    return F2Q_OK;
}

static int ec_fetch(f2q_ctx* c) {
    if (c->ec_drained) return F2Q_OK;
    int rc = f2q_sync(c); if (rc) return rc;
    c->ec_drain_off.assign(1, 0); c->ec_drain_cnt.clear(); c->ec_drain_keys.clear();
    // packed table: compacted on the device, decoded here (2 bits per symbol -> A C T G)
    uint64_t npk = 0;
    if ((rc = ec_compact_packed(c, &npk))) return rc;
    if (npk) {
        std::vector<unsigned long long> pairs(2 * npk);
        CU(c, cudaMemcpy(pairs.data(), reinterpret_cast<const uint8_t*>(c->ec_compact.p) + 16, npk * 16, cudaMemcpyDeviceToHost));
        c->ec_drain_keys.reserve(npk * 24); c->ec_drain_cnt.reserve(npk); c->ec_drain_off.reserve(npk + 1);
        for (uint64_t i = 0; i < npk; i++) {
            const unsigned long long t = pairs[2 * i] - 1;
            const uint32_t len = (uint32_t)(t & 63u);
            const uint64_t codes = t >> 6;
            for (uint32_t k = 0; k < len; k++) c->ec_drain_keys.push_back((uint8_t)("ACTG"[(codes >> (2 * k)) & 3u]));
            c->ec_drain_off.push_back(c->ec_drain_keys.size());
            c->ec_drain_cnt.push_back(pairs[2 * i + 1]);
        }
    }
    if (c->ec_merged) {
        // f2q_ec_merge ran: the byte-arena keys of every rank were merged on the host
        for (size_t k = 0; k < c->ec_extra_cnt.size(); k++) {
            c->ec_drain_keys.insert(c->ec_drain_keys.end(), c->ec_extra_keys.begin() + c->ec_extra_off[k], c->ec_extra_keys.begin() + c->ec_extra_off[k + 1]);
            c->ec_drain_off.push_back(c->ec_drain_keys.size());
            c->ec_drain_cnt.push_back(c->ec_extra_cnt[k]);
        }
    } else {
        std::vector<unsigned long long> ap; std::vector<uint8_t> ar;
        if ((rc = ec_arena_fetch(c, ap, ar))) return rc;
        for (size_t k = 0; k + 1 < ap.size(); k += 2) {
            const uint64_t off = (ap[k] - 1) >> 24, len = (ap[k] - 1) & 0xFFFFFF;
            c->ec_drain_keys.insert(c->ec_drain_keys.end(), ar.begin() + off, ar.begin() + off + len);
            c->ec_drain_off.push_back(c->ec_drain_keys.size());
            c->ec_drain_cnt.push_back(ap[k + 1]);
        }
    }
    c->ec_drained = true;
    return F2Q_OK;
}

F2Q_EXPORT int f2q_ec_size(f2q_ctx* c, uint64_t* n_keys, uint64_t* key_bytes) {
    int rc = check_ctx(c); if (rc) return rc;
    if (c->cfg.mode != F2Q_MODE_EXTRACT_COUNT) return fail(c, F2Q_ESTATE, "not in Extract+Count mode");
    if (!n_keys || !key_bytes) return fail(c, F2Q_EINVAL, "null argument");
    if ((rc = ec_fetch(c))) return rc;
    *n_keys = c->ec_drain_cnt.size(); *key_bytes = c->ec_drain_keys.size();
    return F2Q_OK;
}

F2Q_EXPORT int f2q_ec_drain(f2q_ctx* c, uint8_t* key_bytes, uint64_t* key_offsets, uint64_t* counts) {
    int rc = check_ctx(c); if (rc) return rc;
    if (c->cfg.mode != F2Q_MODE_EXTRACT_COUNT) return fail(c, F2Q_ESTATE, "not in Extract+Count mode");
    if ((rc = ec_fetch(c))) return rc;
    if (!key_offsets || !counts || (!key_bytes && !c->ec_drain_keys.empty())) return fail(c, F2Q_EINVAL, "null argument");
    if (!c->ec_drain_keys.empty()) memcpy(key_bytes, c->ec_drain_keys.data(), c->ec_drain_keys.size());
    memcpy(key_offsets, c->ec_drain_off.data(), c->ec_drain_off.size() * 8);
    if (!c->ec_drain_cnt.empty()) memcpy(counts, c->ec_drain_cnt.data(), c->ec_drain_cnt.size() * 8);
    return F2Q_OK;
}


// ---- multi-GPU: NCCL over NVLink / NVSwitch ---------------------------------------------------------------------------
// The path shards by reads with no data-path collective (SURVEY.md §8e); what crosses GPUs is the RESULT, once per sample:
//   Counter        [counts | stats] summed by one ncclAllReduce(sum, uint64) — merge_feature_dicts, fast2q.py:439-445, 487-495
//   Extract+Count  every rank's key table gathered on every rank (ncclBroadcast per rank inside one group = all-gather of
//                  unequal pieces) and merged on the device into the rank's own packed table (hash insert with count
//                  addition — dict addition again); the few keys of the byte-arena table are merged on the host
// libnccl is loaded at run time (dlopen), so the library itself has no link-time dependency on it: a single-GPU user never
// needs NCCL.  Works for one process per GPU (f2q_comm_unique_id + f2q_comm_init_rank, the id travels by any means the host
// has: MPI, torch.distributed, a file) and for one process driving several contexts (f2q_comm_init).
namespace {

typedef struct f2q_ncclComm* nccl_comm_t;
struct nccl_uid { char internal[128]; };
enum { NCCL_UINT8 = 1, NCCL_UINT64 = 5, NCCL_SUM = 0 };
struct Nccl {
    void* h = nullptr;
    int (*GetUniqueId)(nccl_uid*) = nullptr;
    int (*CommInitRank)(nccl_comm_t*, int, nccl_uid, int) = nullptr;
    int (*CommInitAll)(nccl_comm_t*, int, const int*) = nullptr;
    int (*CommDestroy)(nccl_comm_t) = nullptr;
    int (*AllReduce)(const void*, void*, size_t, int, int, nccl_comm_t, cudaStream_t) = nullptr;
    int (*AllGather)(const void*, void*, size_t, int, nccl_comm_t, cudaStream_t) = nullptr;
    int (*Broadcast)(const void*, void*, size_t, int, int, nccl_comm_t, cudaStream_t) = nullptr;
    int (*GroupStart)() = nullptr;
    int (*GroupEnd)() = nullptr;
    const char* (*GetErrorString)(int) = nullptr;
} g_nccl;
std::mutex g_nccl_mu;

int nccl_load(const char* path) {
    std::lock_guard<std::mutex> l(g_nccl_mu);
    if (g_nccl.h) return F2Q_OK;
    void* h = nullptr;
    if (path && *path) h = dlopen(path, RTLD_NOW | RTLD_GLOBAL);
    if (!h) if (const char* e = getenv("F2Q_NCCL_LIB")) h = dlopen(e, RTLD_NOW | RTLD_GLOBAL);
    if (!h) h = dlopen("libnccl.so.2", RTLD_NOW | RTLD_GLOBAL);
    if (!h) h = dlopen("libnccl.so", RTLD_NOW | RTLD_GLOBAL);
    if (!h) return fail(nullptr, F2Q_EUNSUPPORTED, std::string("libnccl could not be loaded (pass its path to f2q_comm_load or set F2Q_NCCL_LIB): ") + (dlerror() ? dlerror() : ""));
    bool ok = true;
    auto sym = [&](const char* n) { void* p = dlsym(h, n); if (!p) ok = false; return p; };
    g_nccl.GetUniqueId = reinterpret_cast<decltype(g_nccl.GetUniqueId)>(sym("ncclGetUniqueId"));
    g_nccl.CommInitRank = reinterpret_cast<decltype(g_nccl.CommInitRank)>(sym("ncclCommInitRank"));
    g_nccl.CommInitAll = reinterpret_cast<decltype(g_nccl.CommInitAll)>(sym("ncclCommInitAll"));
    g_nccl.CommDestroy = reinterpret_cast<decltype(g_nccl.CommDestroy)>(sym("ncclCommDestroy"));
    g_nccl.AllReduce = reinterpret_cast<decltype(g_nccl.AllReduce)>(sym("ncclAllReduce"));
    g_nccl.AllGather = reinterpret_cast<decltype(g_nccl.AllGather)>(sym("ncclAllGather"));
    g_nccl.Broadcast = reinterpret_cast<decltype(g_nccl.Broadcast)>(sym("ncclBroadcast"));
    g_nccl.GroupStart = reinterpret_cast<decltype(g_nccl.GroupStart)>(sym("ncclGroupStart"));
    g_nccl.GroupEnd = reinterpret_cast<decltype(g_nccl.GroupEnd)>(sym("ncclGroupEnd"));
    g_nccl.GetErrorString = reinterpret_cast<decltype(g_nccl.GetErrorString)>(sym("ncclGetErrorString"));
    if (!ok) { dlclose(h); return fail(nullptr, F2Q_EUNSUPPORTED, "libnccl lacks a symbol this library needs"); }
    g_nccl.h = h;
    return F2Q_OK;
}

#define NC(ctx, call)                                                                                              \
    do {                                                                                                           \
        int r__ = (call);                                                                                          \
        if (r__ != 0) return fail(ctx, F2Q_ECUDA, std::string(#call) + ": " + (g_nccl.GetErrorString ? g_nccl.GetErrorString(r__) : "NCCL error")); \
    } while (0)

int comm_check(f2q_ctx** ctxs, int n) {
    if (!ctxs || n < 1) return F2Q_EINVAL;
    for (int i = 0; i < n; i++) {
        if (!ctxs[i]) return F2Q_EINVAL;
        if (ctxs[i]->sticky) return ctxs[i]->sticky;
        if (!ctxs[i]->comm) return fail(ctxs[i], F2Q_ESTATE, "the context has no communicator (f2q_comm_init / f2q_comm_init_rank first)");
    }
    return F2Q_OK;
}

// merged pairs (tag, count) of every rank -> this rank's packed table (emptied first)
__global__ void __launch_bounds__(256) k_ec_merge_pairs(EcTable E, Outputs O, const unsigned long long* __restrict__ pairs, uint64_t n) {
    for (uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x; i < n; i += (uint64_t)gridDim.x * blockDim.x) {
        const unsigned long long tag = pairs[2 * i];
        if (tag) ec_pk_insert(E, O, tag, pairs[2 * i + 1]);
    }
}

}  // namespace

F2Q_EXPORT int f2q_comm_load(const char* libnccl_path) { return nccl_load(libnccl_path); }

F2Q_EXPORT int f2q_comm_unique_id(uint8_t* id128) {
    if (!id128) return fail(nullptr, F2Q_EINVAL, "null argument");
    int rc = nccl_load(nullptr); if (rc) return rc;
    nccl_uid u;
    NC(nullptr, g_nccl.GetUniqueId(&u));
    memcpy(id128, u.internal, 128);
    return F2Q_OK;
}

F2Q_EXPORT int f2q_comm_init_rank(f2q_ctx* c, const uint8_t* id128, int nranks, int rank) {
    int rc = check_ctx(c); if (rc) return rc;
    if (!id128 || nranks < 1 || rank < 0 || rank >= nranks) return fail(c, F2Q_EINVAL, "bad communicator arguments");
    if (c->comm) return fail(c, F2Q_ESTATE, "the context already has a communicator");
    if ((rc = nccl_load(nullptr))) return fail(c, rc, f2q_last_error(nullptr));
    nccl_uid u;
    memcpy(u.internal, id128, 128);
    nccl_comm_t comm = nullptr;
    NC(c, g_nccl.CommInitRank(&comm, nranks, u, rank));
    c->comm = comm; c->comm_rank = rank; c->comm_size = nranks; c->comm_owner = true;
    return F2Q_OK;
}

F2Q_EXPORT int f2q_comm_init(f2q_ctx** ctxs, int n) {
    if (!ctxs || n < 1) return fail(nullptr, F2Q_EINVAL, "bad communicator arguments");
    int rc = nccl_load(nullptr); if (rc) return rc;
    std::vector<int> devs(n);
    for (int i = 0; i < n; i++) {
        if (!ctxs[i] || ctxs[i]->comm) return fail(ctxs[i], F2Q_ESTATE, "null context, or the context already has a communicator");
        devs[i] = ctxs[i]->device;
        for (int j = 0; j < i; j++) if (devs[j] == devs[i]) return fail(ctxs[i], F2Q_EINVAL, "f2q_comm_init needs one context per device");
    }
    std::vector<nccl_comm_t> comms(n, nullptr);
    NC(ctxs[0], g_nccl.CommInitAll(comms.data(), n, devs.data()));
    for (int i = 0; i < n; i++) { ctxs[i]->comm = comms[i]; ctxs[i]->comm_rank = i; ctxs[i]->comm_size = n; ctxs[i]->comm_owner = true; }
    return F2Q_OK;
}

F2Q_EXPORT int f2q_comm_destroy(f2q_ctx* c) {
    if (!c) return F2Q_EINVAL;
    if (c->comm && c->comm_owner && g_nccl.CommDestroy) { cudaSetDevice(c->device); if (c->stream) cudaStreamSynchronize(c->stream); g_nccl.CommDestroy(static_cast<nccl_comm_t>(c->comm)); }
    c->comm = nullptr; c->comm_size = 1; c->comm_rank = 0; c->comm_owner = false;
    return F2Q_OK;
}

// another context of the same device and process uses `from`'s communicator (which must outlive it): creating a communicator
// costs a rendezvous, a process that runs several configurations needs only one
F2Q_EXPORT int f2q_comm_share(f2q_ctx* c, f2q_ctx* from) {
    int rc = check_ctx(c); if (rc) return rc;
    if (!from || !from->comm) return fail(c, F2Q_ESTATE, "the source context has no communicator");
    if (c->comm) return fail(c, F2Q_ESTATE, "the context already has a communicator");
    if (c->device != from->device) return fail(c, F2Q_EINVAL, "a communicator can only be shared by contexts of one device");
    c->comm = from->comm; c->comm_rank = from->comm_rank; c->comm_size = from->comm_size; c->comm_owner = false;
    return F2Q_OK;
}

// in-place sum over all ranks of [counts[n_keys] | stats[5]], stream-ordered on each context's stream (call it after the
// last submit of the sample and before f2q_end_sample / f2q_end_sample_async)
F2Q_EXPORT int f2q_allreduce_counts(f2q_ctx** ctxs, int n) {
    int rc = comm_check(ctxs, n); if (rc) return rc;
    for (int i = 0; i < n; i++) {
        f2q_ctx* c = ctxs[i];
        if (!c->in_sample) return fail(c, F2Q_ESTATE, "f2q_allreduce_counts outside a sample");
        if (!c->closed) { cudaSetDevice(c->device); if ((rc = process_device_chunk(c, nullptr, 0, 1))) return rc; }      // flush a carried final record first
    }
    NC(ctxs[0], g_nccl.GroupStart());
    for (int i = 0; i < n; i++) {
        f2q_ctx* c = ctxs[i];
        cudaSetDevice(c->device);
        const int r = g_nccl.AllReduce(c->result.p, c->result.p, (size_t)c->n_keys + 5, NCCL_UINT64, NCCL_SUM, static_cast<nccl_comm_t>(c->comm), c->stream);
        if (r != 0) { g_nccl.GroupEnd(); return fail(c, F2Q_ECUDA, std::string("ncclAllReduce: ") + g_nccl.GetErrorString(r)); }
        c->launches++;
    }
    NC(ctxs[0], g_nccl.GroupEnd());
    return F2Q_OK;
}

// Extract+Count: after it every rank's tables hold the keys of ALL ranks with summed counts (f2q_ec_size / f2q_ec_drain then
// return the merged table everywhere).  The five statistics are NOT touched: f2q_allreduce_counts sums them.
F2Q_EXPORT int f2q_ec_merge(f2q_ctx** ctxs, int n) {
    int rc = comm_check(ctxs, n); if (rc) return rc;
    const int W = ctxs[0]->comm_size;
    const bool dbg = getenv("F2Q_DEBUG_MERGE") != nullptr;
    auto now = []() { return std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now().time_since_epoch()).count(); };
    double tp = now();
    auto lap = [&](const char* what) { if (dbg) { for (int i = 0; i < n; i++) { cudaSetDevice(ctxs[i]->device); cudaStreamSynchronize(ctxs[i]->stream); } const double t = now(); fprintf(stderr, "f2q_ec_merge: %-28s %8.2f ms\n", what, t - tp); tp = t; } };
    struct Local { uint64_t npk = 0; std::vector<uint8_t> blob; };     // blob: arena keys as [len u32 | count u64 | bytes]...
    std::vector<Local> L(n);
    std::vector<DevBuf> sizes_d(n), gathered(n), blob_d(n), blobs_all(n);
    std::vector<std::vector<unsigned long long>> sizes_h(n, std::vector<unsigned long long>(2 * (size_t)W, 0));
    auto cleanup = [&]() { for (int i = 0; i < n; i++) { cudaSetDevice(ctxs[i]->device); sizes_d[i].release(); gathered[i].release(); blob_d[i].release(); blobs_all[i].release(); } };
    // 1. local tables: packed keys compacted on the device, arena keys packed into a blob on the host (they are few)
    for (int i = 0; i < n; i++) {
        f2q_ctx* c = ctxs[i];
        if (c->cfg.mode != F2Q_MODE_EXTRACT_COUNT) return fail(c, F2Q_ESTATE, "not in Extract+Count mode");
        if (c->comm_size != W) return fail(c, F2Q_EINVAL, "contexts of different communicators");
        cudaSetDevice(c->device);
        if (c->in_sample && !c->closed && (rc = process_device_chunk(c, nullptr, 0, 1))) return rc;
        CU(c, cudaStreamSynchronize(c->stream));
        {
            std::vector<unsigned long long> ap; std::vector<uint8_t> ar;
            if ((rc = ec_arena_fetch(c, ap, ar))) return rc;           // (first: it uses the compaction buffer the packed keys stay in)
            for (size_t k = 0; k + 1 < ap.size(); k += 2) {
                const uint64_t off = (ap[k] - 1) >> 24; const uint32_t len = (uint32_t)((ap[k] - 1) & 0xFFFFFF);
                const uint64_t cnt = ap[k + 1];
                const uint8_t* p4 = reinterpret_cast<const uint8_t*>(&len); const uint8_t* p8 = reinterpret_cast<const uint8_t*>(&cnt);
                L[i].blob.insert(L[i].blob.end(), p4, p4 + 4); L[i].blob.insert(L[i].blob.end(), p8, p8 + 8);
                L[i].blob.insert(L[i].blob.end(), ar.begin() + off, ar.begin() + off + len);
            }
        }
        if ((rc = ec_compact_packed(c, &L[i].npk))) return rc;
    }
    lap("local tables");
    // 2. sizes of every rank's pieces (two words per rank: packed pairs, blob bytes)
    for (int i = 0; i < n; i++) {
        f2q_ctx* c = ctxs[i];
        cudaSetDevice(c->device);
        if ((rc = dev_alloc(c, sizes_d[i], 16 * (size_t)W + 16))) { cleanup(); return rc; }
        unsigned long long mine[2] = {L[i].npk, L[i].blob.size()};
        CU(c, cudaMemcpyAsync(reinterpret_cast<uint8_t*>(sizes_d[i].p) + 16 * (size_t)W, mine, 16, cudaMemcpyHostToDevice, c->stream));
    }
    NC(ctxs[0], g_nccl.GroupStart());
    for (int i = 0; i < n; i++) {
        f2q_ctx* c = ctxs[i];
        cudaSetDevice(c->device);
        g_nccl.AllGather(reinterpret_cast<uint8_t*>(sizes_d[i].p) + 16 * (size_t)W, sizes_d[i].p, 2, NCCL_UINT64, static_cast<nccl_comm_t>(c->comm), c->stream);
        c->launches++;
    }
    NC(ctxs[0], g_nccl.GroupEnd());
    for (int i = 0; i < n; i++) {
        f2q_ctx* c = ctxs[i];
        cudaSetDevice(c->device);
        CU(c, cudaMemcpyAsync(sizes_h[i].data(), sizes_d[i].p, 16 * (size_t)W, cudaMemcpyDeviceToHost, c->stream));
        CU(c, cudaStreamSynchronize(c->stream));
    }
    lap("sizes all-gather");
    // 3. the pieces themselves: rank r broadcasts its piece into everybody's buffer at r's offset (one NCCL group)
    std::vector<uint64_t> tot_pk(n, 0), tot_blob(n, 0);
    for (int i = 0; i < n; i++) {
        f2q_ctx* c = ctxs[i];
        cudaSetDevice(c->device);
        for (int r = 0; r < W; r++) { tot_pk[i] += sizes_h[i][2 * r]; tot_blob[i] += sizes_h[i][2 * r + 1]; }
        if ((rc = dev_alloc(c, gathered[i], (tot_pk[i] + 1) * 16)) || (rc = dev_alloc(c, blob_d[i], L[i].blob.size() + 16)) ||
            (rc = dev_alloc(c, blobs_all[i], tot_blob[i] + 16))) { cleanup(); return rc; }
        if (!L[i].blob.empty()) CU(c, cudaMemcpyAsync(blob_d[i].p, L[i].blob.data(), L[i].blob.size(), cudaMemcpyHostToDevice, c->stream));
    }
    NC(ctxs[0], g_nccl.GroupStart());
    for (int i = 0; i < n; i++) {
        f2q_ctx* c = ctxs[i];
        cudaSetDevice(c->device);
        uint64_t opk = 0, ob = 0;
        for (int r = 0; r < W; r++) {
            const uint64_t npk = sizes_h[i][2 * r], nb = sizes_h[i][2 * r + 1];
            const void* send_pk = reinterpret_cast<const uint8_t*>(c->ec_compact.p) + 16;      // (only read on the root)
            if (npk) g_nccl.Broadcast(r == c->comm_rank ? send_pk : reinterpret_cast<uint8_t*>(gathered[i].p) + opk * 16, reinterpret_cast<uint8_t*>(gathered[i].p) + opk * 16, npk * 2, NCCL_UINT64, r,
                                      static_cast<nccl_comm_t>(c->comm), c->stream);
            if (nb) g_nccl.Broadcast(r == c->comm_rank ? blob_d[i].p : reinterpret_cast<uint8_t*>(blobs_all[i].p) + ob, reinterpret_cast<uint8_t*>(blobs_all[i].p) + ob, nb, NCCL_UINT8, r,
                                     static_cast<nccl_comm_t>(c->comm), c->stream);
            opk += npk; ob += nb;
            c->launches++;
        }
    }
    NC(ctxs[0], g_nccl.GroupEnd());
    lap("pieces broadcast");
    // 4. merge: the packed table is emptied and every gathered pair inserted (counts add); the arena blobs merge on the host
    for (int i = 0; i < n; i++) {
        f2q_ctx* c = ctxs[i];
        cudaSetDevice(c->device);
        // room for every gathered key (nothing is in flight: the counters are exact)
        while (!c->ec_pend.empty()) { if (c->ec_pend.front().ev) { cudaEventSynchronize(c->ec_pend.front().ev); c->ec_events.push_back(c->ec_pend.front().ev); } c->ec_pend.pop_front(); }
        if (c->ec_meta.p) {
            CU(c, cudaStreamSynchronize(c->stream));
            if (c->ec_pk.p) CU(c, cudaMemsetAsync(c->ec_pk.p, 0, c->ec_pk_cap * 16, c->stream));
            CU(c, cudaMemsetAsync(reinterpret_cast<uint8_t*>(c->ec_meta.p) + 16, 0, 8, c->stream));
            unsigned long long meta[4];
            CU(c, cudaMemcpyAsync(meta, c->ec_meta.p, 32, cudaMemcpyDeviceToHost, c->stream));
            CU(c, cudaStreamSynchronize(c->stream));
            c->ec_known[0] = meta[0]; c->ec_known[1] = meta[1]; c->ec_known[2] = 0;
        }
        if ((rc = ec_reserve(c, tot_pk[i], 0, 0))) { cleanup(); return rc; }
        if (tot_pk[i]) {
            k_ec_merge_pairs<<<(unsigned)std::min<uint64_t>((tot_pk[i] + 255) / 256, (uint64_t)c->sm_count * 16), 256, 0, c->stream>>>(
                c->E, outputs_of(c), reinterpret_cast<const unsigned long long*>(gathered[i].p), tot_pk[i]);
            c->launches++;
        }
        if ((rc = ec_after_chunk(c))) { cleanup(); return rc; }
        std::vector<uint8_t> all(tot_blob[i] + 1);
        if (tot_blob[i]) CU(c, cudaMemcpyAsync(all.data(), blobs_all[i].p, tot_blob[i], cudaMemcpyDeviceToHost, c->stream));
        CU(c, cudaStreamSynchronize(c->stream));
        std::map<std::string, uint64_t> extra;                         // (ordered: every rank gets the same table)
        for (uint64_t p = 0; p + 12 <= tot_blob[i];) {
            uint32_t len; uint64_t cnt;
            memcpy(&len, all.data() + p, 4); memcpy(&cnt, all.data() + p + 4, 8);
            extra[std::string(reinterpret_cast<const char*>(all.data() + p + 12), len)] += cnt;
            p += 12 + len;
        }
        c->ec_extra_keys.clear(); c->ec_extra_off.assign(1, 0); c->ec_extra_cnt.clear();
        for (auto& kv : extra) {
            c->ec_extra_keys.insert(c->ec_extra_keys.end(), kv.first.begin(), kv.first.end());
            c->ec_extra_off.push_back(c->ec_extra_keys.size());
            c->ec_extra_cnt.push_back(kv.second);
        }
        c->ec_merged = true; c->ec_drained = false;
    }
    lap("device merge");
    cleanup();
    lap("free");
    return F2Q_OK;
}

// ---- one file, several contexts ------------------------------------------------------------------------------------
// f2q_submit_file_sharded (DESIGN.md §5): the file is cut into byte ranges, one per context, and every context parses its
// range on its own host thread and its own stream, exactly as f2q_submit_file would.  A range that starts mid-file guesses
// its first record start on the device (k_shard_head); the guesses are verified on the host once every range is parsed,
// the bytes around the cuts (the head before each guess, the partial record behind each range's last whole record) are
// parsed on ctxs[0] in file order, and the other contexts' results are added into ctxs[0].  Anything that cannot be split
// or verified is parsed again, whole, on ctxs[0].
namespace {

constexpr uint64_t SHARD_MIN_BYTES = 64ull << 20;

// file offsets of the blocks of a bgzip file, from their 18-byte headers alone; false unless the file is whole BGZF blocks
// that end with the end-of-file block (a foreign gzip member or a truncated block leave nothing to cut at)
bool bgzf_block_starts(int fd, uint64_t size, std::vector<uint64_t>& starts) {
    starts.clear();
    uint8_t hdr[18];
    for (uint64_t off = 0; off < size;) {
        if (size - off < 28 || pread(fd, hdr, 18, (off_t)off) != 18) return false;
        const size_t bs = bgzf_block_size(hdr, 18);
        if (!bs || bs > size - off) return false;
        starts.push_back(off);
        off += bs;
    }
    uint8_t eof[28];
    return !starts.empty() && starts.back() == size - 28 && pread(fd, eof, 28, (off_t)(size - 28)) == 28 && memcmp(eof, BGZF_EOF, 28) == 0;
}

struct ShardJob { uint64_t beg = 0, end = 0; bool first = false, last = false; int threads = 1; int rc = F2Q_OK; uint64_t bytes = 0; };

// one range of the file -> this context's sample: the first range is parsed as the start of the stream, the last one closes
// it, the others end with their partial record carried (k_carry) and begin with k_shard_head
int shard_run(f2q_ctx* c, const char* path, bool gz, ShardJob& J) {
    int rc = check_ctx(c); if (rc) return rc;
    FILE* f = fopen(path, "rb");
    if (!f) return fail(c, F2Q_EINVAL, std::string("cannot open ") + path + ": " + strerror(errno));
    setvbuf(f, nullptr, _IONBF, 0);
    if ((rc = ensure_ring(c))) { fclose(f); return rc; }
    FileRing& R = *c->file_ring;
    c->shard_head_pending = !J.first;
    if (!gz) {
        // plain file: pread straight into this context's ring
        const int fd = fileno(f);
        for (uint64_t off = J.beg; off < J.end && !rc;) {
            uint8_t* buf; int idx;
            if ((rc = ring_get(c, R, &buf, &idx))) break;
            const size_t want = (size_t)std::min<uint64_t>(R.bytes, J.end - off), got = pread_parallel(fd, buf, want, off, J.threads);
            if (got < want) { rc = fail(c, F2Q_EINVAL, std::string(path) + ": the file ended early (did it change?)"); break; }
            off += got; J.bytes += got;
            rc = ring_submit(c, R, idx, got, (J.last && off == J.end) ? 1 : 0);
        }
    } else {
        uint64_t resume = 0; bool finished = false;
        rc = submit_bgzf_gpu(c, f, R, J.threads, J.beg, J.end, &J.bytes, &resume, &finished);
        if (!rc && !finished) { c->shard_noguess = true; rc = fail(c, F2Q_EINVAL, "a shard is not whole BGZF blocks"); }
        if (!rc && J.last) rc = process_device_chunk(c, nullptr, 0, 1);
    }
    fclose(f);
    c->shard_head_pending = false;
    return rc;
}

int copy_to(f2q_ctx* dst, void* d, const f2q_ctx* src, const void* s, size_t n) {
    if (!n) return F2Q_OK;
    if (dst->device == src->device) CU(dst, cudaMemcpyAsync(d, s, n, cudaMemcpyDeviceToDevice, dst->stream));
    else CU(dst, cudaMemcpyPeerAsync(d, dst->device, s, src->device, n, dst->stream));
    return F2Q_OK;
}

// the arena keys of one context's Extract+Count table, added into `extra` (host)
int ec_arena_collect(f2q_ctx* c, std::map<std::string, uint64_t>& extra) {
    std::vector<unsigned long long> ap; std::vector<uint8_t> ar;
    int rc = ec_arena_fetch(c, ap, ar); if (rc) return rc;
    for (size_t k = 0; k + 1 < ap.size(); k += 2) {
        const uint64_t off = (ap[k] - 1) >> 24, len = (ap[k] - 1) & 0xFFFFFF;
        extra[std::string(reinterpret_cast<const char*>(ar.data() + off), len)] += ap[k + 1];
    }
    return F2Q_OK;
}

}  // namespace

F2Q_EXPORT int f2q_submit_file_sharded(f2q_ctx** ctxs, int n, const char* path, int is_gzip, const uint64_t* cuts, int threads,
                                       int* complete, uint64_t* bytes_out) {
    if (!ctxs || n < 1 || !ctxs[0]) return fail(nullptr, F2Q_EINVAL, "f2q_submit_file_sharded: no contexts");
    f2q_ctx* c0 = ctxs[0];
    int rc;
    for (int i = 0; i < n; i++) {
        f2q_ctx* c = ctxs[i];
        if (!c) return fail(c0, F2Q_EINVAL, "null context");
        for (int j = 0; j < i; j++) if (ctxs[j] == c) return fail(c0, F2Q_EINVAL, "a context appears twice");
        if ((rc = check_ctx(c))) return rc;
        if (!c->in_sample) return fail(c0, F2Q_ESTATE, "f2q_submit_file_sharded: context " + std::to_string(i) + " is not inside a sample");
        if (c->sample_failed) return c->sample_failed;
        if (c->closed) return fail(c0, F2Q_ESTATE, "f2q_submit_file_sharded: the stream of context " + std::to_string(i) + " is already closed");
        if (memcmp(&c->cfg, &c0->cfg, sizeof(f2q_config)) != 0 || c->n_keys != c0->n_keys || c->lib_hash != c0->lib_hash)
            return fail(c0, F2Q_EINVAL, "f2q_submit_file_sharded: context " + std::to_string(i) + " has another configuration or library than context 0");
    }
    if (!path) return fail(c0, F2Q_EINVAL, "null path");
    if (cuts) for (int k = 1; k + 1 < n; k++) if (cuts[k] < cuts[k - 1]) return fail(c0, F2Q_EINVAL, "cuts must not decrease");
    if (complete) *complete = 1;
    if (bytes_out) *bytes_out = 0;
    const bool gz = is_gzip != 0;
    // ---- the plan: range bounds [0 = b_0 < b_1 < ... < b_s = size], empty ranges dropped
    std::vector<uint64_t> bounds(1, 0);
    bool shardable = true;
    {
        FILE* f = fopen(path, "rb");
        if (!f) return fail(c0, F2Q_EINVAL, std::string("cannot open ") + path + ": " + strerror(errno));
        struct stat sb;
        const uint64_t size = fstat(fileno(f), &sb) == 0 ? (uint64_t)sb.st_size : 0;
        std::vector<uint64_t> starts;
        if (gz) {
            // only bgzip can be cut (at block starts; ordinary gzip is one deflate stream), and only when inflated on the device
            uint8_t h[18];
            shardable = c0->gpu_inflate && pread(fileno(f), h, 18, 0) == 18 && bgzf_block_size(h, 18) && bgzf_block_starts(fileno(f), size, starts);
        }
        fclose(f);
        const int want = cuts ? n : (int)std::min<uint64_t>((uint64_t)n, std::max<uint64_t>(1, size / SHARD_MIN_BYTES));
        for (int k = 1; shardable && k < want; k++) {
            uint64_t x = std::min(size, cuts ? cuts[k - 1] : size / want * k);
            if (gz) {
                // the next block start; none before the end-of-file block: the end of the file
                auto it = std::lower_bound(starts.begin(), starts.end() - 1, x);
                x = it == starts.end() - 1 ? size : *it;
            }
            if (x > bounds.back() && x < size) bounds.push_back(x);
        }
        bounds.push_back(size);
    }
    const int ns = (int)bounds.size() - 1;
    // ---- the other contexts end empty and closed; ctxs[0] takes the whole file when there is one range or a fallback
    auto close_others = [&]() -> int {
        for (int k = 1; k < n; k++) {
            f2q_ctx* c = ctxs[k];
            c->ch_from_device = false;                                  // (its geometry was sniffed behind a shard head)
            int r = f2q_begin_sample(c); if (r) return r;
            c->closed = true;
        }
        return F2Q_OK;
    };
    auto whole_on_ctx0 = [&](bool fallback) -> int {
        int r = close_others(); if (r) return r;
        if (fallback && (r = f2q_begin_sample(c0))) return r;
        r = f2q_submit_file(c0, path, is_gzip, 0, threads, complete, bytes_out);
        c0->last_shards = 1; c0->last_shard_fallback = fallback ? 1 : 0;
        return r;
    };
    if (!shardable || ns < 2) return whole_on_ctx0(!shardable);

    // ---- every range on its own context and host thread
    std::atomic<bool> abort{false};
    std::vector<ShardJob> J(ns);
    for (int k = 0; k < ns; k++) {
        J[k].beg = bounds[k]; J[k].end = bounds[k + 1]; J[k].first = k == 0; J[k].last = k == ns - 1;
        J[k].threads = std::max(1, threads / ns);
        ctxs[k]->shard_abort = &abort; ctxs[k]->shard_noguess = false;
    }
    auto run = [&](int k) {
        J[k].rc = shard_run(ctxs[k], path, gz, J[k]);
        if (ctxs[k]->shard_noguess) abort = true;                       // the others need not finish: the file is parsed again
    };
    {
        std::vector<std::thread> pool;
        for (int k = 1; k < ns; k++) pool.emplace_back(run, k);
        run(0);
        for (auto& t : pool) t.join();
    }
    bool noguess = false;
    for (int k = 0; k < ns; k++) { ctxs[k]->shard_abort = nullptr; noguess = noguess || ctxs[k]->shard_noguess; }
    if (noguess) return whole_on_ctx0(true);
    for (int k = 0; k < ns; k++)
        if (J[k].rc) { if (k) c0->err = ctxs[k]->err; return J[k].rc; }
    std::vector<DevState> S(ns);
    bool dev_error = false;                                            // a range failed on the device (a record longer than carry_bytes ...)
    for (int k = 0; k < ns; k++) {
        f2q_ctx* c = ctxs[k];
        uint32_t err = 0;
        cudaSetDevice(c->device);
        CU(c, cudaStreamSynchronize(c->stream));
        CU(c, cudaMemcpy(&S[k], c->dS, sizeof(DevState), cudaMemcpyDeviceToHost));
        CU(c, cudaMemcpy(&err, c->d_error, 4, cudaMemcpyDeviceToHost));
        dev_error = dev_error || err || S[k].error;
    }
    // ---- verification.  Records are every 4 lines from byte 0.  Range 0 starts at byte 0, so at line phase 0.  When range k-1
    // is parsed at the right phase, its carried partial record holds tail_nl[k-1] lines of the record that range k's head
    // completes; range k's guess is a record start exactly when the head adds the missing lines, (tail_nl[k-1] + head_nl[k])
    // % 4 == 0 (head_nl is 1..4, so the head is exactly those lines).  Then range k is parsed at the right phase too: by
    // induction every guess is right, and every record is parsed exactly once, either inside a range or from a tail + head.
    // A range that failed on the device fails the sample: no check, no stitch, its error words reach ctxs[0] with the sum below
    // (a second pass on ctxs[0] could hide the failure where its own chunks happen to be cut elsewhere).
    for (int k = 1; k < ns && !dev_error; k++)
        if (!S[k].head_ok || (S[k - 1].tail_nl + S[k].head_nl) % 4 != 0) return whole_on_ctx0(true);

    // ---- stitch: ctxs[0] (carrying range 0's tail) is fed H1, T1, H2, ..., T(s-2), H(s-1) and closed
    std::vector<std::vector<uint8_t>> piece;
    for (int k = 1; k < ns && !dev_error; k++) {
        f2q_ctx* c = ctxs[k];
        cudaSetDevice(c->device);
        piece.emplace_back(S[k].head_len);
        if (S[k].head_len) CU(c0, cudaMemcpy(piece.back().data(), c->shard_head.p, S[k].head_len, cudaMemcpyDeviceToHost));
        if (k == ns - 1) break;
        piece.emplace_back(S[k].tail_len);
        if (S[k].tail_len) CU(c0, cudaMemcpy(piece.back().data(), c->carry.p, S[k].tail_len, cudaMemcpyDeviceToHost));
    }
    if ((rc = check_ctx(c0))) return rc;
    for (auto& p : piece)
        if (!p.empty() && (rc = submit_host(c0, p.data(), p.size(), 0, nullptr))) { c0->sample_failed = rc; return rc; }
    if ((rc = process_device_chunk(c0, nullptr, 0, 1))) { c0->sample_failed = rc; return rc; }

    // ---- sum: [counts | stats] and the error words of every other range into ctxs[0] (their streams are idle: synchronised above)
    const uint64_t nw = (uint64_t)c0->n_keys + 5;
    DevBuf recv, recv_pk;
    auto release = [&]() { cudaSetDevice(c0->device); cudaStreamSynchronize(c0->stream); recv.release(); recv_pk.release(); };
    if ((rc = dev_alloc(c0, recv, nw * 8 + 16))) return rc;
    uint32_t* recv_err = reinterpret_cast<uint32_t*>(reinterpret_cast<uint8_t*>(recv.p) + nw * 8);
    for (int k = 1; k < ns; k++) {
        f2q_ctx* c = ctxs[k];
        if ((rc = copy_to(c0, recv.p, c, c->result.p, nw * 8)) || (rc = copy_to(c0, recv_err, c, c->d_error, 4)) ||
            (rc = copy_to(c0, recv_err + 1, c, &c->dS->error, 4))) { release(); return rc; }
        k_shard_sum<<<(unsigned)std::min<uint64_t>((nw + 255) / 256, (uint64_t)c0->sm_count * 4), 256, 0, c0->stream>>>(
            reinterpret_cast<unsigned long long*>(c0->result.p), reinterpret_cast<const unsigned long long*>(recv.p), nw, c0->d_error, c0->dS, recv_err);
        c0->launches++;
        CU(c0, cudaGetLastError());
    }
    if (c0->cfg.mode == F2Q_MODE_EXTRACT_COUNT) {
        // Extract+Count: every other packed table compacted on its device, copied over and inserted into ctxs[0]'s (counts
        // add); the few byte-arena keys of every context, ctxs[0]'s own included, merge on the host (as f2q_ec_merge does)
        std::map<std::string, uint64_t> extra;
        CU(c0, cudaStreamSynchronize(c0->stream));
        if ((rc = ec_arena_collect(c0, extra))) { release(); return rc; }
        for (int k = 1; k < ns; k++) {
            f2q_ctx* c = ctxs[k];
            uint64_t npk = 0;
            cudaSetDevice(c->device);
            if ((rc = ec_arena_collect(c, extra)) || (rc = ec_compact_packed(c, &npk))) { c0->err = c->err; release(); return rc; }
            cudaSetDevice(c0->device);
            if (!npk) continue;
            if ((rc = dev_alloc(c0, recv_pk, npk * 16)) || (rc = copy_to(c0, recv_pk.p, c, reinterpret_cast<const uint8_t*>(c->ec_compact.p) + 16, npk * 16)) ||
                (rc = ec_reserve(c0, npk, 0, 0))) { release(); return rc; }
            k_ec_merge_pairs<<<(unsigned)std::min<uint64_t>((npk + 255) / 256, (uint64_t)c0->sm_count * 16), 256, 0, c0->stream>>>(
                c0->E, outputs_of(c0), reinterpret_cast<const unsigned long long*>(recv_pk.p), npk);
            c0->launches++;
            CU(c0, cudaGetLastError());
            if ((rc = ec_after_chunk(c0))) { release(); return rc; }
            CU(c0, cudaStreamSynchronize(c0->stream));                 // (recv_pk is refilled for the next context)
        }
        c0->ec_extra_keys.clear(); c0->ec_extra_off.assign(1, 0); c0->ec_extra_cnt.clear();
        for (auto& kv : extra) {
            c0->ec_extra_keys.insert(c0->ec_extra_keys.end(), kv.first.begin(), kv.first.end());
            c0->ec_extra_off.push_back(c0->ec_extra_keys.size());
            c0->ec_extra_cnt.push_back(kv.second);
        }
        c0->ec_merged = true; c0->ec_drained = false;
    }
    release();
    if ((rc = close_others())) return rc;
    if ((rc = check_ctx(c0))) return rc;
    c0->last_shards = ns; c0->last_shard_fallback = 0;
    uint64_t total = 0;
    for (auto& j : J) total += j.bytes;
    if (bytes_out) *bytes_out = total;
    return F2Q_OK;
}

// ---- memory helpers --------------------------------------------------------------------------------------
F2Q_EXPORT int f2q_host_alloc(void** ptr, uint64_t nbytes) {
    if (!ptr) return F2Q_EINVAL;
    cudaError_t e = cudaHostAlloc(ptr, nbytes ? nbytes : 1, cudaHostAllocDefault);
    if (e != cudaSuccess) { cudaGetLastError(); *ptr = nullptr; return fail(nullptr, F2Q_ENOMEM, std::string("cudaHostAlloc: ") + cudaGetErrorString(e)); }
    return F2Q_OK;
}

namespace {
std::mutex g_near_mu;
std::map<void*, size_t> g_near;                                        // buffers of f2q_host_alloc_near that were mmap'ed + registered

// NUMA node of a CUDA device from sysfs (-1: unknown / the platform shows a single node, as VMs do)
int device_numa_node(int device) {
    char bdf[32] = {0};
    if (cudaDeviceGetPCIBusId(bdf, sizeof(bdf), device) != cudaSuccess) { cudaGetLastError(); return -1; }
    for (char* p = bdf; *p; p++) *p = (char)tolower(*p);
    const std::string path = std::string("/sys/bus/pci/devices/") + bdf + "/numa_node";
    FILE* f = fopen(path.c_str(), "r");
    if (!f) return -1;
    int node = -1;
    if (fscanf(f, "%d", &node) != 1) node = -1;
    fclose(f);
    return node;
}
int numa_nodes_visible() {
    int n = 0;
    for (int k = 0; k < 64; k++) {
        const std::string p = "/sys/devices/system/node/node" + std::to_string(k);
        if (access(p.c_str(), F_OK) == 0) n++;
    }
    return n;
}
}  // namespace

// page-locked host memory for the chunks of ONE device: on the NUMA node of that device when the platform shows more than
// one node (mmap + mbind(MPOL_BIND) + first touch + cudaHostRegister), else plain cudaHostAlloc.  flags bit 0: write-combined
// (the CPU only writes the buffer, the GPU's DMA reads it without snooping the CPU caches).  *numa_node = the node used, -1 none
F2Q_EXPORT int f2q_host_alloc_near(void** ptr, uint64_t nbytes, int device, int flags, int* numa_node) {
    if (!ptr) return F2Q_EINVAL;
    *ptr = nullptr;
    if (numa_node) *numa_node = -1;
    const int node = device_numa_node(device);
    const size_t len = ((nbytes ? nbytes : 1) + 4095) & ~(size_t)4095;
    if (node >= 0 && node < 64 && numa_nodes_visible() > 1 && !(flags & 1)) {
        void* p = mmap(nullptr, len, PROT_READ | PROT_WRITE, MAP_PRIVATE | MAP_ANONYMOUS, -1, 0);
        if (p != MAP_FAILED) {
            unsigned long mask = 1ul << node;
            const long r = syscall(SYS_mbind, p, len, 2 /*MPOL_BIND*/, &mask, 65ul, 0u);
            if (r == 0) {
                memset(p, 0, len);                                     // first touch on the bound node
                if (cudaHostRegister(p, len, cudaHostRegisterDefault) == cudaSuccess) {
                    std::lock_guard<std::mutex> l(g_near_mu);
                    g_near[p] = len;
                    *ptr = p;
                    if (numa_node) *numa_node = node;
                    return F2Q_OK;
                }
                cudaGetLastError();
            }
            munmap(p, len);
        }
    }
    cudaError_t e = cudaHostAlloc(ptr, len, (flags & 1) ? cudaHostAllocWriteCombined : cudaHostAllocDefault);
    if (e != cudaSuccess) { cudaGetLastError(); *ptr = nullptr; return fail(nullptr, F2Q_ENOMEM, std::string("cudaHostAlloc: ") + cudaGetErrorString(e)); }
    return F2Q_OK;
}

F2Q_EXPORT int f2q_host_free(void* ptr) {
    if (!ptr) return F2Q_OK;
    {
        std::lock_guard<std::mutex> l(g_near_mu);
        auto it = g_near.find(ptr);
        if (it != g_near.end()) {
            cudaHostUnregister(ptr);
            munmap(ptr, it->second);
            g_near.erase(it);
            return F2Q_OK;
        }
    }
    cudaFreeHost(ptr);
    return F2Q_OK;
}

F2Q_EXPORT int f2q_device_alloc(f2q_ctx* c, void** dptr, uint64_t nbytes) {
    int rc = check_ctx(c); if (rc) return rc;
    if (!dptr) return fail(c, F2Q_EINVAL, "null argument");
    cudaError_t e = cudaMalloc(dptr, nbytes ? nbytes : 16);
    if (e != cudaSuccess) { cudaGetLastError(); *dptr = nullptr; return fail(c, F2Q_ENOMEM, std::string("cudaMalloc: ") + cudaGetErrorString(e)); }
    return F2Q_OK;
}
F2Q_EXPORT int f2q_device_free(f2q_ctx* c, void* dptr) {
    int rc = check_ctx(c); if (rc) return rc;
    CU(c, cudaStreamSynchronize(c->stream));
    if (dptr) CU(c, cudaFree(dptr));
    return F2Q_OK;
}
F2Q_EXPORT int f2q_memcpy_d2h(f2q_ctx* c, void* host, const void* dptr, uint64_t nbytes) {
    int rc = check_ctx(c); if (rc) return rc;
    CU(c, cudaMemcpyAsync(host, dptr, nbytes, cudaMemcpyDeviceToHost, c->stream));
    CU(c, cudaStreamSynchronize(c->stream));
    return F2Q_OK;
}
F2Q_EXPORT int f2q_memcpy_h2d(f2q_ctx* c, void* dptr, const void* host, uint64_t nbytes) {
    int rc = check_ctx(c); if (rc) return rc;
    CU(c, cudaMemcpyAsync(dptr, host, nbytes, cudaMemcpyHostToDevice, c->stream));
    CU(c, cudaStreamSynchronize(c->stream));
    return F2Q_OK;
}

F2Q_EXPORT uint64_t f2q_launch_count(const f2q_ctx* c) { return c ? c->launches : 0; }

F2Q_EXPORT int f2q_spec_counts(const f2q_ctx* c, uint64_t* committed, uint64_t* fell_back) {
    if (!c || !committed || !fell_back) return F2Q_EINVAL;
    *committed = c->spec_counts[0]; *fell_back = c->spec_counts[1];
    return F2Q_OK;
}

F2Q_EXPORT int f2q_get_info(f2q_ctx* c, const char* name, int64_t* value) {
    int rc = check_ctx(c); if (rc) return rc;
    if (!name || !value) return fail(c, F2Q_EINVAL, "null argument");
    const std::string n(name);
    if (n == "policy") *value = c->policy;
    else if (n == "table") *value = c->T.cuckoo ? (c->T.ck_neighbours ? 3 : 2) : c->T.cslots ? 1 : 0;
    else if (n == "hist") *value = c->hist_used;
    else if (n == "seed_parts") *value = c->T.seed_ncombo ? (int64_t)c->T.seed_parts : 0;
    else if (n == "flex_table") *value = c->T.fx_slots ? 1 : 0;
    else if (n == "shards") *value = c->last_shards;
    else if (n == "shard_fallback") *value = c->last_shard_fallback;
    else if (n == "generic_reads") {
        if (c->in_sample) return fail(c, F2Q_ESTATE, "generic_reads is known once the sample has finished");
        unsigned long long v = 0;
        CU(c, cudaStreamSynchronize(c->stream));
        CU(c, cudaMemcpy(&v, &c->dS->generic_reads, sizeof(v), cudaMemcpyDeviceToHost));
        *value = (int64_t)v;
    } else return fail(c, F2Q_EINVAL, "unknown info " + n);
    return F2Q_OK;
}

F2Q_EXPORT int f2q_memo_counts(const f2q_ctx* c, uint64_t* lookups, uint64_t* hits) {
    if (!c || !lookups || !hits) return F2Q_EINVAL;
    *lookups = c->memo_counts[0]; *hits = c->memo_counts[1];
    return F2Q_OK;
}

F2Q_EXPORT int f2q_kernel_times(f2q_ctx* c, double* ms, uint64_t* launches) {
    if (!c || !ms || !launches) return F2Q_EINVAL;
    for (int k = 0; k < 4; k++) { ms[k] = c->kernel_ms[k]; launches[k] = c->kernel_launches[k]; }
    return F2Q_OK;
}

// ---- K0 synthetic generator ------------------------------------------------------------------------------
F2Q_EXPORT int f2q_synth_fastq(f2q_ctx* c, const f2q_synth_spec* spec, const uint8_t* guides, void* dptr) {
    int rc = check_ctx(c); if (rc) return rc;
    if (!spec || !dptr) return fail(c, F2Q_EINVAL, "null argument");
    if (spec->feat_len < 4 || spec->feat_len > 32 || spec->read_len < spec->feat_len || spec->read_len > 150 || spec->n_guides == 0 || spec->shape > 3)
        return fail(c, F2Q_EINVAL, "synthetic spec out of range");
    for (int k = 0; k < 4; k++) if (spec->delim_len[k] > 16) return fail(c, F2Q_EINVAL, "synthetic spec: search sequence longer than 16");
    const size_t gbytes = (size_t)spec->n_guides * spec->feat_len * (spec->shape >= 2 ? 2 : 1);
    if (guides) {
        // (synchronous: the caller's host array may go away after the call)
        CU(c, cudaStreamSynchronize(c->stream));
        if ((rc = dev_alloc(c, c->synth_guides, gbytes))) return rc;
        CU(c, cudaMemcpy(c->synth_guides.p, guides, gbytes, cudaMemcpyHostToDevice));
        c->synth_guide_bytes = gbytes;
    } else if (!c->synth_guides.p || c->synth_guide_bytes != gbytes)
        return fail(c, F2Q_ESTATE, "f2q_synth_fastq without guides needs an earlier call that uploaded the same table");
    if (spec->n_reads) {
        const unsigned grid = (unsigned)std::min<uint64_t>((spec->n_reads + 255) / 256, (uint64_t)c->sm_count * 16);
        k_synth<<<grid, 256, 0, c->stream>>>(*spec, reinterpret_cast<const uint8_t*>(c->synth_guides.p), reinterpret_cast<uint8_t*>(dptr));
        c->launches++;
    }
    CU(c, cudaGetLastError());
    if (guides) CU(c, cudaStreamSynchronize(c->stream));
    return F2Q_OK;
}

// ---- single-read helpers (README.md:259-298 public helpers of the reference) -----------------------------
F2Q_EXPORT int f2q_border_finder(int device, const uint8_t* seq, uint32_t seq_len, const uint8_t* read, uint32_t read_len,
                                 int32_t mismatch, int32_t start_place, int32_t* pos) {
    if (!pos || (seq_len && !seq) || (read_len && !read)) return fail(nullptr, F2Q_EINVAL, "null argument");
    if (f2q_device_count() == 0) return fail(nullptr, F2Q_ENODEVICE, "no CUDA device: libf2q has no CPU path");
    if (cudaSetDevice(device) != cudaSuccess) return fail(nullptr, F2Q_ECUDA, "cudaSetDevice failed");
    uint8_t* d = nullptr; int* dout = nullptr;
    if (cudaMalloc(&d, (size_t)seq_len + read_len + 16) != cudaSuccess || cudaMalloc(&dout, 16) != cudaSuccess) { cudaFree(d); return fail(nullptr, F2Q_ENOMEM, "cudaMalloc failed"); }
    if (seq_len) cudaMemcpy(d, seq, seq_len, cudaMemcpyHostToDevice);
    if (read_len) cudaMemcpy(d + seq_len, read, read_len, cudaMemcpyHostToDevice);
    k_border_finder<<<1, 32>>>(d, (int)seq_len, d + seq_len, (int)read_len, mismatch, start_place, dout);
    int out = -1;
    cudaError_t e = cudaMemcpy(&out, dout, 4, cudaMemcpyDeviceToHost);
    cudaFree(d); cudaFree(dout);
    if (e != cudaSuccess) return fail(nullptr, F2Q_ECUDA, std::string("k_border_finder: ") + cudaGetErrorString(e));
    *pos = out;
    return F2Q_OK;
}

F2Q_EXPORT int f2q_sequence_tinder(int device, const f2q_config* cfg, int32_t iteration, const uint8_t* read, uint32_t read_len,
                                   const uint8_t* qual, uint32_t qual_len, const uint64_t* set_up, const uint64_t* set_down,
                                   int32_t* found, int32_t* start, int32_t* end) {
    if (!cfg || !found || !start || !end || (read_len && !read) || (qual_len && !qual)) return fail(nullptr, F2Q_EINVAL, "null argument");
    if (iteration < 0 || iteration >= F2Q_MAX_ITER) return fail(nullptr, F2Q_EINVAL, "iteration out of range");
    if (f2q_device_count() == 0) return fail(nullptr, F2Q_ENODEVICE, "no CUDA device: libf2q has no CPU path");
    if (cudaSetDevice(device) != cudaSuccess) return fail(nullptr, F2Q_ECUDA, "cudaSetDevice failed");
    GenericCfg G; std::string why;
    f2q_config tmp = *cfg; if (tmp.n_iter < 1) tmp.n_iter = 1;
    int rc = make_generic_cfg(&tmp, G, why);
    if (rc) return fail(nullptr, rc, why);
    if (set_up) memcpy(G.set_up.w, set_up, 32);
    if (set_down) memcpy(G.set_down.w, set_down, 32);
    uint8_t* d = nullptr; int* dout = nullptr;
    if (cudaMalloc(&d, (size_t)read_len + qual_len + 16) != cudaSuccess || cudaMalloc(&dout, 16) != cudaSuccess) { cudaFree(d); return fail(nullptr, F2Q_ENOMEM, "cudaMalloc failed"); }
    if (read_len) cudaMemcpy(d, read, read_len, cudaMemcpyHostToDevice);
    if (qual_len) cudaMemcpy(d + read_len, qual, qual_len, cudaMemcpyHostToDevice);
    k_sequence_tinder<<<1, 32>>>(G, iteration, d, (int)read_len, d + read_len, (int)qual_len, dout);
    int out[3] = {0, 0, 0};
    cudaError_t e = cudaMemcpy(out, dout, 12, cudaMemcpyDeviceToHost);
    cudaFree(d); cudaFree(dout);
    if (e != cudaSuccess) return fail(nullptr, F2Q_ECUDA, std::string("k_sequence_tinder: ") + cudaGetErrorString(e));
    *found = out[0]; *start = out[1]; *end = out[2];
    return F2Q_OK;
}
