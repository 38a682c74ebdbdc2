// dark_bwt.cu — context, round driver and C ABI (include/dark_bwt.h) of the B200-native forward BWT.
//
// Host-side control flow of one block (replaces saca::Constructor::compute + TransformIterator,
// /root/reference/src/saca.rs:368-378 and src/block/dc.rs:45-50):
//
//   alphabet scan -> initial keys (K symbols per 64-bit key) -> radix sort -> re-rank/compact
//   while (unsettled suffixes remain):  keys (rank[i], rank[i+h]) -> radix sort -> re-rank/compact;  h *= 2
//   BWT gather + origin
//
// All device memory is carved from one arena allocated at create (Constructor::new allocates its
// arena up front too, saca.rs:351-360); the forward calls allocate nothing.
#include <cuda_runtime.h>

#include <algorithm>
#include <atomic>
#include <chrono>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <future>
#include <new>
#include <thread>
#include <vector>

#include "../../include/dark_bwt.h"
#include "common.cuh"
#include "radix_sort.cuh"
#include "onesweep_tma.cuh"
#include "suffix_kernels.cuh"
#include "dc_kernels.cuh"

using namespace dark;

namespace {

constexpr int kSortTile = 3072;  // smallest tile of any pass variant (sizes the status buffer)
#ifndef DARK_SCAN_THREADS
#define DARK_SCAN_THREADS 512
#endif
constexpr int kScanThreads = DARK_SCAN_THREADS;  // tuning builds: -DDARK_SCAN_THREADS=256 (profiles/r1_ncu_rerank_final.md)
constexpr int kScanItems = 8;
constexpr int kScanTile = kScanThreads * kScanItems;
constexpr int kInitThreads = 256;
constexpr int kInitItems = 16;
constexpr int kBuildThreads = 256;
constexpr int kBuildItems = 8;
constexpr int kMaxCounters = 4096;
constexpr u32 kMaxManyBlocks = DARK_BWT_MAX_MANY_BLOCKS;
constexpr int kMaxEvents = 16 + 10 * DARK_BWT_MAX_ROUNDS;

enum Phase { PH_INIT = 0, PH_SORT, PH_PASS, PH_GENPASS, PH_KEYBUILD, PH_RERANK, PH_EMIT, PH_COUNT };

struct Mailbox {  // pinned host memory the device results are copied into
    u32 sigma;
    u32 count;
    u32 trivial[kMaxPasses];
    float collide[kMaxPasses];
    u64 origin;
    unsigned long long bad;
    u32 flag;  // pairs-mode detector: set when some group has three or more members
    u32 not_pairs;  // the same answer from the check queued behind a re-rank (read with the survivor count)
    u32 bad_block;  // inverse_many: the lowest block whose list does not cover its rows (with `count` = how many do not)
};

struct DeviceScalars {  // mirrors Mailbox on the device
    u32 sigma;
    u32 count;
    u32 trivial[kMaxPasses];
    float collide[kMaxPasses];
    u64 origin;
    unsigned long long bad;
};

inline size_t align_up(size_t x, size_t a) { return (x + a - 1) / a * a; }
inline int bit_length(u64 x) {
    int b = 0;
    while (x) {
        ++b;
        x >>= 1;
    }
    return b;
}

}  // namespace

// Test and tuning knobs, resolved ONCE at dark_bwt_create from the environment (never on the hot path).  The test knobs
// force code paths that the block size or content would otherwise choose; none of them changes a result, and each has
// a parity test (tests/test_gpu_parity.py).  The tuning knobs can skip work (garbage output) or select kernels without
// a forward-progress guarantee, so they exist only in builds with -DDARK_BWT_TUNING (tools/, never shipped).
struct Knobs {
    int pass_impl = 1;              // DARK_BWT_PASS_IMPL: 1 = onesweep_tma.cuh, 0 = the round-1 kernel k_onesweep_pass
    bool force_u64_status = false;  // DARK_BWT_FORCE_U64_STATUS=1
    bool fused_init = true;         // DARK_BWT_FUSED_INIT=0 materialises the round-0 keys
    bool gram_hist = true;          // DARK_BWT_GRAM_HIST=0 counts digits key by key
    bool check_hist = false;        // DARK_BWT_CHECK_HIST=1 counts both ways and compares
    bool inline_emit = true;        // DARK_BWT_INLINE_EMIT=0
    bool sparse_rerank = true;      // DARK_BWT_SPARSE_RERANK=0
    int inline_gather = 0;          // DARK_BWT_INLINE_GATHER=1: unpruned blocks emit inline too, gathering T[id-1] in the re-rank
    bool fuse_round0 = true;        // DARK_BWT_FUSE_ROUND0=0: round 0 of an unpruned large block without the fused bucket sink
    bool rerank_chainfree = false;  // DARK_BWT_RERANK_CHAINFREE=1: rounds >= 1 re-ranked by flags + scan + apply kernels (no look-back chain; measured
                                    // equal to the single kernel on C3/C5/C4: profiles/r2_rejected.md)
    int text_div = 8;               // DARK_BWT_TEXT_BUILD=<k>: text-order key build while m > n/k (0 = never, no isa[] tag)
    bool pairs = true;              // DARK_BWT_PAIRS=0
    bool rank_search = true;        // DARK_BWT_RANK_SEARCH=0
    int bucketed = -1;              // DARK_BWT_BUCKETED=0/1 (-1: by block size)
    int host_chunk_mb = 2;          // DARK_BWT_HOST_CHUNK_MB: pinned bytes per staging lane (2 MiB chunks fill the pipeline sooner than 8: 23.1 vs 23.8 ms per C2 call)
    int host_threads = 12;          // DARK_BWT_HOST_THREADS=<t>: staging lanes per direction for pageable host buffers (0: let the driver stage)
    int sort_variant = -1;          // DARK_BWT_SORT_VARIANT=<i>: run the round-1 kernel with tiling i
    int emit_window_mb = 64;        // DARK_BWT_EMIT_WINDOW_MB: text window of the emission
    int ibwt_stride = 48;           // DARK_BWT_IBWT_STRIDE: splitter stride of the inverse BWT
    bool ibwt_two_walks = false;    // DARK_BWT_IBWT_TWO_WALKS=1
    // tuning builds only (-DDARK_BWT_TUNING)
    bool tile_by_blockidx = false;  // DARK_BWT_TILE_BY_BLOCKIDX=1: tiles by blockIdx (no forward-progress guarantee)
    unsigned knockout = 0;          // DARK_BWT_PASS_KNOCKOUT=<mask>: skip phases of k_onesweep_pass (garbage output)
    int pass_prefetch = -1;         // DARK_BWT_PASS_PREFETCH=<tiles>
    int rerank_prefetch = -1;       // DARK_BWT_RERANK_PREFETCH=<tiles>
    bool group_stats = false;       // DARK_BWT_GROUP_STATS=1

    void read_env() {
        auto geti = [](const char* name, int dflt) {
            const char* e = getenv(name);
            return e ? atoi(e) : dflt;
        };
        pass_impl = geti("DARK_BWT_PASS_IMPL", pass_impl);
        force_u64_status = geti("DARK_BWT_FORCE_U64_STATUS", 0) != 0;
        fused_init = geti("DARK_BWT_FUSED_INIT", 1) != 0;
        gram_hist = geti("DARK_BWT_GRAM_HIST", 1) != 0;
        check_hist = geti("DARK_BWT_CHECK_HIST", 0) != 0;
        inline_emit = geti("DARK_BWT_INLINE_EMIT", 1) != 0;
        sparse_rerank = geti("DARK_BWT_SPARSE_RERANK", 1) != 0;
        rerank_chainfree = geti("DARK_BWT_RERANK_CHAINFREE", 0) != 0;
        fuse_round0 = geti("DARK_BWT_FUSE_ROUND0", 1) != 0;
        inline_gather = geti("DARK_BWT_INLINE_GATHER", 0);
        text_div = geti("DARK_BWT_TEXT_BUILD", text_div);
        pairs = geti("DARK_BWT_PAIRS", 1) != 0;
        rank_search = geti("DARK_BWT_RANK_SEARCH", 1) != 0;
        bucketed = geti("DARK_BWT_BUCKETED", -1);
        {
            const unsigned hw = std::thread::hardware_concurrency();
            if (hw > 0) host_threads = (int)std::min<unsigned>((unsigned)host_threads, std::max(1u, hw - 2u));
        }
        host_threads = std::min(std::max(geti("DARK_BWT_HOST_THREADS", host_threads), 0), 16);
        host_chunk_mb = std::min(std::max(geti("DARK_BWT_HOST_CHUNK_MB", host_chunk_mb), 1), 64);
        sort_variant = geti("DARK_BWT_SORT_VARIANT", -1);
        emit_window_mb = std::max(1, geti("DARK_BWT_EMIT_WINDOW_MB", 64));
        ibwt_stride = std::max(2, geti("DARK_BWT_IBWT_STRIDE", 48));
        ibwt_two_walks = geti("DARK_BWT_IBWT_TWO_WALKS", 0) != 0;
#ifdef DARK_BWT_TUNING
        tile_by_blockidx = geti("DARK_BWT_TILE_BY_BLOCKIDX", 0) != 0;
        knockout = (unsigned)geti("DARK_BWT_PASS_KNOCKOUT", 0);
        pass_prefetch = geti("DARK_BWT_PASS_PREFETCH", -1);
        rerank_prefetch = geti("DARK_BWT_RERANK_PREFETCH", -1);
        group_stats = geti("DARK_BWT_GROUP_STATS", 0) != 0;
#endif
    }
};

// Pinned staging for PAGEABLE host buffers (the reference hands over a plain Vec<u8>, src/main.rs:95, and collects into a
// fresh Vec, src/block/dc.rs:47-48).  A cudaMemcpy from pageable memory is staged by the driver through one small
// bounce buffer on the calling thread (a few GB/s); here `lanes` host threads each own one pinned chunk and a stream:
// a thread copies a chunk of the caller's buffer into its pinned chunk and sends it on (or receives a chunk and copies
// it out), so the DMA of one lane overlaps the memcpy of the others.  One set for each direction; allocated on the
// first pageable call of the context (pinning costs milliseconds per 10 MB, contexts that only ever see pinned or
// device buffers should not pay it).
struct HostStage {
    static constexpr int kMaxLanes = 16;
    size_t chunk = 2u << 20;
    int lanes = 0;
    u8* pinned = nullptr;  // lanes x 2 slots x chunk
    cudaStream_t streams[kMaxLanes] = {nullptr};
    cudaEvent_t slot_done[kMaxLanes][2] = {{nullptr}};  // the DMA out of / into a lane's slot has completed
};

struct dark_bwt_ctx {
    int device = 0;
    Knobs knobs;
    HostStage stage_in, stage_out;
    int num_sms = 148;
    u64 capacity = 0;
    u32 flags = 0;
    cudaStream_t stream = nullptr;

    void* arena = nullptr;
    size_t arena_bytes = 0;
    u64* keys[2] = {nullptr, nullptr};
    u32* ids[2] = {nullptr, nullptr};
    u32* ranks = nullptr;      // rank of each active suffix's group (current list)
    u32* ranks_alt = nullptr;  // the re-rank of rounds >= 1 reads `ranks` and writes here, then they swap
    u32* isa = nullptr;
    u32* sa = nullptr;
    u8* d_text = nullptr;  // host-entry staging
    u8* d_bwt = nullptr;
    u8* d_text2 = nullptr;  // second pair for the pipelined batch entry
    u8* d_bwt2 = nullptr;
    cudaStream_t copy_in = nullptr, copy_out = nullptr;
    cudaEvent_t ev_in[2] = {nullptr, nullptr}, ev_comp[2] = {nullptr, nullptr}, ev_out[2] = {nullptr, nullptr};
    u32* hist = nullptr;
    u32* present = nullptr;
    u8* lut = nullptr;
    DeviceScalars* scalars = nullptr;
    void* sort_status = nullptr;
    size_t sort_status_bytes = 0;
    // Sorts of at most 2^31 pairs use 32-bit status words and the buffer as two halves in turn: the workers of a pass zero
    // the rows of the OTHER half (onesweep_tma.cuh), so only what they did not cover is cleared by a memset.  Rows [lo, hi)
    // of half h may hold stale words.
    int status_cur = 0;
    u32 status_dirty_lo[2] = {0u, 0u}, status_dirty_hi[2] = {0u, 0u};
    u32* counters = nullptr;
    u64* scan_words = nullptr;
    long long* pass_trace = nullptr;  // debug: per-tile phase stamps of the radix pass (dark_bwt_debug_trace)
    long long* rerank_trace = nullptr;  // debug: per-tile phase stamps of the round-0 re-rank (dark_bwt_debug_trace_rerank)
    u32* bucket_hist = nullptr;  // 256 counters / cursors of the bucketed rank scatter
    u32* many_starts = nullptr;            // dark_bwt_forward_many: block offsets (kMaxManyBlocks + 1)
    unsigned long long* many_origins = nullptr;  // ... per-block origins
    u16* many_lut = nullptr;               // ... byte -> code 1..sigma
    DcInfoDev* dc_info = nullptr;             // dark_bwt_dc_*: device copy of the result header, followed by the run counter
    u32* bitmap = nullptr;  // n bits: positions whose rank the next round reads; new-head flags of the chain-free re-rank
    u32* bitmap2 = nullptr;  // old-head flags of the chain-free re-rank
    size_t scan_tiles = 0;

    Mailbox* mail = nullptr;      // pinned + mapped host memory: kernels write their scalar results straight into it
    Mailbox* mail_dev = nullptr;  // the device alias of `mail`
    u32* reuse_words = nullptr;
    u64 reuse_count = 0;

    cudaEvent_t events[kMaxEvents];
    int n_events = 0;
    struct Span {
        int phase, e0, e1;
    };
    std::vector<Span> spans;
    int next_counter = 0;
    u32* count_dev = nullptr;  // device copy of the survivor count of the last re-rank launched (nullptr: none)
    u32 tag = 0;  // bit carried by isa[] entries of active suffixes during forward_device (0: not used)
    u32 launches = 0;
    u32 syncs = 0;
    char err[320] = {0};

    int fail_cuda(cudaError_t e, const char* what, int line) {
        snprintf(err, sizeof(err), "CUDA error %d (%s) at dark_bwt.cu:%d: %s", (int)e, cudaGetErrorString(e), line, what);
        return DARK_BWT_E_CUDA;
    }
    int fail_internal(const char* what) {
        snprintf(err, sizeof(err), "internal error: %s", what);
        return DARK_BWT_E_INTERNAL;
    }
};

#define CK(call)                                                              \
    do {                                                                      \
        cudaError_t e__ = (call);                                             \
        if (e__ != cudaSuccess) return ctx->fail_cuda(e__, #call, __LINE__); \
    } while (0)
#define LAUNCHED()            \
    do {                      \
        ctx->launches += 1;   \
        CK(cudaGetLastError()); \
    } while (0)

namespace {

// every host round trip of a forward call goes through here (dark_bwt_stats.host_syncs)
inline cudaError_t sync_counted(dark_bwt_ctx* ctx) {
    ctx->syncs += 1;
    return cudaStreamSynchronize(ctx->stream);
}

int span_begin(dark_bwt_ctx* ctx, int phase) {
    if (ctx->n_events + 2 > kMaxEvents - 4) return -1;  // the last events are reserved for the entry points
    int e0 = ctx->n_events++;
    cudaEventRecord(ctx->events[e0], ctx->stream);
    ctx->spans.push_back({phase, e0, -1});
    return (int)ctx->spans.size() - 1;
}
void span_end(dark_bwt_ctx* ctx, int span) {
    if (span < 0) return;
    int e1 = ctx->n_events++;
    cudaEventRecord(ctx->events[e1], ctx->stream);
    ctx->spans[span].e1 = e1;
}

template <typename K>
int set_smem(dark_bwt_ctx* ctx, K kernel, size_t bytes) {
    CK(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes));
    return 0;
}

int next_counter(dark_bwt_ctx* ctx, u32** out) {
    if (ctx->next_counter >= kMaxCounters) return ctx->fail_internal("tile counters exhausted");
    *out = ctx->counters + ctx->next_counter++;
    return 0;
}

// Tuning variants of the radix pass (threads, items per thread, min CTAs per SM).  The default is
// chosen from measurements (profiles/); DARK_BWT_SORT_VARIANT=<i> selects another one for sweeps.
template <int THREADS, int ITEMS, int MINBLOCKS, int ILP, typename StatusT, bool ALIGNED, bool GEN = false>
int launch_pass_kernel(dark_bwt_ctx* ctx, const u64* kin, const u32* vin, u64* kout, u32* vout, u32 m, int shift,
                       const u32* digit_base, u32* counter, u32 tiles, const u8* prev_text, u32 n_text, KeyGen gen = KeyGen()) {
    typedef OnesweepSmem<THREADS, ITEMS> Smem;
    auto kern = k_onesweep_pass<THREADS, ITEMS, MINBLOCKS, ILP, StatusT, ALIGNED, GEN>;
    CK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(Smem)));  // per device
    const bool by_block_index = ctx->knobs.tile_by_blockidx;
    const u32 knock = ctx->knobs.knockout;  // tuning builds only: skip phases (1 look-back, 2 ranking, 4 stores)
    // persistent grid: as many CTAs as stay resident (SMs x MINBLOCKS), each claiming tiles until none are left
    const u32 grid = by_block_index ? tiles : std::min<u32>(tiles, (u32)ctx->num_sms * MINBLOCKS);
    // L2 prefetch distance in tiles: two thirds of a wave of claims (the persistent grid; 148..444 measured alike, beyond
    // one wave the gain fades) unless DARK_BWT_PASS_PREFETCH says otherwise (0 = off)
    const u32 prefetch_ahead = by_block_index ? 0u : (ctx->knobs.pass_prefetch >= 0 ? (u32)ctx->knobs.pass_prefetch : std::max(1u, grid * 2 / 3));
    kern<<<grid, THREADS, sizeof(Smem), ctx->stream>>>(kin, vin, kout, vout, m, shift, digit_base, (StatusT*)ctx->sort_status,
                                                        by_block_index ? nullptr : counter, ctx->pass_trace, prev_text, n_text, knock, gen,
                                                        prefetch_ahead);
    LAUNCHED();
    return 0;
}

template <int THREADS, int ITEMS, int MINBLOCKS, int ILP>
int launch_pass_variant(dark_bwt_ctx* ctx, const u64* kin, const u32* vin, u64* kout, u32* vout, u32 m, int shift,
                        const u32* digit_base, u32* counter, bool wide, const u8* prev_text, u32 n_text, const KeyGen* gen = nullptr) {
    typedef OnesweepSmem<THREADS, ITEMS> Smem;
    const u32 tiles = (u32)ceil_div(m, Smem::kTile);
    const size_t bytes = (size_t)tiles * kRadix * (wide ? sizeof(u64) : sizeof(u32));
    if (bytes > ctx->sort_status_bytes) return ctx->fail_internal("sort status buffer too small");
    CK(cudaMemsetAsync(ctx->sort_status, 0, bytes, ctx->stream));
    {  // this kernel uses the buffer from its start: both halves of the TMA pass' bookkeeping are stale now
        const u32 half_rows = (u32)(ctx->sort_status_bytes / 2 / (kRadix * sizeof(u32)));
        for (int h = 0; h < 2; ++h) ctx->status_dirty_lo[h] = 0u, ctx->status_dirty_hi[h] = half_rows;
    }
    const bool aligned = (shift & 7) == 0;  // always true for the suffix sorter; the public sort may differ
#define LP(ST, AL) launch_pass_kernel<THREADS, ITEMS, MINBLOCKS, ILP, ST, AL>(ctx, kin, vin, kout, vout, m, shift, digit_base, counter, tiles, prev_text, n_text)
    if (gen != nullptr) {  // keys built from the text inside the pass (default tiling, byte-aligned digits only)
        if (!aligned) return ctx->fail_internal("key-generating pass needs a byte-aligned digit");
        if (wide)
            return launch_pass_kernel<THREADS, ITEMS, MINBLOCKS, ILP, u64, true, true>(ctx, kin, vin, kout, vout, m, shift, digit_base, counter,
                                                                                       tiles, prev_text, n_text, *gen);
        return launch_pass_kernel<THREADS, ITEMS, MINBLOCKS, ILP, u32, true, true>(ctx, kin, vin, kout, vout, m, shift, digit_base, counter,
                                                                                   tiles, prev_text, n_text, *gen);
    }
    if (!aligned) return wide ? LP(u64, false) : LP(u32, false);
    return wide ? LP(u64, true) : LP(u32, true);
#undef LP
}

// The TMA-staged, software-pipelined pass (onesweep_tma.cuh): byte-aligned digits, 16-byte aligned inputs, plain or
// key-generating (GEN mode 0).  Returns 1 if this pass is not eligible (the caller then runs k_onesweep_pass).
template <int THREADS, int ITEMS, int MINBLOCKS, int ILP>
int launch_pass_tma(dark_bwt_ctx* ctx, const u64* kin, const u32* vin, u64* kout, u32* vout, u32 m, int shift, const u32* digit_base,
                    u32* counter, bool wide, const u8* prev_text, const KeyGen* gen) {
    typedef PipeSmem<THREADS, ITEMS> Smem;
    const u32 tiles = (u32)ceil_div(m, Smem::kTile);
    const u32 rows_needed = tiles + 3 * kScannerBatch;  // the scanners read ahead
    const u32 half_rows = (u32)(ctx->sort_status_bytes / 2 / (kRadix * sizeof(u32)));
    void* st_use = ctx->sort_status;
    void* st_clean = nullptr;
    if (wide) {
        const size_t bytes = (size_t)rows_needed * kRadix * sizeof(u64);
        if (bytes > ctx->sort_status_bytes) return ctx->fail_internal("sort status buffer too small");
        CK(cudaMemsetAsync(ctx->sort_status, 0, bytes, ctx->stream));
        for (int h = 0; h < 2; ++h) ctx->status_dirty_lo[h] = 0u, ctx->status_dirty_hi[h] = half_rows;
    } else {
        if (rows_needed > half_rows) return ctx->fail_internal("sort status buffer too small");
        const int h = ctx->status_cur, o = h ^ 1;
        u32* base_h = (u32*)ctx->sort_status + (size_t)h * half_rows * kRadix;
        u32* base_o = (u32*)ctx->sort_status + (size_t)o * half_rows * kRadix;
        if (ctx->status_dirty_hi[h] > ctx->status_dirty_lo[h]) {  // what the previous pass' workers did not zero (usually nothing)
            CK(cudaMemsetAsync(base_h + (size_t)ctx->status_dirty_lo[h] * kRadix, 0,
                               (size_t)(ctx->status_dirty_hi[h] - ctx->status_dirty_lo[h]) * kRadix * sizeof(u32), ctx->stream));
        }
        ctx->status_dirty_lo[h] = 0u;  // this pass writes rows [0, tiles) of its half ...
        ctx->status_dirty_hi[h] = tiles;
        if (ctx->status_dirty_hi[o] <= tiles) ctx->status_dirty_lo[o] = ctx->status_dirty_hi[o] = 0u;  // ... and zeroes rows [0, tiles) of the other
        else ctx->status_dirty_lo[o] = std::max(ctx->status_dirty_lo[o], tiles);
        ctx->status_cur = o;
        st_use = base_h;
        st_clean = base_o;
    }
    const u32 grid = std::min<u32>(tiles + kScanners, (u32)ctx->num_sms * MINBLOCKS);  // kScanners CTAs scan, the rest sort
    const KeyGen g = gen ? *gen : KeyGen();
    const bool hi = shift >= 32;
#define LT(ST, GEN)                                                                                                          \
    do {                                                                                                                     \
        auto kern = hi ? k_onesweep_tma<THREADS, ITEMS, MINBLOCKS, ILP, ST, GEN, true>                                       \
                       : k_onesweep_tma<THREADS, ITEMS, MINBLOCKS, ILP, ST, GEN, false>;                                     \
        CK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(Smem)));                      \
        kern<<<grid, THREADS, sizeof(Smem), ctx->stream>>>(kin, vin, kout, vout, m, shift, digit_base, (ST*)st_use, (ST*)st_clean, \
                                                           counter, g, prev_text, ctx->pass_trace);                          \
    } while (0)
    if (gen) {
        if (wide) LT(u64, true);
        else LT(u32, true);
    } else {
        if (wide) LT(u64, false);
        else LT(u32, false);
    }
#undef LT
    LAUNCHED();
    return 0;
}

#ifndef DARK_PASS_ILP
#define DARK_PASS_ILP 2
#endif
#ifndef DARK_PASS_THREADS
#define DARK_PASS_THREADS 256
#define DARK_PASS_ITEMS 16
#endif
#ifndef DARK_PASS_CTAS
#define DARK_PASS_CTAS 2
#endif
constexpr int kDefaultSortVariant = 1;  // 256 threads x 16 items, 3 CTAs/SM: best of the sweeps in profiles/r1_sort_variants_*.log

// One onesweep pass over m pairs: buffers[cur] -> buffers[cur^1].
int launch_pass(dark_bwt_ctx* ctx, const u64* kin, const u32* vin, u64* kout, u32* vout, u32 m, int shift,
                const u32* digit_base, const u8* prev_text = nullptr, u32 n_text = 0, const KeyGen* gen = nullptr) {
    u32* counter = nullptr;
    if (int rc = next_counter(ctx, &counter)) return rc;
    for (int k = 0; k < kScanners; ++k) {
        u32* scanner_sm = nullptr;  // the words after the tile counter: where the scanner CTAs of onesweep_tma.cuh say which SMs they run on
        if (int rc = next_counter(ctx, &scanner_sm)) return rc;
    }
    // The round-1 kernel's 32-bit status words hold prefixes below 2^30, the pipelined pass' below 2^31 (blocks up to 2 GiB);
    // larger sorts use 64-bit words.
    // DARK_BWT_FORCE_U64_STATUS=1 exercises the wide path on small inputs (tests).
    const bool wide = !(m < (1u << 30)) || ctx->knobs.force_u64_status;
    const bool wide_tma = m > (1u << 31) || ctx->knobs.force_u64_status;  // the pipelined pass keeps 31 bits of prefix in a 4-byte word
    const bool ev = ctx->knobs.sort_variant >= 0;
    const int variant = ev ? ctx->knobs.sort_variant : kDefaultSortVariant;
    {
        // default: the TMA-staged pipelined pass; DARK_BWT_PASS_IMPL=0 keeps the round-1 kernel (k_onesweep_pass)
        const int impl = ctx->knobs.pass_impl;
        const bool eligible = (shift & 7) == 0 && !ev && (gen == nullptr || gen->mode == 0) &&
                              (gen != nullptr || (prev_text == nullptr && ((uintptr_t)kin & 15) == 0 && ((uintptr_t)vin & 15) == 0));
        if (impl != 0 && eligible) {
            return launch_pass_tma<DARK_PASS_THREADS, DARK_PASS_ITEMS, DARK_PASS_CTAS, DARK_PASS_ILP>(ctx, kin, vin, kout, vout, m, shift, digit_base, counter, wide_tma, prev_text, gen);
        }
    }
    if (gen != nullptr) return launch_pass_variant<256, 16, 3, 2>(ctx, kin, vin, kout, vout, m, shift, digit_base, counter, wide, prev_text, n_text, gen);
#define V(T, I, B, L) return launch_pass_variant<T, I, B, L>(ctx, kin, vin, kout, vout, m, shift, digit_base, counter, wide, prev_text, n_text)
    switch (variant) {
        case 0: V(256, 16, 2, 2);
        case 2: V(256, 12, 3, 2);
        case 5: V(512, 12, 2, 2);
        case 42: V(384, 16, 2, 2);
        default: V(256, 16, 3, 2);  // 1
    }
#undef V
}

// Sort passes for a histogram that is already in ctx->hist (counts).  `cur` is the index of the
// (keys, ids) pair holding the input; returns the index holding the output through *cur_out.
//
// Pass pruning (round 0 only, `prune`): an LSD sort of the top t digits alone orders the keys by
// their leading 8t bits; whatever stays tied is finished by the doubling rounds.  With S_p the
// probability that two keys share digit p (from the histogram), about m * prod(S_p) of the keys
// keep a partner after the top t digits, IF the digits are independent.  That holds for
// high-entropy blocks (packed DNA, random bytes) and fails badly for text, where a shallower
// initial sort also slows every later round (h starts smaller).  So the low digits are dropped
// only when every digit is close to uniform (S_p <= 1.5/256) and the estimate leaves < 1/64 of the
// block tied; measured: C2 8 -> 5 passes + one 65,792-element round; C1/C5 unchanged.
// *first_pass_out = index of the lowest digit that was sorted.
int run_sort(dark_bwt_ctx* ctx, u64* const keys[2], u32* const vals[2], int cur, u32 m, int begin_bit, int num_passes,
             int* cur_out, dark_bwt_stats* st, int round, bool prune = false, int* first_pass_out = nullptr,
             const u8* patch_text = nullptr, bool* patched_out = nullptr, const KeyGen* gen = nullptr, bool* gen_used_out = nullptr,
             bool all_passes = false) {
    // Scalar results (flags, counts, origin) are written by the kernels directly into mapped pinned host
    // memory and read after a stream sync.  A cudaMemcpy D2H would queue on the copy engine behind the
    // 256 MB block transfers of the pipelined batch entry (measured: +5 ms per block).
    k_scan_hist<<<num_passes, kRadix, 0, ctx->stream>>>(ctx->hist, m, ctx->mail_dev->trivial, ctx->mail_dev->collide);
    LAUNCHED();
    // all_passes (a round that still holds more than n/8 suffixes): their ranks span at least m slots, so at most the
    // top digit could be constant; every pass runs and the host does not wait for the flags (one round trip less per round)
    if (!all_passes) CK(sync_counted(ctx));
    int first = 0;
    if (prune) {
        for (int p = 0; p < num_passes; ++p)
            if (ctx->mail->collide[p] > 1.5f / 256.0f) prune = false;  // not a high-entropy block
    }
    if (prune) {
        double tied = (double)m;  // m * P(two keys agree on the top t digits) ~ fraction of keys left with a partner
        int t = 0;
        for (int p = num_passes - 1; p >= 0; --p) {
            tied *= (double)ctx->mail->collide[p];
            ++t;
            if (tied * 64.0 <= 1.0) break;
        }
        first = num_passes - t;
        if (first < 0) first = 0;
    }
    if (first_pass_out) *first_pass_out = first;
    // pruned by at least one digit: the first pass that runs also drops the BWT byte into the low key byte
    const u8* patch = (first >= 1) ? patch_text : nullptr;
    int sp = span_begin(ctx, gen ? PH_GENPASS : PH_PASS);
    for (int p = first; p < num_passes; ++p) {
        if (!all_passes && ctx->mail->trivial[p]) continue;  // every key has the same digit: the pass is the identity
        if (int rc = launch_pass(ctx, keys[cur], vals[cur], keys[cur ^ 1], vals[cur ^ 1], m, begin_bit + p * kRadixBits,
                                 ctx->hist + p * kRadix, patch, m, gen))
            return rc;
        if (gen) {  // only the first pass that runs builds its input; the later ones read what it wrote
            if (gen_used_out) *gen_used_out = true;
            gen = nullptr;
            if (st) {
                st->gen_passes += 1;
                st->gen_elements += m;
            }
            span_end(ctx, sp);  // the key-generating launch is timed on its own (13 B per suffix, not 24)
            sp = span_begin(ctx, PH_PASS);
        }
        if (patch) {
            if (patched_out) *patched_out = true;
            patch = nullptr;
        }
        cur ^= 1;
        if (st) {
            st->sort_passes += 1;
            st->sorted_elements += m;
            if (round < DARK_BWT_MAX_ROUNDS) st->passes[round] += 1;
        }
    }
    span_end(ctx, sp);
    *cur_out = cur;
    return 0;
}

struct PairSink {  // where a PAIRS re-rank puts its (id, rank) updates
    u32* ids = nullptr;
    u32* vals = nullptr;
    int shift = 0;
};

template <bool ROUND0, bool PAIRS>
int launch_rerank(dark_bwt_ctx* ctx, const u64* keys, const u32* ids, u32 m, u32 n, int K, int kb, u32* sa, u32* out_ids,
                  const u8* text, u8* bwt_inline, PairSink sink = PairSink()) {
    const u32 tiles = (u32)ceil_div(m, kScanTile);
    if (tiles > ctx->scan_tiles) return ctx->fail_internal("scan tile state too small");
    ScanTileState ts{ctx->scan_words};
    constexpr size_t smem = kRerankSmem<kScanTile>;
    if (!ROUND0 && ctx->knobs.rerank_chainfree) {
        // rounds >= 1: flags + tile aggregates, a scan over the aggregates, apply — no chain between tiles (suffix_kernels.cuh)
        auto kflags = k_rerank<kScanThreads, kScanItems, false, false, 1>;
        auto kapply = k_rerank<kScanThreads, kScanItems, false, PAIRS, 2>;
        if (smem > 48 * 1024) {
            CK(cudaFuncSetAttribute(kflags, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
            CK(cudaFuncSetAttribute(kapply, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        }
        u8* fnew = (u8*)ctx->bitmap;
        u8* fold = (u8*)ctx->bitmap2;
        kflags<<<tiles, kScanThreads, 0, ctx->stream>>>(keys, ids, ctx->ranks, m, n, K, kb, ctx->isa, sa, out_ids, ctx->ranks_alt, ts, nullptr,
                                                           &ctx->mail_dev->count, nullptr, nullptr, nullptr, 0, text, bwt_inline,
                                                           &ctx->mail_dev->origin, 0u, ctx->tag, nullptr, fnew, fold);
        LAUNCHED();
        k_rerank_scan_tiles<<<1, 1024, 0, ctx->stream>>>(ctx->scan_words, tiles, &ctx->mail_dev->count);
        LAUNCHED();
        kapply<<<tiles, kScanThreads, smem, ctx->stream>>>(keys, ids, ctx->ranks, m, n, K, kb, ctx->isa, sa, out_ids, ctx->ranks_alt, ts, nullptr,
                                                           &ctx->mail_dev->count, sink.ids, sink.vals, ctx->bucket_hist, sink.shift, text, bwt_inline,
                                                           &ctx->mail_dev->origin, 0u, ctx->tag, nullptr, fnew, fold);
        LAUNCHED();
        std::swap(ctx->ranks, ctx->ranks_alt);
        ctx->count_dev = nullptr;  // this form leaves the count in the mailbox only
        return 0;
    }
    u32 *counter = nullptr, *count_copy = nullptr;  // two consecutive words: the tile counter, then the survivor count (device copy)
    if (int rc = next_counter(ctx, &counter)) return rc;
    if (int rc = next_counter(ctx, &count_copy)) return rc;
    ctx->count_dev = count_copy;
    CK(cudaMemsetAsync(ctx->scan_words, 0, sizeof(u64) * kScanWordsPerTile * tiles, ctx->stream));
    const u32 prefetch_ahead = ctx->knobs.rerank_prefetch >= 0 ? (u32)ctx->knobs.rerank_prefetch : 2u * (u32)ctx->num_sms;  // one wave of CTAs ahead (-2 %)
    auto kern = k_rerank<kScanThreads, kScanItems, ROUND0, PAIRS>;
    if (smem > 48 * 1024) CK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    kern<<<tiles, kScanThreads, smem, ctx->stream>>>(
        keys, ids, ROUND0 ? nullptr : ctx->ranks, m, n, K, kb, ctx->isa, sa, out_ids, ROUND0 ? ctx->ranks : ctx->ranks_alt, ts, counter,
        &ctx->mail_dev->count, sink.ids, sink.vals,
        ctx->bucket_hist, sink.shift, text, bwt_inline, &ctx->mail_dev->origin, prefetch_ahead, (ROUND0 && !PAIRS) ? 0u : ctx->tag,
        ROUND0 ? ctx->rerank_trace : nullptr, nullptr, nullptr);
    LAUNCHED();
    if (!ROUND0) std::swap(ctx->ranks, ctx->ranks_alt);
    return 0;
}

// Bucketed scatter of round 0: partition the `count` pairs by id >> shift into per-bucket regions of
// (out_ids, out_vals) — region b starts at element b << shift, ctx->bucket_hist[b] is its fill cursor.
int bucket_partition(dark_bwt_ctx* ctx, const u32* pair_ids, const u32* pair_vals, u32 count, int shift, u32* out_ids,
                     u32* out_vals, u32 or_mask = 0) {
    const u32 blocks = (u32)ceil_div(count, 256 * 16);
    if (pair_vals)
        k_partition_pairs<256, 16, false><<<blocks, 256, 0, ctx->stream>>>(pair_ids, pair_vals, count, shift, ctx->bucket_hist,
                                                                           out_ids, out_vals, or_mask);
    else
        k_partition_pairs<256, 16, true><<<blocks, 256, 0, ctx->stream>>>(pair_ids, nullptr, count, shift, ctx->bucket_hist,
                                                                          out_ids, out_vals, 0u);
    LAUNCHED();
    return 0;
}
// Scatter of the per-bucket regions (counts in ctx->bucket_hist) into isa[], bucket by bucket.
int region_scatter(dark_bwt_ctx* ctx, const u32* ids, const u32* vals, u32 upper, int shift) {
    u32* chunk_prefix = ctx->bucket_hist + 256;
    k_region_chunks<<<1, 256, 0, ctx->stream>>>(ctx->bucket_hist, chunk_prefix);
    LAUNCHED();
    // one CTA per chunk, dispatched in chunk order: the chunks in flight stay neighbours, so they write one bucket's slice of
    // isa[] while it sits in L2 (persistent CTAs striding over the chunks drift apart: C5 re-rank phase 9.6 -> 17.6 ms)
    k_scatter_regions<<<(u32)ceil_div(upper, kRegionChunk) + 256, 256, 0, ctx->stream>>>(ids, vals, ctx->bucket_hist, chunk_prefix, shift, ctx->isa);
    LAUNCHED();
    return 0;
}

int fetch_count(dark_bwt_ctx* ctx, u32* out) {
    CK(sync_counted(ctx));
    *out = ctx->mail->count;
    return 0;
}

// Queues the pairs check (suffix_kernels.cuh, k_pairs_detect) behind the re-rank that has just been launched: it reads the
// survivor count from the device copy the re-rank leaves beside its tile counter, and its answer (ctx->mail->not_pairs) arrives with that count in the
// round trip the round makes anyway.  `upper` bounds the count.
int queue_pairs_check(dark_bwt_ctx* ctx, u32 upper, bool* queued) {
    *queued = false;
    if (ctx->count_dev == nullptr) return 0;
    u32* seen = nullptr;
    if (int rc = next_counter(ctx, &seen)) return rc;
    ctx->mail->not_pairs = 0;
    const u32 grid = (u32)std::min<u64>(std::max<u64>(ceil_div(upper, 256), 1), (u64)ctx->num_sms * 4);
    k_pairs_detect<<<grid, 256, 0, ctx->stream>>>(ctx->ranks, 0u, ctx->count_dev, seen, &ctx->mail_dev->not_pairs);
    LAUNCHED();
    *queued = true;
    return 0;
}

int emit(dark_bwt_ctx* ctx, const u8* d_text, u32 n, const u32* d_sa, u8* d_bwt) {
    const u32 blocks = (u32)ceil_div(ceil_div(n, 4), 256);
    const bool aligned = (((uintptr_t)d_bwt) & 3) == 0;
    const int sa16 = (((uintptr_t)d_sa) & 15) == 0 ? 1 : 0;  // else the kernels read the SA word by word
    // text window kept L2-resident per launch (126 MB L2); DARK_BWT_EMIT_WINDOW_MB overrides for sweeps
    const u64 window = (u64)ctx->knobs.emit_window_mb << 20;
    if (!aligned || n <= window + window / 2) {  // small block or odd output pointer: one plain gather launch
        k_emit_bwt<256><<<blocks, 256, 0, ctx->stream>>>(d_text, n, d_sa, d_bwt, &ctx->mail_dev->origin, aligned ? 1 : 0, sa16);
        LAUNCHED();
        return 0;
    }
    // every window launch re-reads the whole SA (4n bytes), so the window count is capped: beyond 8
    // windows (blocks over 512 MiB) they grow past L2 instead (C4: 32 windows cost 93 ms)
    const u32 nwin = (u32)std::min<u64>(ceil_div(n, window), 8);
    const u64 step = ceil_div(n, nwin);
    for (u32 w = 0; w < nwin; ++w) {
        const u32 lo = (u32)(w * step), hi = (u32)std::min<u64>((u64)n, (w + 1) * step);
        if (w == 0)
            k_emit_bwt_window<256, true><<<blocks, 256, 0, ctx->stream>>>(d_text, n, d_sa, d_bwt, &ctx->mail_dev->origin, lo, hi, sa16);
        else
            k_emit_bwt_window<256, false><<<blocks, 256, 0, ctx->stream>>>(d_text, n, d_sa, d_bwt, &ctx->mail_dev->origin, lo, hi, sa16);
        LAUNCHED();
    }
    return 0;
}

void finish_stats(dark_bwt_ctx* ctx, dark_bwt_stats* st, int e_first, int e_last) {
    if (!st) return;
    float ms = 0.f;
    cudaEventElapsedTime(&ms, ctx->events[e_first], ctx->events[e_last]);
    st->device_ms = ms;
    for (const auto& s : ctx->spans) {
        if (s.e1 < 0) continue;
        float t = 0.f;
        cudaEventElapsedTime(&t, ctx->events[s.e0], ctx->events[s.e1]);
        switch (s.phase) {
            case PH_INIT: st->init_ms += t; break;
            case PH_SORT: st->sort_ms += t; break;
            case PH_PASS: st->pass_ms += t; break;
            case PH_GENPASS: st->pass_ms += t; st->gen_pass_ms += t; break;
            case PH_KEYBUILD: st->keybuild_ms += t; break;
            case PH_RERANK: st->rerank_ms += t; break;
            case PH_EMIT: st->emit_ms += t; break;
        }
    }
    st->kernel_launches = ctx->launches;
    st->host_syncs = ctx->syncs;
}

// The whole forward transform on device buffers.  d_sa_user nullable.
int forward_device(dark_bwt_ctx* ctx, const u8* d_text, u64 n64, u8* d_bwt, u64* origin_out, u32* d_sa_user,
                   dark_bwt_stats* st) {
    if (n64 < 2 || n64 > ctx->capacity || n64 > 0xFFFFFFFEull) return DARK_BWT_E_INVALID_N;
    const u32 n = (u32)n64;
    CK(cudaSetDevice(ctx->device));
    ctx->n_events = 0;
    ctx->spans.clear();
    ctx->next_counter = 0;
    ctx->launches = 0;
    ctx->syncs = 0;
    if (st) {
        const float h2d = st->h2d_ms;
        memset(st, 0, sizeof(*st));
        st->h2d_ms = h2d;
        st->n = n;
        st->active[0] = n;
    }
    u32* sa = d_sa_user ? d_sa_user : ctx->sa;

    const int e_first = ctx->n_events++;
    CK(cudaEventRecord(ctx->events[e_first], ctx->stream));

    // ---- alphabet: sigma, dense codes, symbols per key
    int sp = span_begin(ctx, PH_INIT);
    CK(cudaMemsetAsync(ctx->counters, 0, sizeof(u32) * kMaxCounters, ctx->stream));
    CK(cudaMemsetAsync(ctx->present, 0, sizeof(u32) * 256, ctx->stream));
    CK(cudaMemsetAsync(ctx->hist, 0, sizeof(u32) * kMaxPasses * kRadix, ctx->stream));
    const int no_pack = (ctx->flags & DARK_BWT_F_NO_ALPHABET_PACKING) ? 1 : 0;
    {
        const u32 blocks = (u32)std::min<u64>(ceil_div(ceil_div(n, 16), 256), 148 * 8);
        k_symbol_presence<256><<<std::max(blocks, 1u), 256, 0, ctx->stream>>>(d_text, n, ctx->present);
        LAUNCHED();
        k_build_lut<<<1, 256, 0, ctx->stream>>>(ctx->present, ctx->lut, &ctx->mail_dev->sigma, no_pack);
        LAUNCHED();
    }
    CK(sync_counted(ctx));
    const u32 sigma = ctx->mail->sigma;
    if (sigma < 1 || sigma > 256) return ctx->fail_internal("alphabet scan returned an impossible sigma");
    const int s_bits = no_pack ? 8 : std::max(1, bit_length(sigma - 1));
    const int K = 64 / s_bits;
    const int passes0 = kMaxPasses;  // the symbol field is MSB-aligned in the 64-bit key
    if (st) {
        st->sigma = sigma;
        st->bits_per_symbol = s_bits;
        st->symbols_per_key = K;
    }

    // ---- round 0: keys of K symbols, ids descending
    // Fused initial keys (s in {1,2,4,8}): the key builder only counts digits; the first radix pass that runs
    // rebuilds the keys from the text (radix_sort.cuh, GEN).  DARK_BWT_FUSED_INIT=0 materialises them instead.
    const Knobs& kn = ctx->knobs;
    const bool packed_s = s_bits == 1 || s_bits == 2 || s_bits == 4 || s_bits == 8;
    const bool fuse_init = packed_s && kn.fused_init && kn.sort_variant < 0;
    const bool gram_hist = packed_s && kn.gram_hist;  // histograms from the text's q-grams (suffix_kernels.cuh)
    const int lg_s = s_bits == 1 ? 0 : s_bits == 2 ? 1 : s_bits == 4 ? 2 : 3;
    auto init_keys = [&](bool write, bool hist) -> int {
        const u32 blocks = (u32)std::min<u64>(ceil_div(n, kInitThreads * kInitItems), (u64)ctx->num_sms * 8);
#define INIT_PACKED(S)                                                                                                              \
    do {                                                                                                                            \
        if (write && hist)                                                                                                          \
            k_init_keys_packed<kInitThreads, kInitItems, S, true, true><<<blocks, kInitThreads, 0, ctx->stream>>>(                  \
                d_text, n, ctx->lut, ctx->keys[0], ctx->ids[0], ctx->hist);                                                         \
        else if (write)                                                                                                             \
            k_init_keys_packed<kInitThreads, kInitItems, S, true, false><<<blocks, kInitThreads, 0, ctx->stream>>>(                 \
                d_text, n, ctx->lut, ctx->keys[0], ctx->ids[0], ctx->hist);                                                         \
        else                                                                                                                        \
            k_init_keys_packed<kInitThreads, kInitItems, S, false, true><<<blocks, kInitThreads, 0, ctx->stream>>>(d_text, n, ctx->lut, \
                                                                                                               nullptr, nullptr, ctx->hist); \
    } while (0)
        switch (s_bits) {
            case 1: INIT_PACKED(1); break;
            case 2: INIT_PACKED(2); break;
            case 4: INIT_PACKED(4); break;
            case 8: INIT_PACKED(8); break;
            default:
                k_init_keys<kInitThreads, kInitItems><<<blocks, kInitThreads, 0, ctx->stream>>>(
                    d_text, n, ctx->lut, s_bits, K, ctx->keys[0], ctx->ids[0], ctx->hist, passes0);
        }
#undef INIT_PACKED
        LAUNCHED();
        return 0;
    };
    if (gram_hist) {
        u32* gram = ctx->bucket_hist;  // 256 counters, free until the first rank scatter
        CK(cudaMemsetAsync(gram, 0, sizeof(u32) * kRadix, ctx->stream));
        const u32 blocks = (u32)std::min<u64>(ceil_div(n, 256 * 16), (u64)ctx->num_sms * 8);
        switch (s_bits) {
            case 1: k_gram_hist<256, 1><<<blocks, 256, 0, ctx->stream>>>(d_text, n, ctx->lut, gram); break;
            case 2: k_gram_hist<256, 2><<<blocks, 256, 0, ctx->stream>>>(d_text, n, ctx->lut, gram); break;
            case 4: k_gram_hist<256, 4><<<blocks, 256, 0, ctx->stream>>>(d_text, n, ctx->lut, gram); break;
            default: k_gram_hist<256, 8><<<blocks, 256, 0, ctx->stream>>>(d_text, n, ctx->lut, gram); break;
        }
        LAUNCHED();
        k_gram_expand<<<1, kRadix, 0, ctx->stream>>>(d_text, n, ctx->lut, lg_s, gram, ctx->hist);
        LAUNCHED();
        if (kn.check_hist) {  // test hook: compare with the histogram counted key by key
            std::vector<u32> a(kMaxPasses * kRadix), b(kMaxPasses * kRadix);
            CK(cudaMemcpyAsync(a.data(), ctx->hist, a.size() * 4, cudaMemcpyDeviceToHost, ctx->stream));
            CK(cudaMemsetAsync(ctx->hist, 0, sizeof(u32) * kMaxPasses * kRadix, ctx->stream));
            if (int rc = init_keys(false, true)) return rc;
            CK(cudaMemcpyAsync(b.data(), ctx->hist, b.size() * 4, cudaMemcpyDeviceToHost, ctx->stream));
            CK(sync_counted(ctx));
            if (a != b) return ctx->fail_internal("q-gram histogram differs from the per-key histogram");
            CK(cudaMemcpyAsync(ctx->hist, a.data(), a.size() * 4, cudaMemcpyHostToDevice, ctx->stream));
            CK(sync_counted(ctx));
        }
        if (!fuse_init)
            if (int rc = init_keys(true, false)) return rc;
    } else {
        if (int rc = init_keys(!fuse_init, true)) return rc;
    }
    span_end(ctx, sp);

    int cur = 0;
    int first_pass = 0;
    sp = span_begin(ctx, PH_SORT);
    // Inline emission: when the initial sort is pruned by >= 1 digit the BWT byte of each suffix travels in
    // the (unsorted) low key byte and is emitted as the suffix settles; no gather pass at the end.
    const bool want_inline = kn.inline_emit;
    bool emit_inline = false;
    KeyGen gen;
    gen.text = d_text;
    gen.lut = ctx->lut;
    gen.n = n;
    gen.lg_s = lg_s;
    gen.mode = 0;
    gen.origin = 0;
    bool gen_used = false;
    if (int rc = run_sort(ctx, ctx->keys, ctx->ids, cur, n, 0, passes0, &cur, st, 0, /*prune=*/!no_pack, &first_pass,
                          want_inline ? d_text : nullptr, &emit_inline, fuse_init ? &gen : nullptr, &gen_used))
        return rc;
    if (fuse_init && !gen_used) {  // every digit was trivial (one-symbol text): no pass ran, the re-rank still wants the keys
        if (int rc = init_keys(true, false)) return rc;
        cur = 0;
    }
    span_end(ctx, sp);
    // DARK_BWT_INLINE_GATHER=1: an unpruned block emits inline as well, the re-rank gathering T[id-1] for every suffix as it
    // settles.  Measured equal to the final gather pass (C4: re-rank +38 ms, emission -37 ms: one random DRAM sector per
    // suffix wherever the read is issued, profiles/r2_rejected.md), so it stays an option.
    if (want_inline && !emit_inline && kn.inline_gather > 0) emit_inline = true;
    u8* bwt_inline = emit_inline ? d_bwt : nullptr;
    // The sort covered the key bits above `drop`: K0 whole leading symbols are known equal inside a
    // tie group, Kc symbols were touched (a suffix shorter than Kc had padding compared).
    const int drop = first_pass * kRadixBits;
    const int sorted_bits = 64 - drop;
    const int K0 = std::min(K, sorted_bits / s_bits);
    const int Kc = std::min(K, (sorted_bits + s_bits - 1) / s_bits);
    if (K0 < 1) return ctx->fail_internal("initial sort covered less than one symbol");
    if (st) st->initial_symbols = K0;

    const int kb = bit_length(n);  // rank2 = isa+1 in [0, n]
    const int key_bits = kb + bit_length(((u64)n - 1) >> 1);  // high part = rank >> 1 (suffix_kernels.cuh, k_rerank)
    const int passes_r = (key_bits + kRadixBits - 1) / kRadixBits;

    sp = span_begin(ctx, PH_RERANK);
    u32 m = 0;
    bool sparse_done = false;
    bool pairs_checked = false;  // the pairs check of the current list was queued behind its re-rank: the answer is in the mailbox
    // Pruned initial sort with inline emission (high-entropy block: almost everything settles): the chain-free
    // sparse re-rank (suffix_kernels.cuh).  DARK_BWT_SPARSE_RERANK=0 keeps the scan-based kernel.
    if (emit_inline && first_pass >= 1 && kn.sparse_rerank) {
        u32 *total = nullptr, *ovf = nullptr;
        if (int rc = next_counter(ctx, &total)) return rc;
        if (int rc = next_counter(ctx, &ovf)) return rc;
        const u32 tiles = (u32)ceil_div(n, kScanTile);
        k_rerank0_sparse<kScanThreads, kScanItems><<<tiles, kScanThreads, 0, ctx->stream>>>(
            ctx->keys[cur], ctx->ids[cur], n, Kc, drop, sa, bwt_inline, &ctx->mail_dev->origin, (u8*)ctx->bitmap, total);
        LAUNCHED();
        k_copy_u32<<<1, 1, 0, ctx->stream>>>(total, &ctx->mail_dev->count);
        LAUNCHED();
        u32 survivors = 0;
        if (int rc = fetch_count(ctx, &survivors)) return rc;
        if (survivors == 0) {
            sparse_done = true;
        } else if (survivors <= n / 16) {
            const u64 nbytes = ceil_div(n, 8);
            const u32 nblocks = (u32)ceil_div(nbytes, kSparseChunk);
            u32* counts = (u32*)ctx->scan_words;  // n/32768 counters; the scan state is not in use
            u32* pos = ctx->ranks_alt;
            k_sparse_count<<<nblocks, 256, 0, ctx->stream>>>((const u8*)ctx->bitmap, nbytes, counts);
            LAUNCHED();
            k_sparse_scan<<<1, 1024, 0, ctx->stream>>>(counts, nblocks);
            LAUNCHED();
            k_sparse_positions<<<nblocks, 256, 0, ctx->stream>>>((const u8*)ctx->bitmap, nbytes, counts, pos);
            LAUNCHED();
            k_sparse_finalize<<<(u32)ceil_div(survivors, 256), 256, 0, ctx->stream>>>(pos, survivors, ctx->keys[cur], ctx->ids[cur], n, Kc, drop,
                                                                                 ctx->ids[cur ^ 1], ctx->ranks, ovf);
            LAUNCHED();
            k_copy_u32<<<1, 1, 0, ctx->stream>>>(ovf, &ctx->mail_dev->flag);
            LAUNCHED();
            CK(sync_counted(ctx));
            if (ctx->mail->flag == 0) {
                sparse_done = true;
                m = survivors;
            }
        }
    }
    // isa[] entries of active suffixes carry bit 31 (blocks up to 2^31 bytes): the text-order key builder finds
    // them by it.  DARK_BWT_TEXT_BUILD=0 switches tag and builder off; =<k> uses the builder while m > n/k.
    const int text_div = kn.text_div;
    const u32 tag = (text_div > 0 && (u64)n <= (1ull << 31)) ? 0x80000000u : 0u;
    ctx->tag = tag;
    // Scatters of more than n/16 ranks into an isa[] that outgrows L2 go through the bucketed path.
    const bool bucketed = kn.bucketed >= 0 ? kn.bucketed != 0 : ((u64)n * 4 > (96ull << 20));
    const int bshift = std::max(0, bit_length((u64)n - 1) - 8);
    // A large block whose initial sort was not pruned is text-like: most suffixes survive round 0 and every rank is needed.
    // Its round-0 re-rank then feeds the bucket regions of the rank scatter itself (every suffix reports its rank, settled
    // ones their slot) instead of two partition passes over the SA and the survivor list afterwards.  DARK_BWT_FUSE_ROUND0=0
    // keeps the separate passes.
    const bool fused0 = !sparse_done && bucketed && first_pass == 0 && kn.fuse_round0;
    PairSink sink0;
    if (!sparse_done) {
        if (fused0) {
            sink0.ids = (u32*)ctx->keys[cur ^ 1];
            sink0.vals = sink0.ids + align_up((size_t)n, 64);
            sink0.shift = bshift;
            CK(cudaMemsetAsync(ctx->bucket_hist, 0, sizeof(u32) * 256, ctx->stream));
            if (int rc = launch_rerank<true, true>(ctx, ctx->keys[cur], ctx->ids[cur], n, n, Kc, drop, sa, ctx->ids[cur ^ 1], d_text, bwt_inline, sink0)) return rc;
        } else {
            if (int rc = launch_rerank<true, false>(ctx, ctx->keys[cur], ctx->ids[cur], n, n, Kc, drop, sa, ctx->ids[cur ^ 1], d_text, bwt_inline)) return rc;
        }
        if (kn.pairs)
            if (int rc = queue_pairs_check(ctx, n, &pairs_checked)) return rc;
        if (int rc = fetch_count(ctx, &m)) return rc;
    }
    span_end(ctx, sp);
    cur ^= 1;  // the compacted active ids now live in ids[cur]

    // Round 0 wrote no ranks.  If a round follows they are needed: all of them when many suffixes
    // survive; otherwise only the survivors' now, and per round the few that are actually read.
    bool isa_complete = true;
    int selective_rounds = 0;
    const bool use_pairs = kn.pairs;
    bool pairs_mode = false;
    const bool use_search = kn.rank_search;
    if (m > 0 && fused0) {  // the regions hold every suffix's rank already
        sp = span_begin(ctx, PH_RERANK);
        if (int rc = region_scatter(ctx, sink0.ids, sink0.vals, n, bshift)) return rc;
        span_end(ctx, sp);
    } else if (m > 0) {
        sp = span_begin(ctx, PH_RERANK);
        if (m > n / 16) {
            if (bucketed) {  // every suffix gets its rank: settled ones their slot, survivors their group rank
                CK(cudaMemsetAsync(ctx->bucket_hist, 0, sizeof(u32) * 256, ctx->stream));
                u32* oi = (u32*)ctx->keys[0];
                u32* ov = (u32*)ctx->keys[1];
                if (int rc = bucket_partition(ctx, sa, nullptr, n, bshift, oi, ov)) return rc;
                if (int rc = bucket_partition(ctx, ctx->ids[cur], ctx->ranks, m, bshift, oi, ov, tag)) return rc;
                if (int rc = region_scatter(ctx, oi, ov, n, bshift)) return rc;
            } else {
                k_round0_isa<256><<<(u32)ceil_div(n, 256), 256, 0, ctx->stream>>>(sa, n, ctx->ids[cur], ctx->ranks, m, ctx->isa, tag);
                LAUNCHED();
            }
        } else {
            k_scatter_ranks<256><<<(u32)ceil_div(m, 256), 256, 0, ctx->stream>>>(ctx->ids[cur], ctx->ranks, m, ctx->isa, tag);
            LAUNCHED();
            isa_complete = false;
        }
        span_end(ctx, sp);
    }

    // ---- doubling rounds
    u64 h = (u64)K0;
    int round = 1;
    while (m > 0) {
        if (round >= DARK_BWT_MAX_ROUNDS || h >= 2 * (u64)n + 2) return ctx->fail_internal("prefix doubling did not converge");
        if (st) {
            st->active[round] = m;
            st->rounds = round;
        }
        // Once every remaining group is a pair the rounds switch to the pairs kernel for good (groups
        // only ever split).  The check reads the rank list once and costs a host round trip, so it is skipped
        // while most of the block is still active (period-17: ten rounds of giant groups).  The kernel gathers
        // from isa[], so it waits until every rank is there (few survivors after round 0: the selective rounds).
        if (use_pairs && !pairs_mode && isa_complete && (m & 1u) == 0 && (round == 1 || m <= n / 2)) {
            if (pairs_checked) {  // answered in the round trip that fetched m
                if (ctx->mail->not_pairs == 0) pairs_mode = true;
            } else {
                ctx->mail->flag = 0;
                u32* seen = nullptr;
                if (int rc = next_counter(ctx, &seen)) return rc;
                k_pairs_detect<<<(u32)std::min<u64>(ceil_div(m, 256), (u64)ctx->num_sms * 8), 256, 0, ctx->stream>>>(ctx->ranks, m, nullptr, seen,
                                                                                                                    &ctx->mail_dev->flag);
                LAUNCHED();
                CK(sync_counted(ctx));
                if (ctx->mail->flag == 0) {
                    pairs_mode = true;
                }
            }
        }
        pairs_checked = false;
        if (pairs_mode) {
            // every group is a pair: one kernel settles or keeps each pair (suffix_kernels.cuh, "pairs mode")
            sp = span_begin(ctx, PH_RERANK);
            constexpr int kPairThreads = 256, kPairsPerThread = 8;  // 4096 elements per tile, like the re-rank
            const u32 tiles = (u32)ceil_div(m / 2, kPairThreads * kPairsPerThread);
            if (tiles > ctx->scan_tiles) return ctx->fail_internal("scan tile state too small");
            u32* counter = nullptr;
            if (int rc = next_counter(ctx, &counter)) return rc;
            CK(cudaMemsetAsync(ctx->scan_words, 0, sizeof(u64) * kScanWordsPerTile * tiles, ctx->stream));
            ScanTileState ts{ctx->scan_words};
            k_pairs_round<kPairThreads, kPairsPerThread><<<tiles, kPairThreads, 0, ctx->stream>>>(
                ctx->ids[cur], ctx->ranks, m, n, h, ctx->isa, reinterpret_cast<uint2*>(ctx->keys[0]), sa, ctx->ids[cur ^ 1], ctx->ranks_alt, ts, counter,
                &ctx->mail_dev->count, d_text, bwt_inline, &ctx->mail_dev->origin, tag);
            LAUNCHED();
            std::swap(ctx->ranks, ctx->ranks_alt);
            span_end(ctx, sp);
            cur ^= 1;
            if (st) st->pair_rounds += 1;
            const u32 m_before = m;
            if (int rc = fetch_count(ctx, &m)) return rc;
            if (const u32 settled = (m_before - m) / 2) {
                k_pairs_apply<<<(u32)ceil_div(settled, 256), 256, 0, ctx->stream>>>(reinterpret_cast<const uint2*>(ctx->keys[0]), settled, ctx->isa);
                LAUNCHED();
            }
            h *= 2;
            ++round;
            continue;
        }
        if (kn.group_stats) {  // debug: group-size statistics of the active list
            CK(cudaMemsetAsync(ctx->bucket_hist, 0, 8, ctx->stream));
            k_group_stats<<<(u32)ceil_div(m, 256), 256, 0, ctx->stream>>>(ctx->ranks, m, ctx->bucket_hist);
            LAUNCHED();
            u32 gs[2] = {0, 0};
            CK(cudaMemcpyAsync(gs, ctx->bucket_hist, 8, cudaMemcpyDeviceToHost, ctx->stream));
            CK(sync_counted(ctx));
            fprintf(stderr, "[dark_bwt] round %d: h=%llu active=%u groups=%u max_group=%u%s\n", round, (unsigned long long)h, m, gs[1],
                    gs[0], gs[0] >= 4096 ? "+" : "");
        }
        sp = span_begin(ctx, PH_KEYBUILD);
        CK(cudaMemsetAsync(ctx->hist, 0, sizeof(u32) * kMaxPasses * kRadix, ctx->stream));
        bool keys_built = false;
        if (!isa_complete) {
            // ranks of suffixes settled in round 0 exist only where they are about to be read
            if (round == 1 && use_search) {
                // round 1: read the ranks off the sorted round-0 keys (still intact in keys[cur^1] / ids[cur^1])
                k_build_keys_search<256><<<(u32)ceil_div(m, 256), 256, 0, ctx->stream>>>(
                    ctx->ids[cur], ctx->ranks, m, n, h, kb, ctx->keys[cur ^ 1], ctx->ids[cur ^ 1], d_text, ctx->lut, s_bits, K, Kc,
                    drop, ctx->keys[cur], ctx->hist, passes_r);
                LAUNCHED();
                keys_built = true;
            } else if (selective_rounds < 2) {
                const size_t words = (size_t)ceil_div(n, 32);
                CK(cudaMemsetAsync(ctx->bitmap, 0, words * sizeof(u32), ctx->stream));
                k_mark_needed<256><<<(u32)ceil_div(m, 256), 256, 0, ctx->stream>>>(ctx->ids[cur], m, n, h, ctx->bitmap);
                LAUNCHED();
                k_fill_needed<256><<<(u32)ceil_div(n, 256), 256, 0, ctx->stream>>>(sa, n, ctx->bitmap, ctx->isa);
                LAUNCHED();
                ++selective_rounds;
            } else {  // still not done after two rounds: fill every settled rank once
                k_round0_isa<256><<<(u32)ceil_div(n, 256), 256, 0, ctx->stream>>>(sa, n, ctx->ids[cur], ctx->ranks, 0u, ctx->isa, tag);
                LAUNCHED();
                isa_complete = true;
            }
        }
        bool text_built = false;
        if (!keys_built && tag != 0 && isa_complete && (u64)m * (u64)text_div > (u64)n) {
            // many suffixes still active: sweep isa[] in text order instead of gathering from it (k_build_keys_text)
            constexpr int kTextThreads = 512, kTextItems = 8;
            const u32 tiles = (u32)ceil_div(n, kTextThreads * kTextItems);
            if (tiles > ctx->scan_tiles) return ctx->fail_internal("scan tile state too small");
            u32* counter = nullptr;
            if (int rc = next_counter(ctx, &counter)) return rc;
            CK(cudaMemsetAsync(ctx->scan_words, 0, sizeof(u64) * kScanWordsPerTile * tiles, ctx->stream));
            auto kern = k_build_keys_text<kTextThreads, kTextItems>;
            const size_t smem = kBuildTextSmem<kTextThreads, kTextItems>;
            CK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
            const u32 grid = std::min<u32>(tiles, (u32)ctx->num_sms * 3);
            kern<<<grid, kTextThreads, smem, ctx->stream>>>(ctx->isa, n, h, kb, tag, ctx->keys[cur], ctx->ids[cur], ctx->scan_words, counter,
                                                            &ctx->mail_dev->flag, ctx->hist, passes_r);
            LAUNCHED();
            keys_built = true;
            text_built = true;
        }
        if (!keys_built) {
            const u32 blocks = (u32)ceil_div(m, kBuildThreads * kBuildItems);  // one tile per CTA: the gathers want every warp slot filled
            k_build_keys<kBuildThreads, kBuildItems><<<blocks, kBuildThreads, 0, ctx->stream>>>(
                ctx->ids[cur], ctx->ranks, m, n, h, kb, ctx->isa, tag, ctx->keys[cur], ctx->hist, passes_r);
            LAUNCHED();
        }
        span_end(ctx, sp);

        sp = span_begin(ctx, PH_SORT);
        if (int rc = run_sort(ctx, ctx->keys, ctx->ids, cur, m, 0, passes_r, &cur, st, round, false, nullptr, nullptr, nullptr, nullptr, nullptr,
                              /*all_passes=*/text_built))
            return rc;
        span_end(ctx, sp);

        sp = span_begin(ctx, PH_RERANK);
        if (bucketed && m > n / 16) {
            // the re-rank appends each tile's rank updates to per-bucket regions (suffix_kernels.cuh, PAIRS); the
            // regions are then scattered bucket by bucket, each bucket's slice of isa[] staying in L2
            PairSink sink;
            sink.ids = (u32*)ctx->keys[cur ^ 1];
            sink.vals = sink.ids + align_up((size_t)n, 64);
            sink.shift = bshift;
            CK(cudaMemsetAsync(ctx->bucket_hist, 0, sizeof(u32) * 256, ctx->stream));
            if (int rc = launch_rerank<false, true>(ctx, ctx->keys[cur], ctx->ids[cur], m, n, K, kb, sa, ctx->ids[cur ^ 1], d_text, bwt_inline, sink)) return rc;
            if (int rc = region_scatter(ctx, sink.ids, sink.vals, m, bshift)) return rc;
        } else {
            if (int rc = launch_rerank<false, false>(ctx, ctx->keys[cur], ctx->ids[cur], m, n, K, kb, sa, ctx->ids[cur ^ 1], d_text, bwt_inline)) return rc;
        }
        span_end(ctx, sp);
        cur ^= 1;
        const u32 m_sorted = m;
        if (use_pairs && isa_complete && m_sorted <= n / 2) {  // the list that comes out may be all pairs: ask now, read with the count
            if (int rc = queue_pairs_check(ctx, m_sorted, &pairs_checked)) return rc;
        }
        if (int rc = fetch_count(ctx, &m)) return rc;
        if (text_built && ctx->mail->flag != m_sorted) return ctx->fail_internal("tagged isa[] entries disagree with the active list");
        h *= 2;
        ++round;
    }

    // ---- BWT bytes + origin
    sp = span_begin(ctx, PH_EMIT);
    if (!emit_inline)
        if (int rc = emit(ctx, d_text, n, sa, d_bwt)) return rc;
    span_end(ctx, sp);
    const int e_last = ctx->n_events++;
    CK(cudaEventRecord(ctx->events[e_last], ctx->stream));
    CK(sync_counted(ctx));
    *origin_out = ctx->mail->origin;
    finish_stats(ctx, st, e_first, e_last);
    return DARK_BWT_OK;
}

// Many independent blocks in one sort (suffix_kernels.cuh, "many small blocks").  d_text holds the blocks back
// to back, ctx->many_starts their offsets (B + 1 values, already on the device); d_bwt receives the per-block BWTs
// at the same offsets, ctx->many_origins the origins.
int forward_many_device(dark_bwt_ctx* ctx, const u8* d_text, u32 n, u32 B, u8* d_bwt, u32* d_sa_out, dark_bwt_stats* st) {
    CK(cudaSetDevice(ctx->device));
    ctx->n_events = 0;
    ctx->spans.clear();
    ctx->next_counter = 0;
    ctx->launches = 0;
    ctx->tag = 0;
    if (st) {
        const float h2d = st->h2d_ms;
        memset(st, 0, sizeof(*st));
        st->h2d_ms = h2d;
        st->n = n;
        st->active[0] = n;
    }
    const int e_first = ctx->n_events++;
    CK(cudaEventRecord(ctx->events[e_first], ctx->stream));
    int sp = span_begin(ctx, PH_INIT);
    CK(cudaMemsetAsync(ctx->counters, 0, sizeof(u32) * kMaxCounters, ctx->stream));
    CK(cudaMemsetAsync(ctx->present, 0, sizeof(u32) * 256, ctx->stream));
    CK(cudaMemsetAsync(ctx->hist, 0, sizeof(u32) * kMaxPasses * kRadix, ctx->stream));
    {
        const u32 blocks = (u32)std::min<u64>(ceil_div(ceil_div(n, 16), 256), 148 * 8);
        k_symbol_presence<256><<<std::max(blocks, 1u), 256, 0, ctx->stream>>>(d_text, n, ctx->present);
        LAUNCHED();
        k_many_lut<<<1, 256, 0, ctx->stream>>>(ctx->present, ctx->many_lut, &ctx->mail_dev->sigma);
        LAUNCHED();
    }
    CK(cudaStreamSynchronize(ctx->stream));
    const u32 sigma = ctx->mail->sigma;
    if (sigma < 1 || sigma > 256) return ctx->fail_internal("alphabet scan returned an impossible sigma");
    const int s_bits = bit_length(sigma);  // codes 1..sigma, 0 = past the end of the block
    const int K = 64 / s_bits;
    if (st) {
        st->sigma = sigma;
        st->bits_per_symbol = s_bits;
        st->symbols_per_key = K;
        st->initial_symbols = K;
    }
    const u32 grid = (u32)std::min<u64>(ceil_div(n, 256), (u64)ctx->num_sms * 8);
    k_many_init_keys<256><<<grid, 256, 0, ctx->stream>>>(d_text, n, ctx->many_lut, s_bits, K, ctx->many_starts, B, ctx->keys[0], ctx->ids[0],
                                                         ctx->hist);
    LAUNCHED();
    span_end(ctx, sp);

    int cur = 0;
    sp = span_begin(ctx, PH_SORT);
    if (int rc = run_sort(ctx, ctx->keys, ctx->ids, cur, n, 0, kMaxPasses, &cur, st, 0)) return rc;
    span_end(ctx, sp);
    sp = span_begin(ctx, PH_RERANK);
    // no "short suffix" special case (K = 1 disables it): the padding code 0 orders proper prefixes first
    if (int rc = launch_rerank<true, false>(ctx, ctx->keys[cur], ctx->ids[cur], n, n, 1, 0, ctx->sa, ctx->ids[cur ^ 1], d_text, nullptr)) return rc;
    span_end(ctx, sp);
    cur ^= 1;
    u32 m = 0;
    if (int rc = fetch_count(ctx, &m)) return rc;
    if (m > 0) {
        k_round0_isa<256><<<(u32)ceil_div(n, 256), 256, 0, ctx->stream>>>(ctx->sa, n, ctx->ids[cur], ctx->ranks, m, ctx->isa, 0u);
        LAUNCHED();
    }
    const int kb = bit_length((u64)n + B);  // rank2 in [0, n + B]
    const int key_bits = kb + bit_length(((u64)n - 1) >> 1);
    if (key_bits > 64) return ctx->fail_internal("batch too large for 64-bit keys");
    const int passes_r = (key_bits + kRadixBits - 1) / kRadixBits;
    u64 h = (u64)K;
    int round = 1;
    while (m > 0) {
        if (round >= DARK_BWT_MAX_ROUNDS || h >= 2 * (u64)n + 2) return ctx->fail_internal("prefix doubling did not converge");
        if (st) {
            st->active[round] = m;
            st->rounds = round;
        }
        sp = span_begin(ctx, PH_KEYBUILD);
        CK(cudaMemsetAsync(ctx->hist, 0, sizeof(u32) * kMaxPasses * kRadix, ctx->stream));
        const u32 g2 = (u32)std::min<u64>(ceil_div(m, 256), (u64)ctx->num_sms * 8);
        k_many_build_keys<256><<<g2, 256, 0, ctx->stream>>>(ctx->ids[cur], ctx->ranks, m, h, kb, ctx->isa, ctx->many_starts, B, ctx->keys[cur],
                                                            ctx->hist, passes_r);
        LAUNCHED();
        span_end(ctx, sp);
        sp = span_begin(ctx, PH_SORT);
        if (int rc = run_sort(ctx, ctx->keys, ctx->ids, cur, m, 0, passes_r, &cur, st, round)) return rc;
        span_end(ctx, sp);
        sp = span_begin(ctx, PH_RERANK);
        if (int rc = launch_rerank<false, false>(ctx, ctx->keys[cur], ctx->ids[cur], m, n, K, kb, ctx->sa, ctx->ids[cur ^ 1], d_text, nullptr)) return rc;
        span_end(ctx, sp);
        cur ^= 1;
        if (int rc = fetch_count(ctx, &m)) return rc;
        h *= 2;
        ++round;
    }
    // bring every block's suffixes together (stable sort of the interleaved SA by block number), then emit
    sp = span_begin(ctx, PH_EMIT);
    const int bits = std::max(1, bit_length((u64)B - 1));
    const int passes_b = (bits + kRadixBits - 1) / kRadixBits;
    CK(cudaMemsetAsync(ctx->hist, 0, sizeof(u32) * kMaxPasses * kRadix, ctx->stream));
    k_many_blocks_of_sa<256><<<grid, 256, 0, ctx->stream>>>(ctx->sa, n, ctx->many_starts, B, ctx->keys[0], ctx->ids[0], ctx->hist, passes_b);
    LAUNCHED();
    cur = 0;
    if (int rc = run_sort(ctx, ctx->keys, ctx->ids, cur, n, 0, passes_b, &cur, nullptr, 0)) return rc;
    k_many_emit<<<(u32)ceil_div(n, 256), 256, 0, ctx->stream>>>(ctx->keys[cur], ctx->ids[cur], n, d_text, ctx->many_starts, d_bwt,
                                                               ctx->many_origins, d_sa_out);
    LAUNCHED();
    span_end(ctx, sp);
    const int e_last = ctx->n_events++;
    CK(cudaEventRecord(ctx->events[e_last], ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    finish_stats(ctx, st, e_first, e_last);
    return DARK_BWT_OK;
}

// Inverse BWT on device buffers (kernels and method: suffix_kernels.cuh, "inverse BWT").
int inverse_device(dark_bwt_ctx* ctx, const u8* d_bwt, u64 n64, u64 origin64, u8* d_text, float* ms_out) {
    if (n64 < 1 || n64 > ctx->capacity || n64 > 0xFFFFFFFEull) return DARK_BWT_E_INVALID_N;
    if (origin64 >= n64) return DARK_BWT_E_INVALID_ARG;
    const u32 n = (u32)n64, origin = (u32)origin64;
    CK(cudaSetDevice(ctx->device));
    ctx->n_events = 0;
    ctx->spans.clear();
    ctx->next_counter = 0;
    cudaEvent_t ea = ctx->events[kMaxEvents - 1], eb = ctx->events[kMaxEvents - 2];
    CK(cudaEventRecord(ea, ctx->stream));
    CK(cudaMemsetAsync(ctx->counters, 0, sizeof(u32) * kMaxCounters, ctx->stream));
    CK(cudaMemsetAsync(ctx->hist, 0, sizeof(u32) * kMaxPasses * kRadix, ctx->stream));
    // step 1: (last-column symbol, row) pairs; stable partition by symbol -> psi.  The pairs are built inside the
    // radix pass (GEN mode 1) and their digit histogram is the byte histogram of the BWT.
    int cur = 0;
    {
        k_build_lut<<<1, 256, 0, ctx->stream>>>(ctx->present, ctx->lut, &ctx->mail_dev->sigma, 1);  // identity codes
        LAUNCHED();
        u32* gram = ctx->bucket_hist;
        CK(cudaMemsetAsync(gram, 0, sizeof(u32) * kRadix, ctx->stream));
        const u32 blocks = (u32)std::min<u64>(ceil_div(n, 256 * 16), (u64)ctx->num_sms * 8);
        k_gram_hist<256, 8><<<std::max(blocks, 1u), 256, 0, ctx->stream>>>(d_bwt, n, ctx->lut, gram);
        LAUNCHED();
        CK(cudaMemcpyAsync(ctx->hist, gram, sizeof(u32) * kRadix, cudaMemcpyDeviceToDevice, ctx->stream));
        KeyGen gen;
        gen.text = d_bwt;
        gen.lut = ctx->lut;
        gen.n = n;
        gen.lg_s = 3;
        gen.mode = 1;
        gen.origin = origin;
        bool gen_used = false;
        if (int rc = run_sort(ctx, ctx->keys, ctx->ids, 0, n, 0, 1, &cur, nullptr, 0, false, nullptr, nullptr, nullptr, &gen, &gen_used)) return rc;
        if (!gen_used) {  // one-symbol BWT: the pass is the identity and did not run; psi is the row list itself
            k_ibwt_elements<<<(u32)ceil_div(n, 256), 256, 0, ctx->stream>>>(d_bwt, n, origin, ctx->keys[0], ctx->ids[0]);
            LAUNCHED();
            cur = 0;
        }
    }
    const u32* psi1 = ctx->ids[cur];
    // step 2: sublists between splitters
    const u32 stride = (u32)ctx->knobs.ibwt_stride;  // rows between splitters; swept 24..128 with the single walk: 48 (profiles/r1_final.md)
    const u32 head = origin + 1;
    const u32 regular = (u32)ceil_div((u64)n + 1, stride);
    const u32 nodes = regular + 1;
    u32* dist[2] = {ctx->ranks, ctx->sa};
    u32* next[2] = {ctx->isa, ctx->ids[cur ^ 1]};
    // one walk: count the sublists and stash their symbols (DARK_BWT_IBWT_TWO_WALKS=1: count, then a second walk writes)
    u32* len_keep = ctx->ranks_alt;
    u32* stash = (u32*)ctx->keys[cur ^ 1];  // the sort's other key buffer (8 n + 1024 bytes) is free: nodes * 384 <= 6 n + 768
    const u32 cap = (u32)std::min<u64>(kIbwtStashCap, (((u64)n * 8 + 1024) / nodes) & ~3ull);  // smaller strides: smaller chunks
    const bool two_walks = ctx->knobs.ibwt_two_walks || cap < 8;
    // k_ibwt_walk needs the symbol bases (exclusive digit counts of pass 0, left in ctx->hist by run_sort)
    if (two_walks)
        k_ibwt_walk<0><<<(u32)ceil_div(nodes, 128), 128, 0, ctx->stream>>>(psi1, n, head, stride, regular, dist[0], next[0], nullptr, nullptr,
                                                                         nullptr, nullptr, nullptr, 0u, 0u);
    else
        k_ibwt_walk<2><<<(u32)ceil_div(nodes, 128), 128, 0, ctx->stream>>>(psi1, n, head, stride, regular, dist[0], next[0], nullptr, ctx->hist,
                                                                         nullptr, len_keep, stash, 0u, cap);
    LAUNCHED();
    // step 3: suffix sums of the sublist lengths along the splitter list (pointer jumping)
    int w = 0;
    for (u32 span = 1; span < nodes; span <<= 1) {
        k_ibwt_jump<<<(u32)ceil_div(nodes, 256), 256, 0, ctx->stream>>>(dist[w], next[w], dist[w ^ 1], next[w ^ 1], nodes);
        LAUNCHED();
        w ^= 1;
    }
    k_ibwt_report<<<1, 1, 0, ctx->stream>>>(dist[w], regular, &ctx->mail_dev->count);
    LAUNCHED();
    CK(cudaStreamSynchronize(ctx->stream));
    if ((u64)ctx->mail->count != (u64)n + 1) {
        snprintf(ctx->err, sizeof(ctx->err), "inverse BWT: (bwt, origin) is not a forward transform (list covers %u of %llu rows)",
                 ctx->mail->count, (unsigned long long)n + 1);
        return DARK_BWT_E_INVALID_ARG;
    }
    // step 4: the text.  Stashed sublists are copied to their offsets; the few longer ones are walked again.
    if (two_walks) {
        k_ibwt_walk<1><<<(u32)ceil_div(nodes, 128), 128, 0, ctx->stream>>>(psi1, n, head, stride, regular, nullptr, nullptr, dist[w], ctx->hist,
                                                                         d_text, nullptr, nullptr, 0u, 0u);
        LAUNCHED();
    } else {
        k_ibwt_unstash<<<(u32)ceil_div(nodes, 128), 128, 0, ctx->stream>>>(stash, len_keep, dist[w], n, regular, d_text, cap);
        LAUNCHED();
        k_ibwt_walk<1><<<(u32)ceil_div(nodes, 128), 128, 0, ctx->stream>>>(psi1, n, head, stride, regular, nullptr, nullptr, dist[w], ctx->hist,
                                                                         d_text, len_keep, nullptr, cap, 0u);
        LAUNCHED();
    }
    CK(cudaEventRecord(eb, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    if (ms_out) cudaEventElapsedTime(ms_out, ea, eb);
    return DARK_BWT_OK;
}

// Inverse BWT of B blocks in one pass (suffix_kernels.cuh, "inverse BWT of many blocks").  d_bwt holds the blocks back to
// back (n bytes), ctx->many_starts their offsets and ctx->many_origins their origins (validated, on the device); d_text
// receives the texts at the same offsets.  max_nb = the largest block.
//
// Buffers: the rows number R = n + B <= capacity (the entry points check it).  The sort moves n <= capacity pairs.  The
// node arrays (dist and next twice, len_keep) hold `regular + B` entries, and regular = ceil(R / stride) <= (R + 1) / 2 with
// stride >= 2 while every block has at least two rows (B <= R / 2): nodes <= R <= capacity, which the u32 arrays of the
// arena hold.  The stash gets (8 capacity + 1024) / nodes >= 8 bytes a chunk.  So 65,536 blocks of one byte need a
// capacity of 131,072 (rows, not bytes, are what must fit), and sum(ns) <= capacity alone would not be enough.
int inverse_many_device(dark_bwt_ctx* ctx, const u8* d_bwt, u32 n, u32 B, u32 max_nb, u8* d_text, float* ms_out) {
    CK(cudaSetDevice(ctx->device));
    ctx->n_events = 0;
    ctx->spans.clear();
    ctx->next_counter = 0;
    cudaEvent_t ea = ctx->events[kMaxEvents - 1], eb = ctx->events[kMaxEvents - 2];
    CK(cudaEventRecord(ea, ctx->stream));
    CK(cudaMemsetAsync(ctx->counters, 0, sizeof(u32) * kMaxCounters, ctx->stream));
    CK(cudaMemsetAsync(ctx->hist, 0, sizeof(u32) * kMaxPasses * kRadix, ctx->stream));
    // step 1: (block, last symbol) keys of the real rows, one stable sort -> psi and the first symbols
    const int passes = 1 + (B > 1 ? (bit_length((u64)B - 1) + kRadixBits - 1) / kRadixBits : 0);
    const u32 grid = (u32)std::min<u64>(ceil_div(n, 256), (u64)ctx->num_sms * 8);
    k_ibwt_many_elements<256><<<grid, 256, 0, ctx->stream>>>(d_bwt, n, ctx->many_starts, B, ctx->many_origins, ctx->keys[0], ctx->ids[0],
                                                             ctx->hist, passes);
    LAUNCHED();
    int cur = 0;
    // passes whose digit is the same in every key are skipped (one-symbol blocks, a single block): the order stays the row order
    if (int rc = run_sort(ctx, ctx->keys, ctx->ids, 0, n, 0, passes, &cur, nullptr, 0)) return rc;
    const u32* psi = ctx->ids[cur];
    const u64* skeys = ctx->keys[cur];
    // step 2: sublists between splitters (buffers as in inverse_device)
    const u32 stride = (u32)ctx->knobs.ibwt_stride;
    const u32 regular = (u32)ceil_div((u64)n + B, stride);
    const u32 nodes = regular + B;
    u32* dist[2] = {ctx->ranks, ctx->sa};
    u32* next[2] = {ctx->isa, ctx->ids[cur ^ 1]};
    u32* len_keep = ctx->ranks_alt;
    u32* stash = (u32*)ctx->keys[cur ^ 1];
    const u32 cap = (u32)std::min<u64>(kIbwtStashCap, ((ctx->capacity * 8 + 1024) / nodes) & ~3ull);
    const bool two_walks = ctx->knobs.ibwt_two_walks || cap < 8;
    const u32 wgrid = (u32)ceil_div(nodes, 128);
    if (two_walks)
        k_ibwt_many_walk<0><<<wgrid, 128, 0, ctx->stream>>>(psi, skeys, ctx->many_starts, B, ctx->many_origins, stride, regular, dist[0], next[0],
                                                            nullptr, nullptr, nullptr, nullptr, 0u, 0u);
    else
        k_ibwt_many_walk<2><<<wgrid, 128, 0, ctx->stream>>>(psi, skeys, ctx->many_starts, B, ctx->many_origins, stride, regular, dist[0], next[0],
                                                            nullptr, nullptr, len_keep, stash, 0u, cap);
    LAUNCHED();
    // step 3: pointer jumping; a block's list holds at most ceil((max_nb + 1) / stride) + 1 splitters
    const u64 chain = ceil_div((u64)max_nb + 1, stride) + 1;
    int w = 0;
    for (u64 span = 1; span < chain; span <<= 1) {
        k_ibwt_jump<<<(u32)ceil_div(nodes, 256), 256, 0, ctx->stream>>>(dist[w], next[w], dist[w ^ 1], next[w ^ 1], nodes);
        LAUNCHED();
        w ^= 1;
    }
    k_ibwt_many_check<<<1, 1024, 0, ctx->stream>>>(dist[w], regular, ctx->many_starts, B, &ctx->mail_dev->count, &ctx->mail_dev->bad_block);
    LAUNCHED();
    CK(cudaStreamSynchronize(ctx->stream));
    if (ctx->mail->count != 0) {
        snprintf(ctx->err, sizeof(ctx->err), "inverse BWT: block %u is not a forward transform (%u of %u blocks are not)",
                 ctx->mail->bad_block, ctx->mail->count, B);
        return DARK_BWT_E_INVALID_ARG;
    }
    // step 4: the texts
    if (two_walks) {
        k_ibwt_many_walk<1><<<wgrid, 128, 0, ctx->stream>>>(psi, skeys, ctx->many_starts, B, ctx->many_origins, stride, regular, nullptr, nullptr,
                                                            dist[w], d_text, nullptr, nullptr, 0u, 0u);
        LAUNCHED();
    } else {
        k_ibwt_many_unstash<<<wgrid, 128, 0, ctx->stream>>>(stash, len_keep, dist[w], ctx->many_starts, B, stride, regular, d_text, cap);
        LAUNCHED();
        k_ibwt_many_walk<1><<<wgrid, 128, 0, ctx->stream>>>(psi, skeys, ctx->many_starts, B, ctx->many_origins, stride, regular, nullptr, nullptr,
                                                            dist[w], d_text, len_keep, nullptr, cap, 0u);
        LAUNCHED();
    }
    CK(cudaEventRecord(eb, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    if (ms_out) cudaEventElapsedTime(ms_out, ea, eb);
    return DARK_BWT_OK;
}

// Distance coding + MTF of a BWT block on device buffers (dc_kernels.cuh).  Every output pointer is nullable: the
// context's own arena is used for what the caller does not want.  *d_dist_used / *d_pos_used etc. tell where the data is.
struct DcBuffers {
    u32* dist = nullptr;     // n
    u32* item_pos = nullptr; // num_items
    u32* item_dist = nullptr;
    u8* item_sym = nullptr;
    u8* item_rank = nullptr;
};
int dc_device(dark_bwt_ctx* ctx, const u8* d_bwt, u64 n64, DcBuffers* io, dark_bwt_dc_info* info) {
    if (n64 < 1 || n64 > ctx->capacity || n64 > 0xFFFFFFFEull) return DARK_BWT_E_INVALID_N;
    const u32 n = (u32)n64;
    CK(cudaSetDevice(ctx->device));
    const u32 nblocks = (u32)ceil_div(n, kDcBlock);
    // last-occurrence tables: (nblocks + ngroups) x 256 words = n/4 + n/1024 bytes (+ 2 KB): inside the 4n-byte rank buffer for
    // all but tiny blocks, which borrow the sort's status buffer (>= 256 KB)
    u32* tab = ctx->ranks;
    if (n <= 65536u) {
        tab = (u32*)ctx->sort_status;
        for (int h = 0; h < 2; ++h) ctx->status_dirty_lo[h] = 0u, ctx->status_dirty_hi[h] = (u32)(ctx->sort_status_bytes / 2 / (kRadix * sizeof(u32)));
    }
    u32* run_counts = ctx->ranks_alt;
    u32* first = ctx->bucket_hist;
    u32* final_last = ctx->bucket_hist + 256;
    if (!io->dist) io->dist = (u32*)ctx->keys[0];
    if (!io->item_pos) io->item_pos = ctx->isa;
    if (!io->item_dist) io->item_dist = ctx->sa;
    u32* run_start = ctx->ids[0];
    if (!io->item_sym) io->item_sym = (u8*)ctx->ids[1];
    if (!io->item_rank) io->item_rank = (u8*)ctx->ids[1] + (size_t)n;
    unsigned long long* total_runs = (unsigned long long*)((char*)ctx->dc_info + align_up(sizeof(DcInfoDev), 8));
    cudaEvent_t ea = ctx->events[kMaxEvents - 1], eb = ctx->events[kMaxEvents - 2];
    CK(cudaEventRecord(ea, ctx->stream));
    CK(cudaMemsetAsync(first, 0xFF, sizeof(u32) * 256, ctx->stream));
    CK(cudaMemsetAsync(total_runs, 0, sizeof(unsigned long long), ctx->stream));
    k_dc_tables<<<nblocks, 256, 0, ctx->stream>>>(d_bwt, n, tab, first, run_counts, io->dist, total_runs);
    LAUNCHED();
    const u32 ngroups = (u32)ceil_div(nblocks, kDcGroup);
    u32* group_last = tab + (size_t)nblocks * 256;  // ngroups x 256 words behind the table (n/4 + n/1024 bytes of the 4n)
    k_dc_scan_groups<<<ngroups, 256, 0, ctx->stream>>>(tab, nblocks, group_last);
    LAUNCHED();
    k_dc_scan_carry<<<1, 256, 0, ctx->stream>>>(group_last, ngroups, final_last);
    LAUNCHED();
    k_sparse_scan<<<1, 1024, 0, ctx->stream>>>(run_counts, nblocks);  // in place: exclusive run offsets
    LAUNCHED();
    u32* alpha = ctx->bucket_hist + 512;  // 513 words: dense codes of the symbols that occur
    k_dc_alphabet<<<1, 256, 0, ctx->stream>>>(first, alpha);
    LAUNCHED();
    k_dc_ranks<<<(u32)ceil_div(nblocks, 8), 256, 0, ctx->stream>>>(d_bwt, n, tab, group_last, run_counts, nblocks, alpha, io->dist, run_start, io->item_sym, io->item_rank);
    LAUNCHED();
    k_dc_final<<<1, 256, 0, ctx->stream>>>(n, final_last, first, io->dist, total_runs, ctx->dc_info);
    LAUNCHED();
    k_dc_stream<<<(u32)std::min<u64>(ceil_div(n, 256), (u64)ctx->num_sms * 16), 256, 0, ctx->stream>>>(run_start, total_runs, n, io->dist, io->item_pos, io->item_dist);
    LAUNCHED();
    CK(cudaEventRecord(eb, ctx->stream));
    static_assert(offsetof(dark_bwt_dc_info, num_items) == offsetof(DcInfoDev, num_items), "DcInfoDev mirrors the head of dark_bwt_dc_info");
    CK(cudaMemcpyAsync(info, ctx->dc_info, sizeof(DcInfoDev), cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    cudaEventElapsedTime(&info->device_ms, ea, eb);
    return DARK_BWT_OK;
}

// ---- pageable host buffers ---------------------------------------------------------------------
bool is_pageable(const void* p) {
    cudaPointerAttributes a;
    if (cudaPointerGetAttributes(&a, p) != cudaSuccess) {
        cudaGetLastError();
        return true;
    }
    return a.type == cudaMemoryTypeUnregistered;
}

int stage_prepare(dark_bwt_ctx* ctx, HostStage& st) {
    if (st.lanes > 0) return 0;
    const int lanes = ctx->knobs.host_threads;
    if (lanes <= 0) return 1;  // staging switched off
    st.chunk = (size_t)ctx->knobs.host_chunk_mb << 20;
    if (cudaHostAlloc((void**)&st.pinned, st.chunk * lanes * 2, cudaHostAllocDefault) != cudaSuccess) {
        cudaGetLastError();
        st.pinned = nullptr;
        return 1;  // no pinned memory to be had: fall back to the driver's own staging
    }
    for (int i = 0; i < lanes; ++i) {
        if (cudaStreamCreateWithFlags(&st.streams[i], cudaStreamNonBlocking) != cudaSuccess) return ctx->fail_cuda(cudaGetLastError(), "staging stream", __LINE__);
        for (int k = 0; k < 2; ++k)
            if (cudaEventCreateWithFlags(&st.slot_done[i][k], cudaEventDisableTiming) != cudaSuccess)
                return ctx->fail_cuda(cudaGetLastError(), "staging event", __LINE__);
    }
    st.lanes = lanes;
    return 0;
}

void stage_release(HostStage& st) {
    for (int i = 0; i < HostStage::kMaxLanes; ++i) {
        if (st.streams[i]) cudaStreamDestroy(st.streams[i]);
        for (int k = 0; k < 2; ++k)
            if (st.slot_done[i][k]) cudaEventDestroy(st.slot_done[i][k]);
    }
    if (st.pinned) cudaFreeHost(st.pinned);
    st = HostStage();
}

// Copies `bytes` between a pageable host buffer and device memory through the lanes of `st`; returns when done.
// The caller has made sure that the device side is ready (H2D: the buffer is free; D2H: the data is complete).
int staged_copy(dark_bwt_ctx* ctx, HostStage& st, void* dev, void* host, size_t bytes, bool to_device) {
    const size_t chunk = st.chunk;
    const size_t nchunks = (bytes + chunk - 1) / chunk;
    const int lanes = (int)std::min<size_t>((size_t)st.lanes, nchunks);
    std::atomic<size_t> next(0);
    std::atomic<int> failed(0);
    auto work = [&](int lane) {
        if (cudaSetDevice(ctx->device) != cudaSuccess) {
            failed = 1;
            return;
        }
        // two pinned slots per lane: the memcpy of one chunk overlaps the DMA of the lane's other slot
        u8* const slots[2] = {st.pinned + (size_t)(2 * lane) * chunk, st.pinned + (size_t)(2 * lane + 1) * chunk};
        cudaStream_t sm = st.streams[lane];
        cudaEvent_t* done = st.slot_done[lane];
        bool busy[2] = {false, false};            // H2D: a DMA out of the slot is in flight
        size_t p_off = 0, p_len = 0;              // D2H: the chunk whose DMA into slot p_slot was issued last
        int p_slot = -1, cur = 0;
        auto ok = [&](cudaError_t e) {
            if (e != cudaSuccess) failed = 1;
            return e == cudaSuccess;
        };
        for (;;) {
            const size_t c = next.fetch_add(1);
            if (c >= nchunks || failed.load()) break;
            const size_t off = c * chunk, len = std::min(chunk, bytes - off);
            const int sl = cur;
            cur ^= 1;
            if (to_device) {
                if (busy[sl] && !ok(cudaEventSynchronize(done[sl]))) break;
                memcpy(slots[sl], (const u8*)host + off, len);
                if (!ok(cudaMemcpyAsync((u8*)dev + off, slots[sl], len, cudaMemcpyHostToDevice, sm)) || !ok(cudaEventRecord(done[sl], sm))) break;
                busy[sl] = true;
            } else {
                if (!ok(cudaMemcpyAsync(slots[sl], (const u8*)dev + off, len, cudaMemcpyDeviceToHost, sm)) || !ok(cudaEventRecord(done[sl], sm))) break;
                if (p_slot >= 0) {
                    if (!ok(cudaEventSynchronize(done[p_slot]))) break;
                    memcpy((u8*)host + p_off, slots[p_slot], p_len);
                }
                p_slot = sl, p_off = off, p_len = len;
            }
        }
        if (!to_device && p_slot >= 0 && !failed.load() && ok(cudaEventSynchronize(done[p_slot]))) memcpy((u8*)host + p_off, slots[p_slot], p_len);
        ok(cudaStreamSynchronize(sm));
    };
    std::vector<std::thread> pool;
    for (int i = 1; i < lanes; ++i) pool.emplace_back(work, i);
    work(0);
    for (auto& t : pool) t.join();
    if (failed.load()) return ctx->fail_cuda(cudaGetLastError(), "staged host copy", __LINE__);
    return 0;
}

constexpr size_t kStageMinBytes = 1u << 20;  // smaller copies go straight to cudaMemcpyAsync

// host -> device on `stream` semantics: returns after the copy has completed
int copy_in_blocking(dark_bwt_ctx* ctx, u8* dev, const u8* host, size_t bytes, cudaStream_t stream) {
    if (bytes >= kStageMinBytes && is_pageable(host)) {
        const int rc = stage_prepare(ctx, ctx->stage_in);
        if (rc > 1) return rc;
        if (rc == 0) return staged_copy(ctx, ctx->stage_in, dev, (void*)host, bytes, true);
    }
    CK(cudaMemcpyAsync(dev, host, bytes, cudaMemcpyHostToDevice, stream));
    CK(cudaStreamSynchronize(stream));
    return 0;
}
int copy_out_blocking(dark_bwt_ctx* ctx, void* host, const void* dev, size_t bytes, cudaStream_t stream) {
    if (bytes >= kStageMinBytes && is_pageable(host)) {
        const int rc = stage_prepare(ctx, ctx->stage_out);
        if (rc > 1) return rc;
        if (rc == 0) return staged_copy(ctx, ctx->stage_out, (void*)dev, host, bytes, false);
    }
    CK(cudaMemcpyAsync(host, dev, bytes, cudaMemcpyDeviceToHost, stream));
    CK(cudaStreamSynchronize(stream));
    return 0;
}

// A second copy-out of a block that must be complete before the next block is transformed (its device buffer is single).
struct SideCopy {
    void* host = nullptr;
    const void* dev = nullptr;
    size_t bytes = 0;
};

// The pipelined loop of the batch entries: `count` host blocks ins[k] (ns[k] bytes) -> outs[k] (ns[k] bytes).  While block
// k is transformed (transform(k, d_in[b], d_out[b], &side), synchronous on the context's stream), block k+1 is copied into
// the other input buffer and block k-1 out of the other output buffer.  Pinned host buffers ride on the two copy
// streams; pageable ones (>= 1 MiB) are moved by the staging lanes in a helper thread.
template <typename Transform>
int run_pipelined(dark_bwt_ctx* ctx, const u8* const* ins, const uint64_t* ns, u8* const* outs, uint64_t count, u8* const d_in[2],
                  u8* const d_out[2], Transform transform) {
    bool comp_recorded[2] = {false, false}, out_recorded[2] = {false, false};
    std::future<int> fin[2], fout;
    auto staged_in = [&](uint64_t k) { return ns[k] >= kStageMinBytes && is_pageable(ins[k]) && stage_prepare(ctx, ctx->stage_in) == 0; };
    auto staged_out = [&](uint64_t k) { return ns[k] >= kStageMinBytes && is_pageable(outs[k]) && stage_prepare(ctx, ctx->stage_out) == 0; };
    auto start_in = [&](uint64_t k, int buf) -> int {  // the transform that read d_in[buf] has returned (it is synchronous)
        if (staged_in(k)) {
            u8* dst = d_in[buf];
            const u8* src = ins[k];
            const size_t bytes = ns[k];
            fin[buf] = std::async(std::launch::async, [ctx, dst, src, bytes] { return staged_copy(ctx, ctx->stage_in, dst, (void*)src, bytes, true); });
            return 0;
        }
        if (comp_recorded[buf]) CK(cudaStreamWaitEvent(ctx->copy_in, ctx->ev_comp[buf], 0));
        CK(cudaMemcpyAsync(d_in[buf], ins[k], ns[k], cudaMemcpyHostToDevice, ctx->copy_in));
        CK(cudaEventRecord(ctx->ev_in[buf], ctx->copy_in));
        return 0;
    };
    auto drain = [&]() {  // never leave a helper thread behind
        int rc = 0;
        for (int i = 0; i < 2; ++i)
            if (fin[i].valid()) rc |= fin[i].get();
        if (fout.valid()) rc |= fout.get();
        return rc;
    };
    if (int rc = start_in(0, 0)) return rc;
    for (uint64_t k = 0; k < count; ++k) {
        const int b = (int)(k & 1), nb = b ^ 1;
        if (fin[b].valid()) {
            if (int rc = fin[b].get()) { drain(); return rc; }
        } else {
            CK(cudaStreamWaitEvent(ctx->stream, ctx->ev_in[b], 0));
        }
        if (k + 1 < count)
            if (int rc = start_in(k + 1, nb)) { drain(); return rc; }
        // (a staged copy-out of block k-1 may still be reading the OTHER output buffer; this one was drained before it began)
        if (out_recorded[b]) CK(cudaStreamWaitEvent(ctx->stream, ctx->ev_out[b], 0));  // output buffer b drained
        SideCopy side;
        int rc = transform(k, (const u8*)d_in[b], d_out[b], &side);
        if (rc) { drain(); return rc; }
        CK(cudaEventRecord(ctx->ev_comp[b], ctx->stream));
        comp_recorded[b] = true;
        if (fout.valid())
            if (int rc2 = fout.get()) { drain(); return rc2; }  // one staged copy-out at a time (they share the lanes)
        if (staged_out(k)) {
            u8* dst = outs[k];
            const u8* src = d_out[b];
            const size_t bytes = ns[k];
            fout = std::async(std::launch::async, [ctx, dst, src, bytes, side] {
                int r = staged_copy(ctx, ctx->stage_out, (void*)src, dst, bytes, false);
                if (r == 0 && side.host) r = staged_copy(ctx, ctx->stage_out, (void*)side.dev, side.host, side.bytes, false);
                return r;
            });
            if (side.host)
                if (int rc2 = fout.get()) { drain(); return rc2; }  // the side buffer is reused by the next block
            out_recorded[b] = false;
        } else {
            CK(cudaStreamWaitEvent(ctx->copy_out, ctx->ev_comp[b], 0));
            CK(cudaMemcpyAsync(outs[k], d_out[b], ns[k], cudaMemcpyDeviceToHost, ctx->copy_out));
            if (side.host) {  // the side buffer is reused by the next block: drain it before going on
                CK(cudaMemcpyAsync(side.host, side.dev, side.bytes, cudaMemcpyDeviceToHost, ctx->copy_out));
                CK(cudaStreamSynchronize(ctx->copy_out));
            }
            CK(cudaEventRecord(ctx->ev_out[b], ctx->copy_out));
            out_recorded[b] = true;
        }
    }
    if (int rc = drain()) return rc;
    CK(cudaStreamSynchronize(ctx->copy_out));
    CK(cudaStreamSynchronize(ctx->copy_in));
    return DARK_BWT_OK;
}

}  // namespace

// =================================================================================================
extern "C" {

int dark_bwt_abi_version(void) { return DARK_BWT_ABI_VERSION; }

const char* dark_bwt_strerror(int code) {
    switch (code) {
        case DARK_BWT_OK: return "ok";
        case DARK_BWT_E_INVALID_N: return "invalid block length (need 2 <= n <= capacity and n <= 2^32-2)";
        case DARK_BWT_E_INVALID_ARG: return "invalid argument";
        case DARK_BWT_E_CUDA: return "CUDA failure";
        case DARK_BWT_E_NOMEM: return "out of device or pinned host memory";
        case DARK_BWT_E_INTERNAL: return "internal invariant violated";
        default: return "unknown error";
    }
}

const char* dark_bwt_last_error(const dark_bwt_ctx* ctx) { return ctx ? ctx->err : ""; }
uint64_t dark_bwt_capacity(const dark_bwt_ctx* ctx) { return ctx ? ctx->capacity : 0; }
void* dark_bwt_stream(const dark_bwt_ctx* ctx) { return ctx ? (void*)ctx->stream : nullptr; }

int dark_bwt_create(uint64_t max_n, int device, dark_bwt_ctx** out) {
    return dark_bwt_create_ex(max_n, device, DARK_BWT_F_DEFAULT, out);
}

int dark_bwt_create_ex(uint64_t max_n, int device, uint32_t flags, dark_bwt_ctx** out) {
    if (!out) return DARK_BWT_E_INVALID_ARG;
    *out = nullptr;
    if (flags & ~(DARK_BWT_F_NO_ALPHABET_PACKING | DARK_BWT_F_DEVICE_ONLY)) return DARK_BWT_E_INVALID_ARG;
    if (max_n < 2 || max_n > 0xFFFFFFFEull) return DARK_BWT_E_INVALID_N;
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) return DARK_BWT_E_CUDA;  // no CPU fallback
    if (device < 0 || device >= ndev) return DARK_BWT_E_INVALID_ARG;
    if (cudaSetDevice(device) != cudaSuccess) return DARK_BWT_E_CUDA;

    dark_bwt_ctx* ctx = new (std::nothrow) dark_bwt_ctx();
    if (!ctx) return DARK_BWT_E_NOMEM;
    ctx->device = device;
    {
        int sms = 0;
        if (cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, device) == cudaSuccess && sms > 0) ctx->num_sms = sms;
    }
    ctx->capacity = max_n;
    ctx->flags = flags;
    ctx->knobs.read_env();

    const size_t N = (size_t)max_n;
    const size_t sort_tiles = ceil_div(N, kSortTile);
    ctx->sort_status_bytes = (sort_tiles + 128) * kRadix * sizeof(u64);  // + rows the scanner CTA reads ahead
    ctx->scan_tiles = ceil_div(N, std::min(kScanTile, 4096));  // the pairs kernel and the text-order builder scan 4,096-suffix tiles
    const bool staging = !(flags & DARK_BWT_F_DEVICE_ONLY);

    size_t off = 0;
    auto carve = [&](size_t bytes) {
        size_t o = off;
        off = align_up(off + bytes, 256);
        return o;
    };
    const size_t o_keys0 = carve(N * 8 + 1024), o_keys1 = carve(N * 8 + 1024);  // slack: pair lists are split at a 64-aligned offset
    const size_t o_ids0 = carve(N * 4 + 16), o_ids1 = carve(N * 4 + 16);
    const size_t o_ranks = carve(N * 4 + 16), o_ranks2 = carve(N * 4 + 16), o_isa = carve(N * 4 + 16), o_sa = carve(N * 4 + 16);
    const size_t o_text = staging ? carve(N + 16) : 0, o_bwt = staging ? carve(N + 16) : 0;
    const size_t o_text2 = staging ? carve(N + 16) : 0, o_bwt2 = staging ? carve(N + 16) : 0;
    const size_t o_hist = carve(sizeof(u32) * kMaxPasses * kRadix);
    const size_t o_present = carve(sizeof(u32) * 256);
    const size_t o_lut = carve(256);
    const size_t o_scalars = carve(sizeof(DeviceScalars));
    const size_t o_status = carve(ctx->sort_status_bytes);
    const size_t o_counters = carve(sizeof(u32) * kMaxCounters);
    const size_t o_bhist = carve(sizeof(u32) * 1280);  // 256 bucket counters/cursors + 257 chunk prefixes; DC: first/last occurrences + dense alphabet
    const size_t o_bitmap = carve(sizeof(u32) * (ceil_div(N, 32) + 1) + 1024);  // + one tile of flag bytes past the end
    const size_t o_bitmap2 = carve(sizeof(u32) * (ceil_div(N, 32) + 1) + 1024);
    const size_t o_swords = carve(sizeof(u64) * kScanWordsPerTile * ctx->scan_tiles);
    const size_t o_mstarts = carve(sizeof(u32) * (kMaxManyBlocks + 1));
    const size_t o_morigins = carve(sizeof(unsigned long long) * kMaxManyBlocks);
    const size_t o_mlut = carve(sizeof(u16) * 256);
    const size_t o_dcinfo = carve(sizeof(DcInfoDev) + 16);
    ctx->arena_bytes = off;

    auto bail = [&](int code) {
        dark_bwt_destroy(ctx);
        return code;
    };
    if (cudaMalloc(&ctx->arena, ctx->arena_bytes) != cudaSuccess) {
        cudaGetLastError();
        ctx->arena = nullptr;
        return bail(DARK_BWT_E_NOMEM);
    }
    char* base = (char*)ctx->arena;
    ctx->keys[0] = (u64*)(base + o_keys0);
    ctx->keys[1] = (u64*)(base + o_keys1);
    ctx->ids[0] = (u32*)(base + o_ids0);
    ctx->ids[1] = (u32*)(base + o_ids1);
    ctx->ranks = (u32*)(base + o_ranks);
    ctx->ranks_alt = (u32*)(base + o_ranks2);
    ctx->isa = (u32*)(base + o_isa);
    ctx->sa = (u32*)(base + o_sa);
    ctx->d_text = staging ? (u8*)(base + o_text) : nullptr;
    ctx->d_bwt = staging ? (u8*)(base + o_bwt) : nullptr;
    ctx->d_text2 = staging ? (u8*)(base + o_text2) : nullptr;
    ctx->d_bwt2 = staging ? (u8*)(base + o_bwt2) : nullptr;
    ctx->hist = (u32*)(base + o_hist);
    ctx->present = (u32*)(base + o_present);
    ctx->lut = (u8*)(base + o_lut);
    ctx->scalars = (DeviceScalars*)(base + o_scalars);
    ctx->sort_status = base + o_status;
    for (int h = 0; h < 2; ++h) ctx->status_dirty_lo[h] = 0u, ctx->status_dirty_hi[h] = (u32)(ctx->sort_status_bytes / 2 / (kRadix * sizeof(u32)));
    ctx->counters = (u32*)(base + o_counters);
    ctx->scan_words = (u64*)(base + o_swords);
    ctx->bitmap = (u32*)(base + o_bitmap);
    ctx->bitmap2 = (u32*)(base + o_bitmap2);
    ctx->bucket_hist = (u32*)(base + o_bhist);
    ctx->many_starts = (u32*)(base + o_mstarts);
    ctx->many_origins = (unsigned long long*)(base + o_morigins);
    ctx->many_lut = (u16*)(base + o_mlut);
    ctx->dc_info = (DcInfoDev*)(base + o_dcinfo);

    if (cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking) != cudaSuccess) return bail(DARK_BWT_E_CUDA);
    if (staging) {
        if (cudaStreamCreateWithFlags(&ctx->copy_in, cudaStreamNonBlocking) != cudaSuccess ||
            cudaStreamCreateWithFlags(&ctx->copy_out, cudaStreamNonBlocking) != cudaSuccess)
            return bail(DARK_BWT_E_CUDA);
        for (int i = 0; i < 2; ++i)
            if (cudaEventCreateWithFlags(&ctx->ev_in[i], cudaEventDisableTiming) != cudaSuccess ||
                cudaEventCreateWithFlags(&ctx->ev_comp[i], cudaEventDisableTiming) != cudaSuccess ||
                cudaEventCreateWithFlags(&ctx->ev_out[i], cudaEventDisableTiming) != cudaSuccess)
                return bail(DARK_BWT_E_CUDA);
    }
    if (cudaHostAlloc((void**)&ctx->mail, sizeof(Mailbox), cudaHostAllocMapped) != cudaSuccess) return bail(DARK_BWT_E_NOMEM);
    memset(ctx->mail, 0, sizeof(Mailbox));
    if (cudaHostGetDevicePointer((void**)&ctx->mail_dev, ctx->mail, 0) != cudaSuccess) return bail(DARK_BWT_E_CUDA);
    for (int i = 0; i < kMaxEvents; ++i) {
        ctx->events[i] = nullptr;
        if (cudaEventCreate(&ctx->events[i]) != cudaSuccess) return bail(DARK_BWT_E_CUDA);
    }
    if (cudaMemsetAsync(ctx->scalars, 0, sizeof(DeviceScalars), ctx->stream) != cudaSuccess) return bail(DARK_BWT_E_CUDA);
    if (cudaStreamSynchronize(ctx->stream) != cudaSuccess) return bail(DARK_BWT_E_CUDA);
    *out = ctx;
    return DARK_BWT_OK;
}

void dark_bwt_destroy(dark_bwt_ctx* ctx) {
    if (!ctx) return;
    cudaSetDevice(ctx->device);
    if (ctx->stream) cudaStreamSynchronize(ctx->stream);
    for (int i = 0; i < kMaxEvents; ++i)
        if (ctx->events[i]) cudaEventDestroy(ctx->events[i]);
    for (int i = 0; i < 2; ++i) {
        if (ctx->ev_in[i]) cudaEventDestroy(ctx->ev_in[i]);
        if (ctx->ev_comp[i]) cudaEventDestroy(ctx->ev_comp[i]);
        if (ctx->ev_out[i]) cudaEventDestroy(ctx->ev_out[i]);
    }
    stage_release(ctx->stage_in);
    stage_release(ctx->stage_out);
    if (ctx->copy_in) cudaStreamDestroy(ctx->copy_in);
    if (ctx->copy_out) cudaStreamDestroy(ctx->copy_out);
    if (ctx->stream) cudaStreamDestroy(ctx->stream);
    if (ctx->mail) cudaFreeHost(ctx->mail);
    if (ctx->arena) cudaFree(ctx->arena);
    free(ctx->reuse_words);
    delete ctx;
}

int dark_bwt_forward_device(dark_bwt_ctx* ctx, const uint8_t* d_text, uint64_t n, uint8_t* d_bwt_out, uint64_t* origin_out,
                            uint32_t* d_sa_out, dark_bwt_stats* stats) {
    if (!ctx || !d_text || !d_bwt_out || !origin_out) return DARK_BWT_E_INVALID_ARG;
    ctx->err[0] = 0;
    if (stats) stats->h2d_ms = 0.f;
    return forward_device(ctx, d_text, n, d_bwt_out, origin_out, d_sa_out, stats);
}

int dark_bwt_forward(dark_bwt_ctx* ctx, const uint8_t* text, uint64_t n, uint8_t* bwt_out, uint64_t* origin_out,
                     uint32_t* sa_out, dark_bwt_stats* stats) {
    if (!ctx || !text || !bwt_out || !origin_out) return DARK_BWT_E_INVALID_ARG;
    ctx->err[0] = 0;
    if (ctx->flags & DARK_BWT_F_DEVICE_ONLY) return DARK_BWT_E_INVALID_ARG;
    if (n < 2 || n > ctx->capacity || n > 0xFFFFFFFEull) return DARK_BWT_E_INVALID_N;
    CK(cudaSetDevice(ctx->device));
    // pinned (or registered) buffers are copied directly, pageable ones through the context's pinned staging lanes
    typedef std::chrono::steady_clock Clock;
    auto ms_since = [](Clock::time_point t0) { return std::chrono::duration<float, std::milli>(Clock::now() - t0).count(); };
    Clock::time_point t0 = Clock::now();
    if (int rc = copy_in_blocking(ctx, ctx->d_text, text, n, ctx->stream)) return rc;
    const float h2d = ms_since(t0);
    if (stats) stats->h2d_ms = h2d;
    int rc = forward_device(ctx, ctx->d_text, n, ctx->d_bwt, origin_out, nullptr, stats);
    if (rc) return rc;
    t0 = Clock::now();
    if (int rc2 = copy_out_blocking(ctx, bwt_out, ctx->d_bwt, n, ctx->stream)) return rc2;
    if (sa_out)
        if (int rc2 = copy_out_blocking(ctx, sa_out, ctx->sa, n * sizeof(u32), ctx->stream)) return rc2;
    if (stats) stats->d2h_ms = ms_since(t0);
    return DARK_BWT_OK;
}

int dark_bwt_forward_batch(dark_bwt_ctx* ctx, const uint8_t* const* texts, const uint64_t* ns, uint8_t* const* bwt_outs,
                           uint64_t* origins_out, uint32_t* const* sa_outs, uint64_t count, dark_bwt_stats* stats) {
    if (!ctx || !texts || !ns || !bwt_outs || !origins_out) return DARK_BWT_E_INVALID_ARG;
    if (ctx->flags & DARK_BWT_F_DEVICE_ONLY) return DARK_BWT_E_INVALID_ARG;
    ctx->err[0] = 0;
    for (uint64_t k = 0; k < count; ++k) {
        if (!texts[k] || !bwt_outs[k]) return DARK_BWT_E_INVALID_ARG;
        if (ns[k] < 2 || ns[k] > ctx->capacity || ns[k] > 0xFFFFFFFEull) return DARK_BWT_E_INVALID_N;
    }
    if (count == 0) return DARK_BWT_OK;
    CK(cudaSetDevice(ctx->device));
    u8* const d_text[2] = {ctx->d_text, ctx->d_text2};
    u8* const d_bwt[2] = {ctx->d_bwt, ctx->d_bwt2};
    return run_pipelined(ctx, texts, ns, bwt_outs, count, d_text, d_bwt, [&](uint64_t k, const u8* din, u8* dout, SideCopy* side) {
        dark_bwt_stats* st = stats ? stats + k : nullptr;
        if (st) st->h2d_ms = 0.f;
        const int rc = forward_device(ctx, din, ns[k], dout, origins_out + k, nullptr, st);
        if (rc == 0 && sa_outs && sa_outs[k]) {  // the SA of the block is in the context's single SA buffer
            side->host = sa_outs[k];
            side->dev = ctx->sa;
            side->bytes = ns[k] * sizeof(u32);
        }
        return rc;
    });
}

int dark_bwt_inverse_batch(dark_bwt_ctx* ctx, const uint8_t* const* bwts, const uint64_t* ns, const uint64_t* origins,
                           uint8_t* const* text_outs, uint64_t count, float* ms_out) {
    if (!ctx || !bwts || !ns || !origins || !text_outs) return DARK_BWT_E_INVALID_ARG;
    if (ctx->flags & DARK_BWT_F_DEVICE_ONLY) return DARK_BWT_E_INVALID_ARG;
    ctx->err[0] = 0;
    for (uint64_t k = 0; k < count; ++k) {
        if (!bwts[k] || !text_outs[k]) return DARK_BWT_E_INVALID_ARG;
        if (ns[k] < 1 || ns[k] > ctx->capacity || ns[k] > 0xFFFFFFFEull) return DARK_BWT_E_INVALID_N;
        if (origins[k] >= ns[k]) return DARK_BWT_E_INVALID_ARG;
    }
    if (count == 0) return DARK_BWT_OK;
    CK(cudaSetDevice(ctx->device));
    u8* const d_bwt[2] = {ctx->d_bwt, ctx->d_bwt2};
    u8* const d_text[2] = {ctx->d_text, ctx->d_text2};
    return run_pipelined(ctx, bwts, ns, text_outs, count, d_bwt, d_text, [&](uint64_t k, const u8* din, u8* dout, SideCopy*) {
        return inverse_device(ctx, din, ns[k], origins[k], dout, ms_out ? ms_out + k : nullptr);
    });
}

int dark_bwt_forward_many(dark_bwt_ctx* ctx, const uint8_t* const* texts, const uint64_t* ns, uint8_t* const* bwt_outs,
                          uint64_t* origins_out, uint64_t count, dark_bwt_stats* stats) {
    if (!ctx || !texts || !ns || !bwt_outs || !origins_out) return DARK_BWT_E_INVALID_ARG;
    if (ctx->flags & DARK_BWT_F_DEVICE_ONLY) return DARK_BWT_E_INVALID_ARG;
    ctx->err[0] = 0;
    if (count == 0) return DARK_BWT_OK;
    if (count > kMaxManyBlocks) return DARK_BWT_E_INVALID_ARG;
    std::vector<u32> starts(count + 1);
    u64 total = 0;
    for (uint64_t k = 0; k < count; ++k) {
        if (!texts[k] || !bwt_outs[k]) return DARK_BWT_E_INVALID_ARG;
        if (ns[k] < 2) return DARK_BWT_E_INVALID_N;
        starts[k] = (u32)total;
        total += ns[k];
        if (total > ctx->capacity || total > 0xFFFFFFFEull) return DARK_BWT_E_INVALID_N;  // the blocks share one arena
    }
    starts[count] = (u32)total;
    CK(cudaSetDevice(ctx->device));
    cudaEvent_t a = ctx->events[kMaxEvents - 1], b = ctx->events[kMaxEvents - 2];
    CK(cudaEventRecord(a, ctx->stream));
    CK(cudaMemcpyAsync(ctx->many_starts, starts.data(), sizeof(u32) * (count + 1), cudaMemcpyHostToDevice, ctx->stream));
    for (uint64_t k = 0; k < count; ++k)
        CK(cudaMemcpyAsync(ctx->d_text + starts[k], texts[k], ns[k], cudaMemcpyHostToDevice, ctx->stream));
    CK(cudaEventRecord(b, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));  // `starts` may go out of scope only after the copy
    float h2d = 0.f;
    cudaEventElapsedTime(&h2d, a, b);
    if (stats) stats->h2d_ms = h2d;
    if (int rc = forward_many_device(ctx, ctx->d_text, (u32)total, (u32)count, ctx->d_bwt, nullptr, stats)) return rc;
    CK(cudaEventRecord(a, ctx->stream));
    for (uint64_t k = 0; k < count; ++k)
        CK(cudaMemcpyAsync(bwt_outs[k], ctx->d_bwt + starts[k], ns[k], cudaMemcpyDeviceToHost, ctx->stream));
    static_assert(sizeof(unsigned long long) == sizeof(uint64_t), "origins are copied as they are");
    CK(cudaMemcpyAsync(origins_out, ctx->many_origins, sizeof(uint64_t) * count, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaEventRecord(b, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    if (stats) cudaEventElapsedTime(&stats->d2h_ms, a, b);
    return DARK_BWT_OK;
}

int dark_bwt_forward_many_device(dark_bwt_ctx* ctx, const uint8_t* d_text, const uint32_t* d_starts, uint64_t count,
                                 uint8_t* d_bwt_out, uint64_t* d_origins_out, uint32_t* d_sa_out, dark_bwt_stats* stats) {
    if (!ctx || !d_text || !d_starts || !d_bwt_out || !d_origins_out) return DARK_BWT_E_INVALID_ARG;
    ctx->err[0] = 0;
    if (count == 0) return DARK_BWT_OK;
    if (count > kMaxManyBlocks) return DARK_BWT_E_INVALID_ARG;
    CK(cudaSetDevice(ctx->device));
    std::vector<u32> starts(count + 1);
    CK(cudaMemcpyAsync(starts.data(), d_starts, sizeof(u32) * (count + 1), cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    if (starts[0] != 0) return DARK_BWT_E_INVALID_ARG;
    for (uint64_t k = 0; k < count; ++k)
        if (starts[k + 1] < starts[k] + 2) return DARK_BWT_E_INVALID_N;
    const u64 total = starts[count];
    if (total > ctx->capacity || total > 0xFFFFFFFEull) return DARK_BWT_E_INVALID_N;
    CK(cudaMemcpyAsync(ctx->many_starts, d_starts, sizeof(u32) * (count + 1), cudaMemcpyDeviceToDevice, ctx->stream));
    if (stats) stats->h2d_ms = 0.f;
    if (int rc = forward_many_device(ctx, d_text, (u32)total, (u32)count, d_bwt_out, d_sa_out, stats)) return rc;
    CK(cudaMemcpyAsync(d_origins_out, ctx->many_origins, sizeof(uint64_t) * count, cudaMemcpyDeviceToDevice, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    return DARK_BWT_OK;
}

int dark_bwt_inverse_device(dark_bwt_ctx* ctx, const uint8_t* d_bwt, uint64_t n, uint64_t origin, uint8_t* d_text_out,
                            float* ms_out) {
    if (!ctx || !d_bwt || !d_text_out) return DARK_BWT_E_INVALID_ARG;
    ctx->err[0] = 0;
    return inverse_device(ctx, d_bwt, n, origin, d_text_out, ms_out);
}

int dark_bwt_inverse(dark_bwt_ctx* ctx, const uint8_t* bwt, uint64_t n, uint64_t origin, uint8_t* text_out) {
    if (!ctx || !bwt || !text_out) return DARK_BWT_E_INVALID_ARG;
    if (ctx->flags & DARK_BWT_F_DEVICE_ONLY) return DARK_BWT_E_INVALID_ARG;
    if (n < 1 || n > ctx->capacity || n > 0xFFFFFFFEull) return DARK_BWT_E_INVALID_N;
    ctx->err[0] = 0;
    CK(cudaSetDevice(ctx->device));
    if (int rc = copy_in_blocking(ctx, ctx->d_bwt, bwt, n, ctx->stream)) return rc;
    if (int rc = inverse_device(ctx, ctx->d_bwt, n, origin, ctx->d_text, nullptr)) return rc;
    return copy_out_blocking(ctx, text_out, ctx->d_text, n, ctx->stream);
}

int dark_bwt_inverse_many(dark_bwt_ctx* ctx, const uint8_t* const* bwts, const uint64_t* ns, const uint64_t* origins,
                          uint8_t* const* text_outs, uint64_t count, float* ms_out) {
    if (!ctx || !bwts || !ns || !origins || !text_outs) return DARK_BWT_E_INVALID_ARG;
    if (count > kMaxManyBlocks) return DARK_BWT_E_INVALID_ARG;
    if (ctx->flags & DARK_BWT_F_DEVICE_ONLY) return DARK_BWT_E_INVALID_ARG;
    ctx->err[0] = 0;
    if (count == 0) return DARK_BWT_OK;
    std::vector<u32> starts(count + 1);
    u64 total = 0, max_nb = 0;
    for (uint64_t k = 0; k < count; ++k) {
        if (!bwts[k] || !text_outs[k]) return DARK_BWT_E_INVALID_ARG;
        if (ns[k] < 1) return DARK_BWT_E_INVALID_N;
        if (origins[k] >= ns[k]) return DARK_BWT_E_INVALID_ARG;
        starts[k] = (u32)total;
        total += ns[k];
        max_nb = std::max<u64>(max_nb, ns[k]);
        if (total + k + 1 > ctx->capacity) return DARK_BWT_E_INVALID_N;  // the rows (bytes + one '$' row per block) share the arena
    }
    starts[count] = (u32)total;
    CK(cudaSetDevice(ctx->device));
    static_assert(sizeof(unsigned long long) == sizeof(uint64_t), "origins are copied as they are");
    CK(cudaMemcpyAsync(ctx->many_starts, starts.data(), sizeof(u32) * (count + 1), cudaMemcpyHostToDevice, ctx->stream));
    CK(cudaMemcpyAsync(ctx->many_origins, origins, sizeof(uint64_t) * count, cudaMemcpyHostToDevice, ctx->stream));
    for (uint64_t k = 0; k < count; ++k)
        CK(cudaMemcpyAsync(ctx->d_bwt + starts[k], bwts[k], ns[k], cudaMemcpyHostToDevice, ctx->stream));
    if (int rc = inverse_many_device(ctx, ctx->d_bwt, (u32)total, (u32)count, (u32)max_nb, ctx->d_text, ms_out)) return rc;
    for (uint64_t k = 0; k < count; ++k)
        CK(cudaMemcpyAsync(text_outs[k], ctx->d_text + starts[k], ns[k], cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    return DARK_BWT_OK;
}

int dark_bwt_inverse_many_device(dark_bwt_ctx* ctx, const uint8_t* d_bwt, const uint32_t* d_starts, const uint64_t* d_origins,
                                 uint64_t count, uint8_t* d_text_out, float* ms_out) {
    if (!ctx || !d_bwt || !d_starts || !d_origins || !d_text_out) return DARK_BWT_E_INVALID_ARG;
    if (count > kMaxManyBlocks) return DARK_BWT_E_INVALID_ARG;
    ctx->err[0] = 0;
    if (count == 0) return DARK_BWT_OK;
    CK(cudaSetDevice(ctx->device));
    // offsets and origins are checked on the host before any kernel reads them
    std::vector<u32> starts(count + 1);
    std::vector<uint64_t> origins(count);
    CK(cudaMemcpyAsync(starts.data(), d_starts, sizeof(u32) * (count + 1), cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaMemcpyAsync(origins.data(), d_origins, sizeof(uint64_t) * count, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    if (starts[0] != 0) return DARK_BWT_E_INVALID_ARG;
    u64 max_nb = 0;
    for (uint64_t k = 0; k < count; ++k) {
        if ((u64)starts[k + 1] < (u64)starts[k] + 1) return DARK_BWT_E_INVALID_N;
        const u64 nb = (u64)starts[k + 1] - starts[k];
        if (origins[k] >= nb) return DARK_BWT_E_INVALID_ARG;
        max_nb = std::max(max_nb, nb);
    }
    const u64 total = starts[count];
    if (total + count > ctx->capacity) return DARK_BWT_E_INVALID_N;
    CK(cudaMemcpyAsync(ctx->many_starts, d_starts, sizeof(u32) * (count + 1), cudaMemcpyDeviceToDevice, ctx->stream));
    CK(cudaMemcpyAsync(ctx->many_origins, d_origins, sizeof(uint64_t) * count, cudaMemcpyDeviceToDevice, ctx->stream));
    return inverse_many_device(ctx, d_bwt, (u32)total, (u32)count, (u32)max_nb, d_text_out, ms_out);
}

int dark_bwt_dc_encode_device(dark_bwt_ctx* ctx, const uint8_t* d_bwt, uint64_t n, uint32_t* d_dist_out, uint32_t* d_item_pos,
                              uint32_t* d_item_dist, uint8_t* d_item_sym, uint8_t* d_item_rank, dark_bwt_dc_info* info) {
    if (!ctx || !d_bwt || !info) return DARK_BWT_E_INVALID_ARG;
    ctx->err[0] = 0;
    DcBuffers io;
    io.dist = d_dist_out;
    io.item_pos = d_item_pos;
    io.item_dist = d_item_dist;
    io.item_sym = d_item_sym;
    io.item_rank = d_item_rank;
    return dc_device(ctx, d_bwt, n, &io, info);
}

// host buffers; ctx->d_bwt already holds the block when `bwt` is null (dark_bwt_forward_dc)
static int dc_host(dark_bwt_ctx* ctx, const uint8_t* bwt, uint64_t n, uint32_t* dist_out, uint32_t* item_pos, uint32_t* item_dist,
                   uint8_t* item_sym, uint8_t* item_rank, dark_bwt_dc_info* info) {
    if (bwt)
        if (int rc = copy_in_blocking(ctx, ctx->d_bwt, bwt, n, ctx->stream)) return rc;
    DcBuffers io;
    if (int rc = dc_device(ctx, ctx->d_bwt, n, &io, info)) return rc;
    const size_t items = (size_t)info->num_items;
    if (dist_out)
        if (int rc = copy_out_blocking(ctx, dist_out, io.dist, n * sizeof(u32), ctx->stream)) return rc;
    if (item_pos && items)
        if (int rc = copy_out_blocking(ctx, item_pos, io.item_pos, items * sizeof(u32), ctx->stream)) return rc;
    if (item_dist && items)
        if (int rc = copy_out_blocking(ctx, item_dist, io.item_dist, items * sizeof(u32), ctx->stream)) return rc;
    if (item_sym && items)
        if (int rc = copy_out_blocking(ctx, item_sym, io.item_sym, items, ctx->stream)) return rc;
    if (item_rank && items)
        if (int rc = copy_out_blocking(ctx, item_rank, io.item_rank, items, ctx->stream)) return rc;
    return DARK_BWT_OK;
}

int dark_bwt_dc_encode(dark_bwt_ctx* ctx, const uint8_t* bwt, uint64_t n, uint32_t* dist_out, uint32_t* item_pos, uint32_t* item_dist,
                       uint8_t* item_sym, uint8_t* item_rank, dark_bwt_dc_info* info) {
    if (!ctx || !bwt || !info) return DARK_BWT_E_INVALID_ARG;
    if (ctx->flags & DARK_BWT_F_DEVICE_ONLY) return DARK_BWT_E_INVALID_ARG;
    if (n < 1 || n > ctx->capacity || n > 0xFFFFFFFEull) return DARK_BWT_E_INVALID_N;
    ctx->err[0] = 0;
    CK(cudaSetDevice(ctx->device));
    return dc_host(ctx, bwt, n, dist_out, item_pos, item_dist, item_sym, item_rank, info);
}

int dark_bwt_forward_dc(dark_bwt_ctx* ctx, const uint8_t* text, uint64_t n, uint8_t* bwt_out, uint64_t* origin_out, uint32_t* dist_out,
                        uint32_t* item_pos, uint32_t* item_dist, uint8_t* item_sym, uint8_t* item_rank, dark_bwt_dc_info* info,
                        dark_bwt_stats* stats) {
    if (!ctx || !text || !origin_out || !info) return DARK_BWT_E_INVALID_ARG;
    if (ctx->flags & DARK_BWT_F_DEVICE_ONLY) return DARK_BWT_E_INVALID_ARG;
    if (n < 2 || n > ctx->capacity || n > 0xFFFFFFFEull) return DARK_BWT_E_INVALID_N;
    ctx->err[0] = 0;
    CK(cudaSetDevice(ctx->device));
    if (int rc = copy_in_blocking(ctx, ctx->d_text, text, n, ctx->stream)) return rc;
    if (stats) stats->h2d_ms = 0.f;
    if (int rc = forward_device(ctx, ctx->d_text, n, ctx->d_bwt, origin_out, nullptr, stats)) return rc;
    if (bwt_out)
        if (int rc = copy_out_blocking(ctx, bwt_out, ctx->d_bwt, n, ctx->stream)) return rc;
    // the BWT is still in HBM: distance coding reads it there
    return dc_host(ctx, nullptr, n, dist_out, item_pos, item_dist, item_sym, item_rank, info);
}

int dark_bwt_reuse(dark_bwt_ctx* ctx, uint32_t** words_out, uint64_t* count_out) {
    if (!ctx || !words_out || !count_out) return DARK_BWT_E_INVALID_ARG;
    if (!ctx->reuse_words) {
        // same size as the reference arena: n + 0x100 + max(n/4, min(2^15+2^7, n/2))  (saca.rs:353-357)
        const u64 n = ctx->capacity;
        const u64 extra = 0x100 + std::max<u64>(n / 4, std::min<u64>((1ull << 15) + (1ull << 7), n / 2));
        ctx->reuse_words = (u32*)calloc((size_t)(n + extra), sizeof(u32));
        if (!ctx->reuse_words) return DARK_BWT_E_NOMEM;
        ctx->reuse_count = n + extra;
    }
    *words_out = ctx->reuse_words;
    *count_out = ctx->reuse_count;
    return DARK_BWT_OK;
}

int dark_bwt_sort_pairs_device(dark_bwt_ctx* ctx, uint64_t* d_keys, uint32_t* d_vals, uint64_t* d_keys_alt,
                               uint32_t* d_vals_alt, uint64_t count, int begin_bit, int end_bit, int* in_alt_out,
                               float* ms_out) {
    if (!ctx || !d_keys || !d_vals || !d_keys_alt || !d_vals_alt || !in_alt_out) return DARK_BWT_E_INVALID_ARG;
    if (begin_bit < 0 || end_bit > 64 || begin_bit >= end_bit) return DARK_BWT_E_INVALID_ARG;
    if (count == 0 || count > ctx->capacity) return DARK_BWT_E_INVALID_N;
    ctx->err[0] = 0;
    CK(cudaSetDevice(ctx->device));
    const u32 m = (u32)count;
    const int num_passes = (end_bit - begin_bit + kRadixBits - 1) / kRadixBits;
    ctx->next_counter = 0;
    ctx->n_events = 0;
    ctx->spans.clear();
    CK(cudaMemsetAsync(ctx->counters, 0, sizeof(u32) * kMaxCounters, ctx->stream));
    CK(cudaMemsetAsync(ctx->hist, 0, sizeof(u32) * kMaxPasses * kRadix, ctx->stream));
    cudaEvent_t a = ctx->events[kMaxEvents - 1], b = ctx->events[kMaxEvents - 2];
    CK(cudaEventRecord(a, ctx->stream));
    const u32 blocks = (u32)std::min<u64>(ceil_div(m, 256 * 8), 148 * 8);
    k_digit_hist<256><<<blocks, 256, 0, ctx->stream>>>(d_keys, m, begin_bit, num_passes, ctx->hist);
    LAUNCHED();
    u64* keys[2] = {d_keys, d_keys_alt};
    u32* vals[2] = {d_vals, d_vals_alt};
    int cur = 0;
    // note: a partial top digit needs no masking as long as the bits above end_bit are equal in
    // all keys or meant to take part; callers pass end_bit = 64 or keys with zero upper bits.
    if (int rc = run_sort(ctx, keys, vals, 0, m, begin_bit, num_passes, &cur, nullptr, 0)) return rc;
    CK(cudaEventRecord(b, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    if (ms_out) cudaEventElapsedTime(ms_out, a, b);
    *in_alt_out = cur;
    return DARK_BWT_OK;
}

int dark_bwt_verify_sa_device(dark_bwt_ctx* ctx, const uint8_t* d_text, uint64_t n64, const uint32_t* d_sa,
                              uint64_t* bad_out) {
    if (!ctx || !d_text || !d_sa || !bad_out) return DARK_BWT_E_INVALID_ARG;
    if (n64 < 1 || n64 > ctx->capacity) return DARK_BWT_E_INVALID_N;
    ctx->err[0] = 0;
    CK(cudaSetDevice(ctx->device));
    const u32 n = (u32)n64;
    CK(cudaMemsetAsync(&ctx->scalars->bad, 0, sizeof(unsigned long long), ctx->stream));
    CK(cudaMemsetAsync(ctx->isa, 0xFF, sizeof(u32) * (size_t)n, ctx->stream));
    const u32 blocks = (u32)ceil_div(n, 256);
    k_verify_scatter<256><<<blocks, 256, 0, ctx->stream>>>(d_sa, n, ctx->isa, &ctx->scalars->bad);
    LAUNCHED();
    k_verify_order<256><<<blocks, 256, 0, ctx->stream>>>(d_text, d_sa, n, ctx->isa, &ctx->scalars->bad);
    LAUNCHED();
    CK(cudaMemcpyAsync(&ctx->mail->bad, &ctx->scalars->bad, sizeof(unsigned long long), cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    *bad_out = ctx->mail->bad;
    return DARK_BWT_OK;
}

// Debug hook (not in the public header): per-tile clock64() stamps of subsequent radix passes are
// written to d_trace ([tiles][8] long long); nullptr switches tracing off.
int dark_bwt_debug_trace_rerank(dark_bwt_ctx* ctx, long long* d_trace) {
    if (!ctx) return DARK_BWT_E_INVALID_ARG;
#if defined(DARK_BWT_TUNING) || defined(DARK_TUNE_TRACE)
    ctx->rerank_trace = d_trace;
    return DARK_BWT_OK;
#else
    (void)d_trace;
    return DARK_BWT_E_INVALID_ARG;  // tracing exists in tuning builds only
#endif
}

int dark_bwt_debug_trace(dark_bwt_ctx* ctx, long long* d_trace) {
    if (!ctx) return DARK_BWT_E_INVALID_ARG;
#if defined(DARK_BWT_TUNING) || defined(DARK_TUNE_TRACE)
    ctx->pass_trace = d_trace;
    return DARK_BWT_OK;
#else
    (void)d_trace;
    return DARK_BWT_E_INVALID_ARG;  // tracing exists in tuning builds only
#endif
}

int dark_bwt_lcp_profile_device(dark_bwt_ctx* ctx, const uint8_t* d_text, uint64_t n64, const uint32_t* d_sa, uint64_t* m_out,
                                uint32_t* rounds_out, uint64_t* max_lcp_out) {
    if (!ctx || !d_text || !d_sa || !m_out || !rounds_out || !max_lcp_out) return DARK_BWT_E_INVALID_ARG;
    if (n64 < 2 || n64 > ctx->capacity) return DARK_BWT_E_INVALID_N;
    if (((uintptr_t)d_text) & 7) return DARK_BWT_E_INVALID_ARG;  // 64-bit text loads
    ctx->err[0] = 0;
    CK(cudaSetDevice(ctx->device));
    const u32 n = (u32)n64;
    u32* lcp = ctx->ranks;                                             // scratch: n u32
    unsigned long long* buckets = (unsigned long long*)ctx->keys[0];  // scratch: 64 counters
    u32* dmax = (u32*)(buckets + 64);
    CK(cudaMemsetAsync(buckets, 0, 65 * sizeof(unsigned long long), ctx->stream));
    k_lcp_direct<256><<<(u32)ceil_div(n, 256), 256, 0, ctx->stream>>>(d_text, n, d_sa, lcp);
    LAUNCHED();
    k_lcp_buckets<256><<<(u32)std::min<u64>(ceil_div(n, 256 * 8), (u64)ctx->num_sms * 8), 256, 0, ctx->stream>>>(lcp, n, buckets, dmax);
    LAUNCHED();
    unsigned long long host[65];
    CK(cudaMemcpyAsync(host, buckets, sizeof(host), cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    int top = 0;
    for (int k = 0; k < 64; ++k)
        if (host[k]) top = k + 1;
    unsigned long long run = 0;
    for (int k = 63; k >= 0; --k) {
        run += host[k];
        m_out[k] = k < top ? run : 0;
    }
    *rounds_out = (uint32_t)top;
    *max_lcp_out = (uint64_t)(host[64] & 0xFFFFFFFFull);
    return DARK_BWT_OK;
}

int dark_bwt_emit_device(dark_bwt_ctx* ctx, const uint8_t* d_text, uint64_t n, const uint32_t* d_sa, uint8_t* d_bwt_out,
                         uint64_t* origin_out) {
    if (!ctx || !d_text || !d_sa || !d_bwt_out || !origin_out) return DARK_BWT_E_INVALID_ARG;
    if (n < 1 || n > ctx->capacity || n > 0xFFFFFFFEull) return DARK_BWT_E_INVALID_N;
    ctx->err[0] = 0;
    CK(cudaSetDevice(ctx->device));
    if (int rc = emit(ctx, d_text, (u32)n, d_sa, d_bwt_out)) return rc;
    CK(cudaStreamSynchronize(ctx->stream));
    *origin_out = ctx->mail->origin;
    return DARK_BWT_OK;
}

}  // extern "C"
