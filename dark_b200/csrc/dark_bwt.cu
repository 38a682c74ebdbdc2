// dark_bwt.cu — context, round driver and C ABI (include/dark_bwt.h) of the B200-native forward BWT.
//
// Host-side control flow of one block (replaces saca::Constructor::compute + TransformIterator,
// /root/reference/src/saca.rs:368-378 and src/block/dc.rs:45-50):
//
//   scan_alphabet                   sigma, dense codes, K symbols per 64-bit key
//   round0_keys, round0_sort        initial keys / digit histograms -> radix sort (top digits only if high-entropy)
//   round0_rerank                   re-rank/compact (sparse or scan kernel)
//   while (unsettled suffixes remain):
//     doubling_round                keys (rank[i], rank[i+h]) -> radix sort -> re-rank/compact, or pairs_round;  h *= 2
//   emit                            BWT gather + origin (unless the re-ranks emitted the bytes inline)
//
// forward_device drives these phases.  What crosses them lives in one Fwd record; RankFill owns which ranks isa[]
// holds, PairsMode owns pairs mode, SortStatus owns which rows of the radix passes' status buffer may hold stale words.
//
// All device memory is carved from one arena allocated at create (Constructor::new allocates its
// arena up front too, saca.rs:351-360) by carve_arena; the forward calls allocate nothing.  The packed item stream
// (dc_pack) reuses what distance coding has finished with: the host entries' stream lives in keys[1]; the tile counts in
// ranks_alt, or for many blocks (whose item offsets are in ranks_alt) in ranks behind the per-block stream offsets of
// dark_bwt_forward_dc_packed_many and the tile offsets; the first-item bitmap of many blocks in `bitmap`.  Decoding a packed
// stream (dc_decode) parses into keys[0] and re-packs there for its check; the host entry's stream lives in keys[1].
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
#include <type_traits>
#include <vector>

#include "../../include/dark_bwt.h"
#include "common.cuh"
#include "radix_sort.cuh"
#include "onesweep_tma.cuh"
#include "suffix_kernels.cuh"
#include "dc_kernels.cuh"

using namespace dark;

namespace {

constexpr int kSortTile = 3072;  // sizes the status buffer: no radix pass has a smaller tile
constexpr int kScanThreads = 512;
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
    u32 bad_block;  // inverse: the lowest block whose list does not cover its rows (with `count` = how many do not)
    u32 bad_dist;   // inverse: the rows that block's list covers
    unsigned long long packed_bytes;  // distance coding: the size of the packed item stream
    UnpackTotals unpack;              // decoding a packed stream: the parse's totals (k_dc_unpack_chain)
    unsigned long long unpack_diff;   // ... the first byte at which the stream differs from the decoded block's, ~0 if none
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

// Test knobs, resolved ONCE at dark_bwt_create from the environment (never on the hot path).  They force code paths
// that the block size or content would otherwise choose; none of them changes a result, and each has a parity test
// (tests/test_gpu_parity.py).
struct Knobs {
    int pass_impl = 1;              // DARK_BWT_PASS_IMPL: 1 = onesweep_tma.cuh, 0 = the round-1 kernel k_onesweep_pass
    bool force_u64_status = false;  // DARK_BWT_FORCE_U64_STATUS=1
    bool check_hist = false;        // DARK_BWT_CHECK_HIST=1 counts both ways and compares
    bool inline_emit = true;        // DARK_BWT_INLINE_EMIT=0
    bool sparse_rerank = true;      // DARK_BWT_SPARSE_RERANK=0
    bool fuse_round0 = true;        // DARK_BWT_FUSE_ROUND0=0: round 0 of an unpruned large block without the fused bucket sink
    int text_div = 8;               // DARK_BWT_TEXT_BUILD=<k>: text-order key build while m > n/k (0 = never, no isa[] tag)
    bool pairs = true;              // DARK_BWT_PAIRS=0
    bool rank_search = true;        // DARK_BWT_RANK_SEARCH=0
    int bucketed = -1;              // DARK_BWT_BUCKETED=0/1 (-1: by block size)
    int host_chunk_mb = 2;          // DARK_BWT_HOST_CHUNK_MB: pinned bytes per staging lane (2 MiB chunks fill the pipeline sooner than 8: 23.1 vs 23.8 ms per C2 call)
    int host_threads = 12;          // DARK_BWT_HOST_THREADS=<t>: staging lanes per direction for pageable host buffers (0: let the driver stage)
    int emit_window_mb = 64;        // DARK_BWT_EMIT_WINDOW_MB: text window of the emission
    int ibwt_stride = 48;           // DARK_BWT_IBWT_STRIDE: splitter stride of the inverse BWT
    bool ibwt_two_walks = false;    // DARK_BWT_IBWT_TWO_WALKS=1

    void read_env() {
        auto geti = [](const char* name, int dflt) {
            const char* e = getenv(name);
            return e ? atoi(e) : dflt;
        };
        pass_impl = geti("DARK_BWT_PASS_IMPL", pass_impl);
        force_u64_status = geti("DARK_BWT_FORCE_U64_STATUS", 0) != 0;
        check_hist = geti("DARK_BWT_CHECK_HIST", 0) != 0;
        inline_emit = geti("DARK_BWT_INLINE_EMIT", 1) != 0;
        sparse_rerank = geti("DARK_BWT_SPARSE_RERANK", 1) != 0;
        fuse_round0 = geti("DARK_BWT_FUSE_ROUND0", 1) != 0;
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
        emit_window_mb = std::max(1, geti("DARK_BWT_EMIT_WINDOW_MB", 64));
        ibwt_stride = std::max(2, geti("DARK_BWT_IBWT_STRIDE", 48));
        ibwt_two_walks = geti("DARK_BWT_IBWT_TWO_WALKS", 0) != 0;
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

// Where distance coding writes.  Every device pointer is nullable: the context's own arena is used for what the caller does
// not want, and dc_device sets the pointer to where the data is.
struct DcBuffers {
    u32* dist = nullptr;         // n
    u32* item_pos = nullptr;     // num_items
    u32* item_dist = nullptr;
    u8* item_sym = nullptr;
    u8* item_rank = nullptr;
    u32* item_starts = nullptr;  // many blocks: count + 1
};

// The tile status words of the radix passes (decoupled look-back), carved from the arena: every row a pass reads must
// be zero when it starts.  Sorts of at most 2^31 pairs on the TMA pass use the buffer as two halves in turn: the workers
// of a pass zero the rows of the OTHER half (onesweep_tma.cuh), so only what they did not cover is cleared by a memset.
// The round-1 kernel, a TMA pass with 64-bit words and distance coding use the buffer from its start instead.
class SortStatus {
   public:
    void init(void* base, size_t bytes) {
        base_ = base;
        bytes_ = bytes;
        all_stale();
    }
    // The round-1 kernel or a TMA pass with 64-bit words: the first `bytes` of the buffer, zeroed.
    int take_whole(dark_bwt_ctx* ctx, size_t bytes, void** use);
    // A TMA pass with 32-bit words over `tiles` tiles that reads `rows` rows: *use is its half, zero in those rows; *clean
    // the other half, whose rows [0, tiles) the pass' workers zero for the next such pass.
    int take_half(dark_bwt_ctx* ctx, u32 tiles, u32 rows, void** use, void** clean);
    // The whole buffer as scratch (the last-occurrence tables of distance coding on tiny blocks).
    void* borrow() {
        all_stale();
        return base_;
    }

   private:
    u32 half_rows() const { return (u32)(bytes_ / 2 / (kRadix * sizeof(u32))); }
    void all_stale() {
        for (int h = 0; h < 2; ++h) lo_[h] = 0u, hi_[h] = half_rows();
    }

    void* base_ = nullptr;
    size_t bytes_ = 0;
    int cur_ = 0;                              // the half the next TMA pass with 32-bit words uses
    u32 lo_[2] = {0u, 0u}, hi_[2] = {0u, 0u};  // rows [lo_[h], hi_[h]) of half h may hold stale words
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
    u8* d_text2 = nullptr;  // second pair for the pipelined batch entries (== d_text, d_bwt on a one-pair context)
    u8* d_bwt2 = nullptr;
    int pipeline_depth = 0;  // staging pairs: 2, or 1 above 2^31 (the batch entries then run their blocks serially)
    DcBuffers dc_slot[2];  // DARK_BWT_F_DC_BATCH: block k of a pipelined DC batch is coded into slot k & 1 (N entries each)
    cudaStream_t copy_in = nullptr, copy_out = nullptr;
    cudaEvent_t ev_in[2] = {nullptr, nullptr}, ev_comp[2] = {nullptr, nullptr}, ev_out[2] = {nullptr, nullptr};
    u32* hist = nullptr;
    u32* present = nullptr;
    u8* lut = nullptr;
    unsigned long long* bad = nullptr;  // dark_bwt_verify_sa_device: violation counter (device atomics)
    SortStatus status;
    u32* counters = nullptr;
    u64* scan_words = nullptr;
    u32* bucket_hist = nullptr;  // 256 counters / cursors of the bucketed rank scatter
    u32* many_starts = nullptr;            // dark_bwt_forward_many: block offsets (kMaxManyBlocks + 1)
    unsigned long long* many_origins = nullptr;  // ... per-block origins
    u16* many_lut = nullptr;               // ... byte -> code 1..sigma
    DcInfoDev* dc_info = nullptr;             // dark_bwt_dc_*: device copy of the result header, followed by the run counter
    u32* bitmap = nullptr;  // n bits: positions whose rank the next round reads; survivor flags of the sparse round-0 re-rank
    size_t scan_tiles = 0;

    Mailbox* mail = nullptr;      // pinned + mapped host memory: kernels write their scalar results straight into it
    Mailbox* mail_dev = nullptr;  // the device alias of `mail`
    u32* reuse_words = nullptr;
    u64 reuse_count = 0;

    cudaEvent_t events[kMaxEvents];
    cudaEvent_t call_start = nullptr, call_stop = nullptr;  // the last two events: time a whole call (span_begin leaves them free)
    int n_events = 0;
    struct Span {
        int phase, e0, e1;
    };
    std::vector<Span> spans;
    int next_counter = 0;
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

int SortStatus::take_whole(dark_bwt_ctx* ctx, size_t bytes, void** use) {
    if (bytes > bytes_) return ctx->fail_internal("sort status buffer too small");
    CK(cudaMemsetAsync(base_, 0, bytes, ctx->stream));
    all_stale();
    *use = base_;
    return 0;
}

int SortStatus::take_half(dark_bwt_ctx* ctx, u32 tiles, u32 rows, void** use, void** clean) {
    if (rows > half_rows()) return ctx->fail_internal("sort status buffer too small");
    const int h = cur_, o = h ^ 1;
    u32* base_h = (u32*)base_ + (size_t)h * half_rows() * kRadix;
    if (hi_[h] > lo_[h])  // what the previous pass' workers did not zero (usually nothing)
        CK(cudaMemsetAsync(base_h + (size_t)lo_[h] * kRadix, 0, (size_t)(hi_[h] - lo_[h]) * kRadix * sizeof(u32), ctx->stream));
    lo_[h] = 0u;  // this pass writes rows [0, tiles) of its half ...
    hi_[h] = tiles;
    if (hi_[o] <= tiles) lo_[o] = hi_[o] = 0u;  // ... and zeroes rows [0, tiles) of the other
    else lo_[o] = std::max(lo_[o], tiles);
    cur_ = o;
    *use = base_h;
    *clean = (u32*)base_ + (size_t)o * half_rows() * kRadix;
    return 0;
}

namespace {

// every host round trip of a forward call goes through here (dark_bwt_stats.host_syncs)
inline cudaError_t sync_counted(dark_bwt_ctx* ctx) {
    ctx->syncs += 1;
    return cudaStreamSynchronize(ctx->stream);
}

// The start of a call that sorts or inverts: the context's device, fresh per-call bookkeeping (events and spans, tile
// counters, launch and sync counts), the call's clock (call_start) and zeroed tile counters.
int begin_call(dark_bwt_ctx* ctx) {
    CK(cudaSetDevice(ctx->device));
    ctx->n_events = 0;
    ctx->spans.clear();
    ctx->next_counter = 0;
    ctx->launches = 0;
    ctx->syncs = 0;
    CK(cudaEventRecord(ctx->call_start, ctx->stream));
    CK(cudaMemsetAsync(ctx->counters, 0, sizeof(u32) * kMaxCounters, ctx->stream));
    return 0;
}

// Device time from call_start to call_stop; both have completed.
float call_ms(const dark_bwt_ctx* ctx) {
    float ms = 0.f;
    cudaEventElapsedTime(&ms, ctx->call_start, ctx->call_stop);
    return ms;
}

// The stats of a forward call start from zero, but for the host entry's h2d_ms, measured before the transform.
void reset_stats(dark_bwt_stats* st, u32 n) {
    if (!st) return;
    const float h2d = st->h2d_ms;
    memset(st, 0, sizeof(*st));
    st->h2d_ms = h2d;
    st->n = n;
    st->active[0] = n;
}

int span_begin(dark_bwt_ctx* ctx, int phase) {
    if (ctx->n_events + 2 > kMaxEvents - 4) return -1;  // the last events are reserved (call_start, call_stop)
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

int next_counter(dark_bwt_ctx* ctx, u32** out) {
    if (ctx->next_counter >= kMaxCounters) return ctx->fail_internal("tile counters exhausted");
    *out = ctx->counters + ctx->next_counter++;
    return 0;
}

// Tilings of the radix passes: threads, items per thread, CTAs per SM, ranking items in flight per warp.  The pipelined
// pass (onesweep_tma.cuh), and the round-1 kernel k_onesweep_pass (radix_sort.cuh), best of the tiling sweeps in
// profiles/r1_sort_variants_*.log.
constexpr int kPassThreads = 256, kPassItems = 16, kPassCtas = 2, kPassIlp = 2;
constexpr int kRound1Threads = 256, kRound1Items = 16, kRound1Ctas = 3, kRound1Ilp = 2;

// f(BoolC<b>()): a runtime choice as a template argument of the kernel f launches.  A function template, not a lambda:
// the pass kernels are then instantiated after the kernels launched directly, and that order of the module's extern
// shared arrays decides the offset of k_build_keys_text's dynamic shared memory.
template <typename F>
int with_bool(bool b, const F& f) {
    return b ? f(BoolC<true>()) : f(BoolC<false>());
}

// The TMA-staged, software-pipelined pass: byte-aligned digits, 16-byte aligned inputs, plain or key-generating (GEN mode 0).
int launch_pass_tma(dark_bwt_ctx* ctx, const u64* kin, const u32* vin, u64* kout, u32* vout, u32 m, int shift, const u32* digit_base,
                    u32* counter, bool wide, const u8* prev_text, const KeyGen* gen) {
    typedef PipeSmem<kPassThreads, kPassItems> Smem;
    const u32 tiles = (u32)ceil_div(m, Smem::kTile);
    const u32 rows = tiles + 3 * kScannerBatch;  // the scanners read ahead
    void *status = nullptr, *status_clean = nullptr;
    if (int rc = wide ? ctx->status.take_whole(ctx, (size_t)rows * kRadix * sizeof(u64), &status)
                      : ctx->status.take_half(ctx, tiles, rows, &status, &status_clean))
        return rc;
    const u32 grid = std::min<u32>(tiles + kScanners, (u32)ctx->num_sms * kPassCtas);  // kScanners CTAs scan, the rest sort
    const KeyGen g = gen ? *gen : KeyGen();
    auto run = [&](auto wide_c, auto gen_c, auto hi_c) {
        typedef std::conditional_t<decltype(wide_c)::value, u64, u32> StatusT;
        auto kern = k_onesweep_tma<kPassThreads, kPassItems, kPassCtas, kPassIlp, StatusT, decltype(gen_c)::value, decltype(hi_c)::value>;
        CK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(Smem)));
        kern<<<grid, kPassThreads, sizeof(Smem), ctx->stream>>>(kin, vin, kout, vout, m, shift, digit_base, (StatusT*)status,
                                                                 (StatusT*)status_clean, counter, g, prev_text);
        LAUNCHED();
        return 0;
    };
    return with_bool(gen != nullptr, [&](auto gen_c) {
        return with_bool(wide, [&](auto wide_c) {
            return with_bool(shift >= 32, [&](auto hi_c) { return run(wide_c, gen_c, hi_c); });
        });
    });
}

// The round-1 kernel: any digit, any 8-byte aligned input, plain or key-generating (GEN modes 0 and 1).
int launch_pass_round1(dark_bwt_ctx* ctx, const u64* kin, const u32* vin, u64* kout, u32* vout, u32 m, int shift,
                       const u32* digit_base, u32* counter, bool wide, const u8* prev_text, u32 n_text, const KeyGen* gen) {
    typedef OnesweepSmem<kRound1Threads, kRound1Items> Smem;
    const u32 tiles = (u32)ceil_div(m, Smem::kTile);
    void* status = nullptr;
    if (int rc = ctx->status.take_whole(ctx, (size_t)tiles * kRadix * (wide ? sizeof(u64) : sizeof(u32)), &status)) return rc;
    const bool aligned = (shift & 7) == 0;  // always true for the suffix sorter; the public sort may differ
    if (gen && !aligned) return ctx->fail_internal("key-generating pass needs a byte-aligned digit");
    // persistent grid: as many CTAs as stay resident (SMs x CTAs per SM), each claiming tiles until none are left
    const u32 grid = std::min<u32>(tiles, (u32)ctx->num_sms * kRound1Ctas);
    // L2 prefetch distance in tiles: two thirds of a wave of claims (the persistent grid; 148..444 measured alike, beyond
    // one wave the gain fades)
    const u32 prefetch_ahead = std::max(1u, grid * 2 / 3);
    const KeyGen g = gen ? *gen : KeyGen();
    auto run = [&](auto wide_c, auto aligned_c, auto gen_c) {
        typedef std::conditional_t<decltype(wide_c)::value, u64, u32> StatusT;
        auto kern = k_onesweep_pass<kRound1Threads, kRound1Items, kRound1Ctas, kRound1Ilp, StatusT, decltype(aligned_c)::value,
                                    decltype(gen_c)::value>;
        CK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(Smem)));  // per device
        kern<<<grid, kRound1Threads, sizeof(Smem), ctx->stream>>>(kin, vin, kout, vout, m, shift, digit_base, (StatusT*)status, counter,
                                                                   prev_text, n_text, g, prefetch_ahead);
        LAUNCHED();
        return 0;
    };
    if (gen) return with_bool(wide, [&](auto wide_c) { return run(wide_c, BoolC<true>(), BoolC<true>()); });  // keys built from the text inside the pass
    return with_bool(aligned, [&](auto aligned_c) {
        return with_bool(wide, [&](auto wide_c) { return run(wide_c, aligned_c, BoolC<false>()); });
    });
}

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
    // default: the TMA-staged pipelined pass; DARK_BWT_PASS_IMPL=0 keeps the round-1 kernel (k_onesweep_pass)
    const bool eligible = (shift & 7) == 0 && (gen == nullptr || gen->mode == 0) &&
                          (gen != nullptr || (prev_text == nullptr && ((uintptr_t)kin & 15) == 0 && ((uintptr_t)vin & 15) == 0));
    if (ctx->knobs.pass_impl != 0 && eligible)
        return launch_pass_tma(ctx, kin, vin, kout, vout, m, shift, digit_base, counter, wide_tma, prev_text, gen);
    return launch_pass_round1(ctx, kin, vin, kout, vout, m, shift, digit_base, counter, wide, prev_text, n_text, gen);
}

// The digit statistics of the histograms in ctx->hist: mail->trivial[p] (every key has the same digit p) and
// mail->collide[p] (the probability that two keys share it).  `wait`: the host reads them (one round trip).
int scan_digits(dark_bwt_ctx* ctx, u32 m, int num_passes, bool wait) {
    // Scalar results (flags, counts, origin) are written by the kernels directly into mapped pinned host
    // memory and read after a stream sync.  A cudaMemcpy D2H would queue on the copy engine behind the
    // 256 MB block transfers of the pipelined batch entry (measured: +5 ms per block).
    k_scan_hist<<<num_passes, kRadix, 0, ctx->stream>>>(ctx->hist, m, ctx->mail_dev->trivial, ctx->mail_dev->collide);
    LAUNCHED();
    if (wait) CK(sync_counted(ctx));
    return 0;
}

// Radix passes first..num_passes-1 over the (keys, vals) pair *cur, for digits scanned by scan_digits; *cur follows the
// data.  A trivial digit's pass is the identity and is skipped, unless `all_passes` (the flags were not waited for).
// The first pass that runs builds its input from `gen` (if given) and drops the BWT byte from `patch_text` (if given)
// into the low key byte.
int sort_passes(dark_bwt_ctx* ctx, u64* const keys[2], u32* const vals[2], int* cur, u32 m, int begin_bit, int first, int num_passes,
                dark_bwt_stats* st, int round, bool all_passes, const u8* patch_text, const KeyGen* gen) {
    int sp = span_begin(ctx, gen ? PH_GENPASS : PH_PASS);
    for (int p = first; p < num_passes; ++p) {
        if (!all_passes && ctx->mail->trivial[p]) continue;  // every key has the same digit: the pass is the identity
        if (int rc = launch_pass(ctx, keys[*cur], vals[*cur], keys[*cur ^ 1], vals[*cur ^ 1], m, begin_bit + p * kRadixBits,
                                 ctx->hist + p * kRadix, patch_text, m, gen))
            return rc;
        if (gen) {  // only the first pass that runs builds its input; the later ones read what it wrote
            gen = nullptr;
            if (st) {
                st->gen_passes += 1;
                st->gen_elements += m;
            }
            span_end(ctx, sp);  // the key-generating launch is timed on its own (13 B per suffix, not 24)
            sp = span_begin(ctx, PH_PASS);
        }
        patch_text = nullptr;
        *cur ^= 1;
        if (st) {
            st->sort_passes += 1;
            st->sorted_elements += m;
            if (round < DARK_BWT_MAX_ROUNDS) st->passes[round] += 1;
        }
    }
    span_end(ctx, sp);
    return 0;
}

// Sort passes for a histogram that is already in ctx->hist (counts).  `cur` is the index of the
// (keys, ids) pair holding the input; returns the index holding the output through *cur_out.
// all_passes (a round that still holds more than n/8 suffixes): their ranks span at least m slots, so at most the top digit
// could be constant; every pass runs and the host does not wait for the flags (one round trip less per round).
int run_sort(dark_bwt_ctx* ctx, u64* const keys[2], u32* const vals[2], int cur, u32 m, int begin_bit, int num_passes,
             int* cur_out, dark_bwt_stats* st, int round, const KeyGen* gen = nullptr, bool all_passes = false) {
    if (int rc = scan_digits(ctx, m, num_passes, !all_passes)) return rc;
    *cur_out = cur;
    return sort_passes(ctx, keys, vals, cur_out, m, begin_bit, 0, num_passes, st, round, all_passes, nullptr, gen);
}

struct PairSink {  // where a PAIRS re-rank puts its (id, rank) updates
    u32* ids = nullptr;
    u32* vals = nullptr;
    int shift = 0;
};

// `tag`: the bit isa[] entries of active suffixes carry (0: none).  *count_dev (if asked): the device copy of the
// survivor count, beside the tile counter.
template <bool ROUND0, bool PAIRS>
int launch_rerank(dark_bwt_ctx* ctx, const u64* keys, const u32* ids, u32 m, u32 n, int K, int kb, u32* sa, u32* out_ids,
                  const u8* text, u8* bwt_inline, u32 tag, const u32** count_dev, PairSink sink = PairSink()) {
    const u32 tiles = (u32)ceil_div(m, kScanTile);
    if (tiles > ctx->scan_tiles) return ctx->fail_internal("scan tile state too small");
    ScanTileState ts{ctx->scan_words};
    constexpr size_t smem = kRerankSmem<kScanTile>;
    u32 *counter = nullptr, *count_copy = nullptr;  // two consecutive words: the tile counter, then the survivor count (device copy)
    if (int rc = next_counter(ctx, &counter)) return rc;
    if (int rc = next_counter(ctx, &count_copy)) return rc;
    if (count_dev) *count_dev = count_copy;
    CK(cudaMemsetAsync(ctx->scan_words, 0, sizeof(u64) * kScanWordsPerTile * tiles, ctx->stream));
    const u32 prefetch_ahead = 2u * (u32)ctx->num_sms;  // one wave of CTAs ahead (-2 %)
    auto kern = k_rerank<kScanThreads, kScanItems, ROUND0, PAIRS>;
    if (smem > 48 * 1024) CK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    kern<<<tiles, kScanThreads, smem, ctx->stream>>>(
        keys, ids, ROUND0 ? nullptr : ctx->ranks, m, n, K, kb, ctx->isa, sa, out_ids, ROUND0 ? ctx->ranks : ctx->ranks_alt, ts, counter,
        &ctx->mail_dev->count, sink.ids, sink.vals,
        ctx->bucket_hist, sink.shift, text, bwt_inline, &ctx->mail_dev->origin, prefetch_ahead, (ROUND0 && !PAIRS) ? 0u : tag);
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

void finish_stats(dark_bwt_ctx* ctx, dark_bwt_stats* st) {
    if (!st) return;
    st->device_ms = call_ms(ctx);
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

// ---- the forward transform of one block: a driver (forward_device) and one function per phase
// State of one forward_device call that crosses its phases.
struct Fwd {
    const u8* text;
    u32 n;
    u8* bwt;
    u32* sa;
    dark_bwt_stats st = {};  // the call's stats, copied to the caller's record at the end
    int s_bits = 8, K = 8;  // alphabet: bits per symbol code, symbols per 64-bit key
    int cur = 0;            // the (keys, ids) pair holding the active list
    u32 m = 0;              // active suffixes
    u64 h = 0;              // leading symbols known equal inside each group
    int round = 0;
    int kb = 0, passes_r = 0;      // bits of a rank + 1, radix passes of a doubling round
    // The initial sort covered the key bits above `drop`: K0 whole leading symbols are known equal inside a
    // tie group, Kc symbols were touched (a suffix shorter than Kc had padding compared).
    int K0 = 0, Kc = 0, drop = 0;
    bool emit_inline = false;  // the re-ranks emit each suffix's BWT byte as it settles (no gather pass at the end)
    u32 tag = 0;               // bit carried by isa[] entries of active suffixes (0: not used)
    bool bucketed = false;     // rank scatters of more than n/16 ranks go through bucket regions of 2^bshift suffixes
    int bshift = 0;
    PairSink regions = {};     // the regions the fused round-0 re-rank filled with every suffix's rank (ids null: not fused)
};

// Alphabet scan: sigma, dense codes (ctx->lut), bits per symbol and symbols per key.
int scan_alphabet(dark_bwt_ctx* ctx, Fwd& f) {
    CK(cudaMemsetAsync(ctx->present, 0, sizeof(u32) * 256, ctx->stream));
    CK(cudaMemsetAsync(ctx->hist, 0, sizeof(u32) * kMaxPasses * kRadix, ctx->stream));
    const int no_pack = (ctx->flags & DARK_BWT_F_NO_ALPHABET_PACKING) ? 1 : 0;
    const u32 blocks = (u32)std::min<u64>(ceil_div(ceil_div(f.n, 16), 256), 148 * 8);
    k_symbol_presence<256><<<std::max(blocks, 1u), 256, 0, ctx->stream>>>(f.text, f.n, ctx->present);
    LAUNCHED();
    k_build_lut<<<1, 256, 0, ctx->stream>>>(ctx->present, ctx->lut, &ctx->mail_dev->sigma, no_pack);
    LAUNCHED();
    CK(sync_counted(ctx));
    const u32 sigma = ctx->mail->sigma;
    if (sigma < 1 || sigma > 256) return ctx->fail_internal("alphabet scan returned an impossible sigma");
    f.s_bits = no_pack ? 8 : std::max(1, bit_length(sigma - 1));
    f.K = 64 / f.s_bits;
    f.st.sigma = sigma;
    f.st.bits_per_symbol = f.s_bits;
    f.st.symbols_per_key = f.K;
    return 0;
}

// Widths whose keys the packed kernels build: s in {1, 2, 4, 8}
bool packed_width(int s_bits) { return s_bits == 1 || s_bits == 2 || s_bits == 4 || s_bits == 8; }
int lg_width(int s_bits) { return s_bits == 1 ? 0 : s_bits == 2 ? 1 : s_bits == 4 ? 2 : 3; }

// Round-0 keys of K symbols, ids descending, with their digit histograms (packed widths: the keys (write) or the
// digit histograms counted key by key (!write); other widths: both).  The symbol field is MSB-aligned in the 64-bit key.
int init_keys(dark_bwt_ctx* ctx, const Fwd& f, bool write) {
    const u32 blocks = (u32)std::min<u64>(ceil_div(f.n, kInitThreads * kInitItems), (u64)ctx->num_sms * 8);
#define INIT_PACKED(S)                                                                                                              \
    do {                                                                                                                            \
        if (write)                                                                                                                  \
            k_init_keys_packed<kInitThreads, kInitItems, S, true><<<blocks, kInitThreads, 0, ctx->stream>>>(                        \
                f.text, f.n, ctx->lut, ctx->keys[0], ctx->ids[0], ctx->hist);                                                       \
        else                                                                                                                        \
            k_init_keys_packed<kInitThreads, kInitItems, S, false><<<blocks, kInitThreads, 0, ctx->stream>>>(                       \
                f.text, f.n, ctx->lut, nullptr, nullptr, ctx->hist);                                                                \
    } while (0)
    switch (f.s_bits) {
        case 1: INIT_PACKED(1); break;
        case 2: INIT_PACKED(2); break;
        case 4: INIT_PACKED(4); break;
        case 8: INIT_PACKED(8); break;
        default:
            k_init_keys<kInitThreads, kInitItems><<<blocks, kInitThreads, 0, ctx->stream>>>(
                f.text, f.n, ctx->lut, f.s_bits, f.K, ctx->keys[0], ctx->ids[0], ctx->hist, kMaxPasses);
    }
#undef INIT_PACKED
    LAUNCHED();
    return 0;
}

// Round 0, the digit histograms (and, for widths without a fused key build, the keys).  Packed widths: the histograms
// come from the text's q-grams (suffix_kernels.cuh) and the first radix pass that runs builds the keys from the text
// (radix_sort.cuh, GEN).
int round0_keys(dark_bwt_ctx* ctx, const Fwd& f) {
    if (!packed_width(f.s_bits)) return init_keys(ctx, f, true);
    u32* gram = ctx->bucket_hist;  // 256 counters, free until the first rank scatter
    CK(cudaMemsetAsync(gram, 0, sizeof(u32) * kRadix, ctx->stream));
    const u32 blocks = (u32)std::min<u64>(ceil_div(f.n, 256 * 16), (u64)ctx->num_sms * 8);
    switch (f.s_bits) {
        case 1: k_gram_hist<256, 1><<<blocks, 256, 0, ctx->stream>>>(f.text, f.n, ctx->lut, gram); break;
        case 2: k_gram_hist<256, 2><<<blocks, 256, 0, ctx->stream>>>(f.text, f.n, ctx->lut, gram); break;
        case 4: k_gram_hist<256, 4><<<blocks, 256, 0, ctx->stream>>>(f.text, f.n, ctx->lut, gram); break;
        default: k_gram_hist<256, 8><<<blocks, 256, 0, ctx->stream>>>(f.text, f.n, ctx->lut, gram); break;
    }
    LAUNCHED();
    k_gram_expand<<<1, kRadix, 0, ctx->stream>>>(f.text, f.n, ctx->lut, lg_width(f.s_bits), gram, ctx->hist);
    LAUNCHED();
    if (ctx->knobs.check_hist) {  // test hook: compare with the histogram counted key by key
        std::vector<u32> a(kMaxPasses * kRadix), b(kMaxPasses * kRadix);
        CK(cudaMemcpyAsync(a.data(), ctx->hist, a.size() * 4, cudaMemcpyDeviceToHost, ctx->stream));
        CK(cudaMemsetAsync(ctx->hist, 0, sizeof(u32) * kMaxPasses * kRadix, ctx->stream));
        if (int rc = init_keys(ctx, f, false)) return rc;
        CK(cudaMemcpyAsync(b.data(), ctx->hist, b.size() * 4, cudaMemcpyDeviceToHost, ctx->stream));
        CK(sync_counted(ctx));
        if (a != b) return ctx->fail_internal("q-gram histogram differs from the per-key histogram");
        CK(cudaMemcpyAsync(ctx->hist, a.data(), a.size() * 4, cudaMemcpyHostToDevice, ctx->stream));
        CK(sync_counted(ctx));
    }
    return 0;
}

// Pass pruning of the initial sort: an LSD sort of the top t digits alone orders the keys by their leading 8t bits;
// whatever stays tied is finished by the doubling rounds.  With S_p the probability that two keys share digit p (from
// the histogram), about m * prod(S_p) of the keys keep a partner after the top t digits, IF the digits are independent.
// That holds for high-entropy blocks (packed DNA, random bytes) and fails badly for text, where a shallower initial
// sort also slows every later round (h starts smaller).  So the low digits are dropped only when every digit is close
// to uniform (S_p <= 1.5/256) and the estimate leaves < 1/64 of the block tied; measured: C2 8 -> 5 passes + one
// 65,792-element round; C1/C5 unchanged.  Returns the lowest digit to sort.
int round0_first_digit(const Mailbox* mail, u32 m) {
    for (int p = 0; p < kMaxPasses; ++p)
        if (mail->collide[p] > 1.5f / 256.0f) return 0;  // not a high-entropy block
    double tied = (double)m;  // m * P(two keys agree on the top t digits) ~ fraction of keys left with a partner
    int t = 0;
    for (int p = kMaxPasses - 1; p >= 0; --p) {
        tied *= (double)mail->collide[p];
        ++t;
        if (tied * 64.0 <= 1.0) break;
    }
    return std::max(0, kMaxPasses - t);
}

// Round 0, the sort: every digit, or the top ones of a pruned block (round0_first_digit; not without alphabet packing).
int round0_sort(dark_bwt_ctx* ctx, Fwd& f) {
    int sp = span_begin(ctx, PH_SORT);
    if (int rc = scan_digits(ctx, f.n, kMaxPasses, true)) return rc;
    const int first = (ctx->flags & DARK_BWT_F_NO_ALPHABET_PACKING) ? 0 : round0_first_digit(ctx->mail, f.n);
    // Inline emission: when the initial sort is pruned by >= 1 digit the BWT byte of each suffix travels in
    // the (unsorted) low key byte and is emitted as the suffix settles; no gather pass at the end.
    // An unpruned block emits in a final gather pass.  Emitting it inline instead, the re-rank gathering T[id-1] for every
    // suffix as it settles, measured equal (C4: re-rank +38 ms, emission -37 ms: one random DRAM sector per suffix wherever
    // the read is issued, profiles/r2_rejected.md).
    const bool patch = first >= 1 && ctx->knobs.inline_emit;
    const bool packed = packed_width(f.s_bits);
    const KeyGen gen{f.text, ctx->lut, f.n, lg_width(f.s_bits), 0, 0};
    if (int rc = sort_passes(ctx, ctx->keys, ctx->ids, &f.cur, f.n, 0, first, kMaxPasses, &f.st, 0, false, patch ? f.text : nullptr,
                             packed ? &gen : nullptr))
        return rc;
    const bool sorted = f.st.passes[0] > 0;  // some digit was not trivial
    f.emit_inline = patch && sorted;
    if (packed && !sorted) {  // every digit was trivial (one-symbol text): no pass ran, the re-rank still wants the keys
        if (int rc = init_keys(ctx, f, true)) return rc;
        f.cur = 0;
    }
    span_end(ctx, sp);
    f.drop = first * kRadixBits;
    const int sorted_bits = 64 - f.drop;
    f.K0 = std::min(f.K, sorted_bits / f.s_bits);
    f.Kc = std::min(f.K, (sorted_bits + f.s_bits - 1) / f.s_bits);
    if (f.K0 < 1) return ctx->fail_internal("initial sort covered less than one symbol");
    f.st.initial_symbols = f.K0;
    f.kb = bit_length(f.n);  // rank2 = isa+1 in [0, n]
    const int key_bits = f.kb + bit_length(((u64)f.n - 1) >> 1);  // high part = rank >> 1 (suffix_kernels.cuh, k_rerank)
    f.passes_r = (key_bits + kRadixBits - 1) / kRadixBits;
    return 0;
}

// Pairs mode: once every remaining group is a pair the rounds switch to the pairs kernel for good (groups only ever
// split).  The check reads the rank list once; queued behind a re-rank (k_pairs_detect reads the survivor count from the
// device copy the re-rank leaves), its answer (mail->not_pairs) arrives with that count in the round trip the round makes
// anyway.  Otherwise it costs a round trip of its own, so it is skipped while most of the block is still active
// (period-17: ten rounds of giant groups).  The kernel gathers from isa[], so it waits until every rank is there (few
// survivors after round 0: the selective rounds).  DARK_BWT_PAIRS=0 switches it off.
struct PairsMode {
    bool enabled = true;
    bool on = false;
    bool checked = false;  // the check of the current list was queued behind its re-rank: the answer is in the mailbox

    // After the re-rank of round f.round has been launched, with `upper` >= its survivor count.
    int queue(dark_bwt_ctx* ctx, const Fwd& f, bool isa_complete, const u32* count_dev, u32 upper) {
        if (!enabled || (f.round > 0 && !(isa_complete && upper <= f.n / 2))) return 0;
        u32* seen = nullptr;
        if (int rc = next_counter(ctx, &seen)) return rc;
        ctx->mail->not_pairs = 0;
        const u32 grid = (u32)std::min<u64>(std::max<u64>(ceil_div(upper, 256), 1), (u64)ctx->num_sms * 4);
        k_pairs_detect<<<grid, 256, 0, ctx->stream>>>(ctx->ranks, 0u, count_dev, seen, &ctx->mail_dev->not_pairs);
        LAUNCHED();
        checked = true;
        return 0;
    }

    // At the top of a round, with its f.m active suffixes: switches pairs mode on if every group is a pair.
    int decide(dark_bwt_ctx* ctx, const Fwd& f, bool isa_complete) {
        if (enabled && !on && isa_complete && (f.m & 1u) == 0 && (f.round == 1 || f.m <= f.n / 2)) {
            if (checked) {  // answered in the round trip that fetched m
                on = ctx->mail->not_pairs == 0;
            } else {
                ctx->mail->flag = 0;
                u32* seen = nullptr;
                if (int rc = next_counter(ctx, &seen)) return rc;
                k_pairs_detect<<<(u32)std::min<u64>(ceil_div(f.m, 256), (u64)ctx->num_sms * 8), 256, 0, ctx->stream>>>(
                    ctx->ranks, f.m, nullptr, seen, &ctx->mail_dev->flag);
                LAUNCHED();
                CK(sync_counted(ctx));
                on = ctx->mail->flag == 0;
            }
        }
        checked = false;
        return 0;
    }
};

// Round 0, the re-rank: settles the suffixes whose group is a singleton, compacts the others into ids[cur ^ 1] and
// fetches their count.
int round0_rerank(dark_bwt_ctx* ctx, Fwd& f, PairsMode& pairs) {
    const Knobs& kn = ctx->knobs;
    u8* bwt_inline = f.emit_inline ? f.bwt : nullptr;
    int sp = span_begin(ctx, PH_RERANK);
    bool sparse_done = false;
    // Pruned initial sort with inline emission (high-entropy block: almost everything settles): the chain-free
    // sparse re-rank (suffix_kernels.cuh).  DARK_BWT_SPARSE_RERANK=0 keeps the scan-based kernel.
    if (f.emit_inline && kn.sparse_rerank) {
        u32 *total = nullptr, *ovf = nullptr;
        if (int rc = next_counter(ctx, &total)) return rc;
        if (int rc = next_counter(ctx, &ovf)) return rc;
        const u32 tiles = (u32)ceil_div(f.n, kScanTile);
        k_rerank0_sparse<kScanThreads, kScanItems><<<tiles, kScanThreads, 0, ctx->stream>>>(
            ctx->keys[f.cur], ctx->ids[f.cur], f.n, f.Kc, f.drop, f.sa, bwt_inline, &ctx->mail_dev->origin, (u8*)ctx->bitmap, total);
        LAUNCHED();
        k_copy_u32<<<1, 1, 0, ctx->stream>>>(total, &ctx->mail_dev->count);
        LAUNCHED();
        u32 survivors = 0;
        if (int rc = fetch_count(ctx, &survivors)) return rc;
        if (survivors == 0) {
            sparse_done = true;
        } else if (survivors <= f.n / 16) {
            const u64 nbytes = ceil_div(f.n, 8);
            const u32 nblocks = (u32)ceil_div(nbytes, kSparseChunk);
            u32* counts = (u32*)ctx->scan_words;  // n/32768 counters; the scan state is not in use
            u32* pos = ctx->ranks_alt;
            k_sparse_count<<<nblocks, 256, 0, ctx->stream>>>((const u8*)ctx->bitmap, nbytes, counts);
            LAUNCHED();
            k_sparse_scan<<<1, 1024, 0, ctx->stream>>>(counts, nblocks);
            LAUNCHED();
            k_sparse_positions<<<nblocks, 256, 0, ctx->stream>>>((const u8*)ctx->bitmap, nbytes, counts, pos);
            LAUNCHED();
            k_sparse_finalize<<<(u32)ceil_div(survivors, 256), 256, 0, ctx->stream>>>(pos, survivors, ctx->keys[f.cur], ctx->ids[f.cur], f.n,
                                                                                 f.Kc, f.drop, ctx->ids[f.cur ^ 1], ctx->ranks, ovf);
            LAUNCHED();
            k_copy_u32<<<1, 1, 0, ctx->stream>>>(ovf, &ctx->mail_dev->flag);
            LAUNCHED();
            CK(sync_counted(ctx));
            if (ctx->mail->flag == 0) {
                sparse_done = true;
                f.m = survivors;
            }
        }
    }
    // isa[] entries of active suffixes carry bit 31 (blocks up to 2^31 bytes): the text-order key builder finds
    // them by it.  DARK_BWT_TEXT_BUILD=0 switches tag and builder off; =<k> uses the builder while m > n/k.
    f.tag = (kn.text_div > 0 && (u64)f.n <= (1ull << 31)) ? 0x80000000u : 0u;
    // Scatters of more than n/16 ranks into an isa[] that outgrows L2 go through the bucketed path.
    f.bucketed = kn.bucketed >= 0 ? kn.bucketed != 0 : ((u64)f.n * 4 > (96ull << 20));
    f.bshift = std::max(0, bit_length((u64)f.n - 1) - 8);
    if (!sparse_done) {
        // A large block whose initial sort was not pruned is text-like: most suffixes survive round 0 and every rank is
        // needed.  Its round-0 re-rank then feeds the bucket regions of the rank scatter itself (every suffix reports its
        // rank, settled ones their slot) instead of two partition passes over the SA and the survivor list afterwards.
        // DARK_BWT_FUSE_ROUND0=0 keeps the separate passes.
        const u32* count_dev = nullptr;
        if (f.bucketed && f.drop == 0 && kn.fuse_round0) {
            u32* ids = (u32*)ctx->keys[f.cur ^ 1];
            f.regions = PairSink{ids, ids + align_up((size_t)f.n, 64), f.bshift};
            CK(cudaMemsetAsync(ctx->bucket_hist, 0, sizeof(u32) * 256, ctx->stream));
            if (int rc = launch_rerank<true, true>(ctx, ctx->keys[f.cur], ctx->ids[f.cur], f.n, f.n, f.Kc, f.drop, f.sa, ctx->ids[f.cur ^ 1],
                                                   f.text, bwt_inline, f.tag, &count_dev, f.regions))
                return rc;
        } else {
            if (int rc = launch_rerank<true, false>(ctx, ctx->keys[f.cur], ctx->ids[f.cur], f.n, f.n, f.Kc, f.drop, f.sa, ctx->ids[f.cur ^ 1],
                                                    f.text, bwt_inline, f.tag, &count_dev))
                return rc;
        }
        if (int rc = pairs.queue(ctx, f, true, count_dev, f.n)) return rc;
        if (int rc = fetch_count(ctx, &f.m)) return rc;
    }
    span_end(ctx, sp);
    f.cur ^= 1;  // the compacted active ids now live in ids[cur]
    return 0;
}

// Which ranks isa[] holds.  Round 0 writes none.  If a round follows they are needed: all of them when many suffixes
// survive; otherwise only the survivors' now, and per round the few that are actually read.
struct RankFill {
    bool complete = true;  // every rank a round may read is in isa[]
    int selective_rounds = 0;

    // After round 0 (f.round == 0, survivors left), or before the key build of round f.round; *keys_built: this fill
    // built the round's keys too.
    int fill(dark_bwt_ctx* ctx, const Fwd& f, bool* keys_built) {
        if (f.round == 0) {
            int sp = span_begin(ctx, PH_RERANK);
            if (f.regions.ids) {  // the regions hold every suffix's rank already
                if (int rc = region_scatter(ctx, f.regions.ids, f.regions.vals, f.n, f.bshift)) return rc;
            } else if (f.m > f.n / 16) {
                if (f.bucketed) {  // every suffix gets its rank: settled ones their slot, survivors their group rank
                    CK(cudaMemsetAsync(ctx->bucket_hist, 0, sizeof(u32) * 256, ctx->stream));
                    u32* oi = (u32*)ctx->keys[0];
                    u32* ov = (u32*)ctx->keys[1];
                    if (int rc = bucket_partition(ctx, f.sa, nullptr, f.n, f.bshift, oi, ov)) return rc;
                    if (int rc = bucket_partition(ctx, ctx->ids[f.cur], ctx->ranks, f.m, f.bshift, oi, ov, f.tag)) return rc;
                    if (int rc = region_scatter(ctx, oi, ov, f.n, f.bshift)) return rc;
                } else {
                    k_round0_isa<256><<<(u32)ceil_div(f.n, 256), 256, 0, ctx->stream>>>(f.sa, f.n, ctx->ids[f.cur], ctx->ranks, f.m, ctx->isa, f.tag);
                    LAUNCHED();
                }
            } else {
                k_scatter_ranks<256><<<(u32)ceil_div(f.m, 256), 256, 0, ctx->stream>>>(ctx->ids[f.cur], ctx->ranks, f.m, ctx->isa, f.tag);
                LAUNCHED();
                complete = false;
            }
            span_end(ctx, sp);
            return 0;
        }
        if (complete) return 0;
        // ranks of suffixes settled in round 0 exist only where they are about to be read
        if (f.round == 1 && ctx->knobs.rank_search) {
            // round 1: read the ranks off the sorted round-0 keys (still intact in keys[cur^1] / ids[cur^1])
            k_build_keys_search<256><<<(u32)ceil_div(f.m, 256), 256, 0, ctx->stream>>>(
                ctx->ids[f.cur], ctx->ranks, f.m, f.n, f.h, f.kb, ctx->keys[f.cur ^ 1], ctx->ids[f.cur ^ 1], f.text, ctx->lut, f.s_bits, f.K,
                f.Kc, f.drop, ctx->keys[f.cur], ctx->hist, f.passes_r);
            LAUNCHED();
            *keys_built = true;
        } else if (selective_rounds < 2) {
            const size_t words = (size_t)ceil_div(f.n, 32);
            CK(cudaMemsetAsync(ctx->bitmap, 0, words * sizeof(u32), ctx->stream));
            k_mark_needed<256><<<(u32)ceil_div(f.m, 256), 256, 0, ctx->stream>>>(ctx->ids[f.cur], f.m, f.n, f.h, ctx->bitmap);
            LAUNCHED();
            k_fill_needed<256><<<(u32)ceil_div(f.n, 256), 256, 0, ctx->stream>>>(f.sa, f.n, ctx->bitmap, ctx->isa);
            LAUNCHED();
            ++selective_rounds;
        } else {  // still not done after two rounds: fill every settled rank once
            k_round0_isa<256><<<(u32)ceil_div(f.n, 256), 256, 0, ctx->stream>>>(f.sa, f.n, ctx->ids[f.cur], ctx->ranks, 0u, ctx->isa, f.tag);
            LAUNCHED();
            complete = true;
        }
        return 0;
    }
};

// A doubling round in pairs mode: one kernel settles or keeps each pair (suffix_kernels.cuh, "pairs mode").
int pairs_round(dark_bwt_ctx* ctx, Fwd& f) {
    int sp = span_begin(ctx, PH_RERANK);
    constexpr int kPairThreads = 256, kPairsPerThread = 8;  // 4096 elements per tile, like the re-rank
    const u32 tiles = (u32)ceil_div(f.m / 2, kPairThreads * kPairsPerThread);
    if (tiles > ctx->scan_tiles) return ctx->fail_internal("scan tile state too small");
    u32* counter = nullptr;
    if (int rc = next_counter(ctx, &counter)) return rc;
    CK(cudaMemsetAsync(ctx->scan_words, 0, sizeof(u64) * kScanWordsPerTile * tiles, ctx->stream));
    ScanTileState ts{ctx->scan_words};
    k_pairs_round<kPairThreads, kPairsPerThread><<<tiles, kPairThreads, 0, ctx->stream>>>(
        ctx->ids[f.cur], ctx->ranks, f.m, f.n, f.h, ctx->isa, reinterpret_cast<uint2*>(ctx->keys[0]), f.sa, ctx->ids[f.cur ^ 1], ctx->ranks_alt,
        ts, counter, &ctx->mail_dev->count, f.text, f.emit_inline ? f.bwt : nullptr, &ctx->mail_dev->origin, f.tag);
    LAUNCHED();
    std::swap(ctx->ranks, ctx->ranks_alt);
    span_end(ctx, sp);
    f.cur ^= 1;
    f.st.pair_rounds += 1;
    const u32 m_before = f.m;
    if (int rc = fetch_count(ctx, &f.m)) return rc;
    if (const u32 settled = (m_before - f.m) / 2) {
        k_pairs_apply<<<(u32)ceil_div(settled, 256), 256, 0, ctx->stream>>>(reinterpret_cast<const uint2*>(ctx->keys[0]), settled, ctx->isa);
        LAUNCHED();
    }
    return 0;
}

// One doubling round: keys (rank[i], rank[i+h]) -> radix sort -> re-rank/compact, or a pairs round.
int doubling_round(dark_bwt_ctx* ctx, Fwd& f, RankFill& ranks, PairsMode& pairs) {
    if (f.round >= DARK_BWT_MAX_ROUNDS || f.h >= 2 * (u64)f.n + 2) return ctx->fail_internal("prefix doubling did not converge");
    f.st.active[f.round] = f.m;
    f.st.rounds = f.round;
    if (int rc = pairs.decide(ctx, f, ranks.complete)) return rc;
    if (pairs.on) return pairs_round(ctx, f);
    int sp = span_begin(ctx, PH_KEYBUILD);
    CK(cudaMemsetAsync(ctx->hist, 0, sizeof(u32) * kMaxPasses * kRadix, ctx->stream));
    bool keys_built = false;
    if (int rc = ranks.fill(ctx, f, &keys_built)) return rc;
    const bool text_built = !keys_built && f.tag != 0 && ranks.complete && (u64)f.m * (u64)ctx->knobs.text_div > (u64)f.n;
    if (text_built) {
        // many suffixes still active: sweep isa[] in text order instead of gathering from it (k_build_keys_text)
        constexpr int kTextThreads = 512, kTextItems = 8;
        const u32 tiles = (u32)ceil_div(f.n, kTextThreads * kTextItems);
        if (tiles > ctx->scan_tiles) return ctx->fail_internal("scan tile state too small");
        u32* counter = nullptr;
        if (int rc = next_counter(ctx, &counter)) return rc;
        CK(cudaMemsetAsync(ctx->scan_words, 0, sizeof(u64) * kScanWordsPerTile * tiles, ctx->stream));
        auto kern = k_build_keys_text<kTextThreads, kTextItems>;
        const size_t smem = kBuildTextSmem<kTextThreads, kTextItems>;
        CK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        const u32 grid = std::min<u32>(tiles, (u32)ctx->num_sms * 3);
        kern<<<grid, kTextThreads, smem, ctx->stream>>>(ctx->isa, f.n, f.h, f.kb, f.tag, ctx->keys[f.cur], ctx->ids[f.cur], ctx->scan_words,
                                                        counter, &ctx->mail_dev->flag, ctx->hist, f.passes_r);
        LAUNCHED();
    } else if (!keys_built) {
        const u32 blocks = (u32)ceil_div(f.m, kBuildThreads * kBuildItems);  // one tile per CTA: the gathers want every warp slot filled
        k_build_keys<kBuildThreads, kBuildItems><<<blocks, kBuildThreads, 0, ctx->stream>>>(
            ctx->ids[f.cur], ctx->ranks, f.m, f.n, f.h, f.kb, ctx->isa, f.tag, ctx->keys[f.cur], ctx->hist, f.passes_r);
        LAUNCHED();
    }
    span_end(ctx, sp);

    sp = span_begin(ctx, PH_SORT);
    if (int rc = run_sort(ctx, ctx->keys, ctx->ids, f.cur, f.m, 0, f.passes_r, &f.cur, &f.st, f.round, nullptr, /*all_passes=*/text_built))
        return rc;
    span_end(ctx, sp);

    sp = span_begin(ctx, PH_RERANK);
    u8* bwt_inline = f.emit_inline ? f.bwt : nullptr;
    const u32* count_dev = nullptr;
    if (f.bucketed && f.m > f.n / 16) {
        // the re-rank appends each tile's rank updates to per-bucket regions (suffix_kernels.cuh, PAIRS); the
        // regions are then scattered bucket by bucket, each bucket's slice of isa[] staying in L2
        u32* ids = (u32*)ctx->keys[f.cur ^ 1];
        const PairSink sink{ids, ids + align_up((size_t)f.n, 64), f.bshift};
        CK(cudaMemsetAsync(ctx->bucket_hist, 0, sizeof(u32) * 256, ctx->stream));
        if (int rc = launch_rerank<false, true>(ctx, ctx->keys[f.cur], ctx->ids[f.cur], f.m, f.n, f.K, f.kb, f.sa, ctx->ids[f.cur ^ 1], f.text,
                                                bwt_inline, f.tag, &count_dev, sink))
            return rc;
        if (int rc = region_scatter(ctx, sink.ids, sink.vals, f.m, f.bshift)) return rc;
    } else {
        if (int rc = launch_rerank<false, false>(ctx, ctx->keys[f.cur], ctx->ids[f.cur], f.m, f.n, f.K, f.kb, f.sa, ctx->ids[f.cur ^ 1], f.text,
                                                 bwt_inline, f.tag, &count_dev))
            return rc;
    }
    span_end(ctx, sp);
    f.cur ^= 1;
    const u32 m_sorted = f.m;
    if (int rc = pairs.queue(ctx, f, ranks.complete, count_dev, m_sorted)) return rc;  // the list that comes out may be all pairs
    if (int rc = fetch_count(ctx, &f.m)) return rc;
    if (text_built && ctx->mail->flag != m_sorted) return ctx->fail_internal("tagged isa[] entries disagree with the active list");
    return 0;
}

// The whole forward transform on device buffers (2 <= n <= capacity).  d_sa_user and st_out nullable.
int forward_device(dark_bwt_ctx* ctx, const u8* d_text, u32 n, u8* d_bwt, u64* origin_out, u32* d_sa_user, dark_bwt_stats* st_out) {
    if (int rc = begin_call(ctx)) return rc;
    Fwd f{d_text, n, d_bwt, d_sa_user ? d_sa_user : ctx->sa};
    f.st.h2d_ms = st_out ? st_out->h2d_ms : 0.f;
    reset_stats(&f.st, n);

    int sp = span_begin(ctx, PH_INIT);
    if (int rc = scan_alphabet(ctx, f)) return rc;
    if (int rc = round0_keys(ctx, f)) return rc;
    span_end(ctx, sp);
    PairsMode pairs{ctx->knobs.pairs};
    RankFill ranks;
    if (int rc = round0_sort(ctx, f)) return rc;
    if (int rc = round0_rerank(ctx, f, pairs)) return rc;
    if (f.m > 0)
        if (int rc = ranks.fill(ctx, f, nullptr)) return rc;
    for (f.h = (u64)f.K0, f.round = 1; f.m > 0; f.h *= 2, ++f.round)
        if (int rc = doubling_round(ctx, f, ranks, pairs)) return rc;

    // ---- BWT bytes + origin
    sp = span_begin(ctx, PH_EMIT);
    if (!f.emit_inline)
        if (int rc = emit(ctx, d_text, n, f.sa, d_bwt)) return rc;
    span_end(ctx, sp);
    CK(cudaEventRecord(ctx->call_stop, ctx->stream));
    CK(sync_counted(ctx));
    *origin_out = ctx->mail->origin;
    finish_stats(ctx, &f.st);
    if (st_out) *st_out = f.st;
    return DARK_BWT_OK;
}

// Many independent blocks in one sort (suffix_kernels.cuh, "many small blocks").  d_text holds the blocks back
// to back, ctx->many_starts their offsets (B + 1 values, already on the device); d_bwt receives the per-block BWTs
// at the same offsets, ctx->many_origins the origins.
int forward_many_device(dark_bwt_ctx* ctx, const u8* d_text, u32 n, u32 B, u8* d_bwt, u32* d_sa_out, dark_bwt_stats* st) {
    if (int rc = begin_call(ctx)) return rc;
    reset_stats(st, n);
    int sp = span_begin(ctx, PH_INIT);
    CK(cudaMemsetAsync(ctx->present, 0, sizeof(u32) * 256, ctx->stream));
    CK(cudaMemsetAsync(ctx->hist, 0, sizeof(u32) * kMaxPasses * kRadix, ctx->stream));
    {
        const u32 blocks = (u32)std::min<u64>(ceil_div(ceil_div(n, 16), 256), 148 * 8);
        k_symbol_presence<256><<<std::max(blocks, 1u), 256, 0, ctx->stream>>>(d_text, n, ctx->present);
        LAUNCHED();
        k_many_lut<<<1, 256, 0, ctx->stream>>>(ctx->present, ctx->many_lut, &ctx->mail_dev->sigma);
        LAUNCHED();
    }
    CK(sync_counted(ctx));
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
    if (int rc = launch_rerank<true, false>(ctx, ctx->keys[cur], ctx->ids[cur], n, n, 1, 0, ctx->sa, ctx->ids[cur ^ 1], d_text, nullptr, 0u, nullptr)) return rc;
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
        if (int rc = launch_rerank<false, false>(ctx, ctx->keys[cur], ctx->ids[cur], m, n, K, kb, ctx->sa, ctx->ids[cur ^ 1], d_text, nullptr, 0u, nullptr)) return rc;
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
    CK(cudaEventRecord(ctx->call_stop, ctx->stream));
    CK(sync_counted(ctx));
    finish_stats(ctx, st);
    return DARK_BWT_OK;
}

// ---- argument checks of the entry points --------------------------------------------------------
// The length of a single block: min_n (1 or 2) <= n <= capacity, and n <= 2^32-2 (suffixes and rows are u32).
int check_n(const dark_bwt_ctx* ctx, u64 n, u64 min_n) {
    return (n < min_n || n > ctx->capacity || n > 0xFFFFFFFEull) ? DARK_BWT_E_INVALID_N : DARK_BWT_OK;
}

// The host-buffer entries stage through device buffers that a DARK_BWT_F_DEVICE_ONLY context does not have.
int check_staging(const dark_bwt_ctx* ctx) { return (ctx->flags & DARK_BWT_F_DEVICE_ONLY) ? DARK_BWT_E_INVALID_ARG : DARK_BWT_OK; }

// A packed item stream of stream_bytes for a block of n bytes (the decode entries, after their pointer checks).
int check_decode_args(const dark_bwt_ctx* ctx, uint64_t stream_bytes, uint64_t n) {
    if (int rc = check_n(ctx, n, 1)) return rc;
    if (stream_bytes == 0 || stream_bytes > DARK_BWT_DC_PACKED_MAX(n)) return DARK_BWT_E_INVALID_ARG;  // no valid stream is that long
    return DARK_BWT_OK;
}

// The blocks of a many-block entry, back to back: block k is [starts[k], starts[k+1]).
struct BlockList {
    std::vector<u32> starts;              // count + 1 offsets
    std::vector<uint64_t> origins;        // the inverse's, one per block
    const u32* d_starts = nullptr;        // device entries: the caller's offsets and origins, which load_blocks copies
    const uint64_t* d_origins = nullptr;
    u64 max_nb = 0;                       // the largest block
    u32 count() const { return (u32)starts.size() - 1; }
    u32 total() const { return starts.back(); }
};

// The one check of a many-block list, before any kernel reads it.  The offsets come from the host lengths `ns`, or from
// `d_starts` on the device, read back here; `origins` (the inverse's, else null) lives where the offsets do.  `ins` and
// `outs` (nullable) are host blocks and outputs, one per block.  Every block has at least min_n bytes and adds `extra_rows`
// rows beyond them (the inverse's '$' row); the rows must fit the arena and u32 offsets.  u64 arithmetic throughout, so
// no offset, length or sum wraps.  In the order checked: count > DARK_BWT_MAX_MANY_BLOCKS, starts[0] != 0, a null block or
// output pointer or an origin outside its block is DARK_BWT_E_INVALID_ARG; a shorter block (decreasing offsets included)
// or too many rows is DARK_BWT_E_INVALID_N.
int check_blocks(dark_bwt_ctx* ctx, u64 count, const uint64_t* ns, const u32* d_starts, const uint64_t* origins, u64 min_n,
                 u64 extra_rows, const uint8_t* const* ins, uint8_t* const* outs, BlockList* bl) {
    if (count > kMaxManyBlocks) return DARK_BWT_E_INVALID_ARG;
    std::vector<u64> s(count + 1, 0);
    bl->starts.resize(count + 1);
    bl->origins.resize(origins ? count : 0);
    if (d_starts) {
        CK(cudaSetDevice(ctx->device));
        CK(cudaMemcpyAsync(bl->starts.data(), d_starts, sizeof(u32) * (count + 1), cudaMemcpyDeviceToHost, ctx->stream));
        if (origins) CK(cudaMemcpyAsync(bl->origins.data(), origins, sizeof(uint64_t) * count, cudaMemcpyDeviceToHost, ctx->stream));
        CK(cudaStreamSynchronize(ctx->stream));
        std::copy(bl->starts.begin(), bl->starts.end(), s.begin());
        bl->d_starts = d_starts;
        bl->d_origins = origins;
    } else {
        // a block of 2^32 bytes or more fails below whatever its length: clamped there, the lengths add up without wrapping
        for (u64 k = 0; k < count; ++k) s[k + 1] = s[k] + std::min<u64>(ns[k], 1ull << 32);
        if (origins) std::copy(origins, origins + count, bl->origins.begin());
    }
    if (s[0] != 0) return DARK_BWT_E_INVALID_ARG;
    const u64 max_rows = std::min<u64>(ctx->capacity, 0xFFFFFFFEull);
    bl->max_nb = 0;
    for (u64 k = 0; k < count; ++k) {
        if ((ins && !ins[k]) || (outs && !outs[k])) return DARK_BWT_E_INVALID_ARG;
        if (s[k + 1] < s[k] + min_n) return DARK_BWT_E_INVALID_N;
        const u64 nb = s[k + 1] - s[k];
        if (origins && bl->origins[k] >= nb) return DARK_BWT_E_INVALID_ARG;
        bl->max_nb = std::max(bl->max_nb, nb);
        if (s[k + 1] + extra_rows * (k + 1) > max_rows) return DARK_BWT_E_INVALID_N;  // the blocks share one arena
    }
    for (u64 k = 0; k <= count; ++k) bl->starts[k] = (u32)s[k];
    return DARK_BWT_OK;
}

// Puts a checked list where the kernels read it: the offsets into ctx->many_starts, the inverse's origins into ctx->many_origins.
int load_blocks(dark_bwt_ctx* ctx, const BlockList& bl) {
    const size_t count = bl.count();
    if (bl.d_starts) CK(cudaMemcpyAsync(ctx->many_starts, bl.d_starts, sizeof(u32) * (count + 1), cudaMemcpyDeviceToDevice, ctx->stream));
    else CK(cudaMemcpyAsync(ctx->many_starts, bl.starts.data(), sizeof(u32) * (count + 1), cudaMemcpyHostToDevice, ctx->stream));
    static_assert(sizeof(unsigned long long) == sizeof(uint64_t), "origins are copied as they are");
    if (bl.d_origins) CK(cudaMemcpyAsync(ctx->many_origins, bl.d_origins, sizeof(uint64_t) * count, cudaMemcpyDeviceToDevice, ctx->stream));
    else if (!bl.origins.empty())
        CK(cudaMemcpyAsync(ctx->many_origins, bl.origins.data(), sizeof(uint64_t) * count, cudaMemcpyHostToDevice, ctx->stream));
    return 0;
}

// ---- inverse BWT --------------------------------------------------------------------------------
// Inverse BWT on device buffers (kernels and method: suffix_kernels.cuh, "inverse BWT") of one block d_bwt[0..n) with origin
// `origin` (`blocks` null; 1 <= n <= capacity, origin < n), or in one pass of the checked list `blocks`, back to back in d_bwt
// (n bytes) and loaded into ctx->many_starts and ctx->many_origins ("inverse BWT of many blocks"; `origin` unused).  d_text
// receives the texts at the same offsets.
//
// Buffers: the rows number R = n + B <= capacity (the entry points check it).  The sort moves n <= capacity pairs.  The
// node arrays (dist and next twice, len_keep) hold `regular + B` entries, and regular = ceil(R / stride) <= (R + 1) / 2 with
// stride >= 2 while every block has at least two rows (B <= R / 2; one block: regular + 1 <= R): nodes <= R <= capacity,
// which the u32 arrays of the arena hold.  The stash gets (8 capacity + 1024) / nodes >= 8 bytes a chunk.  So 65,536 blocks
// of one byte need a capacity of 131,072 (rows, not bytes, are what must fit), and sum(ns) <= capacity alone would not be
// enough.
int inverse_device(dark_bwt_ctx* ctx, const u8* d_bwt, u32 n, u32 origin, const BlockList* blocks, u8* d_text, float* ms_out) {
    if (int rc = begin_call(ctx)) return rc;
    CK(cudaMemsetAsync(ctx->hist, 0, sizeof(u32) * kMaxPasses * kRadix, ctx->stream));
    const u32 B = blocks ? blocks->count() : 1u;
    int cur = 0;
    IbwtMany many{};  // zero in the single-block instantiations
    if (!blocks) {
        // step 1: (last-column symbol, row) pairs; stable partition by symbol -> psi.  The pairs are built inside the
        // radix pass (GEN mode 1) and their digit histogram is the byte histogram of the BWT.
        k_build_lut<<<1, 256, 0, ctx->stream>>>(ctx->present, ctx->lut, &ctx->mail_dev->sigma, 1);  // identity codes
        LAUNCHED();
        u32* gram = ctx->bucket_hist;
        CK(cudaMemsetAsync(gram, 0, sizeof(u32) * kRadix, ctx->stream));
        const u32 grid = (u32)std::min<u64>(ceil_div(n, 256 * 16), (u64)ctx->num_sms * 8);
        k_gram_hist<256, 8><<<std::max(grid, 1u), 256, 0, ctx->stream>>>(d_bwt, n, ctx->lut, gram);
        LAUNCHED();
        CK(cudaMemcpyAsync(ctx->hist, gram, sizeof(u32) * kRadix, cudaMemcpyDeviceToDevice, ctx->stream));
        KeyGen gen;
        gen.text = d_bwt;
        gen.lut = ctx->lut;
        gen.n = n;
        gen.lg_s = 3;
        gen.mode = 1;
        gen.origin = origin;
        if (int rc = run_sort(ctx, ctx->keys, ctx->ids, 0, n, 0, 1, &cur, nullptr, 0, &gen)) return rc;
        if (cur == 0) {  // one-symbol BWT: the pass is the identity and did not run; psi is the row list itself
            k_ibwt_elements<<<(u32)ceil_div(n, 256), 256, 0, ctx->stream>>>(d_bwt, n, origin, ctx->keys[0], ctx->ids[0]);
            LAUNCHED();
        }
        // k_ibwt_walk finds first symbols in the symbol bases (exclusive digit counts of pass 0, left in ctx->hist by run_sort)
    } else {
        // step 1: (block, last symbol) keys of the real rows, one stable sort -> psi and the first symbols
        const int passes = 1 + (B > 1 ? (bit_length((u64)B - 1) + kRadixBits - 1) / kRadixBits : 0);
        const u32 grid = (u32)std::min<u64>(ceil_div(n, 256), (u64)ctx->num_sms * 8);
        k_ibwt_many_elements<256><<<grid, 256, 0, ctx->stream>>>(d_bwt, n, ctx->many_starts, B, ctx->many_origins, ctx->keys[0],
                                                                 ctx->ids[0], ctx->hist, passes);
        LAUNCHED();
        // passes whose digit is the same in every key are skipped (one-symbol blocks, a single block): the order stays the row order
        if (int rc = run_sort(ctx, ctx->keys, ctx->ids, 0, n, 0, passes, &cur, nullptr, 0)) return rc;
        many = IbwtMany{ctx->many_starts, ctx->many_origins, B, ctx->keys[cur]};
    }
    const u32* psi = ctx->ids[cur];
// Launches a kernel template on MANY: with MANY = true for a block list, false for one block.
#define IBWT_LAUNCH(...)                                \
    do {                                                \
        if (blocks) { constexpr bool MANY = true; __VA_ARGS__; }   \
        else { constexpr bool MANY = false; __VA_ARGS__; }         \
        LAUNCHED();                                     \
    } while (0)
    // step 2: sublists between splitters
    const u32 stride = (u32)ctx->knobs.ibwt_stride;  // rows between splitters; swept 24..128 with the single walk: 48 (profiles/r1_final.md)
    const u32 regular = (u32)ceil_div((u64)n + B, stride);
    const u32 nodes = regular + B;
    const u32 grid = (u32)ceil_div(nodes, 128);
    u32* dist[2] = {ctx->ranks, ctx->sa};
    u32* next[2] = {ctx->isa, ctx->ids[cur ^ 1]};
    // one walk: count the sublists and stash their symbols (DARK_BWT_IBWT_TWO_WALKS=1: count, then a second walk writes)
    u32* len_keep = ctx->ranks_alt;
    u32* stash = (u32*)ctx->keys[cur ^ 1];  // the sort's other key buffer (8 capacity + 1024 bytes) is free
    const u32 cap = (u32)std::min<u64>(kIbwtStashCap, ((ctx->capacity * 8 + 1024) / nodes) & ~3ull);  // smaller strides: smaller chunks
    const bool two_walks = ctx->knobs.ibwt_two_walks || cap < 8;
    if (two_walks)
        IBWT_LAUNCH(k_ibwt_walk<0, MANY><<<grid, 128, 0, ctx->stream>>>(psi, n, origin, stride, regular, dist[0], next[0], nullptr, nullptr,
                                                                       nullptr, nullptr, nullptr, 0u, 0u, many));
    else
        IBWT_LAUNCH(k_ibwt_walk<2, MANY><<<grid, 128, 0, ctx->stream>>>(psi, n, origin, stride, regular, dist[0], next[0], nullptr, ctx->hist,
                                                                       nullptr, len_keep, stash, 0u, cap, many));
    // step 3: suffix sums of the sublist lengths along the splitter lists (pointer jumping); a list holds at most
    // ceil((max n_b + 1) / stride) + 1 splitters (one block: all of them)
    const u64 chain = ceil_div((u64)(blocks ? blocks->max_nb : n) + 1, stride) + 1;
    int w = 0;
    for (u64 span = 1; span < chain; span <<= 1) {
        k_ibwt_jump<<<(u32)ceil_div(nodes, 256), 256, 0, ctx->stream>>>(dist[w], next[w], dist[w ^ 1], next[w ^ 1], nodes);
        LAUNCHED();
        w ^= 1;
    }
    IBWT_LAUNCH(k_ibwt_check<MANY><<<1, 1024, 0, ctx->stream>>>(dist[w], n, regular, &ctx->mail_dev->count, &ctx->mail_dev->bad_block,
                                                                &ctx->mail_dev->bad_dist, many));
    CK(cudaStreamSynchronize(ctx->stream));
    if (ctx->mail->count != 0) {
        if (blocks)
            snprintf(ctx->err, sizeof(ctx->err), "inverse BWT: block %u is not a forward transform (%u of %u blocks are not)",
                     ctx->mail->bad_block, ctx->mail->count, B);
        else
            snprintf(ctx->err, sizeof(ctx->err), "inverse BWT: (bwt, origin) is not a forward transform (list covers %u of %llu rows)",
                     ctx->mail->bad_dist, (unsigned long long)n + 1);
        return DARK_BWT_E_INVALID_ARG;
    }
    // step 4: the text.  Stashed sublists are copied to their offsets; the few longer ones are walked again.
    if (two_walks) {
        IBWT_LAUNCH(k_ibwt_walk<1, MANY><<<grid, 128, 0, ctx->stream>>>(psi, n, origin, stride, regular, nullptr, nullptr, dist[w], ctx->hist,
                                                                       d_text, nullptr, nullptr, 0u, 0u, many));
    } else {
        IBWT_LAUNCH(k_ibwt_unstash<MANY><<<grid, 128, 0, ctx->stream>>>(stash, len_keep, dist[w], n, stride, regular, d_text, cap, many));
        IBWT_LAUNCH(k_ibwt_walk<1, MANY><<<grid, 128, 0, ctx->stream>>>(psi, n, origin, stride, regular, nullptr, nullptr, dist[w], ctx->hist,
                                                                       d_text, len_keep, nullptr, cap, 0u, many));
    }
#undef IBWT_LAUNCH
    CK(cudaEventRecord(ctx->call_stop, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    if (ms_out) *ms_out = call_ms(ctx);
    return DARK_BWT_OK;
}

// ---- distance coding ----------------------------------------------------------------------------
// The per-block records of the many-block pass are staged in the sort's second key buffer (8 N + 1 KiB bytes), which distance
// coding leaves free: count * sizeof(DcRecDev) <= 8 * capacity + 1024.
bool dc_many_records_fit(const dark_bwt_ctx* ctx, u64 count) {
    return count * sizeof(DcRecDev) <= ctx->capacity * 8 + 1024;
}

// Distance coding + MTF on device buffers (dc_kernels.cuh) of one BWT block d_bwt[0..n) (`blocks` null; 1 <= n <= capacity),
// or in one pass of the checked list `blocks`, back to back in d_bwt and loaded into ctx->many_starts (the records fit).
// One block: infos[0] gets the result header.  Many: infos[0..count) get the per-block records, *item_starts_host the
// item offsets, read back.  Neither it nor dc_pack writes ctx->d_bwt or ctx->many_origins: the forward + DC host entries
// copy the BWTs and origins out with the DC outputs.
int dc_device(dark_bwt_ctx* ctx, const u8* d_bwt, u32 n, const BlockList* blocks, DcBuffers* io, dark_bwt_dc_info* infos,
              std::vector<u32>* item_starts_host) {
    CK(cudaSetDevice(ctx->device));
    const u32 nblocks = (u32)ceil_div(n, kDcBlock);
    // last-occurrence tables: (nblocks + ngroups) x 256 words = n/4 + n/1024 bytes (+ 2 KB): inside the 4n-byte rank buffer for
    // all but tiny blocks, which borrow the sort's status buffer (>= 256 KB)
    u32* tab = n <= 65536u ? (u32*)ctx->status.borrow() : ctx->ranks;
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
    DcMany many{};  // zero in the single-block instantiations
    if (blocks) {
        // behind the run counts (4 N + 16 bytes): align4(nblocks) + count + 1 words fit, as the records bound count to capacity / 160
        if (!io->item_starts) io->item_starts = ctx->ranks_alt + align_up(nblocks, 4);
        many = DcMany{ctx->many_starts, blocks->count(), ctx->bitmap, (DcRecDev*)ctx->keys[1], io->item_starts};
    }
    CK(cudaEventRecord(ctx->call_start, ctx->stream));
    CK(cudaMemsetAsync(first, 0xFF, sizeof(u32) * 256, ctx->stream));
    CK(cudaMemsetAsync(total_runs, 0, sizeof(unsigned long long), ctx->stream));
    if (blocks) {
        CK(cudaMemsetAsync(ctx->bitmap, 0, sizeof(u32) * ceil_div(n, 32), ctx->stream));
        k_dc_mark_starts<<<(u32)ceil_div(many.count, 256), 256, 0, ctx->stream>>>(ctx->many_starts, many.count, ctx->bitmap, io->item_starts);
        LAUNCHED();
    }
#define DC_LAUNCH(KERNEL, GRID, ...)                                                          \
    do {                                                                                      \
        if (blocks) KERNEL<true><<<GRID, 256, 0, ctx->stream>>>(__VA_ARGS__, many);           \
        else KERNEL<false><<<GRID, 256, 0, ctx->stream>>>(__VA_ARGS__, many);                 \
        LAUNCHED();                                                                           \
    } while (0)
    DC_LAUNCH(k_dc_tables, nblocks, d_bwt, n, tab, first, run_counts, io->dist, total_runs);
    const u32 ngroups = (u32)ceil_div(nblocks, kDcGroup);
    u32* group_last = tab + (size_t)nblocks * 256;  // ngroups x 256 words behind the table (n/4 + n/1024 bytes of the 4n)
    k_dc_scan_groups<<<ngroups, 256, 0, ctx->stream>>>(tab, nblocks, group_last);
    LAUNCHED();
    k_dc_scan_carry<<<1, 256, 0, ctx->stream>>>(group_last, ngroups, final_last);
    LAUNCHED();
    k_sparse_scan<<<1, 1024, 0, ctx->stream>>>(run_counts, nblocks);  // in place: exclusive run offsets
    LAUNCHED();
    u32* alpha = ctx->bucket_hist + 512;  // 513 words: dense codes of the symbols that occur (in any block)
    k_dc_alphabet<<<1, 256, 0, ctx->stream>>>(first, alpha);
    LAUNCHED();
    const u32 rgrid = (u32)ceil_div(nblocks, 8);
    DC_LAUNCH(k_dc_ranks, rgrid, d_bwt, n, tab, group_last, run_counts, nblocks, alpha, io->dist, run_start, io->item_sym, io->item_rank);
    if (!blocks) {  // many blocks: k_dc_ranks finalises each block at its end
        k_dc_final<<<1, 256, 0, ctx->stream>>>(n, final_last, first, io->dist, total_runs, ctx->dc_info);
        LAUNCHED();
    }
    const u32 sgrid = (u32)std::min<u64>(ceil_div(n, 256), (u64)ctx->num_sms * 16);
    DC_LAUNCH(k_dc_stream, sgrid, run_start, total_runs, n, io->dist, io->item_pos, io->item_dist);
#undef DC_LAUNCH
    CK(cudaEventRecord(ctx->call_stop, ctx->stream));
    if (!blocks) {
        static_assert(offsetof(dark_bwt_dc_info, num_items) == offsetof(DcInfoDev, num_items), "DcInfoDev mirrors the head of dark_bwt_dc_info");
        CK(cudaMemcpyAsync(infos, ctx->dc_info, sizeof(DcInfoDev), cudaMemcpyDeviceToHost, ctx->stream));
        CK(cudaStreamSynchronize(ctx->stream));
        infos->device_ms = call_ms(ctx);
        return DARK_BWT_OK;
    }
    const u32 count = many.count;
    std::vector<DcRecDev> recs(count);
    std::vector<u32>& hs = *item_starts_host;
    hs.resize((size_t)count + 1);
    CK(cudaMemcpyAsync(recs.data(), many.recs, sizeof(DcRecDev) * count, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaMemcpyAsync(hs.data(), io->item_starts, sizeof(u32) * ((size_t)count + 1), cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    const float ms = call_ms(ctx);
    for (u32 k = 0; k < count; ++k) {
        dark_bwt_dc_info& info = infos[k];
        for (int c = 0; c < 256; ++c) info.init[c] = recs[k].init[c];
        memcpy(info.mtf_symbols, recs[k].mtf_symbols, 256);
        info.num_unique = recs[k].num_unique;
        info.reserved_ = 0;
        info.num_items = hs[k + 1] - hs[k];
        info.device_ms = ms;
        info.reserved2_ = 0;
    }
    return DARK_BWT_OK;
}

// The packed item stream (include/dark_bwt.h; kernels in dc_kernels.cuh) of the `items` items dc_device left in `io`, into
// d_out, which holds `capacity` bytes.  *bytes_out = the stream's size, which the scan leaves in the mailbox; a size above
// the capacity is DARK_BWT_E_INVALID_ARG before anything is written.  The tile sums and offsets go to ranks_alt and ranks
// (at most 12 bytes per 2,048 items), which dc_device has finished with.  Returns after the stream is complete; adds the
// pack's device time to *ms.
// Many blocks (d_stream_starts non-null): the items of the `count` blocks of a many-block pass, at io.item_starts.  Each
// block's stream is what the block alone packs to, the streams back to back; d_stream_starts[0..count] (device) gets their
// offsets, [count] = the total, only when the stream fits.  The first-item bitmap goes to ctx->bitmap, which the pass has
// finished with.  ranks_alt holds the item starts, so the tile sums go to ranks instead: ranks holds count + 1 words of 8
// bytes first (where dark_bwt_forward_dc_packed_many keeps the offsets), then the tile offsets, then the tile sums.
int dc_pack(dark_bwt_ctx* ctx, const DcBuffers& io, u64 items, u8* d_out, u64 capacity, uint64_t* bytes_out, float* ms,
            u32 count = 0, u64* d_stream_starts = nullptr) {
    const u32 ntiles = (u32)ceil_div(items, kPackTile);
    const bool many = d_stream_starts != nullptr;
    u64* tile_off = (u64*)ctx->ranks + (many ? count + 1 : 0);
    u32* tile_bytes = many ? (u32*)(tile_off + ntiles) : ctx->ranks_alt;
    PackMany pm{};  // zero in the single-block instantiations
    CK(cudaEventRecord(ctx->call_start, ctx->stream));
    if (many) {
        pm = PackMany{ctx->bitmap, io.item_starts, count, d_stream_starts};
        CK(cudaMemsetAsync(ctx->bitmap, 0, sizeof(u32) * ceil_div(items, 32), ctx->stream));
        k_dc_mark_items<<<(u32)ceil_div(count, 256), 256, 0, ctx->stream>>>(io.item_starts, count, ctx->bitmap);
        LAUNCHED();
        k_dc_pack_sizes<true><<<ntiles, kPackThreads, 0, ctx->stream>>>(io.item_pos, io.item_dist, items, tile_bytes, pm);
    } else {
        k_dc_pack_sizes<false><<<ntiles, kPackThreads, 0, ctx->stream>>>(io.item_pos, io.item_dist, items, tile_bytes, pm);
    }
    LAUNCHED();
    k_dc_pack_scan<<<1, 1024, 0, ctx->stream>>>(tile_bytes, ntiles, tile_off, &ctx->mail_dev->packed_bytes);
    LAUNCHED();
    CK(cudaStreamSynchronize(ctx->stream));
    *bytes_out = ctx->mail->packed_bytes;
    if (*bytes_out > capacity) {
        snprintf(ctx->err, sizeof(ctx->err), "the packed item stream needs %llu bytes, the buffer holds %llu",
                 (unsigned long long)*bytes_out, (unsigned long long)capacity);
        return DARK_BWT_E_INVALID_ARG;
    }
    if (many) {
        static_assert(sizeof(ctx->mail->packed_bytes) == sizeof(u64), "the total is copied as it is");
        CK(cudaMemcpyAsync(d_stream_starts + count, &ctx->mail->packed_bytes, sizeof(u64), cudaMemcpyHostToDevice, ctx->stream));
        k_dc_pack_write<true><<<ntiles, kPackThreads, 0, ctx->stream>>>(io.item_pos, io.item_dist, io.item_sym, io.item_rank, items,
                                                                        tile_off, d_out, pm);
    } else {
        k_dc_pack_write<false><<<ntiles, kPackThreads, 0, ctx->stream>>>(io.item_pos, io.item_dist, io.item_sym, io.item_rank, items,
                                                                         tile_off, d_out, pm);
    }
    LAUNCHED();
    CK(cudaEventRecord(ctx->call_stop, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    *ms += call_ms(ctx);
    return DARK_BWT_OK;
}

// dc_pack of the `count` blocks dc_device coded in one pass (item offsets `starts`, read back): every infos[k].device_ms, and
// *ms_out (nullable), becomes the time of the pass and the pack.
int dc_pack_many(dark_bwt_ctx* ctx, const DcBuffers& io, const std::vector<u32>& starts, u8* d_out, u64 capacity,
                 u64* d_stream_starts, uint64_t* bytes_out, dark_bwt_dc_info* infos, float* ms_out) {
    const u32 count = (u32)starts.size() - 1;
    float ms = infos[0].device_ms;
    if (int rc = dc_pack(ctx, io, starts.back(), d_out, capacity, bytes_out, &ms, count, d_stream_starts)) return rc;
    for (u32 k = 0; k < count; ++k) infos[k].device_ms = ms;
    if (ms_out) *ms_out = ms;
    return DARK_BWT_OK;
}

// The inverse of dark_bwt_dc_encode_packed_device (kernels in dc_kernels.cuh, DESIGN.md §3.9): d_bwt[0..n) gets the block
// whose packed stream is d_stream[0..bytes), 1 <= bytes <= 8 n, or the call is DARK_BWT_E_INVALID_ARG with ctx->err saying
// why.  Parse (tiles, chain), one host round trip for the chain's totals, which must be those of a stream of n bytes, and
// only then the items and the expansion into d_bwt; the check is dc_device + dc_pack of d_bwt and a byte compare with the
// stream.  *info = what the encoder gives for the block, device_ms = the whole call.
// Scratch: run starts (4 n), symbols (n) and the tile summaries and bases (96 bytes per 8 KiB of stream: <= 0.1 n + 96) in
// keys[0] (8 N + 1 KiB), which the check then takes for DC's distances and the re-pack (<= 8 n): the pack reads neither.  A
// host entry's stream in keys[1] and the caller's buffers are only read.
int dc_decode(dark_bwt_ctx* ctx, const u8* d_stream, u64 bytes, u32 n, u8* d_bwt, dark_bwt_dc_info* info) {
    if (int rc = begin_call(ctx)) return rc;
    cudaEvent_t ev_start = ctx->events[0], ev_stop = ctx->events[1];
    CK(cudaEventRecord(ev_start, ctx->stream));
    u8* const scratch = (u8*)ctx->keys[0];
    u32* const run_start = (u32*)scratch;
    u8* const run_sym = scratch + (size_t)n * 4;
    const u32 ntiles = (u32)ceil_div(bytes, kUnpackTile);
    UnpackSum* const tiles = (UnpackSum*)(scratch + align_up((size_t)n * 5, 16));
    UnpackBase* const bases = (UnpackBase*)(tiles + ntiles);
    k_dc_unpack_tiles<<<ntiles, kUnpackThreads, 0, ctx->stream>>>(d_stream, bytes, tiles);
    LAUNCHED();
    k_dc_unpack_chain<<<1, kChainThreads, 0, ctx->stream>>>(tiles, ntiles, bases, &ctx->mail_dev->unpack);
    LAUNCHED();
    CK(cudaStreamSynchronize(ctx->stream));
    const UnpackTotals t = ctx->mail->unpack;
    if (t.err != ~0ull) {
        snprintf(ctx->err, sizeof(ctx->err), "packed item stream: malformed item at byte %llu (a varint of more than 5 bytes or "
                 "above 2^32 - 1, or an item cut off by the end)", t.err);
        return DARK_BWT_E_INVALID_ARG;
    }
    if (t.state != 0) {
        snprintf(ctx->err, sizeof(ctx->err), "packed item stream: the %llu bytes end inside an item", (unsigned long long)bytes);
        return DARK_BWT_E_INVALID_ARG;
    }
    if (t.sum != n) {
        snprintf(ctx->err, sizeof(ctx->err), "packed item stream: the run lengths of its %llu items add up to %s%llu, not n = %u",
                 t.items, t.sum >= kUnpackSumCap ? "at least " : "", t.sum, n);
        return DARK_BWT_E_INVALID_ARG;
    }
    // every item is well formed and the run lengths (each >= 1) add up to n: at most n items, run starts increasing below n
    k_dc_unpack_items<<<ntiles, kUnpackThreads, 0, ctx->stream>>>(d_stream, bytes, bases, n, run_start, run_sym);
    LAUNCHED();
    k_dc_unpack_expand<<<(u32)ceil_div((u64)n + ((uintptr_t)d_bwt & 15u), kExpandWords * 16), kExpandWords, 0, ctx->stream>>>(
        run_start, run_sym, (u32)t.items, n, d_bwt);
    LAUNCHED();
    // the check: the decoded block's own stream must be the input, byte for byte (distances and ranks have no cheaper test)
    DcBuffers io;
    if (int rc = dc_device(ctx, d_bwt, n, nullptr, &io, info, nullptr)) return rc;
    u8* const repack = (u8*)ctx->keys[0];
    u64 repacked = 0;
    float pack_ms = 0.f;
    if (int rc = dc_pack(ctx, io, info->num_items, repack, (u64)n * 8, &repacked, &pack_ms)) return rc;
    if (repacked != bytes) {
        snprintf(ctx->err, sizeof(ctx->err), "packed item stream: the decoded block packs to %llu bytes, the stream has %llu",
                 (unsigned long long)repacked, (unsigned long long)bytes);
        return DARK_BWT_E_INVALID_ARG;
    }
    u32* done = nullptr;
    if (int rc = next_counter(ctx, &done)) return rc;
    CK(cudaMemsetAsync(ctx->bad, 0xFF, sizeof(unsigned long long), ctx->stream));
    const u32 cgrid = (u32)std::min<u64>(ceil_div(bytes, 256), (u64)ctx->num_sms * 8);
    k_dc_unpack_compare<<<cgrid, 256, 0, ctx->stream>>>(d_stream, repack, bytes, ctx->bad, done, &ctx->mail_dev->unpack_diff);
    LAUNCHED();
    CK(cudaEventRecord(ev_stop, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    if (ctx->mail->unpack_diff != ~0ull) {
        snprintf(ctx->err, sizeof(ctx->err), "packed item stream: differs from the decoded block's own stream at byte %llu",
                 ctx->mail->unpack_diff);
        return DARK_BWT_E_INVALID_ARG;
    }
    cudaEventElapsedTime(&info->device_ms, ev_start, ev_stop);
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

void stage_release(HostStage& st) {
    for (int i = 0; i < HostStage::kMaxLanes; ++i) {
        if (st.streams[i]) cudaStreamDestroy(st.streams[i]);
        for (int k = 0; k < 2; ++k)
            if (st.slot_done[i][k]) cudaEventDestroy(st.slot_done[i][k]);
    }
    if (st.pinned) cudaFreeHost(st.pinned);
    st = HostStage();
}

// Sets up the lanes of `st` once: 0 when they are ready, 1 when there are none (switched off, or no pinned memory), or a
// CUDA error code.  A failure part-way releases what was made, so that the next call starts from a clean state.
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
    auto release = [&](int rc) {
        stage_release(st);
        return rc;
    };
    for (int i = 0; i < lanes; ++i) {
        if (cudaStreamCreateWithFlags(&st.streams[i], cudaStreamNonBlocking) != cudaSuccess)
            return release(ctx->fail_cuda(cudaGetLastError(), "staging stream", __LINE__));
        for (int k = 0; k < 2; ++k)
            if (cudaEventCreateWithFlags(&st.slot_done[i][k], cudaEventDisableTiming) != cudaSuccess)
                return release(ctx->fail_cuda(cudaGetLastError(), "staging event", __LINE__));
    }
    st.lanes = lanes;
    return 0;
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

// The staging rule of every host copy in direction `kind`: a pageable host buffer of kStageMinBytes or more goes through the
// context's lanes for that direction (*stage), anything else straight to cudaMemcpyAsync (*stage null), and so does every
// buffer when the lanes are switched off or no pinned memory is to be had.  Returns 0 or a CUDA error code.
int stage_for(dark_bwt_ctx* ctx, const void* host, size_t bytes, cudaMemcpyKind kind, HostStage** stage) {
    *stage = nullptr;
    if (bytes < kStageMinBytes || !is_pageable(host)) return 0;
    HostStage& st = kind == cudaMemcpyHostToDevice ? ctx->stage_in : ctx->stage_out;
    const int rc = stage_prepare(ctx, st);
    if (rc == 0) *stage = &st;
    return rc == 1 ? 0 : rc;
}

// Copies between caller host buffers and device buffers in one direction, issued in order.  Absent buffers (null host
// pointers) and empty copies are left out.  `serial` (the pipelined copy-out): a source is single-buffered (the next block
// overwrites it), so the copies must be complete before the next block is transformed.
struct CopyList {
    struct Copy {
        void* host;
        void* dev;
        size_t bytes;
    };
    std::vector<Copy> list;  // the many-block entries: one copy per block
    bool serial = false;
    CopyList& add(const void* host, const void* dev, size_t bytes) {
        if (host && bytes) list.push_back(Copy{(void*)host, (void*)dev, bytes});
        return *this;
    }
    // The blocks of `bl` between the caller's host blocks hosts[k] and `dev` at their offsets (`hosts` and its entries nullable).
    CopyList& add_blocks(const BlockList& bl, const uint8_t* const* hosts, const u8* dev) {
        if (hosts)
            for (u32 k = 0; k < bl.count(); ++k) add(hosts[k], dev + bl.starts[k], bl.starts[k + 1] - bl.starts[k]);
        return *this;
    }
};

// Runs `copies` in direction `kind` and returns when every one has completed: the staged ones through the lanes, the others
// with cudaMemcpyAsync on `stream` and one synchronise.  The caller has made sure that the device side is ready.
int copy_blocking(dark_bwt_ctx* ctx, const CopyList& copies, cudaMemcpyKind kind, cudaStream_t stream) {
    const bool to_device = kind == cudaMemcpyHostToDevice;
    bool direct = false;
    for (const CopyList::Copy& c : copies.list) {
        HostStage* st;
        if (int rc = stage_for(ctx, c.host, c.bytes, kind, &st)) return rc;
        if (st) {
            if (int rc = staged_copy(ctx, *st, c.dev, c.host, c.bytes, to_device)) return rc;
        } else {
            CK(cudaMemcpyAsync(to_device ? c.dev : c.host, to_device ? c.host : c.dev, c.bytes, kind, stream));
            direct = true;
        }
    }
    if (direct) CK(cudaStreamSynchronize(stream));
    return 0;
}

// The frame of every blocking host entry: the caller's buffers `in` to the device, then device(&out), which runs the device
// drivers (they return with their work complete) and adds the call's outputs to `out`, then `out` to the caller's buffers.
// st (nullable) gets the host-clock time of each direction's copies in h2d_ms and d2h_ms.
template <typename Device>
int run_blocking(dark_bwt_ctx* ctx, const CopyList& in, dark_bwt_stats* st, Device device) {
    typedef std::chrono::steady_clock Clock;
    auto ms_since = [](Clock::time_point t0) { return std::chrono::duration<float, std::milli>(Clock::now() - t0).count(); };
    CK(cudaSetDevice(ctx->device));
    Clock::time_point t0 = Clock::now();
    if (int rc = copy_blocking(ctx, in, cudaMemcpyHostToDevice, ctx->stream)) return rc;
    if (st) st->h2d_ms = ms_since(t0);
    CopyList out;
    if (int rc = device(&out)) return rc;
    t0 = Clock::now();
    if (int rc = copy_blocking(ctx, out, cudaMemcpyDeviceToHost, ctx->stream)) return rc;
    if (st) st->d2h_ms = ms_since(t0);
    return DARK_BWT_OK;
}

// A block's distance-coding outputs, where dc_device left them in `io`, to the caller's host arrays (each nullable): the
// distances (n entries) and the four item arrays (`items` entries).
void add_dc_outputs(CopyList* out, const DcBuffers& io, u64 n, u64 items, uint32_t* dist, uint32_t* item_pos,
                    uint32_t* item_dist, uint8_t* item_sym, uint8_t* item_rank) {
    out->add(dist, io.dist, n * sizeof(u32));
    out->add(item_pos, io.item_pos, items * sizeof(u32));
    out->add(item_dist, io.item_dist, items * sizeof(u32));
    out->add(item_sym, io.item_sym, items);
    out->add(item_rank, io.item_rank, items);
}

// The pipelined loop of the batch entries: `count` host blocks ins[k] (ns[k] bytes).  While block k is transformed
// (transform(k, b, d_in[b], &copies), synchronous on the context's stream; b = k & 1 selects the block's device buffers),
// block k+1 is copied into the other input buffer and the copies of block k-1 run out of the other buffers.  Pinned host
// buffers ride on the two copy streams; a list with a staged copy (stage_for) is sent by a helper thread through
// copy_blocking.  A context with one staging pair (pipeline_depth 1: above 2^31) has only b = 0: the copy-in of block k+1
// starts once transform k has returned and the copies of block k have drained.
template <typename Transform>
int run_pipelined(dark_bwt_ctx* ctx, const u8* const* ins, const uint64_t* ns, uint64_t count, u8* const d_in[2], Transform transform) {
    bool comp_recorded[2] = {false, false}, out_recorded[2] = {false, false};
    std::future<int> fin[2], fout;
    auto start_in = [&](uint64_t k, int buf) -> int {  // the transform that read d_in[buf] has returned (it is synchronous)
        HostStage* st;
        if (int rc = stage_for(ctx, ins[k], ns[k], cudaMemcpyHostToDevice, &st)) return rc;
        if (st) {
            fin[buf] = std::async(std::launch::async, [ctx, st, dst = d_in[buf], src = ins[k], bytes = ns[k]] {
                return staged_copy(ctx, *st, dst, (void*)src, bytes, true);
            });
            return 0;
        }
        if (comp_recorded[buf]) CK(cudaStreamWaitEvent(ctx->copy_in, ctx->ev_comp[buf], 0));
        CK(cudaMemcpyAsync(d_in[buf], ins[k], ns[k], cudaMemcpyHostToDevice, ctx->copy_in));
        CK(cudaEventRecord(ctx->ev_in[buf], ctx->copy_in));
        return 0;
    };
    auto drain = [&]() {  // never leave a helper thread or a copy behind: on an error, the blocks before it are complete
        int rc = 0;
        for (int i = 0; i < 2; ++i)
            if (fin[i].valid()) rc |= fin[i].get();
        if (fout.valid()) rc |= fout.get();
        cudaStreamSynchronize(ctx->copy_out);
        cudaStreamSynchronize(ctx->copy_in);
        return rc;
    };
    const uint64_t depth = (uint64_t)ctx->pipeline_depth;
    if (int rc = start_in(0, 0)) return rc;
    for (uint64_t k = 0; k < count; ++k) {
        const int b = (int)(k % depth), nb = (int)((k + 1) % depth);
        if (fin[b].valid()) {
            if (int rc = fin[b].get()) { drain(); return rc; }
        } else {
            CK(cudaStreamWaitEvent(ctx->stream, ctx->ev_in[b], 0));
        }
        if (depth == 2 && k + 1 < count)
            if (int rc = start_in(k + 1, nb)) { drain(); return rc; }
        // (a staged copy-out of block k-1 may still be reading the OTHER buffers; these were drained before it began)
        if (out_recorded[b]) CK(cudaStreamWaitEvent(ctx->stream, ctx->ev_out[b], 0));  // output buffers b drained
        CopyList oc;
        int rc = transform(k, b, (const u8*)d_in[b], &oc);
        if (rc) { drain(); return rc; }
        if (depth == 1) oc.serial = true;
        CK(cudaEventRecord(ctx->ev_comp[b], ctx->stream));
        comp_recorded[b] = true;
        if (fout.valid())
            if (int rc2 = fout.get()) { drain(); return rc2; }  // one staged copy-out at a time (they share the lanes)
        HostStage* staged = nullptr;  // one staged copy sends the whole list to the helper thread
        for (size_t i = 0; i < oc.list.size() && !staged; ++i)
            if (int rc2 = stage_for(ctx, oc.list[i].host, oc.list[i].bytes, cudaMemcpyDeviceToHost, &staged)) { drain(); return rc2; }
        if (staged) {
            fout = std::async(std::launch::async, [ctx, oc] {
                if (cudaSetDevice(ctx->device) != cudaSuccess) return ctx->fail_cuda(cudaGetLastError(), "helper thread device", __LINE__);
                return copy_blocking(ctx, oc, cudaMemcpyDeviceToHost, ctx->copy_out);
            });
            if (oc.serial)
                if (int rc2 = fout.get()) { drain(); return rc2; }
            out_recorded[b] = false;
        } else {
            CK(cudaStreamWaitEvent(ctx->copy_out, ctx->ev_comp[b], 0));
            for (const CopyList::Copy& c : oc.list)
                CK(cudaMemcpyAsync(c.host, c.dev, c.bytes, cudaMemcpyDeviceToHost, ctx->copy_out));
            if (oc.serial) CK(cudaStreamSynchronize(ctx->copy_out));
            CK(cudaEventRecord(ctx->ev_out[b], ctx->copy_out));
            out_recorded[b] = true;
        }
        if (depth == 1 && k + 1 < count)
            if (int rc2 = start_in(k + 1, nb)) { drain(); return rc2; }
    }
    if (int rc = drain()) return rc;
    CK(cudaStreamSynchronize(ctx->copy_out));
    CK(cudaStreamSynchronize(ctx->copy_in));
    return DARK_BWT_OK;
}

// The arguments dark_bwt_create_ex checks before it looks for a device, in its order: DARK_BWT_OK or the code it returns.
int check_create_args(uint64_t max_n, uint32_t flags) {
    if (flags & ~(DARK_BWT_F_NO_ALPHABET_PACKING | DARK_BWT_F_DEVICE_ONLY | DARK_BWT_F_DC_BATCH)) return DARK_BWT_E_INVALID_ARG;
    // the DC batch is a host-buffer entry: it needs the staging a device-only context does not have
    if ((flags & DARK_BWT_F_DC_BATCH) && (flags & DARK_BWT_F_DEVICE_ONLY)) return DARK_BWT_E_INVALID_ARG;
    if (max_n < 2 || max_n > 0xFFFFFFFEull) return DARK_BWT_E_INVALID_N;
    return DARK_BWT_OK;
}

// The arena of a context of ctx->capacity and ctx->flags (checked): every device buffer, carved in one order.  Returns the
// arena's bytes.  With ctx->arena null it only sizes (dark_bwt_arena_bytes, and create before its cudaMalloc); with the
// allocation it also points the context's buffers into it.
size_t carve_arena(dark_bwt_ctx* ctx) {
    const size_t N = (size_t)ctx->capacity;
    const bool staging = !(ctx->flags & DARK_BWT_F_DEVICE_ONLY);
    const bool dc_batch = ctx->flags & DARK_BWT_F_DC_BATCH;
    // Above 2^31 the second pair (2 N bytes) is what keeps a context of 2^32 - 2 inside a B200: the batch entries then run
    // their blocks one after another through one pair.  The DC batch keeps two pairs: its output slots pair with them.
    ctx->pipeline_depth = !staging ? 0 : (ctx->capacity > (1ull << 31) && !dc_batch) ? 1 : 2;
    ctx->scan_tiles = ceil_div(N, std::min(kScanTile, 4096));  // the pairs kernel and the text-order builder scan 4,096-suffix tiles

    char* const base = (char*)ctx->arena;
    size_t off = 0;
    auto carve = [&](auto& ptr, size_t bytes) {
        if (base) ptr = (std::remove_reference_t<decltype(ptr)>)(base + off);
        off = align_up(off + bytes, 256);
    };
    for (u64*& k : ctx->keys) carve(k, N * 8 + 1024);  // slack: pair lists are split at a 64-aligned offset
    for (u32*& i : ctx->ids) carve(i, N * 4 + 16);
    carve(ctx->ranks, N * 4 + 16), carve(ctx->ranks_alt, N * 4 + 16), carve(ctx->isa, N * 4 + 16), carve(ctx->sa, N * 4 + 16);
    if (staging) carve(ctx->d_text, N + 16), carve(ctx->d_bwt, N + 16);  // host-entry staging
    if (ctx->pipeline_depth == 2) carve(ctx->d_text2, N + 16), carve(ctx->d_bwt2, N + 16);
    else ctx->d_text2 = ctx->d_text, ctx->d_bwt2 = ctx->d_bwt;  // one pair (or none)
    carve(ctx->hist, sizeof(u32) * kMaxPasses * kRadix);
    carve(ctx->present, sizeof(u32) * 256);
    carve(ctx->lut, 256);
    carve(ctx->bad, sizeof(unsigned long long));
    const size_t status_bytes = (ceil_div(N, kSortTile) + 128) * kRadix * sizeof(u64);  // + rows the scanner CTA reads ahead
    void* status = nullptr;
    carve(status, status_bytes);
    ctx->status.init(status, status_bytes);
    carve(ctx->counters, sizeof(u32) * kMaxCounters);
    carve(ctx->bucket_hist, sizeof(u32) * 1280);  // 256 bucket counters/cursors + 257 chunk prefixes; DC: first/last occurrences + dense alphabet
    carve(ctx->bitmap, sizeof(u32) * (ceil_div(N, 32) + 1) + 1024);  // + one tile of flag bytes past the end
    carve(ctx->scan_words, sizeof(u64) * kScanWordsPerTile * ctx->scan_tiles);
    carve(ctx->many_starts, sizeof(u32) * (kMaxManyBlocks + 1));
    carve(ctx->many_origins, sizeof(unsigned long long) * kMaxManyBlocks);
    carve(ctx->many_lut, sizeof(u16) * 256);
    carve(ctx->dc_info, sizeof(DcInfoDev) + 16);
    if (dc_batch)
        for (DcBuffers& s : ctx->dc_slot) {
            carve(s.dist, N * 4 + 16), carve(s.item_pos, N * 4 + 16), carve(s.item_dist, N * 4 + 16);
            carve(s.item_sym, N + 16), carve(s.item_rank, N + 16);
        }
    return off;
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

uint64_t dark_bwt_arena_bytes(uint64_t max_n, uint32_t flags) {
    if (check_create_args(max_n, flags) != DARK_BWT_OK) return 0;
    dark_bwt_ctx sizing;
    sizing.capacity = max_n;
    sizing.flags = flags;
    return carve_arena(&sizing);
}

int dark_bwt_create(uint64_t max_n, int device, dark_bwt_ctx** out) {
    return dark_bwt_create_ex(max_n, device, DARK_BWT_F_DEFAULT, out);
}

int dark_bwt_create_ex(uint64_t max_n, int device, uint32_t flags, dark_bwt_ctx** out) {
    if (!out) return DARK_BWT_E_INVALID_ARG;
    *out = nullptr;
    if (int rc = check_create_args(max_n, flags)) return rc;
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

    ctx->arena_bytes = carve_arena(ctx);
    auto bail = [&](int code) {
        dark_bwt_destroy(ctx);
        return code;
    };
    if (cudaMalloc(&ctx->arena, ctx->arena_bytes) != cudaSuccess) {
        cudaGetLastError();
        ctx->arena = nullptr;
        return bail(DARK_BWT_E_NOMEM);
    }
    carve_arena(ctx);

    if (cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking) != cudaSuccess) return bail(DARK_BWT_E_CUDA);
    if (!(flags & DARK_BWT_F_DEVICE_ONLY)) {
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
    ctx->call_start = ctx->events[kMaxEvents - 1];
    ctx->call_stop = ctx->events[kMaxEvents - 2];
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
    if (int rc = check_n(ctx, n, 2)) return rc;
    ctx->err[0] = 0;
    if (stats) stats->h2d_ms = 0.f;
    return forward_device(ctx, d_text, (u32)n, d_bwt_out, origin_out, d_sa_out, stats);
}

int dark_bwt_forward(dark_bwt_ctx* ctx, const uint8_t* text, uint64_t n, uint8_t* bwt_out, uint64_t* origin_out,
                     uint32_t* sa_out, dark_bwt_stats* stats) {
    if (!ctx || !text || !bwt_out || !origin_out) return DARK_BWT_E_INVALID_ARG;
    if (int rc = check_staging(ctx)) return rc;
    if (int rc = check_n(ctx, n, 2)) return rc;
    ctx->err[0] = 0;
    return run_blocking(ctx, CopyList().add(text, ctx->d_text, n), stats, [&](CopyList* out) {
        if (int rc = forward_device(ctx, ctx->d_text, (u32)n, ctx->d_bwt, origin_out, nullptr, stats)) return rc;
        out->add(bwt_out, ctx->d_bwt, n);
        out->add(sa_out, ctx->sa, n * sizeof(u32));
        return 0;
    });
}

int dark_bwt_forward_batch(dark_bwt_ctx* ctx, const uint8_t* const* texts, const uint64_t* ns, uint8_t* const* bwt_outs,
                           uint64_t* origins_out, uint32_t* const* sa_outs, uint64_t count, dark_bwt_stats* stats) {
    if (!ctx || !texts || !ns || !bwt_outs || !origins_out) return DARK_BWT_E_INVALID_ARG;
    if (int rc = check_staging(ctx)) return rc;
    ctx->err[0] = 0;
    for (uint64_t k = 0; k < count; ++k) {
        if (!texts[k] || !bwt_outs[k]) return DARK_BWT_E_INVALID_ARG;
        if (int rc = check_n(ctx, ns[k], 2)) return rc;
    }
    if (count == 0) return DARK_BWT_OK;
    CK(cudaSetDevice(ctx->device));
    u8* const d_text[2] = {ctx->d_text, ctx->d_text2};
    u8* const d_bwt[2] = {ctx->d_bwt, ctx->d_bwt2};
    return run_pipelined(ctx, texts, ns, count, d_text, [&](uint64_t k, int b, const u8* din, CopyList* out) {
        dark_bwt_stats* st = stats ? stats + k : nullptr;
        if (st) st->h2d_ms = 0.f;
        if (int rc = forward_device(ctx, din, (u32)ns[k], d_bwt[b], origins_out + k, nullptr, st)) return rc;
        out->add(bwt_outs[k], d_bwt[b], ns[k]);
        if (sa_outs && sa_outs[k]) {  // the SA of the block is in the context's single SA buffer
            out->add(sa_outs[k], ctx->sa, ns[k] * sizeof(u32));
            out->serial = true;
        }
        return 0;
    });
}

int dark_bwt_inverse_batch(dark_bwt_ctx* ctx, const uint8_t* const* bwts, const uint64_t* ns, const uint64_t* origins,
                           uint8_t* const* text_outs, uint64_t count, float* ms_out) {
    if (!ctx || !bwts || !ns || !origins || !text_outs) return DARK_BWT_E_INVALID_ARG;
    if (int rc = check_staging(ctx)) return rc;
    ctx->err[0] = 0;
    for (uint64_t k = 0; k < count; ++k) {
        if (!bwts[k] || !text_outs[k]) return DARK_BWT_E_INVALID_ARG;
        if (int rc = check_n(ctx, ns[k], 1)) return rc;
        if (origins[k] >= ns[k]) return DARK_BWT_E_INVALID_ARG;
    }
    if (count == 0) return DARK_BWT_OK;
    CK(cudaSetDevice(ctx->device));
    u8* const d_bwt[2] = {ctx->d_bwt, ctx->d_bwt2};
    u8* const d_text[2] = {ctx->d_text, ctx->d_text2};
    return run_pipelined(ctx, bwts, ns, count, d_bwt, [&](uint64_t k, int b, const u8* din, CopyList* out) {
        if (int rc = inverse_device(ctx, din, (u32)ns[k], (u32)origins[k], nullptr, d_text[b], ms_out ? ms_out + k : nullptr)) return rc;
        out->add(text_outs[k], d_text[b], ns[k]);
        return 0;
    });
}

int dark_bwt_forward_many(dark_bwt_ctx* ctx, const uint8_t* const* texts, const uint64_t* ns, uint8_t* const* bwt_outs,
                          uint64_t* origins_out, uint64_t count, dark_bwt_stats* stats) {
    if (!ctx || !texts || !ns || !bwt_outs || !origins_out) return DARK_BWT_E_INVALID_ARG;
    if (int rc = check_staging(ctx)) return rc;
    ctx->err[0] = 0;
    if (count == 0) return DARK_BWT_OK;
    BlockList bl;
    if (int rc = check_blocks(ctx, count, ns, nullptr, nullptr, 2, 0, texts, bwt_outs, &bl)) return rc;
    return run_blocking(ctx, CopyList().add_blocks(bl, texts, ctx->d_text), stats, [&](CopyList* out) {
        if (int rc = load_blocks(ctx, bl)) return rc;
        if (int rc = forward_many_device(ctx, ctx->d_text, bl.total(), bl.count(), ctx->d_bwt, nullptr, stats)) return rc;
        out->add_blocks(bl, bwt_outs, ctx->d_bwt);
        out->add(origins_out, ctx->many_origins, sizeof(uint64_t) * count);
        return 0;
    });
}

int dark_bwt_forward_many_device(dark_bwt_ctx* ctx, const uint8_t* d_text, const uint32_t* d_starts, uint64_t count,
                                 uint8_t* d_bwt_out, uint64_t* d_origins_out, uint32_t* d_sa_out, dark_bwt_stats* stats) {
    if (!ctx || !d_text || !d_starts || !d_bwt_out || !d_origins_out) return DARK_BWT_E_INVALID_ARG;
    ctx->err[0] = 0;
    if (count == 0) return DARK_BWT_OK;
    BlockList bl;
    if (int rc = check_blocks(ctx, count, nullptr, d_starts, nullptr, 2, 0, nullptr, nullptr, &bl)) return rc;
    if (int rc = load_blocks(ctx, bl)) return rc;
    if (stats) stats->h2d_ms = 0.f;
    if (int rc = forward_many_device(ctx, d_text, bl.total(), bl.count(), d_bwt_out, d_sa_out, stats)) return rc;
    CK(cudaMemcpyAsync(d_origins_out, ctx->many_origins, sizeof(uint64_t) * count, cudaMemcpyDeviceToDevice, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    return DARK_BWT_OK;
}

int dark_bwt_inverse_device(dark_bwt_ctx* ctx, const uint8_t* d_bwt, uint64_t n, uint64_t origin, uint8_t* d_text_out,
                            float* ms_out) {
    if (!ctx || !d_bwt || !d_text_out) return DARK_BWT_E_INVALID_ARG;
    if (int rc = check_n(ctx, n, 1)) return rc;
    if (origin >= n) return DARK_BWT_E_INVALID_ARG;
    ctx->err[0] = 0;
    return inverse_device(ctx, d_bwt, (u32)n, (u32)origin, nullptr, d_text_out, ms_out);
}

int dark_bwt_inverse(dark_bwt_ctx* ctx, const uint8_t* bwt, uint64_t n, uint64_t origin, uint8_t* text_out) {
    if (!ctx || !bwt || !text_out) return DARK_BWT_E_INVALID_ARG;
    if (int rc = check_staging(ctx)) return rc;
    if (int rc = check_n(ctx, n, 1)) return rc;
    if (origin >= n) return DARK_BWT_E_INVALID_ARG;
    ctx->err[0] = 0;
    return run_blocking(ctx, CopyList().add(bwt, ctx->d_bwt, n), nullptr, [&](CopyList* out) {
        if (int rc = inverse_device(ctx, ctx->d_bwt, (u32)n, (u32)origin, nullptr, ctx->d_text, nullptr)) return rc;
        out->add(text_out, ctx->d_text, n);
        return 0;
    });
}

int dark_bwt_inverse_many(dark_bwt_ctx* ctx, const uint8_t* const* bwts, const uint64_t* ns, const uint64_t* origins,
                          uint8_t* const* text_outs, uint64_t count, float* ms_out) {
    if (!ctx || !bwts || !ns || !origins || !text_outs) return DARK_BWT_E_INVALID_ARG;
    if (int rc = check_staging(ctx)) return rc;
    ctx->err[0] = 0;
    if (count == 0) return DARK_BWT_OK;
    BlockList bl;
    if (int rc = check_blocks(ctx, count, ns, nullptr, origins, 1, 1, bwts, text_outs, &bl)) return rc;
    return run_blocking(ctx, CopyList().add_blocks(bl, bwts, ctx->d_bwt), nullptr, [&](CopyList* out) {
        if (int rc = load_blocks(ctx, bl)) return rc;
        if (int rc = inverse_device(ctx, ctx->d_bwt, bl.total(), 0, &bl, ctx->d_text, ms_out)) return rc;
        out->add_blocks(bl, text_outs, ctx->d_text);
        return 0;
    });
}

int dark_bwt_inverse_many_device(dark_bwt_ctx* ctx, const uint8_t* d_bwt, const uint32_t* d_starts, const uint64_t* d_origins,
                                 uint64_t count, uint8_t* d_text_out, float* ms_out) {
    if (!ctx || !d_bwt || !d_starts || !d_origins || !d_text_out) return DARK_BWT_E_INVALID_ARG;
    ctx->err[0] = 0;
    if (count == 0) return DARK_BWT_OK;
    BlockList bl;
    if (int rc = check_blocks(ctx, count, nullptr, d_starts, d_origins, 1, 1, nullptr, nullptr, &bl)) return rc;
    if (int rc = load_blocks(ctx, bl)) return rc;
    return inverse_device(ctx, d_bwt, bl.total(), 0, &bl, d_text_out, ms_out);
}

int dark_bwt_dc_encode_device(dark_bwt_ctx* ctx, const uint8_t* d_bwt, uint64_t n, uint32_t* d_dist_out, uint32_t* d_item_pos,
                              uint32_t* d_item_dist, uint8_t* d_item_sym, uint8_t* d_item_rank, dark_bwt_dc_info* info) {
    if (!ctx || !d_bwt || !info) return DARK_BWT_E_INVALID_ARG;
    if (int rc = check_n(ctx, n, 1)) return rc;
    ctx->err[0] = 0;
    DcBuffers io{d_dist_out, d_item_pos, d_item_dist, d_item_sym, d_item_rank};
    return dc_device(ctx, d_bwt, (u32)n, nullptr, &io, info, nullptr);
}

int dark_bwt_dc_encode(dark_bwt_ctx* ctx, const uint8_t* bwt, uint64_t n, uint32_t* dist_out, uint32_t* item_pos, uint32_t* item_dist,
                       uint8_t* item_sym, uint8_t* item_rank, dark_bwt_dc_info* info) {
    if (!ctx || !bwt || !info) return DARK_BWT_E_INVALID_ARG;
    if (int rc = check_staging(ctx)) return rc;
    if (int rc = check_n(ctx, n, 1)) return rc;
    ctx->err[0] = 0;
    return run_blocking(ctx, CopyList().add(bwt, ctx->d_bwt, n), nullptr, [&](CopyList* out) {
        DcBuffers io;
        if (int rc = dc_device(ctx, ctx->d_bwt, (u32)n, nullptr, &io, info, nullptr)) return rc;
        add_dc_outputs(out, io, n, info->num_items, dist_out, item_pos, item_dist, item_sym, item_rank);
        return 0;
    });
}

int dark_bwt_forward_dc(dark_bwt_ctx* ctx, const uint8_t* text, uint64_t n, uint8_t* bwt_out, uint64_t* origin_out, uint32_t* dist_out,
                        uint32_t* item_pos, uint32_t* item_dist, uint8_t* item_sym, uint8_t* item_rank, dark_bwt_dc_info* info,
                        dark_bwt_stats* stats) {
    if (!ctx || !text || !origin_out || !info) return DARK_BWT_E_INVALID_ARG;
    if (int rc = check_staging(ctx)) return rc;
    if (int rc = check_n(ctx, n, 2)) return rc;
    ctx->err[0] = 0;
    return run_blocking(ctx, CopyList().add(text, ctx->d_text, n), stats, [&](CopyList* out) {
        if (int rc = forward_device(ctx, ctx->d_text, (u32)n, ctx->d_bwt, origin_out, nullptr, stats)) return rc;
        DcBuffers io;
        if (int rc = dc_device(ctx, ctx->d_bwt, (u32)n, nullptr, &io, info, nullptr)) return rc;
        out->add(bwt_out, ctx->d_bwt, n);
        add_dc_outputs(out, io, n, info->num_items, dist_out, item_pos, item_dist, item_sym, item_rank);
        return 0;
    });
}

int dark_bwt_forward_dc_batch(dark_bwt_ctx* ctx, const uint8_t* const* texts, const uint64_t* ns, uint64_t count, uint8_t* const* bwt_outs,
                              uint64_t* origins_out, uint32_t* const* dist_outs, uint32_t* const* item_pos, uint32_t* const* item_dist,
                              uint8_t* const* item_sym, uint8_t* const* item_rank, dark_bwt_dc_info* infos, dark_bwt_stats* stats) {
    if (!ctx || !texts || !ns || !origins_out || !infos) return DARK_BWT_E_INVALID_ARG;
    if (int rc = check_staging(ctx)) return rc;
    if (!(ctx->flags & DARK_BWT_F_DC_BATCH)) return DARK_BWT_E_INVALID_ARG;  // no DC output slots
    ctx->err[0] = 0;
    for (uint64_t k = 0; k < count; ++k) {
        if (!texts[k]) return DARK_BWT_E_INVALID_ARG;
        if (int rc = check_n(ctx, ns[k], 2)) return rc;
    }
    if (count == 0) return DARK_BWT_OK;
    CK(cudaSetDevice(ctx->device));
    u8* const d_text[2] = {ctx->d_text, ctx->d_text2};
    u8* const d_bwt[2] = {ctx->d_bwt, ctx->d_bwt2};
    // Block k: the forward into d_bwt[b], then distance coding of it into slot b (b = k & 1).  Its scratch (run starts,
    // tables, run counts, the status buffer a small block borrows) is consumed before block k+1's forward starts on the
    // same stream; what the copies read stays untouched until the wait on ev_out[b] before block k+2.
    return run_pipelined(ctx, texts, ns, count, d_text, [&](uint64_t k, int b, const u8* din, CopyList* out) {
        const u64 n = ns[k];
        dark_bwt_stats* st = stats ? stats + k : nullptr;
        if (st) st->h2d_ms = 0.f;
        if (int rc = forward_device(ctx, din, (u32)n, d_bwt[b], origins_out + k, nullptr, st)) return rc;
        DcBuffers io = ctx->dc_slot[b];
        if (int rc = dc_device(ctx, d_bwt[b], (u32)n, nullptr, &io, infos + k, nullptr)) return rc;
        out->add(bwt_outs ? bwt_outs[k] : nullptr, d_bwt[b], n);
        add_dc_outputs(out, io, n, infos[k].num_items, dist_outs ? dist_outs[k] : nullptr, item_pos ? item_pos[k] : nullptr,
                       item_dist ? item_dist[k] : nullptr, item_sym ? item_sym[k] : nullptr, item_rank ? item_rank[k] : nullptr);
        return 0;
    });
}

int dark_bwt_dc_encode_packed_device(dark_bwt_ctx* ctx, const uint8_t* d_bwt, uint64_t n, uint8_t* d_stream_out, uint64_t stream_capacity,
                                     uint64_t* stream_bytes_out, dark_bwt_dc_info* info) {
    if (!ctx || !d_bwt || !d_stream_out || !stream_bytes_out || !info) return DARK_BWT_E_INVALID_ARG;
    if (int rc = check_n(ctx, n, 1)) return rc;
    ctx->err[0] = 0;
    DcBuffers io;
    if (int rc = dc_device(ctx, d_bwt, (u32)n, nullptr, &io, info, nullptr)) return rc;
    return dc_pack(ctx, io, info->num_items, d_stream_out, stream_capacity, stream_bytes_out, &info->device_ms);
}

int dark_bwt_forward_dc_packed(dark_bwt_ctx* ctx, const uint8_t* text, uint64_t n, uint8_t* bwt_out, uint64_t* origin_out, uint8_t* stream_out,
                               uint64_t stream_capacity, uint64_t* stream_bytes_out, dark_bwt_dc_info* info, dark_bwt_stats* stats) {
    if (!ctx || !text || !origin_out || !stream_out || !stream_bytes_out || !info) return DARK_BWT_E_INVALID_ARG;
    if (int rc = check_staging(ctx)) return rc;
    if (int rc = check_n(ctx, n, 2)) return rc;
    ctx->err[0] = 0;
    return run_blocking(ctx, CopyList().add(text, ctx->d_text, n), stats, [&](CopyList* out) {
        if (int rc = forward_device(ctx, ctx->d_text, (u32)n, ctx->d_bwt, origin_out, nullptr, stats)) return rc;
        DcBuffers io;
        if (int rc = dc_device(ctx, ctx->d_bwt, (u32)n, nullptr, &io, info, nullptr)) return rc;
        // the sort's second key buffer (8 N + 1 KiB), which single-block distance coding leaves free, holds any stream (<= 8 n)
        u8* const d_stream = (u8*)ctx->keys[1];
        if (int rc = dc_pack(ctx, io, info->num_items, d_stream, stream_capacity, stream_bytes_out, &info->device_ms)) return rc;
        out->add(bwt_out, ctx->d_bwt, n);
        out->add(stream_out, d_stream, *stream_bytes_out);
        return 0;
    });
}

int dark_bwt_forward_dc_packed_batch(dark_bwt_ctx* ctx, const uint8_t* const* texts, const uint64_t* ns, uint64_t count,
                                     uint8_t* const* bwt_outs, uint64_t* origins_out, uint8_t* const* stream_outs,
                                     const uint64_t* stream_capacities, uint64_t* stream_bytes_out, dark_bwt_dc_info* infos,
                                     dark_bwt_stats* stats) {
    if (!ctx || !texts || !ns || !origins_out || !stream_outs || !stream_capacities || !stream_bytes_out || !infos)
        return DARK_BWT_E_INVALID_ARG;
    if (int rc = check_staging(ctx)) return rc;
    if (!(ctx->flags & DARK_BWT_F_DC_BATCH)) return DARK_BWT_E_INVALID_ARG;  // no DC output slots
    ctx->err[0] = 0;
    for (uint64_t k = 0; k < count; ++k) {
        if (!texts[k] || !stream_outs[k]) return DARK_BWT_E_INVALID_ARG;
        if (int rc = check_n(ctx, ns[k], 2)) return rc;
    }
    if (count == 0) return DARK_BWT_OK;
    CK(cudaSetDevice(ctx->device));
    u8* const d_text[2] = {ctx->d_text, ctx->d_text2};
    u8* const d_bwt[2] = {ctx->d_bwt, ctx->d_bwt2};
    // Block k: the forward into d_bwt[b], distance coding into the context's scratch as in the single call, and the pack into
    // slot b (b = k & 1): its dist and item_pos arrays, carved back to back, are 8 N + 32 bytes or more, room for any stream.
    // The scratch is consumed before block k+1's forward starts on the same stream; what the copies read stays untouched
    // until the wait on ev_out[b] before block k+2.
    return run_pipelined(ctx, texts, ns, count, d_text, [&](uint64_t k, int b, const u8* din, CopyList* out) {
        const u64 n = ns[k];
        dark_bwt_stats* st = stats ? stats + k : nullptr;
        if (st) st->h2d_ms = 0.f;
        if (int rc = forward_device(ctx, din, (u32)n, d_bwt[b], origins_out + k, nullptr, st)) return rc;
        DcBuffers io;
        if (int rc = dc_device(ctx, d_bwt[b], (u32)n, nullptr, &io, infos + k, nullptr)) return rc;
        u8* const d_stream = (u8*)ctx->dc_slot[b].dist;
        if (int rc = dc_pack(ctx, io, infos[k].num_items, d_stream, stream_capacities[k], stream_bytes_out + k, &infos[k].device_ms)) {
            if (rc == DARK_BWT_E_INVALID_ARG) {
                char what[sizeof(ctx->err)];
                memcpy(what, ctx->err, sizeof(what));
                snprintf(ctx->err, sizeof(ctx->err), "block %llu: %.280s", (unsigned long long)k, what);
            }
            return rc;
        }
        out->add(stream_outs[k], d_stream, stream_bytes_out[k]);
        out->add(bwt_outs ? bwt_outs[k] : nullptr, d_bwt[b], n);
        return 0;
    });
}

int dark_bwt_dc_decode_packed_device(dark_bwt_ctx* ctx, const uint8_t* d_stream, uint64_t stream_bytes, uint64_t n, uint8_t* d_bwt_out,
                                     dark_bwt_dc_info* info) {
    if (!ctx || !d_stream || !d_bwt_out) return DARK_BWT_E_INVALID_ARG;
    if (int rc = check_decode_args(ctx, stream_bytes, n)) return rc;
    ctx->err[0] = 0;
    dark_bwt_dc_info local;
    return dc_decode(ctx, d_stream, stream_bytes, (u32)n, d_bwt_out, info ? info : &local);
}

int dark_bwt_inverse_dc_packed(dark_bwt_ctx* ctx, const uint8_t* stream, uint64_t stream_bytes, uint64_t n, uint64_t origin,
                               uint8_t* text_out, uint8_t* bwt_out, dark_bwt_dc_info* info) {
    if (!ctx || !stream || !text_out) return DARK_BWT_E_INVALID_ARG;
    if (int rc = check_staging(ctx)) return rc;
    if (int rc = check_decode_args(ctx, stream_bytes, n)) return rc;
    if (origin >= n) return DARK_BWT_E_INVALID_ARG;
    ctx->err[0] = 0;
    dark_bwt_dc_info local;
    // the stream goes to the sort's second key buffer (8 N + 1 KiB >= 8 n), the block to d_bwt, which the inverse reads
    u8* const d_stream = (u8*)ctx->keys[1];
    return run_blocking(ctx, CopyList().add(stream, d_stream, stream_bytes), nullptr, [&](CopyList* out) {
        if (int rc = dc_decode(ctx, d_stream, stream_bytes, (u32)n, ctx->d_bwt, info ? info : &local)) return rc;
        if (int rc = inverse_device(ctx, ctx->d_bwt, (u32)n, (u32)origin, nullptr, ctx->d_text, nullptr)) return rc;
        out->add(text_out, ctx->d_text, n);
        out->add(bwt_out, ctx->d_bwt, n);
        return 0;
    });
}

int dark_bwt_dc_encode_many_device(dark_bwt_ctx* ctx, const uint8_t* d_bwt, const uint32_t* d_starts, uint64_t count, uint32_t* d_dist_out,
                                   uint32_t* d_item_starts, uint32_t* d_item_pos, uint32_t* d_item_dist, uint8_t* d_item_sym,
                                   uint8_t* d_item_rank, dark_bwt_dc_info* infos, float* ms_out) {
    if (!ctx || !d_bwt || !d_starts || !infos) return DARK_BWT_E_INVALID_ARG;
    ctx->err[0] = 0;
    if (count == 0) return DARK_BWT_OK;
    BlockList bl;
    if (int rc = check_blocks(ctx, count, nullptr, d_starts, nullptr, 1, 0, nullptr, nullptr, &bl)) return rc;
    if (!dc_many_records_fit(ctx, count)) return DARK_BWT_E_INVALID_N;
    if (int rc = load_blocks(ctx, bl)) return rc;
    DcBuffers io{d_dist_out, d_item_pos, d_item_dist, d_item_sym, d_item_rank, d_item_starts};
    std::vector<u32> starts;
    if (int rc = dc_device(ctx, d_bwt, bl.total(), &bl, &io, infos, &starts)) return rc;
    if (ms_out) *ms_out = infos[0].device_ms;
    return DARK_BWT_OK;
}

int dark_bwt_dc_encode_many(dark_bwt_ctx* ctx, const uint8_t* const* bwts, const uint64_t* ns, uint64_t count, uint32_t* dist_out,
                            uint32_t* item_starts, uint32_t* item_pos, uint32_t* item_dist, uint8_t* item_sym, uint8_t* item_rank,
                            dark_bwt_dc_info* infos, float* ms_out) {
    if (!ctx || !bwts || !ns || !infos) return DARK_BWT_E_INVALID_ARG;
    if (int rc = check_staging(ctx)) return rc;
    ctx->err[0] = 0;
    if (count == 0) {
        if (item_starts) item_starts[0] = 0;
        return DARK_BWT_OK;
    }
    BlockList bl;
    if (int rc = check_blocks(ctx, count, ns, nullptr, nullptr, 1, 0, bwts, nullptr, &bl)) return rc;
    if (!dc_many_records_fit(ctx, count)) return DARK_BWT_E_INVALID_N;
    return run_blocking(ctx, CopyList().add_blocks(bl, bwts, ctx->d_bwt), nullptr, [&](CopyList* out) {
        if (int rc = load_blocks(ctx, bl)) return rc;
        DcBuffers io;
        std::vector<u32> starts;
        if (int rc = dc_device(ctx, ctx->d_bwt, bl.total(), &bl, &io, infos, &starts)) return rc;
        if (ms_out) *ms_out = infos[0].device_ms;
        if (item_starts) memcpy(item_starts, starts.data(), starts.size() * sizeof(u32));
        add_dc_outputs(out, io, bl.total(), starts.back(), dist_out, item_pos, item_dist, item_sym, item_rank);
        return 0;
    });
}

int dark_bwt_forward_dc_many(dark_bwt_ctx* ctx, const uint8_t* const* texts, const uint64_t* ns, uint64_t count, uint8_t* const* bwt_outs,
                             uint64_t* origins_out, uint32_t* dist_out, uint32_t* item_starts, uint32_t* item_pos, uint32_t* item_dist,
                             uint8_t* item_sym, uint8_t* item_rank, dark_bwt_dc_info* infos, dark_bwt_stats* stats) {
    if (!ctx || !texts || !ns || !origins_out || !infos) return DARK_BWT_E_INVALID_ARG;
    if (int rc = check_staging(ctx)) return rc;
    ctx->err[0] = 0;
    if (count == 0) {
        if (item_starts) item_starts[0] = 0;
        return DARK_BWT_OK;
    }
    BlockList bl;
    if (int rc = check_blocks(ctx, count, ns, nullptr, nullptr, 2, 0, texts, nullptr, &bl)) return rc;
    if (!dc_many_records_fit(ctx, count)) return DARK_BWT_E_INVALID_N;
    return run_blocking(ctx, CopyList().add_blocks(bl, texts, ctx->d_text), stats, [&](CopyList* out) {
        if (int rc = load_blocks(ctx, bl)) return rc;
        if (int rc = forward_many_device(ctx, ctx->d_text, bl.total(), bl.count(), ctx->d_bwt, nullptr, stats)) return rc;
        DcBuffers io;
        std::vector<u32> starts;
        if (int rc = dc_device(ctx, ctx->d_bwt, bl.total(), &bl, &io, infos, &starts)) return rc;
        if (item_starts) memcpy(item_starts, starts.data(), starts.size() * sizeof(u32));
        out->add_blocks(bl, bwt_outs, ctx->d_bwt);
        out->add(origins_out, ctx->many_origins, sizeof(uint64_t) * count);
        add_dc_outputs(out, io, bl.total(), starts.back(), dist_out, item_pos, item_dist, item_sym, item_rank);
        return 0;
    });
}

int dark_bwt_dc_encode_packed_many_device(dark_bwt_ctx* ctx, const uint8_t* d_bwt, const uint32_t* d_starts, uint64_t count,
                                          uint8_t* d_stream_out, uint64_t stream_capacity, uint64_t* d_stream_starts,
                                          uint64_t* stream_bytes_out, dark_bwt_dc_info* infos, float* ms_out) {
    if (!ctx || !d_bwt || !d_starts || !d_stream_out || !d_stream_starts || !stream_bytes_out || !infos) return DARK_BWT_E_INVALID_ARG;
    ctx->err[0] = 0;
    if (count == 0) {
        *stream_bytes_out = 0;
        return DARK_BWT_OK;
    }
    BlockList bl;
    if (int rc = check_blocks(ctx, count, nullptr, d_starts, nullptr, 1, 0, nullptr, nullptr, &bl)) return rc;
    if (!dc_many_records_fit(ctx, count)) return DARK_BWT_E_INVALID_N;
    if (int rc = load_blocks(ctx, bl)) return rc;
    DcBuffers io;
    std::vector<u32> starts;
    if (int rc = dc_device(ctx, d_bwt, bl.total(), &bl, &io, infos, &starts)) return rc;
    return dc_pack_many(ctx, io, starts, d_stream_out, stream_capacity, d_stream_starts, stream_bytes_out, infos, ms_out);
}

int dark_bwt_forward_dc_packed_many(dark_bwt_ctx* ctx, const uint8_t* const* texts, const uint64_t* ns, uint64_t count,
                                    uint8_t* const* bwt_outs, uint64_t* origins_out, uint8_t* stream_out, uint64_t stream_capacity,
                                    uint64_t* stream_starts, uint64_t* stream_bytes_out, dark_bwt_dc_info* infos, dark_bwt_stats* stats) {
    if (!ctx || !texts || !ns || !origins_out || !stream_out || !stream_starts || !stream_bytes_out || !infos) return DARK_BWT_E_INVALID_ARG;
    if (int rc = check_staging(ctx)) return rc;
    ctx->err[0] = 0;
    if (count == 0) {
        *stream_bytes_out = 0;
        stream_starts[0] = 0;
        return DARK_BWT_OK;
    }
    BlockList bl;
    if (int rc = check_blocks(ctx, count, ns, nullptr, nullptr, 2, 0, texts, nullptr, &bl)) return rc;
    if (!dc_many_records_fit(ctx, count)) return DARK_BWT_E_INVALID_N;
    return run_blocking(ctx, CopyList().add_blocks(bl, texts, ctx->d_text), stats, [&](CopyList* out) {
        if (int rc = load_blocks(ctx, bl)) return rc;
        if (int rc = forward_many_device(ctx, ctx->d_text, bl.total(), bl.count(), ctx->d_bwt, nullptr, stats)) return rc;
        DcBuffers io;
        std::vector<u32> starts;
        if (int rc = dc_device(ctx, ctx->d_bwt, bl.total(), &bl, &io, infos, &starts)) return rc;
        // dc_device has read the per-block records back out of the sort's second key buffer (8 N + 1 KiB): it holds any stream
        // (<= 8 sum(ns)).  The offsets go to the head of ranks, in front of the pack's tile scratch (dc_pack).
        u8* const d_stream = (u8*)ctx->keys[1];
        u64* const d_offsets = (u64*)ctx->ranks;
        if (int rc = dc_pack_many(ctx, io, starts, d_stream, stream_capacity, d_offsets, stream_bytes_out, infos, nullptr)) return rc;
        out->add_blocks(bl, bwt_outs, ctx->d_bwt);
        out->add(origins_out, ctx->many_origins, sizeof(uint64_t) * count);
        out->add(stream_out, d_stream, *stream_bytes_out);
        out->add(stream_starts, d_offsets, sizeof(u64) * (count + 1));
        return 0;
    });
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
    if (int rc = check_n(ctx, count, 1)) return rc;
    ctx->err[0] = 0;
    const u32 m = (u32)count;
    const int num_passes = (end_bit - begin_bit + kRadixBits - 1) / kRadixBits;
    if (int rc = begin_call(ctx)) return rc;
    CK(cudaMemsetAsync(ctx->hist, 0, sizeof(u32) * kMaxPasses * kRadix, ctx->stream));
    const u32 blocks = (u32)std::min<u64>(ceil_div(m, 256 * 8), 148 * 8);
    k_digit_hist<256><<<blocks, 256, 0, ctx->stream>>>(d_keys, m, begin_bit, num_passes, ctx->hist);
    LAUNCHED();
    u64* keys[2] = {d_keys, d_keys_alt};
    u32* vals[2] = {d_vals, d_vals_alt};
    int cur = 0;
    // note: a partial top digit needs no masking as long as the bits above end_bit are equal in
    // all keys or meant to take part; callers pass end_bit = 64 or keys with zero upper bits.
    if (int rc = run_sort(ctx, keys, vals, 0, m, begin_bit, num_passes, &cur, nullptr, 0)) return rc;
    CK(cudaEventRecord(ctx->call_stop, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    if (ms_out) *ms_out = call_ms(ctx);
    *in_alt_out = cur;
    return DARK_BWT_OK;
}

int dark_bwt_verify_sa_device(dark_bwt_ctx* ctx, const uint8_t* d_text, uint64_t n64, const uint32_t* d_sa,
                              uint64_t* bad_out) {
    if (!ctx || !d_text || !d_sa || !bad_out) return DARK_BWT_E_INVALID_ARG;
    if (int rc = check_n(ctx, n64, 1)) return rc;
    ctx->err[0] = 0;
    CK(cudaSetDevice(ctx->device));
    const u32 n = (u32)n64;
    CK(cudaMemsetAsync(ctx->bad, 0, sizeof(unsigned long long), ctx->stream));
    CK(cudaMemsetAsync(ctx->isa, 0xFF, sizeof(u32) * (size_t)n, ctx->stream));
    const u32 blocks = (u32)ceil_div(n, 256);
    k_verify_scatter<256><<<blocks, 256, 0, ctx->stream>>>(d_sa, n, ctx->isa, ctx->bad);
    LAUNCHED();
    k_verify_order<256><<<blocks, 256, 0, ctx->stream>>>(d_text, d_sa, n, ctx->isa, ctx->bad);
    LAUNCHED();
    CK(cudaMemcpyAsync(&ctx->mail->bad, ctx->bad, sizeof(unsigned long long), cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    *bad_out = ctx->mail->bad;
    return DARK_BWT_OK;
}

int dark_bwt_lcp_profile_device(dark_bwt_ctx* ctx, const uint8_t* d_text, uint64_t n64, const uint32_t* d_sa, uint64_t* m_out,
                                uint32_t* rounds_out, uint64_t* max_lcp_out) {
    if (!ctx || !d_text || !d_sa || !m_out || !rounds_out || !max_lcp_out) return DARK_BWT_E_INVALID_ARG;
    if (int rc = check_n(ctx, n64, 2)) return rc;
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
    if (int rc = check_n(ctx, n, 1)) return rc;
    ctx->err[0] = 0;
    CK(cudaSetDevice(ctx->device));
    if (int rc = emit(ctx, d_text, (u32)n, d_sa, d_bwt_out)) return rc;
    CK(cudaStreamSynchronize(ctx->stream));
    *origin_out = ctx->mail->origin;
    return DARK_BWT_OK;
}

}  // extern "C"
