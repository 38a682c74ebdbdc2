// radix_sort.cuh — LSD radix sort of (u64 key, u32 value) pairs in "onesweep" form:
// one upfront multi-digit histogram, then ONE kernel per 8-bit digit that reads each pair
// once and writes it once, chaining the per-tile digit counts with a decoupled look-back.
//
// This is the sort under the prefix-doubling suffix sorter that replaces the induced-sorting
// sweeps of the reference (put_substr/induce_low/induce_sup, /root/reference/src/saca.rs:60-163):
// keys are packed (rank[i], rank[i+h]) pairs, values are suffix indices.
//
// Roofline: HBM-bound.  Algorithmic bytes per pass launch = 24 B/pair (12 read + 12 written);
// the histogram adds one 8 B/pair read per sort (fused into the key builders on the hot path).
#pragma once

#include "common.cuh"

namespace dark {

__device__ __forceinline__ u32 digit_of(u64 key, int shift) { return (u32)(key >> shift) & (kRadix - 1); }

// ---- shared-memory digit histogram for all passes of a sort -----------------------------------
// s_hist: [kMaxPasses][kRadix] u32, zeroed by the caller.
__device__ __forceinline__ void hist_add_key(u32* s_hist, u64 key, int begin_bit, int num_passes) {
#pragma unroll
    for (int p = 0; p < kMaxPasses; ++p) {
        if (p < num_passes) atomicAdd(&s_hist[p * kRadix + digit_of(key, begin_bit + p * kRadixBits)], 1u);
    }
}
__device__ __forceinline__ void hist_clear(u32* s_hist, int tid, int nthreads) {
    for (int i = tid; i < kMaxPasses * kRadix; i += nthreads) s_hist[i] = 0;
}
__device__ __forceinline__ void hist_flush(u32* s_hist, u32* g_hist, int num_passes, int tid, int nthreads) {
    for (int i = tid; i < num_passes * kRadix; i += nthreads) {
        u32 c = s_hist[i];
        if (c) atomicAdd(&g_hist[i], c);
    }
}

// Stand-alone histogram (used when the keys were not produced by one of the fused builders).
template <int THREADS>
__global__ void __launch_bounds__(THREADS) k_digit_hist(const u64* __restrict__ keys, u32 m, int begin_bit,
                                                        int num_passes, u32* __restrict__ g_hist) {
    __shared__ u32 s_hist[kMaxPasses * kRadix];
    hist_clear(s_hist, threadIdx.x, THREADS);
    __syncthreads();
    const u64 stride = (u64)gridDim.x * THREADS;
    for (u64 i = (u64)blockIdx.x * THREADS + threadIdx.x; i < m; i += stride)
        hist_add_key(s_hist, ld_stream(keys + i), begin_bit, num_passes);
    __syncthreads();
    hist_flush(s_hist, g_hist, num_passes, threadIdx.x, THREADS);
}

// Counts -> exclusive digit bases, in place; one CTA of kRadix threads per pass.
// trivial[p] = 1 when a single digit holds all m keys (the pass would be the identity).
// collide[p] = sum_d (c_d / m)^2: the probability that two random keys share digit p — used by the
// host to decide how many of the low digits of the initial sort can be skipped (pass pruning).
__global__ void __launch_bounds__(kRadix) k_scan_hist(u32* __restrict__ g_hist, u32 m, u32* __restrict__ trivial,
                                                      float* __restrict__ collide) {
    __shared__ u32 s_warp[kRadix / 32];
    __shared__ float s_sq[kRadix / 32];
    __shared__ u32 s_triv;
    const int d = threadIdx.x, lane = d & 31, warp = d >> 5;
    u32* row = g_hist + blockIdx.x * kRadix;
    if (d == 0) s_triv = 0;
    __syncthreads();
    const u32 c = row[d];
    if (c == m) s_triv = 1;
    u32 incl = c;
    const float f = (float)c / (float)m;
    float sq = f * f;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        u32 t = __shfl_up_sync(0xffffffffu, incl, o);
        if (lane >= o) incl += t;
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) sq += __shfl_xor_sync(0xffffffffu, sq, o);
    if (lane == 31) s_warp[warp] = incl;
    if (lane == 0) s_sq[warp] = sq;
    __syncthreads();
    u32 base = 0;
    for (int w = 0; w < warp; ++w) base += s_warp[w];
    row[d] = base + incl - c;
    if (d == 0) {
        trivial[blockIdx.x] = s_triv;
        float tot = 0.f;
        for (int w = 0; w < kRadix / 32; ++w) tot += s_sq[w];
        collide[blockIdx.x] = tot;
    }
}

// ---- the onesweep pass ------------------------------------------------------------------------
// Tile status word: [flag | value]; flag 0 = not ready, 1 = tile aggregate, 2 = inclusive prefix.
template <typename StatusT>
struct StatusTraits;
template <>
struct StatusTraits<u32> {
    static constexpr int kShift = 30;
    static constexpr u32 kMask = (1u << 30) - 1;
};
template <>
struct StatusTraits<u64> {
    static constexpr int kShift = 62;
    static constexpr u64 kMask = (1ull << 62) - 1;
};

template <int THREADS, int ITEMS>
struct OnesweepSmem {
    static constexpr int kTile = THREADS * ITEMS;
    static constexpr int kWarps = THREADS / 32;
    u64 keys[kTile];             // tile re-ordered by digit (so the global scatter is run-coalesced)
    u32 vals[kTile];
    u32 raw_vals[kTile];         // values as loaded (cp.async), consumed by the re-order
    u32 warp_hist[kWarps][kRadix];  // per-warp digit counters -> exclusive warp offsets
    u32 digit_start[kRadix];        // exclusive scan of the tile's digit counts
    u32 global_off[kRadix];         // output index of local position 0 of each digit (mod 2^32)
    u32 warp_sum[kRadix / 32];
    u32 tile;
};

// Lanes whose 8-bit digit equals mine, restricted to `peers`: one test + one vote + a predicated NOT +
// an AND per bit.  Written in PTX because the C++ form (`bit ? vote : ~vote`) compiled to 6 instructions
// per bit (bit tested twice, a SEL to build the mask).
template <int BIT>
__device__ __forceinline__ u32 match_digit_bit(u32 peers, u32 d) {
    asm("{\n"
        ".reg .pred p;\n"
        ".reg .b32 v;\n"
        "and.b32 v, %1, %2;\n"
        "setp.ne.u32 p, v, 0;\n"
        "vote.sync.ballot.b32 v, p, 0xffffffff;\n"
        "@!p not.b32 v, v;\n"
        "and.b32 %0, %0, v;\n"
        "}\n"
        : "+r"(peers)
        : "r"(d), "n"(1 << BIT));
    return peers;
}
__device__ __forceinline__ u32 match_digit_bits(u32 peers, u32 d) {
    peers = match_digit_bit<0>(peers, d);
    peers = match_digit_bit<1>(peers, d);
    peers = match_digit_bit<2>(peers, d);
    peers = match_digit_bit<3>(peers, d);
    peers = match_digit_bit<4>(peers, d);
    peers = match_digit_bit<5>(peers, d);
    peers = match_digit_bit<6>(peers, d);
    peers = match_digit_bit<7>(peers, d);
    return peers;
}

// Digit selection.  ALIGNED (shift a multiple of 8, the only case the suffix sorter uses): the digit
// is one byte of the high or low key word, a single PRMT.  Otherwise a generic 64-bit shift.
template <bool ALIGNED>
struct DigitSel {
    int shift;
    u32 bsel;  // __byte_perm selector: 0x4440 | byte index inside the word
    bool hi;
    __device__ __forceinline__ explicit DigitSel(int sh) : shift(sh), bsel(0x4440u | ((u32)(sh & 31) >> 3)), hi(sh >= 32) {}
    __device__ __forceinline__ u32 operator()(u64 key) const {
        if (ALIGNED) {
            const u32 w = hi ? (u32)(key >> 32) : (u32)key;  // `hi` is launch-uniform
            return __byte_perm(w, 0u, bsel);
        }
        return (u32)(key >> shift) & (kRadix - 1);
    }
};

// Batched decoupled look-back of one digit column: kBatch predecessor status words per L2 round trip.
// issue() only starts the loads; consume() folds them (aggregates up to the nearest inclusive prefix)
// and moves the cursor, so the round trip can be overlapped with other work.
template <typename StatusT, int kBatch>
struct DigitLookback {
    typedef StatusTraits<StatusT> ST;
    StatusT v[kBatch];
    StatusT excl;
    int t;
    bool found, pending;
    __device__ __forceinline__ void init(u32 tile) {
        excl = 0;
        t = (int)tile - 1;
        found = tile == 0;
        pending = false;
    }
    __device__ __forceinline__ void issue(const StatusT* __restrict__ status, int tid) {
#pragma unroll
        for (int j = 0; j < kBatch; ++j)
            v[j] = (t - j >= 0) ? ld_relaxed(status + (size_t)(t - j) * kRadix + tid) : ((StatusT)2 << ST::kShift);
        pending = true;
    }
    __device__ __forceinline__ void consume() {
        int used = kBatch;
#pragma unroll
        for (int j = 0; j < kBatch; ++j) {
            if (j < used && !found) {
                const u32 flag = (u32)(v[j] >> ST::kShift);
                if (flag == 0) {
                    used = j;  // not published yet: poll again from this tile
                } else {
                    excl += v[j] & ST::kMask;
                    if (flag == 2) found = true;
                }
            }
        }
        t -= used;
        pending = false;
    }
    // one overlapped step: fold what has arrived, start the next batch if still searching
    __device__ __forceinline__ void step(const StatusT* __restrict__ status, int tid) {
        if (found) return;
        if (pending) consume();
        if (!found) issue(status, tid);
    }
    __device__ __forceinline__ void finish(const StatusT* __restrict__ status, int tid) {
        while (!found) {
            if (!pending) issue(status, tid);
            consume();
        }
    }
};

// GEN (first pass of the suffix sorter's round 0): the (key, id) pairs are not read from memory but
// built from the text on the fly — element j is suffix id = n-1-j, its key the first 64/s symbols as dense
// s-bit codes (exactly what k_init_keys_packed would have written, suffix_kernels.cuh).  Saves the 12 B per
// suffix the key builder would write and the 12 B this pass would read back.
struct KeyGen {
    const u8* text;
    const u8* lut;  // byte -> dense code
    u32 n;
    int lg_s;       // log2(bits per symbol): s in {1, 2, 4, 8}
    int mode;       // 0: suffix keys of round 0;  1: inverse BWT — element e is (last-column symbol, row) of the e-th real row
    u32 origin;     // mode 1: origin index of the transform (`text` is the BWT)
};

// The body of one tile.  FULL = all THREADS*ITEMS slots hold a pair (every tile but the last):
// no validity predicates anywhere on that path.
// Tried and rejected (measurements in profiles/r1_pass_trace_v4.md): publishing the aggregate from a
// shared-atomic pre-count and starting the look-back before the ranking loop (1.22-1.40 ms per 2^27
// pairs instead of 1.07: the prefix still appears only after the ranking, so walks get longer), and a
// dedicated scan warp doing the look-back beside the ranking warps (2.1 ms: one warp cannot keep enough
// status loads in flight).
template <int THREADS, int ITEMS, int ILP, typename StatusT, bool ALIGNED, bool FULL, bool GEN>
__device__ __forceinline__ void onesweep_tile(OnesweepSmem<THREADS, ITEMS>& s, const u64* __restrict__ keys_in,
                                              const u32* __restrict__ vals_in, u64* __restrict__ keys_out,
                                              u32* __restrict__ vals_out, const u32 tile, const u32 nvalid, const int shift,
                                              const u32* __restrict__ digit_base, StatusT* __restrict__ status,
                                              const u8* __restrict__ prev_text, const u32 n_text, const KeyGen gen) {
    typedef OnesweepSmem<THREADS, ITEMS> Smem;
    typedef StatusTraits<StatusT> ST;
    constexpr int TILE = Smem::kTile;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const u64 tile_base = (u64)tile * TILE;
    const DigitSel<ALIGNED> digit(shift);

    // warp-striped arrangement: element (warp, k, lane) has tile-local index warp*32*ITEMS + k*32 + lane,
    // so every load instruction of a warp covers 32 consecutive pairs and rank order == index order.
    const u32 local0 = warp * (32 * ITEMS) + lane;
    u64 key[ITEMS];
    if (GEN && gen.mode == 1) {
        // inverse BWT, step 1 (suffix_kernels.cuh): row r(e) = 0, e, or e+1 around the origin; key = that row's last symbol
#pragma unroll
        for (int k = 0; k < ITEMS; ++k) {
            const u32 jl = local0 + k * 32;
            key[k] = ~0ull;
            if (FULL || jl < nvalid) {
                const u32 e = (u32)tile_base + jl;
                const u32 r = e == 0 ? 0u : (e <= gen.origin ? e : e + 1u);
                key[k] = (u64)__ldg(gen.text + (e == 0 ? gen.origin : r - 1));
                s.raw_vals[jl] = r;
            }
        }
    } else if (GEN) {
        // the tile's symbol codes, packed MSB-first into 32-bit words (s.keys is free until the re-order);
        // a key is a 64-bit window of that bit stream
        u32* words = reinterpret_cast<u32*>(s.keys);
        const int lg_s = gen.lg_s, sbits = 1 << lg_s, spw = 32 >> lg_s;
        const u64 i_lo = (u64)gen.n - tile_base - nvalid;  // lowest text position of this tile
        const u32 nwords = ((u32)(TILE + (64 >> lg_s)) >> (5 - lg_s)) + 3;
        for (u32 w = tid; w < nwords; w += THREADS) {
            u32 word = 0;
            const u64 pos0 = i_lo + ((u64)w << (5 - lg_s));
            for (int c = 0; c < spw; c += 4) {
                u32 code[4];
#pragma unroll
                for (int e = 0; e < 4; ++e) code[e] = pos0 + c + e < gen.n ? (u32)__ldg(gen.text + pos0 + c + e) : 0x100u;
#pragma unroll
                for (int e = 0; e < 4; ++e) code[e] = code[e] < 0x100u ? (u32)__ldg(gen.lut + code[e]) : 0u;
#pragma unroll
                for (int e = 0; e < 4; ++e) word = (word << sbits) | code[e];
            }
            words[w] = word;
        }
        __syncthreads();
#pragma unroll
        for (int k = 0; k < ITEMS; ++k) {
            const u32 jl = local0 + k * 32;
            key[k] = ~0ull;
            if (FULL || jl < nvalid) {
                const u32 x = nvalid - 1 - jl;
                const u32 bit = x << lg_s;
                const u32 wi = bit >> 5, sh = bit & 31;
                const u32 w0 = words[wi], w1 = words[wi + 1], w2 = words[wi + 2];
                key[k] = ((u64)__funnelshift_l(w1, w0, sh) << 32) | __funnelshift_l(w2, w1, sh);
                s.raw_vals[jl] = (u32)(i_lo + x);
            }
        }
        // (the words are dead once every thread has passed the barrier that follows the ranking loop)
    } else {
        const u64* kp = keys_in + tile_base + local0;
#pragma unroll
        for (int k = 0; k < ITEMS; ++k) key[k] = (FULL || local0 + k * 32 < nvalid) ? ld_stream(kp + k * 32) : ~0ull;
    }
    if (prev_text != nullptr) {
        // First pass of a pruned initial sort (the low key byte is not sorted): element j is still suffix
        // n-1-j, so its BWT byte T[id-1] is a contiguous read; it rides in the low key byte from here on
        // and the round-0 re-rank emits it for every suffix it settles — no gather for those.
#pragma unroll
        for (int k = 0; k < ITEMS; ++k) {
            const u64 j = tile_base + local0 + k * 32;
            if (FULL || local0 + k * 32 < nvalid) {
                const u32 id = n_text - 1 - (u32)j;
                key[k] = (key[k] & ~0xFFull) | (u64)__ldg(prev_text + (id == 0 ? n_text - 1 : id - 1));
            }
        }
    }
    // The values go straight to shared memory with cp.async (no registers held across the ranking
    // loop, latency hidden behind it); each thread later reads back exactly the words it copied.
    if (!GEN) {
        const u32* vp = vals_in + tile_base + local0;
        const u32 dst = smem_addr(&s.raw_vals[local0]);
#pragma unroll
        for (int k = 0; k < ITEMS; ++k)
            if (FULL || local0 + k * 32 < nvalid)
                asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"(dst + k * 128), "l"(vp + k * 32) : "memory");
        asm volatile("cp.async.commit_group;" ::: "memory");
    }

    constexpr int kLookbackBatch = 8;
    DigitLookback<StatusT, kLookbackBatch> lb;
    lb.init(tile);
    u32 count = 0;

    // ---- rank inside the warp.  Lanes with equal digits are found with 8 ballots (one per digit bit;
    // match.any is microcoded per distinct value and was the top stall of the first version,
    // profiles/r1_ncu_c2_v1.md).  Every lane reads its digit's counter, the lowest lane of each group
    // then bumps it.  Ranks are < 32*ITEMS and packed two per register.
    static_assert(ITEMS % 2 == 0 && 32 * ITEMS < 65536, "ranks are packed two per register");
    u32 rank2[ITEMS / 2];
    u32* whist = s.warp_hist[warp];
    const u32 lt = lanemask_lt();
#pragma unroll
    for (int k = 0; k < ITEMS; ++k) {
        const bool valid = FULL || (local0 + k * 32) < nvalid;
        u32 d = digit(key[k]);
        // Tie this item's ballots to the result of item k-ILP: without the false dependency the
        // compiler hoists the votes of all ITEMS items to the top (150+ registers, one CTA per SM);
        // ILP items stay in flight per warp.
        if (k >= ILP) asm volatile("" : "+r"(d) : "r"(rank2[(k - ILP) / 2]));
        u32 peers = FULL ? 0xffffffffu : __ballot_sync(0xffffffffu, valid);
        peers = match_digit_bits(peers, d);
        const u32 prev = whist[d];  // every lane reads (padding lanes harmlessly), then the group's lowest lane bumps
        const u32 below = peers & lt;
        const u32 r = prev + __popc(below);
        __syncwarp();
        if (valid && below == 0) whist[d] = prev + __popc(peers);
        if (k & 1) rank2[k / 2] |= r << 16;
        else rank2[k / 2] = r;
        __syncwarp();
    }
    __syncthreads();

    // ---- per digit: exclusive offsets across warps, tile total, publish the aggregate
    if (tid < kRadix) {
        u32 run = 0;
#pragma unroll
        for (int w = 0; w < Smem::kWarps; ++w) {
            const u32 c = s.warp_hist[w][tid];
            s.warp_hist[w][tid] = run;
            run += c;
        }
        count = run;
        st_relaxed(status + (size_t)tile * kRadix + tid, ((StatusT)(tile == 0 ? 2 : 1) << ST::kShift) | (StatusT)count);
    }
    // exclusive scan of the 256 digit counts (threads >= 256 contribute 0 and are ignored)
    u32 incl = count;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        u32 t = __shfl_up_sync(0xffffffffu, incl, o);
        if (lane >= o) incl += t;
    }
    if (tid < kRadix && lane == 31) s.warp_sum[warp] = incl;
    __syncthreads();
    u32 dstart = 0;
    if (tid < kRadix) {
        u32 wbase = 0;
        for (int w = 0; w < warp; ++w) wbase += s.warp_sum[w];
        dstart = wbase + incl - count;
        // fold the digit start into the per-warp offsets: one table lookup per element in the re-order
#pragma unroll
        for (int w = 0; w < Smem::kWarps; ++w) s.warp_hist[w][tid] += dstart;
    }
    __syncthreads();

    // ---- re-order the tile by digit in shared memory (needs only tile-local offsets, so it runs
    // before the look-back and gives the predecessor tiles time to publish)
    asm volatile("cp.async.wait_group 0;" ::: "memory");
#pragma unroll
    for (int k = 0; k < ITEMS; ++k) {
        if (FULL || (local0 + k * 32) < nvalid) {
            const u32 pos = whist[digit(key[k])] + ((rank2[k / 2] >> (16 * (k & 1))) & 0xFFFFu);
            s.keys[pos] = key[k];
            s.vals[pos] = s.raw_vals[local0 + k * 32];
        }
    }

    // ---- decoupled look-back over the predecessors' digit counts.  Tiles finish every ~60 cycles
    // chip-wide while a status read costs an L2 round trip (600+ cycles, more under load), so the
    // nearest inclusive prefix is 10-25 tiles back: walking them one load at a time cost 34 % of the
    // tile time (profiles/r1_pass_trace_v3.log); 8 predecessors are read per round trip.
    if (tid < kRadix) {
        if (tile > 0) {
            lb.finish(status, tid);
            st_relaxed(status + (size_t)tile * kRadix + tid, ((StatusT)2 << ST::kShift) | (lb.excl + count));
        }
        s.global_off[tid] = digit_base[tid] + (u32)lb.excl - dstart;
    }
    __syncthreads();

    // ---- scatter: consecutive threads write consecutive addresses inside each digit run
#pragma unroll
    for (int k = 0; k < ITEMS; ++k) {
        const u32 p = k * THREADS + tid;
        if (FULL || p < nvalid) {
            const u64 kk = s.keys[p];
            const u32 idx = s.global_off[digit(kk)] + p;
            keys_out[idx] = kk;
            vals_out[idx] = s.vals[p];
        }
    }
}

template <int THREADS, int ITEMS, int MINBLOCKS, int ILP, typename StatusT, bool ALIGNED, bool GEN = false>
__global__ void __launch_bounds__(THREADS, MINBLOCKS)
k_onesweep_pass(const u64* __restrict__ keys_in, const u32* __restrict__ vals_in, u64* __restrict__ keys_out,
                u32* __restrict__ vals_out, u32 m, int shift, const u32* __restrict__ digit_base,
                StatusT* __restrict__ status, u32* __restrict__ tile_counter, const u8* __restrict__ prev_text, u32 n_text,
                KeyGen gen, u32 prefetch_ahead) {
    static_assert(THREADS >= kRadix && THREADS % 32 == 0, "one thread per digit is assumed");
    typedef OnesweepSmem<THREADS, ITEMS> Smem;
    constexpr int TILE = Smem::kTile;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    Smem& s = *reinterpret_cast<Smem*>(smem_raw);
    const int tid = threadIdx.x;

    // Persistent CTAs: the grid is (SMs x resident CTAs) and every CTA claims tiles from a counter until
    // none are left.  Tiles are thereby numbered in the order they are started, so the look-back only
    // ever waits on tiles that are already running; and a CTA no longer has to drain its scattered
    // stores and be re-launched between tiles — with one tile per CTA the SMs held only 1.8 of 3
    // resident tiles on average (profiles/r1_pass_trace_v4.log).
    const u32 num_tiles = (u32)(((u64)m + TILE - 1) / TILE);
    for (;;) {
        if (tid == 0) s.tile = atomicAdd(tile_counter, 1u);
        for (int i = tid; i < Smem::kWarps * kRadix; i += THREADS) (&s.warp_hist[0][0])[i] = 0;
        __syncthreads();
        const u32 tile = s.tile;
        if (tile >= num_tiles) break;
        const u32 nvalid = (u32)min((u64)TILE, (u64)m - (u64)tile * TILE);
        if (!GEN) {
            // Pull the pairs of the tile this CTA is likely to claim next (one wave of claims ahead) into L2, a
            // 128-byte line per thread: its loads then miss only L1.  Measured: C2 sort phase 10.1 -> 9.4 ms at a
            // distance of one wave (444 tiles); no gain at two waves (profiles/r1_final.md).
            const u64 q = ((u64)tile + prefetch_ahead) * TILE;
            if (q + TILE <= m) {
                for (int c = tid; c < TILE / 16; c += THREADS) asm volatile("prefetch.global.L2 [%0];" ::"l"(keys_in + q + (u64)c * 16));
                for (int c = tid; c < TILE / 32; c += THREADS) asm volatile("prefetch.global.L2 [%0];" ::"l"(vals_in + q + (u64)c * 32));
            }
        }
        if (nvalid == TILE)
            onesweep_tile<THREADS, ITEMS, ILP, StatusT, ALIGNED, true, GEN>(s, keys_in, vals_in, keys_out, vals_out, tile, nvalid,
                                                                            shift, digit_base, status, prev_text, n_text, gen);
        else
            onesweep_tile<THREADS, ITEMS, ILP, StatusT, ALIGNED, false, GEN>(s, keys_in, vals_in, keys_out, vals_out, tile, nvalid,
                                                                             shift, digit_base, status, prev_text, n_text, gen);
        __syncthreads();  // the scatter has read the shared tile: it may be overwritten now
    }
}

}  // namespace dark
