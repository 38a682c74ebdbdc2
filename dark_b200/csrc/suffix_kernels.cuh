// suffix_kernels.cuh — the prefix-doubling suffix sorter around the radix sort, and BWT emission.
//
// Replaces (results, not internals) the reference's SA-IS `saca()` (/root/reference/src/saca.rs:270-340)
// and `compress::bwt::TransformIterator` (call sites src/block/dc.rs:45-50, src/block/raw.rs:39-44).
//
// Order convention (SURVEY.md App. A.1/A.3): plain lexicographic order of suffixes, a proper prefix
// sorts first.  There is no in-band sentinel: "beyond the end" is rank 0, real ranks are stored
// 0-based in isa[] and read as isa[i]+1.
#pragma once

#include "common.cuh"
#include "radix_sort.cuh"

namespace dark {

// Staging of compacted elements in shared memory.  A thread owns ITEMS = 8 consecutive elements, so the lanes of a warp
// store at a stride of up to 8 words: eight lanes per bank.  One pad word per 32 (one 8-byte pad per 16 for 64-bit
// elements) spreads a stride-8 warp store over all banks and leaves the lane-consecutive read-out conflict-free.
__host__ __device__ constexpr u32 stage_pad32(u32 i) { return i + (i >> 5); }
__host__ __device__ constexpr u32 stage_pad64(u32 i) { return i + (i >> 4); }

// ---- alphabet ---------------------------------------------------------------------------------
// Which byte values occur?  (HBM: N bytes read.)  Plain racing stores of the constant 1 are fine.
template <int THREADS>
__global__ void __launch_bounds__(THREADS) k_symbol_presence(const u8* __restrict__ text, u64 n, u32* __restrict__ present) {
    __shared__ u32 s_present[256];
    for (int i = threadIdx.x; i < 256; i += THREADS) s_present[i] = 0;
    __syncthreads();
    // 16-byte aligned body, scalar head and tail
    const u64 addr = (u64)text;
    u64 head = (16 - (addr & 15)) & 15;
    if (head > n) head = n;
    const u64 nvec = (n - head) / 16;
    const uint4* body = reinterpret_cast<const uint4*>(text + head);
    const u64 gtid = (u64)blockIdx.x * THREADS + threadIdx.x, gstride = (u64)gridDim.x * THREADS;
    for (u64 v = gtid; v < nvec; v += gstride) {
        const uint4 q = __ldg(body + v);
        const u32 w[4] = {q.x, q.y, q.z, q.w};
#pragma unroll
        for (int a = 0; a < 4; ++a) {
            s_present[w[a] & 255] = 1;
            s_present[(w[a] >> 8) & 255] = 1;
            s_present[(w[a] >> 16) & 255] = 1;
            s_present[w[a] >> 24] = 1;
        }
    }
    if (gtid < head) s_present[text[gtid]] = 1;
    const u64 tail0 = head + nvec * 16;
    if (tail0 + gtid < n && gtid < 16) s_present[text[tail0 + gtid]] = 1;
    __syncthreads();
    for (int i = threadIdx.x; i < 256; i += THREADS)
        if (s_present[i]) present[i] = 1;
}

// present[256] -> dense codes (rank among the present symbols) and sigma.  One CTA of 256 threads.
__global__ void __launch_bounds__(256) k_build_lut(const u32* __restrict__ present, u8* __restrict__ lut, u32* __restrict__ sigma_out,
                                                   int identity) {
    __shared__ u32 s_warp[8];
    const int d = threadIdx.x, lane = d & 31, warp = d >> 5;
    const u32 c = present[d] ? 1u : 0u;
    u32 incl = c;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        u32 t = __shfl_up_sync(0xffffffffu, incl, o);
        if (lane >= o) incl += t;
    }
    if (lane == 31) s_warp[warp] = incl;
    __syncthreads();
    u32 base = 0;
    for (int w = 0; w < warp; ++w) base += s_warp[w];
    lut[d] = identity ? (u8)d : (u8)(base + incl - c);
    if (d == 255) *sigma_out = base + incl;
}

// ---- round 0: initial keys ----------------------------------------------------------------------
// Element j of the sort input is suffix id = n-1-j (descending), key = the first K symbols of the
// suffix as dense s-bit codes, most significant first, zero-padded past the end of the text.
// The descending order makes the STABLE LSD sort break ties between a short (padded) suffix and
// longer ones with the same key the right way: the shorter suffix comes first (App. A.3).
// Fused: digit histogram of all passes.  HBM: N read, 12 N written.
template <int THREADS, int ITEMS>
__global__ void __launch_bounds__(THREADS)
k_init_keys(const u8* __restrict__ text, u32 n, const u8* __restrict__ lut, int s_bits, int K, u64* __restrict__ keys_out,
            u32* __restrict__ ids_out, u32* __restrict__ g_hist, int num_passes) {
    constexpr int TILE = THREADS * ITEMS;
    __shared__ u8 s_code[TILE + 64];
    __shared__ u8 s_lut[256];
    __shared__ u32 s_hist[kMaxPasses * kRadix];
    const int tid = threadIdx.x;
    hist_clear(s_hist, tid, THREADS);
    for (int i = tid; i < 256; i += THREADS) s_lut[i] = lut[i];
    __syncthreads();

    // a capped grid loops over the tiles, so the shared histogram is flushed (2,048 global atomics)
    // once per CTA instead of once per tile — the flush was a third of this kernel's stalls
    const u32 ntiles = (u32)(((u64)n + TILE - 1) / TILE);
    for (u32 tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
        const u64 jb = (u64)tile * TILE;
        const u32 cnt = (u32)min((u64)TILE, (u64)n - jb);
        const u64 i_lo = (u64)n - jb - cnt;  // lowest text position of this tile
        const u32 span = cnt + K - 1;
        for (u32 x = tid; x < span; x += THREADS) {
            const u64 pos = i_lo + x;
            s_code[x] = pos < n ? s_lut[text[pos]] : (u8)0;
        }
        __syncthreads();
#pragma unroll 4
        for (int k = 0; k < ITEMS; ++k) {
            const u32 jl = k * THREADS + tid;
            if (jl < cnt) {
                const u32 x = cnt - 1 - jl;  // position i = i_lo + x
                u64 key = 0;
                for (int c = 0; c < K; ++c) key = (key << s_bits) | s_code[x + c];
                key <<= (64 - s_bits * K);  // symbol field MSB-aligned, so "the top 8t bits" are whole leading symbols
                keys_out[jb + jl] = key;
                ids_out[jb + jl] = (u32)(i_lo + x);
                hist_add_key(s_hist, key, 0, num_passes);
            }
        }
        __syncthreads();
    }
    hist_flush(s_hist, g_hist, num_passes, tid, THREADS);
}

// Fast path for s in {1,2,4,8} bits per symbol (sigma <= 2, 4, 16, 256): the tile's codes are first
// packed MSB-first into 32-bit words in shared memory; a key is then a 64-bit window of that bit
// stream (3 LDS + 2 funnel shifts instead of K byte loads — the byte loop made the first version
// of this kernel issue-bound at K = 32, profiles/r1_ncu_c2_v1.md).
// WRITE = true: keys only (the histograms came from k_gram_hist; the keys are needed when no radix pass builds them,
// radix_sort.cuh GEN).  WRITE = false: the digit histograms only, counted key by key (DARK_BWT_CHECK_HIST).
template <int THREADS, int ITEMS, int S, bool WRITE>
__global__ void __launch_bounds__(THREADS)
k_init_keys_packed(const u8* __restrict__ text, u32 n, const u8* __restrict__ lut, u64* __restrict__ keys_out,
                   u32* __restrict__ ids_out, u32* __restrict__ g_hist) {
    constexpr int TILE = THREADS * ITEMS;
    constexpr int SPW = 32 / S;   // symbols per word
    constexpr int K = 64 / S;     // symbols per key: exactly two words
    constexpr int NWORDS = (TILE + K) / SPW + 3;
    __shared__ u32 s_words[NWORDS];
    __shared__ u8 s_lut[256];
    __shared__ u32 s_hist[kMaxPasses * kRadix];
    const int tid = threadIdx.x;
    hist_clear(s_hist, tid, THREADS);
    for (int i = tid; i < 256; i += THREADS) s_lut[i] = lut[i];
    __syncthreads();

    const u32 ntiles = (u32)(((u64)n + TILE - 1) / TILE);
    for (u32 tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {  // capped grid: one histogram flush per CTA
        const u64 jb = (u64)tile * TILE;
        const u32 cnt = (u32)min((u64)TILE, (u64)n - jb);
        const u64 i_lo = (u64)n - jb - cnt;
        for (int w = tid; w < NWORDS; w += THREADS) {
            u32 word = 0;
            const u64 pos0 = i_lo + (u64)w * SPW;
#pragma unroll
            for (int c = 0; c < SPW; ++c) {
                const u64 pos = pos0 + c;
                const u32 code = pos < n ? (u32)s_lut[text[pos]] : 0u;
                word = (S == 32 ? 0u : (word << (S & 31))) | code;
            }
            s_words[w] = word;
        }
        __syncthreads();
#pragma unroll 4
        for (int k = 0; k < ITEMS; ++k) {
            const u32 jl = k * THREADS + tid;
            if (jl < cnt) {
                const u32 x = cnt - 1 - jl;
                const u32 bit = x * S;
                const u32 wi = bit >> 5, sh = bit & 31;
                const u32 w0 = s_words[wi], w1 = s_words[wi + 1], w2 = s_words[wi + 2];
                const u32 hi = __funnelshift_l(w1, w0, sh);
                const u32 lo = __funnelshift_l(w2, w1, sh);
                const u64 key = ((u64)hi << 32) | lo;
                if (WRITE) {
                    keys_out[jb + jl] = key;
                    ids_out[jb + jl] = (u32)(i_lo + x);
                } else {
                    hist_add_key(s_hist, key, 0, kMaxPasses);
                }
            }
        }
        __syncthreads();
    }
    if (!WRITE) hist_flush(s_hist, g_hist, kMaxPasses, tid, THREADS);
}

// Digit histograms of the initial keys without building a key.  For s in {1,2,4,8} a radix digit is a whole
// number Q = 8/s of symbols, so digit t (from the top) of the key of suffix i is the Q-gram at text position
// i + tQ (zero-padded past the end): all eight histograms are the ONE Q-gram histogram G of the text, minus
// the grams of the first tQ positions, plus tQ padding grams.  One shared-memory atomic per text byte
// instead of eight per key (the fused count in the key builder was bank-conflict bound at 0.95 ms per 2^28).
template <int THREADS, int S>
__global__ void __launch_bounds__(THREADS)
k_gram_hist(const u8* __restrict__ text, u32 n, const u8* __restrict__ lut, u32* __restrict__ g_gram) {
    constexpr int Q = 8 / S;
    constexpr int WARPS = THREADS / 32;
    constexpr int PER = 16;  // text positions per thread and step
    __shared__ u32 s_h[WARPS][kRadix];
    __shared__ u8 s_lut[256];
    const int tid = threadIdx.x, warp = tid >> 5;
    for (int i = tid; i < WARPS * kRadix; i += THREADS) (&s_h[0][0])[i] = 0;
    for (int i = tid; i < 256; i += THREADS) s_lut[i] = lut[i];
    __syncthreads();
    const bool vec = (((uintptr_t)text) & 15) == 0;
    for (u64 base = (u64)blockIdx.x * (THREADS * PER); base < n; base += (u64)gridDim.x * (THREADS * PER)) {
        const u64 i0 = base + (u64)tid * PER;
        if (i0 >= n) continue;
        u32 code[PER + Q - 1];
        if (vec && i0 + PER <= n) {
            const uint4 v = *reinterpret_cast<const uint4*>(text + i0);
            const u32 w[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
            for (int e = 0; e < PER; ++e) code[e] = s_lut[(w[e >> 2] >> (8 * (e & 3))) & 0xFFu];
        } else {
#pragma unroll
            for (int e = 0; e < PER; ++e) code[e] = i0 + e < n ? (u32)s_lut[text[i0 + e]] : 0u;
        }
#pragma unroll
        for (int e = PER; e < PER + Q - 1; ++e) code[e] = i0 + e < n ? (u32)s_lut[text[i0 + e]] : 0u;
#pragma unroll
        for (int e = 0; e < PER; ++e) {
            u32 gram = 0;
#pragma unroll
            for (int c = 0; c < Q; ++c) gram = (gram << S) | code[e + c];
            if (i0 + e < n) atomicAdd(&s_h[warp][gram & 0xFFu], 1u);
        }
    }
    __syncthreads();
    for (int d = tid; d < kRadix; d += THREADS) {
        u32 c = 0;
#pragma unroll
        for (int w = 0; w < WARPS; ++w) c += s_h[w][d];
        if (c) atomicAdd(&g_gram[d], c);
    }
}

// G -> the eight digit histograms (row p = digit at bit 8p, i.e. t = 7-p from the top); one CTA of 256 threads.
__global__ void __launch_bounds__(kRadix) k_gram_expand(const u8* __restrict__ text, u32 n, const u8* __restrict__ lut, int lg_s,
                                                        const u32* __restrict__ g_gram, u32* __restrict__ g_hist) {
    __shared__ u32 s_code[72];
    __shared__ u32 s_gram[64];
    const int v = threadIdx.x;
    const int S = 1 << lg_s, Q = 8 >> lg_s;
    if (v < 72) s_code[v] = (u32)v < n ? (u32)lut[text[v]] : 0u;
    __syncthreads();
    if (v < 64) {
        u32 gram = 0;
        for (int c = 0; c < Q; ++c) gram = (gram << S) | s_code[v + c];
        s_gram[v] = gram & 0xFFu;
    }
    __syncthreads();
    const u32 G = g_gram[v];
    for (int t = 0; t < kMaxPasses; ++t) {
        const u32 c = min((u32)(t * Q), n);  // leading positions that digit t never sees = padding grams it sees instead
        u32 lead = 0;
        for (u32 j = 0; j < c; ++j) lead += s_gram[j] == (u32)v ? 1u : 0u;
        g_hist[(kMaxPasses - 1 - t) * kRadix + v] = G - lead + (v == 0 ? c : 0u);
    }
}

// ---- round r >= 1: keys (rank[i], rank[i+h]) ------------------------------------------------------
// Active element p: suffix ids[p] in a group of rank ranks[p].  key = rank << kb | (isa[i+h]+1 or 0).
// Fused: digit histogram.  HBM: 8 B read + one 4-byte gather (a 32 B sector) + 8 B written per element.
template <int THREADS, int ITEMS>
__global__ void __launch_bounds__(THREADS)
k_build_keys(const u32* __restrict__ ids, const u32* __restrict__ ranks, u32 m, u32 n, u64 h, int kb,
             const u32* __restrict__ isa, u32 tag, u64* __restrict__ keys_out, u32* __restrict__ g_hist, int num_passes) {
    __shared__ u32 s_hist[kMaxPasses * kRadix];
    const int tid = threadIdx.x;
    hist_clear(s_hist, tid, THREADS);
    __syncthreads();
    const u32 ntiles = (u32)(((u64)m + THREADS * ITEMS - 1) / (THREADS * ITEMS));
    for (u32 tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {  // capped grid: one histogram flush per CTA
        const u64 base = (u64)tile * (THREADS * ITEMS);
        u32 id[ITEMS], r2[ITEMS];
#pragma unroll
        for (int k = 0; k < ITEMS; ++k) {
            const u64 p = base + k * THREADS + tid;
            id[k] = p < m ? ld_stream(ids + p) : 0u;
        }
#pragma unroll
        for (int k = 0; k < ITEMS; ++k) {
            const u64 p = base + k * THREADS + tid;
            const u64 pos2 = (u64)id[k] + h;
            r2[k] = (p < m && pos2 < n) ? (__ldg(isa + pos2) & ~tag) + 1u : 0u;
        }
#pragma unroll
        for (int k = 0; k < ITEMS; ++k) {
            const u64 p = base + k * THREADS + tid;
            if (p < m) {
                const u64 key = ((u64)(ld_stream(ranks + p) >> 1) << kb) | r2[k];  // >>1: see k_rerank
                keys_out[p] = key;
                hist_add_key(s_hist, key, 0, num_passes);
            }
        }
    }
    __syncthreads();
    hist_flush(s_hist, g_hist, num_passes, tid, THREADS);
}

// The same keys built in TEXT order.  isa[] entries of active suffixes carry `tag` (bit 31, blocks of at most
// 2^31 bytes), so a sweep over isa[] finds them; rank2 = isa[i+h] is then a second sequential stream instead
// of a random gather (110 B of DRAM traffic per gathered rank once isa[] outgrows L2,
// profiles/r1_ncu_c5_c3_v2.md).  The active list comes out in text order instead of rank order, which the sort
// does not care about: it orders by (rank, rank2) from scratch, and the re-rank reads the exact ranks
// position-wise from the old list, whose group layout the sorted list reproduces.
// HBM: 4n read (+ the second stream, mostly L2 hits), 12 m written.  Used while m > n/8.
template <int THREADS, int ITEMS>
constexpr size_t kBuildTextSmem = (size_t)stage_pad64(THREADS * ITEMS) * 8 + (size_t)stage_pad32(THREADS * ITEMS) * 4 + (size_t)kMaxPasses * kRadix * 4;
template <int THREADS, int ITEMS>
__global__ void __launch_bounds__(THREADS)
k_build_keys_text(const u32* __restrict__ isa, u32 n, u64 h, int kb, u32 tag, u64* __restrict__ keys_out, u32* __restrict__ ids_out,
                  u64* __restrict__ scan_words, u32* __restrict__ tile_counter, u32* __restrict__ out_count,
                  u32* __restrict__ g_hist, int num_passes) {
    constexpr int TILE = THREADS * ITEMS;
    constexpr int WARPS = THREADS / 32;
    static_assert(ITEMS % 4 == 0, "128-bit loads");
    extern __shared__ __align__(16) unsigned char smem_text_build[];  // kBuildTextSmem<THREADS, ITEMS> bytes
    u64* s_key = reinterpret_cast<u64*>(smem_text_build);
    u32* s_id = reinterpret_cast<u32*>(s_key + stage_pad64(TILE));
    u32* s_hist = s_id + stage_pad32(TILE);
    __shared__ u32 s_warp[WARPS];
    __shared__ u32 s_excl, s_total, s_tile;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    hist_clear(s_hist, tid, THREADS);
    const u32 ntiles = (u32)(((u64)n + TILE - 1) / TILE);
    for (;;) {  // persistent CTAs: one histogram flush per CTA, tiles numbered in claim order for the look-back
        __syncthreads();
        if (tid == 0) s_tile = atomicAdd(tile_counter, 1u);
        __syncthreads();
        const u32 tile = s_tile;
        if (tile >= ntiles) break;
        {   // L2 prefetch of the tile this CTA is likely to claim next, both streams (as in the radix pass)
            const u64 q = ((u64)tile + (gridDim.x * 2u) / 3u) * TILE;
            if (q + TILE <= n && tid < TILE / 32) {
                asm volatile("prefetch.global.L2 [%0];" ::"l"(isa + q + (u64)tid * 32));
                if (q + h + TILE <= n) asm volatile("prefetch.global.L2 [%0];" ::"l"(isa + q + h + (u64)tid * 32));
            }
        }
        const u64 i0 = (u64)tile * TILE + (u64)tid * ITEMS;  // blocked: a thread owns ITEMS consecutive suffixes
        u32 r1[ITEMS], r2[ITEMS];
        if (i0 + ITEMS <= n) {
            const uint4* v = reinterpret_cast<const uint4*>(isa + i0);
#pragma unroll
            for (int k = 0; k < ITEMS / 4; ++k) {
                const uint4 q = v[k];
                r1[4 * k] = q.x;
                r1[4 * k + 1] = q.y;
                r1[4 * k + 2] = q.z;
                r1[4 * k + 3] = q.w;
            }
        } else {
#pragma unroll
            for (int k = 0; k < ITEMS; ++k) r1[k] = i0 + k < n ? isa[i0 + k] : 0u;
        }
        u32 act = 0;
#pragma unroll
        for (int k = 0; k < ITEMS; ++k)
            if (r1[k] & tag) act |= 1u << k;
        const u64 j0 = i0 + h;
        if (act) {
            if ((h & 3) == 0 && j0 + ITEMS <= n) {
                const uint4* v = reinterpret_cast<const uint4*>(isa + j0);
#pragma unroll
                for (int k = 0; k < ITEMS / 4; ++k) {
                    const uint4 q = v[k];
                    r2[4 * k] = (q.x & ~tag) + 1u;
                    r2[4 * k + 1] = (q.y & ~tag) + 1u;
                    r2[4 * k + 2] = (q.z & ~tag) + 1u;
                    r2[4 * k + 3] = (q.w & ~tag) + 1u;
                }
            } else {
#pragma unroll
                for (int k = 0; k < ITEMS; ++k) r2[k] = (((act >> k) & 1u) && j0 + k < n) ? (__ldg(isa + j0 + k) & ~tag) + 1u : 0u;
            }
        }
        // exclusive scan of the active counts: thread -> warp -> tile -> look-back on one self-flagged word
        const u32 mine = __popc(act);
        u32 incl = mine;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const u32 t = __shfl_up_sync(0xffffffffu, incl, o);
            if (lane >= o) incl += t;
        }
        if (lane == 31) s_warp[warp] = incl;
        __syncthreads();
        u32 wprefix = 0;
        for (int w = 0; w < warp; ++w) wprefix += s_warp[w];
        if (warp == 0) {
            u32 total = 0;
            for (int w = 0; w < WARPS; ++w) total += s_warp[w];
            u64* word = scan_words + (size_t)tile * 4 + 2;
            u32 excl = 0;
            if (tile == 0) {
                if (lane == 0) st_relaxed(word, ((u64)2 << 62) | total);
            } else {
                if (lane == 0) st_relaxed(word, ((u64)1 << 62) | total);
                int base = (int)tile - 1;
                for (;;) {
                    const int t = base - lane;
                    u64 w2 = (u64)2 << 62;
                    if (t >= 0) {
                        const u64* theirs = scan_words + (size_t)t * 4 + 2;
                        do { w2 = ld_relaxed(theirs); } while ((w2 >> 62) == 0);
                    }
                    const u32 im = __ballot_sync(0xffffffffu, (w2 >> 62) == 2);
                    const int first = im ? (__ffs(im) - 1) : 31;
                    excl += __reduce_add_sync(0xffffffffu, lane <= first ? (u32)w2 : 0u);
                    if (im) break;
                    base -= 32;
                }
                if (lane == 0) st_relaxed(word, ((u64)2 << 62) | (excl + total));
            }
            if (lane == 0) {
                s_excl = excl;
                s_total = total;
                if (tile + 1 == ntiles) *out_count = excl + total;
            }
        }
        // stage the tile's keys compacted in shared memory, then write them out lane-consecutively
        u32 lq = wprefix + incl - mine;
#pragma unroll
        for (int k = 0; k < ITEMS; ++k) {
            if ((act >> k) & 1u) {
                const u64 key = ((u64)((r1[k] & ~tag) >> 1) << kb) | r2[k];
                s_key[stage_pad64(lq)] = key;
                s_id[stage_pad32(lq)] = (u32)(i0 + k);
                hist_add_key(s_hist, key, 0, num_passes);
                ++lq;
            }
        }
        __syncthreads();
        const u32 total = s_total, excl = s_excl;
        for (u32 i = tid; i < total; i += THREADS) {
            keys_out[excl + i] = s_key[stage_pad64(i)];
            ids_out[excl + i] = s_id[stage_pad32(i)];
        }
    }
    __syncthreads();
    hist_flush(s_hist, g_hist, num_passes, tid, THREADS);
}

// Round 1 after a pruned round 0 with few survivors: no rank array exists yet (round 0 scatters none), and
// filling even the needed part of it means a pass over the whole suffix array.  The rank of suffix
// j = i+h after round 0 is the slot of the head of its tie group, which can be read off the SORTED
// round-0 keys directly: lower bound of j's key prefix, then past the (at most Kc-1) short suffixes that
// tie with it.  ~log2(n) dependent reads per survivor instead of a 4n-byte sweep.
template <int THREADS>
__global__ void __launch_bounds__(THREADS)
k_build_keys_search(const u32* __restrict__ ids, const u32* __restrict__ ranks, u32 m, u32 n, u64 h, int kb,
                    const u64* __restrict__ sorted_keys, const u32* __restrict__ sorted_ids, const u8* __restrict__ text,
                    const u8* __restrict__ lut, int s_bits, int K, int Kc, int drop, u64* __restrict__ keys_out,
                    u32* __restrict__ g_hist, int num_passes) {
    __shared__ u32 s_hist[kMaxPasses * kRadix];
    __shared__ u8 s_lut[256];
    const int tid = threadIdx.x;
    hist_clear(s_hist, tid, THREADS);
    for (int i = tid; i < 256; i += THREADS) s_lut[i] = lut[i];
    __syncthreads();
    const u64 p = (u64)blockIdx.x * THREADS + tid;
    if (p < m) {
        const u64 j = (u64)ids[p] + h;
        u32 r2 = 0;
        if (j < n) {
            // key prefix of suffix j exactly as the initial key builder packs it (MSB-aligned, zero padded)
            u64 kj = 0;
            for (int c = 0; c < K; ++c) {
                const u64 pos = j + c;
                kj = (kj << s_bits) | (pos < n && c < Kc ? (u64)s_lut[text[pos]] : 0ull);
            }
            kj <<= (64 - s_bits * K);
            const u64 want = kj >> drop;
            u32 lo = 0, hi = n;  // first slot whose sorted prefix is >= want
            while (lo < hi) {
                const u32 mid = lo + ((hi - lo) >> 1);
                if ((sorted_keys[mid] >> drop) < want) lo = mid + 1;
                else hi = mid;
            }
            const u64 short_from = (u64)n >= (u64)Kc ? (u64)n - Kc + 1 : 0;
            u32 slot = lo;
            if (j >= short_from) {
                while (slot < n && sorted_ids[slot] != (u32)j) ++slot;          // a short suffix is its own group
            } else {
                while (slot < n && (sorted_keys[slot] >> drop) == want && sorted_ids[slot] >= short_from) ++slot;  // skip tied shorts
            }
            r2 = slot + 1;
        }
        const u64 key = ((u64)(ranks[p] >> 1) << kb) | r2;
        keys_out[p] = key;
        hist_add_key(s_hist, key, 0, num_passes);
    }
    __syncthreads();
    hist_flush(s_hist, g_hist, num_passes, tid, THREADS);
}

// ---- re-rank + compaction: one decoupled look-back scan ------------------------------------------
// Input: the active list sorted by key.  A "new head" starts a run of equal keys (= a group of
// suffixes still tied after 2h symbols); an "old head" starts a run of equal key>>kb (the group the
// run was split from).  With gs/hs the indices of the latest old/new head at or before p:
//     new rank(p) = old rank + (hs - gs)        (= global SA slot of the new group's first member)
// A new group of size 1 is settled: SA[rank] = id, and it is dropped from the active list.
// The scan carries (latest old head + 1, latest new head + 1, survivors so far).
struct ScanTriple {
    u32 gs1, hs1, cnt;
};
__device__ __forceinline__ ScanTriple scan_combine(ScanTriple a, ScanTriple b) {  // a earlier, b later
    ScanTriple r;
    r.gs1 = max(a.gs1, b.gs1);
    r.hs1 = max(a.hs1, b.hs1);
    r.cnt = a.cnt + b.cnt;
    return r;
}
__device__ __forceinline__ ScanTriple shfl_up_triple(ScanTriple v, int o) {
    ScanTriple r;
    r.gs1 = __shfl_up_sync(0xffffffffu, v.gs1, o);
    r.hs1 = __shfl_up_sync(0xffffffffu, v.hs1, o);
    r.cnt = __shfl_up_sync(0xffffffffu, v.cnt, o);
    return r;
}
// Scan tile descriptors: three self-describing 64-bit words per tile, one per scanned quantity:
// [flag:2 | value:32], flag 0 = empty, 1 = tile aggregate, 2 = inclusive prefix.  Value and flag
// travel in one word, so relaxed gpu-scope accesses suffice and no fence sits on the look-back
// path (the first version published a 16-byte payload behind a flag with three __threadfence()
// per tile and ran at 1.2 TB/s, profiles/r1_ncu_c5_c3_v2.md).  The three words of a tile may be
// observed in different states; each quantity is therefore resolved independently.
template <int TILE>
constexpr size_t kRerankSmem = (size_t)stage_pad32(TILE) * 8;
struct ScanTileState {
    u64* words;  // [tiles][4]  (gs1, hs1, cnt, pad)
};
constexpr int kScanWordsPerTile = 4;
constexpr int kLookbackWarps = 4;  // 32 x this many predecessor tiles polled per look-back step
__device__ __forceinline__ u64 scan_pack(u32 flag, u32 value) { return ((u64)flag << 62) | value; }

// PAIRS (large rounds >= 1): changed ranks are not scattered into isa[] here.  The tile partitions its
// (id, new rank) updates by bucket = id >> pair_shift in shared memory and appends each bucket's run to that
// bucket's region of pair_ids/pair_vals (region b starts at element b << pair_shift and can hold every id
// of the bucket; pair_hist[b] is its fill cursor).  The bucketed scatter that follows reads the regions.
// A chain-free form of rounds >= 1 (flags and tile aggregates, a scan over the aggregates, then an apply kernel) was
// measured equal to this one (C3 45.1 vs 44.6 ms, C5 33.0 vs 32.9, C4 345.5 vs 345.2: what bounds the re-rank of a large
// round is the apply phase - shared-memory partition and scattered stores - not the chain, profiles/r2_rejected.md).
template <int THREADS, int ITEMS, bool ROUND0, bool PAIRS>
__global__ void __launch_bounds__(THREADS, 1024 / THREADS)
k_rerank(const u64* __restrict__ keys, const u32* __restrict__ ids, const u32* __restrict__ ranks_in, u32 m, u32 n, int K, int kb,
         u32* __restrict__ isa, u32* __restrict__ sa, u32* __restrict__ out_ids, u32* __restrict__ out_ranks, ScanTileState ts,
         u32* __restrict__ tile_counter, u32* __restrict__ out_count, u32* __restrict__ pair_ids,
         u32* __restrict__ pair_vals, u32* __restrict__ pair_hist, int pair_shift, const u8* __restrict__ text,
         u8* __restrict__ bwt_inline, u64* __restrict__ origin, u32 prefetch_ahead, u32 tag) {
    constexpr int TILE = THREADS * ITEMS;
    constexpr int WARPS = THREADS / 32;
    static_assert(TILE / 8 <= THREADS, "one prefetch per thread covers the tile");
    static_assert(THREADS / 32 <= 32, "warp aggregates are combined by one loop per thread");
    __shared__ ScanTriple s_warp[WARPS];
    __shared__ ScanTriple s_excl;
    __shared__ u32 s_tile;
    __shared__ u64 s_lb[2][kLookbackWarps][3];
    extern __shared__ __align__(16) u32 smem_rerank[];  // kRerankSmem<TILE> bytes
    u32* s_oid = smem_rerank;         // this tile's survivors, staged for coalesced stores
    u32* s_ork = smem_rerank + stage_pad32(TILE);
    __shared__ u32 s_tile_cnt;
    __shared__ u32 s_bhist[PAIRS ? 256 : 1], s_bcur[PAIRS ? 256 : 1], s_goff[PAIRS ? 256 : 1];
    __shared__ u32 s_bwarp[8], s_btotal;
    static_assert(WARPS >= kLookbackWarps, "look-back warps");
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    if (tid == 0) s_tile = atomicAdd(tile_counter, 1u);
    if (PAIRS)
        for (int i = tid; i < 256; i += THREADS) s_bhist[i] = 0;
    __syncthreads();
    const u32 tile = s_tile;
    const u64 p0 = (u64)tile * TILE + (u64)tid * ITEMS;  // blocked arrangement
    {
        // pull the input of the tile that will be claimed ~one wave from now into L2: a tile's lifetime is
        // load latency + look-back, and only two CTAs fit on an SM
        const u64 q0 = ((u64)tile + prefetch_ahead) * TILE;
        if (q0 + TILE <= m) {
            const void* a = nullptr;
            if (tid < TILE / 16) a = keys + q0 + (u64)tid * 16;  // 128 B lines
            else if (tid < TILE / 16 + TILE / 32) a = ids + q0 + (u64)(tid - TILE / 16) * 32;
            else if (!ROUND0 && tid < TILE / 16 + TILE / 16) a = ranks_in + q0 + (u64)(tid - TILE / 16 - TILE / 32) * 32;
            if (a) asm volatile("prefetch.global.L2 [%0];" ::"l"(a));
        }
    }

    // keys[p0-1 .. p0+ITEMS], ids[p0 .. p0+ITEMS) (+ neighbours in round 0)
    u64 key[ITEMS + 2];
    u32 id[ITEMS + 2];
    if (p0 + ITEMS <= m) {
        const ulonglong2* kv = reinterpret_cast<const ulonglong2*>(keys + p0);
#pragma unroll
        for (int k = 0; k < ITEMS / 2; ++k) {
            const ulonglong2 q = kv[k];
            key[1 + 2 * k] = q.x;
            key[2 + 2 * k] = q.y;
        }
        if (ROUND0) {
            const uint4* iv = reinterpret_cast<const uint4*>(ids + p0);
#pragma unroll
            for (int k = 0; k < ITEMS / 4; ++k) {
                const uint4 q = iv[k];
                id[1 + 4 * k] = q.x;
                id[2 + 4 * k] = q.y;
                id[3 + 4 * k] = q.z;
                id[4 + 4 * k] = q.w;
            }
        }
    } else {
#pragma unroll
        for (int k = 0; k < ITEMS; ++k) {
            key[1 + k] = (p0 + k < m) ? keys[p0 + k] : 0;
            if (ROUND0) id[1 + k] = (p0 + k < m) ? ids[p0 + k] : 0;
        }
    }
    key[0] = (p0 > 0 && p0 - 1 < m) ? keys[p0 - 1] : 0;
    key[ITEMS + 1] = (p0 + ITEMS < m) ? keys[p0 + ITEMS] : 0;
    if (ROUND0) {
        id[0] = (p0 > 0 && p0 - 1 < m) ? ids[p0 - 1] : 0;
        id[ITEMS + 1] = (p0 + ITEMS < m) ? ids[p0 + ITEMS] : 0;
    }

    // Old group ranks (rounds >= 1).  The key carries only rank>>1 in its high part — active groups
    // have at least two members, so their head slots differ by >= 2 and rank>>1 is still strictly
    // increasing from group to group; that saves a key bit (8 -> 7 radix passes at n = 2^28).  The exact
    // rank comes from the list itself: sorting permutes elements only inside their group, and every
    // member of a group holds the same rank, so ranks_in[p] is the rank of whatever lands at index p.
    u32 rold[ITEMS];
    // head flags for p0 .. p0+ITEMS (the last one is the look-ahead of item ITEMS-1)
    const u32 short_from = n >= (u32)K ? n - (u32)K + 1u : 0u;  // suffix i is "short" (key padded) iff i >= short_from
    const u32 navail = p0 >= m ? 0u : (u32)min((u64)ITEMS + 1, (u64)m - p0);  // of p0 .. p0+ITEMS, how many are inside the list
    const u32 nvalid = min(navail, (u32)ITEMS);                                // ... of this thread's own ITEMS elements
    u64 hi[ITEMS + 2];  // the compared key part: bits above kb
#pragma unroll
    for (int k = 0; k < ITEMS + 2; ++k) hi[k] = key[k] >> kb;
    u32 newh = 0, oldh = 0;  // bit k: element p0+k starts a new / an old group
#pragma unroll
    for (int k = 0; k <= ITEMS; ++k) {
        bool nh, oh;
        if (ROUND0) {
            // round 0 sorted only the bits above kb (pass pruning): ties on those bits are groups
            nh = hi[k + 1] != hi[k] || id[k + 1] >= short_from || id[k] >= short_from;
            oh = false;
        } else {
            nh = key[k + 1] != key[k];
            oh = hi[k + 1] != hi[k];
        }
        newh |= (nh ? 1u : 0u) << k;
        oldh |= (oh ? 1u : 0u) << k;
    }
    // list boundaries: position 0 and everything from m on are heads
    if (p0 == 0) {
        newh |= 1u;
        oldh |= 1u;
    }
    if (navail < (u32)ITEMS + 1u) {  // p0+k >= m for k >= navail
        const u32 tail = ~((1u << navail) - 1u) & ((2u << ITEMS) - 1u);
        newh |= tail;
        oldh |= tail;
    }

    // thread aggregate, from the flag words: latest old/new head among the valid elements, survivors
    ScanTriple agg = {0u, 0u, 0u};
    {
        const u32 vmask = (1u << nvalid) - 1u;
        const u32 oh = oldh & vmask, nh = newh & vmask;
        if (oh) agg.gs1 = (u32)p0 + (32u - __clz(oh));  // index of the highest set bit, plus one
        if (nh) agg.hs1 = (u32)p0 + (32u - __clz(nh));
        const u32 singles = newh & (newh >> 1) & vmask;  // head whose successor is a head too
        agg.cnt = nvalid - __popc(singles);
    }
    // block-wide exclusive scan of the thread aggregates
    ScanTriple incl = agg;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        ScanTriple t = shfl_up_triple(incl, o);
        if (lane >= o) incl = scan_combine(t, incl);
    }
    if (lane == 31) s_warp[warp] = incl;
    __syncthreads();
    if (!ROUND0) {
        // Rounds >= 1: the head flags need the keys only.  The ids and the old ranks are fetched AFTER the tile's
        // aggregate is on its way (below), so that fewer bytes stand between a tile's start and its publish — every later
        // tile's look-back waits for the slowest recent tile to publish (profiles/r1_ncu_rerank_final.md) — and their
        // latency hides behind the look-back.
        if (p0 + ITEMS <= m) {
            const uint4* iv = reinterpret_cast<const uint4*>(ids + p0);
#pragma unroll
            for (int k = 0; k < ITEMS / 4; ++k) {
                const uint4 q = iv[k];
                id[1 + 4 * k] = q.x;
                id[2 + 4 * k] = q.y;
                id[3 + 4 * k] = q.z;
                id[4 + 4 * k] = q.w;
            }
            const uint4* rv = reinterpret_cast<const uint4*>(ranks_in + p0);
#pragma unroll
            for (int k = 0; k < ITEMS / 4; ++k) {
                const uint4 q = rv[k];
                rold[4 * k] = q.x;
                rold[4 * k + 1] = q.y;
                rold[4 * k + 2] = q.z;
                rold[4 * k + 3] = q.w;
            }
        } else {
#pragma unroll
            for (int k = 0; k < ITEMS; ++k) {
                id[1 + k] = (p0 + k < m) ? ids[p0 + k] : 0u;
                rold[k] = (p0 + k < m) ? ranks_in[p0 + k] : 0u;
            }
        }
    }
    ScanTriple wprefix = {0u, 0u, 0u};
    for (int w = 0; w < warp; ++w) wprefix = scan_combine(wprefix, s_warp[w]);
    ScanTriple texcl = shfl_up_triple(incl, 1);
    if (lane == 0) texcl = ScanTriple{0u, 0u, 0u};
    texcl = scan_combine(wprefix, texcl);  // exclusive prefix of this thread inside the tile

    // tile aggregate -> publish, look back.  The scan does almost no arithmetic per tile, so every
    // resident CTA soon waits on its predecessors and throughput becomes (window x tile) elements per
    // L2 round trip: the "inclusive prefix known" frontier advances one window per polling step.  A
    // 32-tile window of 2,048-element tiles ran at 1.5-1.9 TB/s (profiles/r1_ncu_c5_c3_v2.md), hence
    // kLookbackWarps warps poll kLookbackWarps*32 predecessors per step and the tiles are 4,096 wide.
    if (warp < kLookbackWarps) {
        ScanTriple tile_agg = {0u, 0u, 0u};
        for (int w = 0; w < WARPS; ++w) tile_agg = scan_combine(tile_agg, s_warp[w]);
        ScanTriple excl = {0u, 0u, 0u};
        u64* mine = ts.words + (size_t)tile * kScanWordsPerTile;
        if (tile == 0) {
            if (warp == 0 && lane < 3)
                st_relaxed(mine + lane, scan_pack(2u, lane == 0 ? tile_agg.gs1 : lane == 1 ? tile_agg.hs1 : tile_agg.cnt));
        } else {
            if (warp == 0 && lane < 3)
                st_relaxed(mine + lane, scan_pack(1u, lane == 0 ? tile_agg.gs1 : lane == 1 ? tile_agg.hs1 : tile_agg.cnt));
            int base = (int)tile - 1;
            u32 pending = 7u;  // bit c set: quantity c has not met an inclusive prefix yet
            int it = 0;
            while (pending) {
                const int t = base - (warp * 32 + lane);
                u64 w0 = scan_pack(2u, 0u), w1 = w0, w2 = w0;  // virtual tiles before tile 0: inclusive identity
                if (t >= 0) {
                    const u64* theirs = ts.words + (size_t)t * kScanWordsPerTile;
                    // the three loads of a poll are issued together: one L2 round trip per poll, not three
                    do {
                        w0 = ld_relaxed(theirs + 0);
                        w1 = ld_relaxed(theirs + 1);
                        w2 = ld_relaxed(theirs + 2);
                    } while (((w0 >> 62) == 0) | ((w1 >> 62) == 0) | ((w2 >> 62) == 0));
                }
                // per warp: value up to (and including) its nearest inclusive prefix, and whether it has one
                u64 part0, part1, part2;
                {
                    const u32 im = __ballot_sync(0xffffffffu, (w0 >> 62) == 2);
                    const int first = im ? (__ffs(im) - 1) : 31;
                    part0 = (u64)__reduce_max_sync(0xffffffffu, lane <= first ? (u32)w0 : 0u) | (im ? (1ull << 63) : 0ull);
                }
                {
                    const u32 im = __ballot_sync(0xffffffffu, (w1 >> 62) == 2);
                    const int first = im ? (__ffs(im) - 1) : 31;
                    part1 = (u64)__reduce_max_sync(0xffffffffu, lane <= first ? (u32)w1 : 0u) | (im ? (1ull << 63) : 0ull);
                }
                {
                    const u32 im = __ballot_sync(0xffffffffu, (w2 >> 62) == 2);
                    const int first = im ? (__ffs(im) - 1) : 31;
                    part2 = (u64)__reduce_add_sync(0xffffffffu, lane <= first ? (u32)w2 : 0u) | (im ? (1ull << 63) : 0ull);
                }
                if (lane < 3) s_lb[it & 1][warp][lane] = lane == 0 ? part0 : lane == 1 ? part1 : part2;
                asm volatile("bar.sync 1, %0;" ::"n"(kLookbackWarps * 32) : "memory");
                // nearest window first; a quantity stops at the first warp that met an inclusive prefix
#pragma unroll
                for (int w = 0; w < kLookbackWarps; ++w) {
                    if (pending & 1u) {
                        const u64 x = s_lb[it & 1][w][0];
                        excl.gs1 = max(excl.gs1, (u32)x);
                        if (x >> 63) pending &= ~1u;
                    }
                    if (pending & 2u) {
                        const u64 x = s_lb[it & 1][w][1];
                        excl.hs1 = max(excl.hs1, (u32)x);
                        if (x >> 63) pending &= ~2u;
                    }
                    if (pending & 4u) {
                        const u64 x = s_lb[it & 1][w][2];
                        excl.cnt += (u32)x;
                        if (x >> 63) pending &= ~4u;
                    }
                }
                base -= 32 * kLookbackWarps;
                ++it;
            }
            const ScanTriple inc = scan_combine(excl, tile_agg);
            if (warp == 0 && lane < 3)
                st_relaxed(mine + lane, scan_pack(2u, lane == 0 ? inc.gs1 : lane == 1 ? inc.hs1 : inc.cnt));
        }
        if (warp == 0 && lane == 0) {
            s_excl = excl;
            s_tile_cnt = tile_agg.cnt;
            if ((u64)(tile + 1) * TILE >= m) {  // last tile: survivors in total, for the host (mapped memory) and, in
                *out_count = excl.cnt + tile_agg.cnt;  // device memory beside the tile counter, for kernels queued behind this one
                tile_counter[1] = excl.cnt + tile_agg.cnt;
            }
        }
    }
    __syncthreads();
    ScanTriple run = scan_combine(s_excl, texcl);

    // apply.  Stores are shaped for L2: a thread's 8 consecutive words leave as two 128-bit stores,
    // and the compacted survivors are staged in shared memory and written out lane-consecutively
    // (per-lane 4-byte stores at a 32 B stride cost one L2 sector operation each; the first version
    // spent its time there: 3 sector writes per element, profiles/r1_ncu_c5_c3_v2.md).
    const u32 tile_cnt0 = s_excl.cnt;  // survivors before this tile
    // bwt_inline != nullptr: BWT bytes are emitted as suffixes settle.  Round 0 emits only after a pruned initial sort
    // (kb >= 8), where the byte T[id-1] sits in the low key byte (see the radix pass); later rounds gather it.
    u32 v_sa[ITEMS], v_pid[ITEMS], v_pval[ITEMS];
    u32 v_b0 = 0, v_b1 = 0;  // round 0: the 8 BWT bytes of this thread's slots
#pragma unroll
    for (int k = 0; k < ITEMS; ++k) {
        const u64 p = p0 + k;
        v_sa[k] = 0xFFFFFFFFu;
        v_pid[k] = 0xFFFFFFFFu;
        v_pval[k] = 0u;
        if (p < m) {
            if ((oldh >> k) & 1) run.gs1 = (u32)p + 1;
            if ((newh >> k) & 1) run.hs1 = (u32)p + 1;
            const u32 r_old = ROUND0 ? 0u : rold[k];
            const u32 r_new = r_old + (run.hs1 - run.gs1);
            const u32 sid = id[k + 1];
            const bool single = ((newh >> k) & 1) && ((newh >> (k + 1)) & 1);
            // Round 0 leaves isa[] alone: if nothing survives (DNA-like blocks) the ranks are never
            // read, otherwise they are scattered afterwards.  It writes every SA slot
            // (SUF_INVALID for unsettled ones) so that the later fill can tell which slots are final.
            // isa[] entries of suffixes that stay active carry `tag` (k_build_keys_text finds them by it); a
            // suffix that settles with its rank unchanged is therefore rewritten too, to drop the tag
            // (round 0 with the bucket sink: every suffix reports its rank - its slot if settled - since isa[] is still empty)
            const bool changed = ROUND0 || r_new != r_old || (tag != 0 && single);
            const u32 r_tagged = r_new | (single ? 0u : tag);
            if (PAIRS) {
                if (changed) {
                    v_pid[k] = sid;
                    atomicAdd(&s_bhist[sid >> pair_shift], 1u);
                }
                v_pval[k] = r_tagged;
            } else if (!ROUND0 && changed) {
                DARK_ASSERT(sid < n);
                isa[sid] = r_tagged;
            }
            if (ROUND0 && single) v_sa[k] = sid;
            if (bwt_inline != nullptr && single) {
                if (ROUND0) {
                    const u32 byte = (u32)key[k + 1] & 0xFFu;
                    if (k < 4) v_b0 |= byte << (8 * k);
                    else v_b1 |= byte << (8 * (k - 4));
                    if (sid == 0) *origin = p;
                } else {
                    bwt_inline[r_new] = __ldg(text + (sid == 0 ? n - 1 : sid - 1));
                    if (sid == 0) *origin = r_new;
                }
            }
            if (single) {
                DARK_ASSERT(r_new < n && sid < n);
                if (!ROUND0) sa[r_new] = sid;
            } else {
                const u32 lq = stage_pad32(run.cnt - tile_cnt0);  // position among this tile's survivors
                s_oid[lq] = sid;
                s_ork[lq] = r_new;
                run.cnt += 1;
            }
        }
    }
    static_assert(ITEMS == 8, "two 128-bit stores per thread");
    if (ROUND0) {
        if (p0 + ITEMS <= m && (((uintptr_t)sa) & 15) == 0) {
            uint4* o = reinterpret_cast<uint4*>(sa + p0);
            o[0] = make_uint4(v_sa[0], v_sa[1], v_sa[2], v_sa[3]);
            o[1] = make_uint4(v_sa[4], v_sa[5], v_sa[6], v_sa[7]);
        } else {
#pragma unroll
            for (int k = 0; k < ITEMS; ++k)
                if (p0 + k < m) sa[p0 + k] = v_sa[k];
        }
    }
    if (ROUND0 && bwt_inline != nullptr) {  // unsettled slots get a placeholder now and their byte when they settle
        if (p0 + ITEMS <= m && (((uintptr_t)bwt_inline) & 7) == 0) {
            *reinterpret_cast<uint2*>(bwt_inline + p0) = make_uint2(v_b0, v_b1);
        } else {
#pragma unroll
            for (int k = 0; k < ITEMS; ++k)
                if (p0 + k < m) bwt_inline[p0 + k] = (u8)((k < 4 ? v_b0 >> (8 * k) : v_b1 >> (8 * (k - 4))) & 0xFFu);
        }
    }
    __syncthreads();
    {
        const u32 tile_cnt = s_tile_cnt;
        for (u32 i = tid; i < tile_cnt; i += THREADS) {
            out_ids[tile_cnt0 + i] = s_oid[stage_pad32(i)];
            out_ranks[tile_cnt0 + i] = s_ork[stage_pad32(i)];
        }
    }
    if (PAIRS) {
        static_assert(!PAIRS || THREADS >= 256, "one thread per bucket");
        // bucket starts inside the tile; one global atomicAdd per (tile, bucket) reserves the run
        const u32 c = tid < 256 ? s_bhist[tid] : 0u;
        u32 incl = c;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const u32 t = __shfl_up_sync(0xffffffffu, incl, o);
            if (lane >= o) incl += t;
        }
        if (tid < 256 && lane == 31) s_bwarp[warp] = incl;
        __syncthreads();  // also: the survivors have left s_oid/s_ork
        if (tid < 256) {
            u32 wbase = 0;
            for (int w = 0; w < warp; ++w) wbase += s_bwarp[w];
            const u32 start = wbase + incl - c;
            s_bcur[tid] = start;
            s_goff[tid] = ((u32)tid << pair_shift) + (c ? atomicAdd(&pair_hist[tid], c) : 0u) - start;
            if (tid == 255) s_btotal = start + c;
        }
        __syncthreads();
#pragma unroll
        for (int k = 0; k < ITEMS; ++k) {
            if (v_pid[k] != 0xFFFFFFFFu) {
                const u32 q = atomicAdd(&s_bcur[v_pid[k] >> pair_shift], 1u);
                s_oid[q] = v_pid[k];
                s_ork[q] = v_pval[k];
            }
        }
        __syncthreads();
        const u32 total = s_btotal;
        for (u32 i = tid; i < total; i += THREADS) {
            const u32 v = s_oid[i];
            const u32 o = s_goff[v >> pair_shift] + i;
            pair_ids[o] = v;
            pair_vals[o] = s_ork[i];
        }
    }
}

// ---- sparse round-0 re-rank (pruned initial sort: almost every suffix settles) -------------------------------
// After a pruned round 0 of a high-entropy block (C2: 65,792 survivors of 2^28) the scan of k_rerank carries almost
// nothing, yet its look-back chain sets the kernel's pace (1.66 ms per 2^28 against 0.8 ms of memory time,
// profiles/r1_ncu_rerank_final.md).  What a SETTLED suffix writes depends on its own head flags only, so the tiles
// run without any chain: k_rerank0_sparse writes the SA slots and BWT bytes of the singletons and one survivor bit
// per slot; the few survivors are then listed in slot order from the bitmap (count / scan / positions) and each
// finds its group head by walking left over equal keys (k_sparse_finalize).  The driver falls back to k_rerank when
// more than n/16 suffixes survive or a group turns out longer than kSparseMaxWalk.
template <int THREADS, int ITEMS>
__global__ void __launch_bounds__(THREADS, 1024 / THREADS)
k_rerank0_sparse(const u64* __restrict__ keys, const u32* __restrict__ ids, u32 n, int K, int kb, u32* __restrict__ sa,
                 u8* __restrict__ bwt_inline, u64* __restrict__ origin, u8* __restrict__ surv_bits, u32* __restrict__ surv_total) {
    static_assert(ITEMS == 8, "one survivor byte and two 128-bit SA stores per thread");
    constexpr int TILE = THREADS * ITEMS;
    const int tid = threadIdx.x;
    const u32 m = n;
    const u64 p0 = (u64)blockIdx.x * TILE + (u64)tid * ITEMS;
    if (p0 >= m) return;
    u64 key[ITEMS + 2];
    u32 id[ITEMS + 2];
    if (p0 + ITEMS <= m) {
        const ulonglong2* kv = reinterpret_cast<const ulonglong2*>(keys + p0);
#pragma unroll
        for (int k = 0; k < ITEMS / 2; ++k) {
            const ulonglong2 q = kv[k];
            key[1 + 2 * k] = q.x;
            key[2 + 2 * k] = q.y;
        }
        const uint4* iv = reinterpret_cast<const uint4*>(ids + p0);
#pragma unroll
        for (int k = 0; k < ITEMS / 4; ++k) {
            const uint4 q = iv[k];
            id[1 + 4 * k] = q.x;
            id[2 + 4 * k] = q.y;
            id[3 + 4 * k] = q.z;
            id[4 + 4 * k] = q.w;
        }
    } else {
#pragma unroll
        for (int k = 0; k < ITEMS; ++k) {
            key[1 + k] = (p0 + k < m) ? keys[p0 + k] : 0;
            id[1 + k] = (p0 + k < m) ? ids[p0 + k] : 0;
        }
    }
    key[0] = p0 > 0 ? keys[p0 - 1] : 0;
    key[ITEMS + 1] = (p0 + ITEMS < m) ? keys[p0 + ITEMS] : 0;
    id[0] = p0 > 0 ? ids[p0 - 1] : 0;
    id[ITEMS + 1] = (p0 + ITEMS < m) ? ids[p0 + ITEMS] : 0;
    // head flags exactly as k_rerank<ROUND0> computes them
    const u32 short_from = n >= (u32)K ? n - (u32)K + 1u : 0u;
    const u32 navail = (u32)min((u64)ITEMS + 1, (u64)m - p0);
    const u32 nvalid = min(navail, (u32)ITEMS);
    u32 newh = 0;
#pragma unroll
    for (int k = 0; k <= ITEMS; ++k) {
        const bool nh = (key[k + 1] >> kb) != (key[k] >> kb) || id[k + 1] >= short_from || id[k] >= short_from;
        newh |= (nh ? 1u : 0u) << k;
    }
    if (p0 == 0) newh |= 1u;
    if (navail < (u32)ITEMS + 1u) newh |= ~((1u << navail) - 1u) & ((2u << ITEMS) - 1u);
    const u32 vmask = (1u << nvalid) - 1u;
    const u32 singles = newh & (newh >> 1) & vmask;
    u32 v_sa[ITEMS];
    u32 v_b0 = 0, v_b1 = 0;
#pragma unroll
    for (int k = 0; k < ITEMS; ++k) {
        const bool single = (singles >> k) & 1u;
        v_sa[k] = single ? id[k + 1] : 0xFFFFFFFFu;
        if (single) {
            const u32 byte = (u32)key[k + 1] & 0xFFu;
            if (k < 4) v_b0 |= byte << (8 * k);
            else v_b1 |= byte << (8 * (k - 4));
            if (id[k + 1] == 0) *origin = p0 + k;
        }
    }
    if (p0 + ITEMS <= m && (((uintptr_t)sa) & 15) == 0) {
        uint4* o = reinterpret_cast<uint4*>(sa + p0);
        o[0] = make_uint4(v_sa[0], v_sa[1], v_sa[2], v_sa[3]);
        o[1] = make_uint4(v_sa[4], v_sa[5], v_sa[6], v_sa[7]);
    } else {
#pragma unroll
        for (int k = 0; k < ITEMS; ++k)
            if (p0 + k < m) sa[p0 + k] = v_sa[k];
    }
    if (p0 + ITEMS <= m && (((uintptr_t)bwt_inline) & 7) == 0) {
        *reinterpret_cast<uint2*>(bwt_inline + p0) = make_uint2(v_b0, v_b1);
    } else {
#pragma unroll
        for (int k = 0; k < ITEMS; ++k)
            if (p0 + k < m) bwt_inline[p0 + k] = (u8)((k < 4 ? v_b0 >> (8 * k) : v_b1 >> (8 * (k - 4))) & 0xFFu);
    }
    const u32 surv = ~singles & vmask;
    surv_bits[p0 >> 3] = (u8)surv;
    if (surv) atomicAdd(surv_total, (u32)__popc(surv));
}

constexpr u32 kSparseChunk = 4096;   // bitmap bytes per CTA of the compaction kernels (256 threads x 16 bytes)
constexpr u32 kSparseMaxWalk = 64;   // longest group the sparse path resolves itself
__device__ __forceinline__ uint4 sparse_load16(const u8* __restrict__ bits, u64 nbytes, u64 c0) {
    if (c0 + 16 <= nbytes) return *reinterpret_cast<const uint4*>(bits + c0);
    u32 w[4] = {0u, 0u, 0u, 0u};
    for (u32 e = 0; e < 16; ++e)
        if (c0 + e < nbytes) w[e >> 2] |= (u32)bits[c0 + e] << (8 * (e & 3));
    return make_uint4(w[0], w[1], w[2], w[3]);
}
__global__ void __launch_bounds__(256) k_sparse_count(const u8* __restrict__ bits, u64 nbytes, u32* __restrict__ counts) {
    __shared__ u32 s_sum;
    if (threadIdx.x == 0) s_sum = 0;
    __syncthreads();
    const u64 c0 = (u64)blockIdx.x * kSparseChunk + (u64)threadIdx.x * 16;
    u32 c = 0;
    if (c0 < nbytes) {
        const uint4 v = sparse_load16(bits, nbytes, c0);
        c = __popc(v.x) + __popc(v.y) + __popc(v.z) + __popc(v.w);
    }
    c = __reduce_add_sync(0xffffffffu, c);
    if ((threadIdx.x & 31) == 0 && c) atomicAdd(&s_sum, c);
    __syncthreads();
    if (threadIdx.x == 0) counts[blockIdx.x] = s_sum;
}
__global__ void __launch_bounds__(1024) k_sparse_scan(u32* __restrict__ counts, u32 nblocks) {  // in place: exclusive offsets
    __shared__ u32 s_warp[32];
    __shared__ u32 s_carry;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    if (tid == 0) s_carry = 0;
    __syncthreads();
    for (u32 b0 = 0; b0 < nblocks; b0 += 1024) {
        const u32 i = b0 + tid;
        const u32 c = i < nblocks ? counts[i] : 0u;
        u32 incl = c;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const u32 t = __shfl_up_sync(0xffffffffu, incl, o);
            if (lane >= o) incl += t;
        }
        if (lane == 31) s_warp[warp] = incl;
        __syncthreads();
        u32 wbase = 0;
        for (int w = 0; w < warp; ++w) wbase += s_warp[w];
        const u32 carry = s_carry;
        if (i < nblocks) counts[i] = carry + wbase + incl - c;
        __syncthreads();
        if (tid == 1023) s_carry = carry + wbase + incl;
        __syncthreads();
    }
}
__global__ void __launch_bounds__(256)
k_sparse_positions(const u8* __restrict__ bits, u64 nbytes, const u32* __restrict__ offsets, u32* __restrict__ pos_out) {
    __shared__ u32 s_warp[8];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const u64 c0 = (u64)blockIdx.x * kSparseChunk + (u64)tid * 16;
    uint4 v = make_uint4(0u, 0u, 0u, 0u);
    if (c0 < nbytes) v = sparse_load16(bits, nbytes, c0);
    const u32 c = __popc(v.x) + __popc(v.y) + __popc(v.z) + __popc(v.w);
    u32 incl = c;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const u32 t = __shfl_up_sync(0xffffffffu, incl, o);
        if (lane >= o) incl += t;
    }
    if (lane == 31) s_warp[warp] = incl;
    __syncthreads();
    u32 wbase = 0;
    for (int w = 0; w < warp; ++w) wbase += s_warp[w];
    u32 out = offsets[blockIdx.x] + wbase + incl - c;
    const u32 w4[4] = {v.x, v.y, v.z, v.w};
    const u64 bit0 = c0 * 8;  // slot of bit 0 of this thread's first byte
#pragma unroll
    for (int q = 0; q < 4; ++q) {
        u32 word = w4[q];
        while (word) {
            const int b = __ffs(word) - 1;
            word &= word - 1;
            pos_out[out++] = (u32)(bit0 + 32 * q + b);
        }
    }
}
// survivor j sits at slot pos[j]; its rank is the slot of its group's head: walk left while the key prefix stays equal
__global__ void __launch_bounds__(256)
k_sparse_finalize(const u32* __restrict__ pos, u32 count, const u64* __restrict__ keys, const u32* __restrict__ ids, u32 n, int K, int kb,
                  u32* __restrict__ out_ids, u32* __restrict__ out_ranks, u32* __restrict__ overflow) {
    const u32 j = blockIdx.x * 256 + threadIdx.x;
    if (j >= count) return;
    const u32 short_from = n >= (u32)K ? n - (u32)K + 1u : 0u;
    const u32 p = pos[j];
    const u32 id = ids[p];
    const u64 hk = keys[p] >> kb;
    u32 q = p, steps = 0;
    // slot q is not a head iff slot q-1 has the same key prefix and neither suffix is short (k_rerank<ROUND0>)
    while (q > 0 && id < short_from) {
        if ((keys[q - 1] >> kb) != hk || ids[q - 1] >= short_from) break;
        --q;
        if (++steps > kSparseMaxWalk) {
            *overflow = 1;
            break;
        }
    }
    out_ids[j] = id;
    out_ranks[j] = q;
}
__global__ void k_copy_u32(const u32* __restrict__ src, u32* __restrict__ dst) { *dst = *src; }

// Deferred rank scatter of round 0 (only launched when suffixes survive round 0):
// settled slots give isa[SA[p]] = p, survivors give isa[id] = rank of their group.
template <int THREADS>
__global__ void __launch_bounds__(THREADS)
k_round0_isa(const u32* __restrict__ sa, u32 n, const u32* __restrict__ act_ids, const u32* __restrict__ act_ranks, u32 m,
             u32* __restrict__ isa, u32 tag) {
    const u64 p = (u64)blockIdx.x * THREADS + threadIdx.x;
    if (p < n) {
        const u32 v = ld_stream(sa + p);
        if (v != 0xFFFFFFFFu) isa[v] = (u32)p;
    }
    if (p < m) isa[ld_stream(act_ids + p)] = ld_stream(act_ranks + p) | tag;
}

// Rank scatter of the survivors alone: isa[id] = rank of its group (m elements).
template <int THREADS>
__global__ void __launch_bounds__(THREADS)
k_scatter_ranks(const u32* __restrict__ act_ids, const u32* __restrict__ act_ranks, u32 m, u32* __restrict__ isa, u32 tag) {
    const u64 p = (u64)blockIdx.x * THREADS + threadIdx.x;
    if (p < m) isa[ld_stream(act_ids + p)] = ld_stream(act_ranks + p) | tag;
}

// Scatter of bucket regions filled by the PAIRS re-rank: region b holds counts[b] pairs from element
// b << shift on.  chunk_prefix[b] = number of kRegionChunk-sized chunks in the regions before b (k_region_chunks);
// block x finds its (bucket, chunk) in it.  The grid is the host-side bound ceil(m / chunk) + 256.
constexpr u32 kRegionChunk = 1024;  // one 128-bit load pair and four stores per thread
__global__ void __launch_bounds__(256) k_region_chunks(const u32* __restrict__ counts, u32* __restrict__ chunk_prefix) {
    __shared__ u32 s_warp[8];
    const int d = threadIdx.x, lane = d & 31, warp = d >> 5;
    const u32 c = (counts[d] + kRegionChunk - 1) / kRegionChunk;
    u32 incl = c;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const u32 t = __shfl_up_sync(0xffffffffu, incl, o);
        if (lane >= o) incl += t;
    }
    if (lane == 31) s_warp[warp] = incl;
    __syncthreads();
    u32 base = 0;
    for (int w = 0; w < warp; ++w) base += s_warp[w];
    chunk_prefix[d] = base + incl - c;
    if (d == 255) chunk_prefix[256] = base + incl;
}
__global__ void __launch_bounds__(256)
k_scatter_regions(const u32* __restrict__ ids, const u32* __restrict__ vals, const u32* __restrict__ counts,
                  const u32* __restrict__ chunk_prefix, int shift, u32* __restrict__ isa) {
    __shared__ u32 s_prefix[257];
    const int tid = threadIdx.x;
    s_prefix[tid] = chunk_prefix[tid];
    if (tid == 0) s_prefix[256] = chunk_prefix[256];
    __syncthreads();
    const u32 x = blockIdx.x;
    if (x >= s_prefix[256]) return;
    int lo = 0, hi = 255;  // last bucket whose prefix is <= x (empty buckets share a prefix with their successor)
    while (lo < hi) {
        const int mid = (lo + hi + 1) >> 1;
        if (s_prefix[mid] <= x) lo = mid;
        else hi = mid - 1;
    }
    const u32 b = (u32)lo;
    const u32 first = (x - s_prefix[b]) * kRegionChunk, count = counts[b];
    const u64 base = ((u64)b << shift) + first;
    const u32 len = min(kRegionChunk, count - first);
    const bool vec = (base & 3) == 0;  // regions of tiny blocks (shift < 2) may start unaligned
    for (u32 q = tid * 4; q < len; q += 256 * 4) {
        if (vec && q + 4 <= len) {
            uint4 i4, v4;
            asm volatile("ld.global.cs.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(i4.x), "=r"(i4.y), "=r"(i4.z), "=r"(i4.w) : "l"(ids + base + q));
            asm volatile("ld.global.cs.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(v4.x), "=r"(v4.y), "=r"(v4.z), "=r"(v4.w) : "l"(vals + base + q));
            DARK_ASSERT((i4.x >> shift) == b && (i4.y >> shift) == b && (i4.z >> shift) == b && (i4.w >> shift) == b);
            isa[i4.x] = v4.x;
            isa[i4.y] = v4.y;
            isa[i4.z] = v4.z;
            isa[i4.w] = v4.w;
        } else {
            for (u32 e = q; e < min(q + 4, len); ++e) isa[ids[base + e]] = vals[base + e];
        }
    }
}

// Selective rank fill (few survivors after round 0): the next round reads isa[i+h] for the
// active i only, so mark those positions in an n-bit map (L2-resident: n/8 bytes) ...
template <int THREADS>
__global__ void __launch_bounds__(THREADS)
k_mark_needed(const u32* __restrict__ act_ids, u32 m, u32 n, u64 h, u32* __restrict__ bitmap) {
    const u64 p = (u64)blockIdx.x * THREADS + threadIdx.x;
    if (p >= m) return;
    const u64 j = (u64)ld_stream(act_ids + p) + h;
    if (j < n) atomicOr(bitmap + (j >> 5), 1u << (j & 31));
}
// ... then stream over the suffix array once and write the rank (= slot) of the marked suffixes
// that are already settled.  Unsettled ones had their rank scattered as survivors.
template <int THREADS>
__global__ void __launch_bounds__(THREADS)
k_fill_needed(const u32* __restrict__ sa, u32 n, const u32* __restrict__ bitmap, u32* __restrict__ isa) {
    const u64 p = (u64)blockIdx.x * THREADS + threadIdx.x;
    if (p >= n) return;
    const u32 v = ld_stream(sa + p);
    if (v != 0xFFFFFFFFu && ((__ldg(bitmap + (v >> 5)) >> (v & 31)) & 1u)) isa[v] = (u32)p;
}

// ---- bucketed rank scatter --------------------------------------------------------------------------
// isa[id] = rank over ids in SA order is a random 4-byte scatter: every store costs a 32 B sector fill
// plus write-back once isa[] outgrows L2 (17 GB of DRAM traffic for 2^28 ranks, profiles/r1_ncu_c2_v1.md).
// Large scatters are therefore done in two steps: (1) partition the (id, rank) pairs by the top 8 bits
// of id — unstable, so shared-memory atomics give the in-tile position and one global atomicAdd per
// (tile, bucket) reserves the output run: no look-back chain; (2) scatter bucket by bucket, where
// each bucket's slice of isa[] (n/256 ranks) stays in L2 and leaves as full sectors.
// VAL_IS_INDEX: the value of element i is i itself (rank of a settled suffix = its SA slot).
template <int THREADS, int ITEMS, bool VAL_IS_INDEX>
__global__ void __launch_bounds__(THREADS)
k_partition_pairs(const u32* __restrict__ ids, const u32* __restrict__ vals, u32 count, int shift, u32* __restrict__ cursor,
                  u32* __restrict__ out_ids, u32* __restrict__ out_vals, u32 or_mask) {
    constexpr int TILE = THREADS * ITEMS;
    __shared__ u32 s_ids[TILE];
    __shared__ u32 s_vals[TILE];
    __shared__ u32 s_cnt[256];
    __shared__ u32 s_start[256];
    __shared__ u32 s_goff[256];
    __shared__ u32 s_warp[8];
    static_assert(THREADS == 256, "one thread per bucket");
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    s_cnt[tid] = 0;
    __syncthreads();
    const u64 base = (u64)blockIdx.x * TILE;
    u32 id[ITEMS], val[ITEMS], pos[ITEMS];
#pragma unroll
    for (int k = 0; k < ITEMS; ++k) {
        const u64 i = base + k * THREADS + tid;
        id[k] = i < count ? ld_stream(ids + i) : 0xFFFFFFFFu;
    }
#pragma unroll
    for (int k = 0; k < ITEMS; ++k) {
        const u64 i = base + k * THREADS + tid;
        val[k] = VAL_IS_INDEX ? (u32)i : (i < count ? ld_stream(vals + i) | or_mask : 0u);
    }
#pragma unroll
    for (int k = 0; k < ITEMS; ++k) pos[k] = id[k] != 0xFFFFFFFFu ? atomicAdd(&s_cnt[id[k] >> shift], 1u) : 0u;
    __syncthreads();
    const u32 c = s_cnt[tid];
    u32 incl = c;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        u32 t = __shfl_up_sync(0xffffffffu, incl, o);
        if (lane >= o) incl += t;
    }
    if (lane == 31) s_warp[warp] = incl;
    __syncthreads();
    u32 wbase = 0;
    for (int w = 0; w < warp; ++w) wbase += s_warp[w];
    const u32 start = wbase + incl - c;
    s_start[tid] = start;
    // cursor[b] counts from 0; bucket b's region starts at element b << shift (it can hold every id of the bucket)
    s_goff[tid] = ((u32)tid << shift) + (c ? atomicAdd(&cursor[tid], c) : 0u) - start;
    u32 total = 0;
    for (int w = 0; w < 8; ++w) total += s_warp[w];
    __syncthreads();
#pragma unroll
    for (int k = 0; k < ITEMS; ++k) {
        if (id[k] != 0xFFFFFFFFu) {
            const u32 q = s_start[id[k] >> shift] + pos[k];
            s_ids[q] = id[k];
            s_vals[q] = val[k];
        }
    }
    __syncthreads();
#pragma unroll
    for (int k = 0; k < ITEMS; ++k) {
        const u32 q = k * THREADS + tid;
        if (q < total) {
            const u32 v = s_ids[q];
            const u32 o = s_goff[v >> shift] + q;
            out_ids[o] = v;
            out_vals[o] = s_vals[q];
        }
    }
}

// ---- BWT emission ---------------------------------------------------------------------------------
// bwt[j] = T[SA[j]-1]; the single j with SA[j]==0 takes T[n-1] and is the origin
// (TransformIterator; known answers /root/reference/src/saca.rs:411-412).
// HBM: 4 N read (SA, 128-bit loads), N random byte gathers (one 32 B sector each), N written.
template <int THREADS>
__global__ void __launch_bounds__(THREADS)
k_emit_bwt(const u8* __restrict__ text, u32 n, const u32* __restrict__ sa, u8* __restrict__ bwt, u64* __restrict__ origin,
           int bwt_aligned4, int sa_aligned16) {
    const u64 j0 = ((u64)blockIdx.x * THREADS + threadIdx.x) * 4;
    if (j0 >= n) return;
    u32 s[4];
    if (j0 + 4 <= n && sa_aligned16) {  // 128-bit SA loads need a 16-byte aligned SA (a caller's d_sa may be a 4-byte aligned slice)
        const uint4 q = *reinterpret_cast<const uint4*>(sa + j0);
        s[0] = q.x; s[1] = q.y; s[2] = q.z; s[3] = q.w;
    } else {
#pragma unroll
        for (int k = 0; k < 4; ++k) s[k] = (j0 + k < n) ? sa[j0 + k] : 1u;
    }
    u32 b[4];
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        const u32 pos = s[k] == 0 ? n - 1 : s[k] - 1;
        b[k] = (j0 + k < n) ? (u32)__ldg(text + pos) : 0u;
        if (s[k] == 0 && j0 + k < n) *origin = j0 + k;
    }
    if (j0 + 4 <= n && bwt_aligned4) {
        *reinterpret_cast<u32*>(bwt + j0) = b[0] | (b[1] << 8) | (b[2] << 16) | (b[3] << 24);
    } else {
#pragma unroll
        for (int k = 0; k < 4; ++k)
            if (j0 + k < n) bwt[j0 + k] = (u8)b[k];
    }
}

// Windowed emission for blocks much larger than L2: the gather T[SA[j]-1] is a random one-byte read,
// and every miss costs a 64 B DRAM granule (92 B per gather measured on C2, profiles/r1_ncu_c2_v1.md).
// The block is therefore emitted in W launches; launch w serves only the positions that fall into
// text window w (<= 64 MiB, kept in L2 with an evict_last policy) while SA and the output stream
// through with evict-first hints.  Each thread owns one aligned 4-byte output word and
// read-modify-writes it (the first launch writes without reading).
__device__ __forceinline__ u64 l2_policy_evict_last() {
    u64 pol;
    asm volatile("createpolicy.fractional.L2::evict_last.b64 %0, 1.0;" : "=l"(pol));
    return pol;
}
__device__ __forceinline__ u32 ld_u8_keep(const u8* p, u64 pol) {
    u32 v;
    asm volatile("ld.global.nc.L2::cache_hint.u8 %0, [%1], %2;" : "=r"(v) : "l"(p), "l"(pol));
    return v;
}
template <int THREADS, bool FIRST>
__global__ void __launch_bounds__(THREADS)
k_emit_bwt_window(const u8* __restrict__ text, u32 n, const u32* __restrict__ sa, u8* __restrict__ bwt, u64* __restrict__ origin,
                  u32 win_lo, u32 win_hi, int sa_aligned16) {
    const u64 j0 = ((u64)blockIdx.x * THREADS + threadIdx.x) * 4;
    if (j0 >= n) return;
    const u64 pol = l2_policy_evict_last();
    u32 s[4];
    if (j0 + 4 <= n && sa_aligned16) {
        uint4 q;
        asm volatile("ld.global.cs.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(q.x), "=r"(q.y), "=r"(q.z), "=r"(q.w) : "l"(sa + j0));
        s[0] = q.x; s[1] = q.y; s[2] = q.z; s[3] = q.w;
    } else {
#pragma unroll
        for (int k = 0; k < 4; ++k) s[k] = (j0 + k < n) ? sa[j0 + k] : 1u;
    }
    u32 pos[4];
    u32 hit = 0;
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        pos[k] = s[k] == 0 ? n - 1 : s[k] - 1;
        if (j0 + k < n && pos[k] >= win_lo && pos[k] < win_hi) hit |= 1u << k;
        if (FIRST && s[k] == 0 && j0 + k < n) *origin = j0 + k;
    }
    if (!FIRST && hit == 0) return;
    u32 b[4] = {0u, 0u, 0u, 0u};
#pragma unroll
    for (int k = 0; k < 4; ++k)
        if ((hit >> k) & 1) b[k] = ld_u8_keep(text + pos[k], pol);
    const u32 fresh = b[0] | (b[1] << 8) | (b[2] << 16) | (b[3] << 24);
    if (j0 + 4 <= n) {
        u32* out = reinterpret_cast<u32*>(bwt + j0);
        u32 word = 0;
        if (!FIRST && hit != 15u) word = ld_stream(out);
        st_stream(out, word | fresh);
    } else {
#pragma unroll
        for (int k = 0; k < 4; ++k)
            if ((hit >> k) & 1) bwt[j0 + k] = (u8)b[k];
    }
}

// ---- inverse BWT (SURVEY.md 8f: the unpack side, compress::bwt::decode at src/block/dc.rs:154-156) -------
// The rows of the forward transform are the suffixes with end-of-text lowest, i.e. the sorted rotations of
// T$ without the "$T" row.  With that row put back (row 0; its last symbol is bwt[origin]) and the row of
// suffix 0 (row origin+1) ending in '$', a STABLE partition of the n real last-column symbols by value
// gives psi: sorted slot q (= row q+1) <- the row whose last symbol it is.  Following psi from row
// origin+1 spells T forwards: T[i] = first symbol of the i-th row visited.
//   step 1  k_ibwt_elements: (symbol, row) pairs in row order            -> one radix pass -> psi
//   step 2  k_ibwt_walk<2>: every STRIDE-th row (and the head) is a splitter; one thread walks from each
//           splitter to the next: sublist length + successor splitter      (dependent random reads)
//   step 3  k_ibwt_jump: pointer jumping over the splitter list only        (n/STRIDE nodes)
//   check   k_ibwt_check: the list from the head covers all n + 1 rows
//   step 4  k_ibwt_unstash, k_ibwt_walk<1>: the text at the known offsets
// The walk, unstash and check kernels serve the many-block form too (MANY = true, "inverse BWT of many blocks" below).
__global__ void __launch_bounds__(256)
k_ibwt_elements(const u8* __restrict__ bwt, u32 n, u32 origin, u64* __restrict__ keys, u32* __restrict__ rows) {
    const u64 e = (u64)blockIdx.x * 256 + threadIdx.x;
    if (e >= n) return;
    const u32 r = e == 0 ? 0u : (e <= origin ? (u32)e : (u32)e + 1u);
    keys[e] = e == 0 ? bwt[origin] : bwt[r - 1];
    rows[e] = r;
}

constexpr u32 kIbwtNil = 0xFFFFFFFFu;

// first symbol of row r >= 1: the symbol whose bucket [base[c], base[c+1]) holds sorted slot r-1
__device__ __forceinline__ u32 ibwt_first_symbol(const u32* s_base, u32 r) {
    const u32 q = r - 1;
    u32 lo = 0, hi = 255;  // largest c with s_base[c] <= q
    while (lo < hi) {
        const u32 mid = (lo + hi + 1) >> 1;
        if (s_base[mid] <= q) lo = mid;
        else hi = mid - 1;
    }
    return lo;
}

// What only the many-block form reads (zero in the single-block instantiations; "inverse BWT of many blocks" below): block b
// is bytes [starts[b], starts[b+1]) of the BWTs with origin origins[b], and sorted slot q holds the key (b << 8) | symbol.
struct IbwtMany {
    const u32* starts;  // count + 1
    const unsigned long long* origins;
    u32 count;
    const u64* sorted_keys;
};

__device__ __forceinline__ u32 row_block_of(const u32* __restrict__ starts, u32 B, u32 row) {  // largest b with starts[b] + b <= row
    u32 lo = 0, hi = B - 1;
    while (lo < hi) {
        const u32 mid = (lo + hi + 1) >> 1;
        if (__ldg(starts + mid) + mid <= row) lo = mid;
        else hi = mid - 1;
    }
    return lo;
}
__device__ __forceinline__ u32 ibwt_many_block(const u32* __restrict__ starts, u32 B, u32 stride, u32 regular, u32 s) {
    return s < regular ? row_block_of(starts, B, s * stride) : s - regular;
}

// MODE 0: count only (sublist length + successor splitter).
// MODE 1: write the text at the known offset (second walk; with `only_longer_than` > 0 just the sublists longer than that).
// MODE 2: count AND stash the symbols of the sublist in the splitter's private chunk of `stash` (kIbwtStashCap bytes):
//         the text offset is not known yet, k_ibwt_unstash copies the chunk once it is.  One walk instead of two —
//         a walk is n dependent random reads of psi and runs at the memory system's transaction rate (~55 G/s).
// Splitter s < regular starts at row s * stride, splitter regular + b at the head row of block b.  A block b owns the rows from
// its '$' row starts[b] + b on, and psi of its row r is at psi[r - b - 1], its sorted slot.  One block (MANY = false) is block
// 0 of n bytes with origin `origin`: '$' row 0, head row origin + 1, and the first symbol of a row is found in the symbol
// bases `base` (no second load per step).  Many blocks read it from the sorted key; `n` and `origin` are then unused.
constexpr u32 kIbwtStashCap = 384;  // bytes per chunk at the default stride: sublists are ~geometric with mean `stride` (48 by default),
                                    // 0.03 % are longer and are walked again (the driver passes min(this, what the buffer allows))
template <int MODE, bool MANY>
__global__ void __launch_bounds__(128)
k_ibwt_walk(const u32* __restrict__ psi, u32 n, u32 origin, u32 stride, u32 regular, u32* __restrict__ len, u32* __restrict__ next,
            const u32* __restrict__ dist, const u32* __restrict__ base, u8* __restrict__ text_out, u32* __restrict__ len_keep,
            u32* __restrict__ stash, u32 only_longer_than, u32 cap, IbwtMany many) {
    constexpr bool WRITE = MODE == 1, COUNT = MODE != 1, STASH = MODE == 2;
    __shared__ u32 s_base[256];
    if constexpr (!MANY) {
        if (!COUNT || STASH) {
            for (int i = threadIdx.x; i < 256; i += 128) s_base[i] = base[i];
            __syncthreads();
        }
    }
    const u32 s = blockIdx.x * 128 + threadIdx.x;
    if (s > regular + (MANY ? many.count - 1 : 0u)) return;
    u32 b = 0, first = 0, nb = n, head = origin + 1;  // the block of splitter s: bytes [first, first + nb)
    if constexpr (MANY) {
        b = ibwt_many_block(many.starts, many.count, stride, regular, s);
        first = __ldg(many.starts + b);
        nb = __ldg(many.starts + b + 1) - first;
        head = first + b + (u32)__ldg(many.origins + b) + 1u;
    }
    const u32 dollar = first + b;  // the block's '$' row
    // the first symbol of row r (not the '$' row)
    auto first_symbol = [&](u32 r) -> u32 {
        if constexpr (MANY) {
            const u64 key = __ldg(many.sorted_keys + (r - b - 1));
            DARK_ASSERT((u32)(key >> 8) == b);
            return (u32)(key & 0xFFu);
        } else {
            return ibwt_first_symbol(s_base, r);
        }
    };
    u32 r = s < regular ? s * stride : head;
    if (s < regular && r == head) {  // the head row is owned by its block's head splitter
        if (COUNT) {
            len[s] = 0;
            next[s] = kIbwtNil;
            if (STASH) len_keep[s] = 0;
        }
        return;
    }
    if (WRITE && only_longer_than && len_keep[s] <= only_longer_than) return;
    u64 pos = 0;
    if (WRITE) pos = (u64)(nb + 1) - dist[s];  // block-relative text position of this splitter's row
    u32 cnt = 0;
    // WRITE: a sublist spells consecutive text positions; the bytes are gathered into aligned 32-bit words and
    // stored once per word (a byte store per step made the writing walk 9.3 ms against 5.2 ms for the counting one)
    const bool word_stores = WRITE && (((uintptr_t)text_out) & 3) == 0;
    u32 acc = 0, have = 0;
    u64 wbase = 0;  // text offset of the word being gathered
    u32* const chunk = STASH ? stash + (size_t)s * (cap / 4) : nullptr;  // cap: chunk bytes, a multiple of 4
    do {
        const u32 nx = r == dollar ? head : __ldg(psi + (r - b - 1));  // issued before the symbol is found, so the two overlap
        DARK_ASSERT(nx >= dollar && nx <= dollar + nb);
        if (WRITE && r != dollar && pos + cnt < nb) {
            const u64 q = (u64)first + pos + cnt;
            DARK_ASSERT(pos <= nb);
            const u32 sym = first_symbol(r);
            if (word_stores) {
                acc |= sym << (8 * (u32)(q & 3));
                have |= 1u << (u32)(q & 3);
                wbase = q & ~3ull;
                if ((q & 3) == 3) {
                    if (have == 0xFu) {
                        *reinterpret_cast<u32*>(text_out + (q & ~3ull)) = acc;
                    } else {
                        for (u32 e = 0; e < 4; ++e)
                            if ((have >> e) & 1u) text_out[(q & ~3ull) + e] = (u8)(acc >> (8 * e));
                    }
                    acc = 0;
                    have = 0;
                }
            } else {
                text_out[q] = (u8)sym;
            }
        }
        if (STASH && cnt < cap) {  // byte cnt of the chunk (the '$' row leaves a placeholder)
            const u32 sym = r != dollar ? first_symbol(r) : 0u;
            acc |= sym << (8 * (cnt & 3));
            if ((cnt & 3) == 3) {
                chunk[cnt >> 2] = acc;
                acc = 0;
            }
        }
        ++cnt;
        r = nx;
    } while (!(r % stride == 0 || r == head) && cnt <= nb);  // cnt bound: corrupt input must not hang
    if (WRITE && have) {  // the last, partial word of the sublist
        for (u32 e = 0; e < 4; ++e)
            if ((have >> e) & 1u) text_out[wbase + e] = (u8)(acc >> (8 * e));
    }
    if (STASH && (cnt & 3) != 0 && cnt < cap) chunk[cnt >> 2] = acc;  // partial last word: the chunk is private
    if (COUNT) {
        len[s] = cnt;
        if (STASH) len_keep[s] = cnt;
        // Only the '$' row leads to the head, so the walk that reaches it ends its block's list.  This holds for any input:
        // the rows psi lists are fixed by the origins, and the head row is not among them.  With one block that walk is
        // the one from splitter 0, the '$' row.
        next[s] = r == head ? kIbwtNil : r / stride;
    }
}

// Copy L bytes of a stash chunk to dst: with `words`, aligned 32-bit stores composed from two neighbouring chunk words,
// single bytes only at the two ends.
__device__ __forceinline__ void ibwt_copy_chunk(const u32* __restrict__ src, u8* __restrict__ dst, u32 L, bool words) {
    auto byte_at = [&](u32 i) { return (u8)(src[i >> 2] >> (8 * (i & 3))); };
    u32 i = 0;
    if (words) {
        while ((((uintptr_t)dst + i) & 3) != 0 && i < L) {
            dst[i] = byte_at(i);
            ++i;
        }
        const u32 sh = 8 * (i & 3);  // constant from here on: source and destination differ by a fixed byte offset
        for (; i + 4 <= L; i += 4) {
            const u32 lo = src[i >> 2], hi = sh ? src[(i >> 2) + 1] : 0u;  // (the word after the last is inside the chunk or unused)
            *reinterpret_cast<u32*>(dst + i) = sh ? __funnelshift_r(lo, hi, sh) : lo;
        }
    }
    for (; i < L; ++i) dst[i] = byte_at(i);
}

// Copy every stashed sublist (length <= cap) to its place in the text.
template <bool MANY>
__global__ void __launch_bounds__(128)
k_ibwt_unstash(const u32* __restrict__ stash, const u32* __restrict__ len_keep, const u32* __restrict__ dist, u32 n, u32 stride,
               u32 regular, u8* __restrict__ text_out, u32 cap, IbwtMany many) {
    const u32 s = blockIdx.x * 128 + threadIdx.x;
    if (s > regular + (MANY ? many.count - 1 : 0u)) return;
    const u32 len = len_keep[s];
    if (len == 0 || len > cap) return;  // longer sublists are written by a second walk
    u32 first = 0, nb = n;
    if constexpr (MANY) {
        const u32 b = ibwt_many_block(many.starts, many.count, stride, regular, s);
        first = __ldg(many.starts + b);
        nb = __ldg(many.starts + b + 1) - first;
    }
    const u64 pos = (u64)(nb + 1) - dist[s];
    if (pos >= nb) return;
    const u32 L = (u32)min((u64)len, (u64)nb - pos);  // the '$' row's placeholder falls off the block's end
    ibwt_copy_chunk(stash + (size_t)s * (cap / 4), text_out + first + pos, L, (((uintptr_t)text_out) & 3) == 0);
}

// one pointer-jumping round over the splitter list: suffix sums of the sublist lengths
__global__ void __launch_bounds__(256)
k_ibwt_jump(const u32* __restrict__ dist_in, const u32* __restrict__ next_in, u32* __restrict__ dist_out,
            u32* __restrict__ next_out, u32 count) {
    const u32 s = blockIdx.x * 256 + threadIdx.x;
    if (s >= count) return;
    const u32 nx = next_in[s];
    u32 d = dist_in[s];
    u32 nn = kIbwtNil;
    if (nx != kIbwtNil) {
        d += dist_in[nx];
        nn = next_in[nx];
    }
    dist_out[s] = d;
    next_out[s] = nn;
}

// Every block's list must cover its n_b + 1 rows: dist[regular + b] == n_b + 1.  *bad_out = the blocks whose list does not,
// *first_bad_out = the lowest of them and *first_dist_out = the rows its list covers.
template <bool MANY>
__global__ void __launch_bounds__(1024)
k_ibwt_check(const u32* __restrict__ dist, u32 n, u32 regular, u32* __restrict__ bad_out, u32* __restrict__ first_bad_out,
             u32* __restrict__ first_dist_out, IbwtMany many) {
    __shared__ u32 s_bad, s_first;
    if (threadIdx.x == 0) {
        s_bad = 0;
        s_first = 0xFFFFFFFFu;
    }
    __syncthreads();
    u32 bad = 0, first = 0xFFFFFFFFu;
    for (u32 b = threadIdx.x; b < (MANY ? many.count : 1u); b += 1024) {
        const u64 nb = MANY ? (u64)__ldg(many.starts + b + 1) - __ldg(many.starts + b) : (u64)n;
        if ((u64)dist[regular + b] != nb + 1) {
            ++bad;
            first = min(first, b);
        }
    }
    if (bad) {
        atomicAdd(&s_bad, bad);
        atomicMin(&s_first, first);
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        *bad_out = s_bad;
        *first_bad_out = s_first;
        *first_dist_out = s_bad ? dist[regular + s_first] : 0u;
    }
}

// ---- LCP profile (SURVEY.md 8d / 8f rank 4): the data-defined round structure m_r ------------------------
// LCP[j] = lcp(SA[j-1], SA[j]) by direct comparison, 8 bytes per step (two aligned 64-bit loads and a
// funnel shift per side; the text is read through L1/L2).  Work is sum(LCP)/8 steps: fine as a tool even
// for the period-17 block (mean LCP 5,254).  Then v_j = max(LCP[j], LCP[j+1]) is bucketed by
// floor(log2(v/8)); m_r of the profiler is the suffix sum of the buckets.
__device__ __forceinline__ u64 load_u64_unaligned(const u8* __restrict__ text, u64 pos, u64 n) {
    // bytes text[pos .. pos+8) little-endian, zero beyond n (callers stop at the end of either suffix)
    const u64 base = pos & ~7ull;
    const u64* w = reinterpret_cast<const u64*>(text) + (base >> 3);
    const u64 lo = base < n ? __ldg(w) : 0ull;  // reads up to 7 bytes past n only inside the same aligned word
    const unsigned sh = (unsigned)(pos & 7) * 8;
    if (sh == 0) return lo;
    const u64 hi = base + 8 < n ? __ldg(w + 1) : 0ull;
    return (lo >> sh) | (hi << (64 - sh));
}

template <int THREADS>
__global__ void __launch_bounds__(THREADS)
k_lcp_direct(const u8* __restrict__ text, u32 n, const u32* __restrict__ sa, u32* __restrict__ lcp) {
    const u64 j = (u64)blockIdx.x * THREADS + threadIdx.x;
    if (j >= n) return;
    if (j == 0) {
        lcp[0] = 0;
        return;
    }
    const u64 a = sa[j - 1], b = sa[j];
    const u64 limit = (u64)n - max(a, b);  // the shorter suffix ends here
    u64 l = 0;
    while (l < limit) {
        const u64 x = load_u64_unaligned(text, a + l, n) ^ load_u64_unaligned(text, b + l, n);
        if (x) {
            l += (u64)(__ffsll((long long)x) - 1) >> 3;  // first differing byte (little-endian)
            break;
        }
        l += 8;
    }
    lcp[j] = (u32)min(l, limit);
}

template <int THREADS>
__global__ void __launch_bounds__(THREADS)
k_lcp_buckets(const u32* __restrict__ lcp, u32 n, unsigned long long* __restrict__ buckets /*[64]*/, u32* __restrict__ max_out) {
    __shared__ unsigned long long s_b[64];
    __shared__ u32 s_max;
    if (threadIdx.x < 64) s_b[threadIdx.x] = 0;
    if (threadIdx.x == 0) s_max = 0;
    __syncthreads();
    const u64 stride = (u64)gridDim.x * THREADS;
    u32 mx = 0;
    for (u64 j = (u64)blockIdx.x * THREADS + threadIdx.x; j < n; j += stride) {
        const u32 cur = lcp[j];
        const u32 nxt = j + 1 < n ? lcp[j + 1] : 0u;
        const u32 v = max(cur, nxt);
        mx = max(mx, cur);
        if (v >= 8) atomicAdd(&s_b[31 - __clz(v >> 3)], 1ull);
    }
    atomicMax(&s_max, mx);
    __syncthreads();
    if (threadIdx.x < 64 && s_b[threadIdx.x]) atomicAdd(&buckets[threadIdx.x], s_b[threadIdx.x]);
    if (threadIdx.x == 0) atomicMax(max_out, s_max);
}

// ---- pairs mode -----------------------------------------------------------------------------------
// Long repeats leave an active list made of PAIRS only (two suffixes tied over a long common prefix:
// the mixed 256 MiB block has nothing but pairs from round 4 on, for 8 more rounds).  Sorting a
// group of two needs no sort: one kernel per round gathers both second ranks, settles the pair when they
// differ and keeps it otherwise.  Replaces key build + 7 radix passes + re-rank for those rounds.
// m_ptr != nullptr: the length of the list is read from device memory (the count the re-rank before this launch has just
// written), so the check can be queued behind the re-rank and its answer read with the survivor count in ONE round trip.
__global__ void __launch_bounds__(256) k_pairs_detect(const u32* __restrict__ ranks, u32 m, const u32* __restrict__ m_ptr,
                                                      u32* __restrict__ seen, u32* __restrict__ not_pairs) {
    if (m_ptr != nullptr) {  // mapped host memory: one read per CTA
        __shared__ u32 s_m;
        if (threadIdx.x == 0) s_m = ld_relaxed(m_ptr);
        __syncthreads();
        m = s_m;
    }
    int big = 0;
    for (u64 p = (u64)blockIdx.x * 256 + threadIdx.x; p + 2 < m; p += (u64)gridDim.x * 256)
        big |= ranks[p] == ranks[p + 2];  // a group of three or more
    // `not_pairs` lives in mapped host memory: exactly one thread of the grid writes it
    if (__syncthreads_or(big) && threadIdx.x == 0 && ld_relaxed(seen) == 0 && atomicExch(seen, 1u) == 0) *not_pairs = 1;
}

__global__ void __launch_bounds__(256) k_pairs_apply(const uint2* __restrict__ pending, u32 count, u32* __restrict__ isa) {
    const u64 i = (u64)blockIdx.x * 256 + threadIdx.x;
    if (i < count) {
        const uint2 e = pending[i];
        isa[e.x] = e.y;
    }
}

template <int THREADS, int PPT>  // PPT pairs per thread
__global__ void __launch_bounds__(THREADS)
k_pairs_round(const u32* __restrict__ ids, const u32* __restrict__ ranks, u32 m, u32 n, u64 h, const u32* __restrict__ isa_ro,
              uint2* __restrict__ pending, u32* __restrict__ sa, u32* __restrict__ out_ids, u32* __restrict__ out_ranks,
              ScanTileState ts, u32* __restrict__ tile_counter, u32* __restrict__ out_count, const u8* __restrict__ text,
              u8* __restrict__ bwt_inline, u64* __restrict__ origin, u32 tag) {
    constexpr int TILE_PAIRS = THREADS * PPT;
    constexpr int WARPS = THREADS / 32;
    __shared__ u32 s_warp[WARPS];
    __shared__ u32 s_excl, s_tile;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    if (tid == 0) s_tile = atomicAdd(tile_counter, 1u);
    __syncthreads();
    const u32 tile = s_tile;
    const u32 npairs = m >> 1;
    const u64 q0 = (u64)tile * TILE_PAIRS + (u64)tid * PPT;  // first pair of this thread

    u32 a[PPT], b[PPT], r[PPT], ra[PPT], rb[PPT];
#pragma unroll
    for (int k = 0; k < PPT; ++k) {
        const u64 q = q0 + k;
        if (q < npairs) {
            const uint2 id2 = *reinterpret_cast<const uint2*>(ids + 2 * q);
            a[k] = id2.x;
            b[k] = id2.y;
            r[k] = ranks[2 * q];
        } else {
            a[k] = b[k] = r[k] = 0;
        }
    }
#pragma unroll
    for (int k = 0; k < PPT; ++k) {
        const u64 pa = (u64)a[k] + h, pb = (u64)b[k] + h;
        ra[k] = (q0 + k < npairs && pa < n) ? (__ldg(isa_ro + pa) & ~tag) + 1u : 0u;
        rb[k] = (q0 + k < npairs && pb < n) ? (__ldg(isa_ro + pb) & ~tag) + 1u : 0u;
    }
    u32 tied = 0;
#pragma unroll
    for (int k = 0; k < PPT; ++k)
        if (q0 + k < npairs && ra[k] == rb[k]) tied |= 1u << k;
    const u32 mine = __popc(tied);

    // exclusive scan of the surviving pairs: warp, CTA, then a 32-tile look-back window on one word
    u32 incl = mine;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const u32 t = __shfl_up_sync(0xffffffffu, incl, o);
        if (lane >= o) incl += t;
    }
    if (lane == 31) s_warp[warp] = incl;
    __syncthreads();
    u32 wprefix = 0;
    for (int w = 0; w < warp; ++w) wprefix += s_warp[w];
    if (warp == 0) {
        u32 total = 0;
        for (int w = 0; w < WARPS; ++w) total += s_warp[w];
        u64* word = ts.words + (size_t)tile * kScanWordsPerTile + 2;
        u32 excl = 0;
        if (tile == 0) {
            if (lane == 0) st_relaxed(word, scan_pack(2u, total));
        } else {
            if (lane == 0) st_relaxed(word, scan_pack(1u, total));
            int base = (int)tile - 1;
            for (;;) {
                const int t = base - lane;
                u64 w2 = scan_pack(2u, 0u);
                if (t >= 0) {
                    const u64* theirs = ts.words + (size_t)t * kScanWordsPerTile + 2;
                    do { w2 = ld_relaxed(theirs); } while ((w2 >> 62) == 0);
                }
                const u32 im = __ballot_sync(0xffffffffu, (w2 >> 62) == 2);
                const int first = im ? (__ffs(im) - 1) : 31;
                excl += __reduce_add_sync(0xffffffffu, lane <= first ? (u32)w2 : 0u);
                if (im) break;
                base -= 32;
            }
            if (lane == 0) st_relaxed(word, scan_pack(2u, excl + total));
        }
        if (lane == 0) {
            s_excl = excl;
            if ((u64)(tile + 1) * TILE_PAIRS >= npairs) *out_count = 2u * (excl + total);  // survivors (elements)
        }
    }
    __syncthreads();
    u32 slot = s_excl + wprefix + incl - mine;  // index of this thread's first surviving pair

#pragma unroll
    for (int k = 0; k < PPT; ++k) {
        if (q0 + k >= npairs) continue;
        if ((tied >> k) & 1u) {  // still tied: the pair survives with its rank
            *reinterpret_cast<uint2*>(out_ids + 2 * (u64)slot) = make_uint2(a[k], b[k]);
            *reinterpret_cast<uint2*>(out_ranks + 2 * (u64)slot) = make_uint2(r[k], r[k]);
            ++slot;
        } else {  // settled: the smaller second rank takes slot r, the other r+1
            const bool a_first = ra[k] < rb[k];
            const u32 lo = a_first ? a[k] : b[k], hi = a_first ? b[k] : a[k];
            sa[r[k]] = lo;
            sa[r[k] + 1] = hi;
            // lo keeps rank r; hi's new rank is applied after the kernel (k_pairs_apply) so that every
            // gather of this round sees the ranks of the previous round: the round count stays canonical
            pending[q0 + k - slot] = make_uint2(hi, r[k] + 1);
            if (bwt_inline != nullptr) {
                bwt_inline[r[k]] = __ldg(text + (lo == 0 ? n - 1 : lo - 1));
                bwt_inline[r[k] + 1] = __ldg(text + (hi == 0 ? n - 1 : hi - 1));
                if (lo == 0) *origin = r[k];
                if (hi == 0) *origin = (u64)r[k] + 1;
            }
        }
    }
}

// ---- many small blocks in one sort (dark_bwt_forward_many) ----------------------------------------
// B independent blocks are concatenated (block b = text[starts[b] .. starts[b+1])) and their suffixes sorted
// together; a suffix ends at the end of ITS block.  Symbols get dense codes 1..sigma and code 0 pads a key past
// the block end, so a suffix that is a proper prefix of another sorts first without the single-block
// descending-id device (App. A.3).  In the doubling rounds "past the end of block b" reads as rank 1+b and real
// ranks as isa+1+B: equal suffixes of different blocks are ordered by block number, so the sort terminates.
// The resulting suffix array interleaves the blocks; one stable radix sort by block number brings every block's
// suffixes together, in their own lexicographic order, at the block's offsets (k_many_blocks_of_sa, k_many_emit).
// These kernels favour simplicity: a C1-sized block is launch-latency bound on its own (33 launches for 768 KB).
__device__ __forceinline__ u32 block_of(const u32* __restrict__ starts, u32 B, u32 i) {  // largest b with starts[b] <= i
    u32 lo = 0, hi = B - 1;
    while (lo < hi) {
        const u32 mid = (lo + hi + 1) >> 1;
        if (__ldg(starts + mid) <= i) lo = mid;
        else hi = mid - 1;
    }
    return lo;
}
__global__ void __launch_bounds__(256) k_many_lut(const u32* __restrict__ present, u16* __restrict__ lut16, u32* __restrict__ sigma_out) {
    __shared__ u32 s_warp[8];
    const int d = threadIdx.x, lane = d & 31, warp = d >> 5;
    const u32 c = present[d] ? 1u : 0u;
    u32 incl = c;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const u32 t = __shfl_up_sync(0xffffffffu, incl, o);
        if (lane >= o) incl += t;
    }
    if (lane == 31) s_warp[warp] = incl;
    __syncthreads();
    u32 base = 0;
    for (int w = 0; w < warp; ++w) base += s_warp[w];
    lut16[d] = (u16)(c ? base + incl : 0u);  // codes 1..sigma
    if (d == 255) *sigma_out = base + incl;
}
template <int THREADS>
__global__ void __launch_bounds__(THREADS)
k_many_init_keys(const u8* __restrict__ text, u32 n, const u16* __restrict__ lut16, int s_bits, int K, const u32* __restrict__ starts,
                 u32 B, u64* __restrict__ keys_out, u32* __restrict__ ids_out, u32* __restrict__ g_hist) {
    __shared__ u32 s_hist[kMaxPasses * kRadix];
    __shared__ u16 s_lut[256];
    const int tid = threadIdx.x;
    hist_clear(s_hist, tid, THREADS);
    for (int i = tid; i < 256; i += THREADS) s_lut[i] = lut16[i];
    __syncthreads();
    for (u64 i = (u64)blockIdx.x * THREADS + tid; i < n; i += (u64)gridDim.x * THREADS) {
        const u32 b = block_of(starts, B, (u32)i);
        const u64 end = __ldg(starts + b + 1);
        u64 key = 0;
        for (int c = 0; c < K; ++c) key = (key << s_bits) | (i + c < end ? (u64)s_lut[text[i + c]] : 0ull);
        key <<= (64 - s_bits * K);
        keys_out[i] = key;
        ids_out[i] = (u32)i;
        hist_add_key(s_hist, key, 0, kMaxPasses);
    }
    __syncthreads();
    hist_flush(s_hist, g_hist, kMaxPasses, tid, THREADS);
}
template <int THREADS>
__global__ void __launch_bounds__(THREADS)
k_many_build_keys(const u32* __restrict__ ids, const u32* __restrict__ ranks, u32 m, u64 h, int kb, const u32* __restrict__ isa,
                  const u32* __restrict__ starts, u32 B, u64* __restrict__ keys_out, u32* __restrict__ g_hist, int num_passes) {
    __shared__ u32 s_hist[kMaxPasses * kRadix];
    const int tid = threadIdx.x;
    hist_clear(s_hist, tid, THREADS);
    __syncthreads();
    for (u64 p = (u64)blockIdx.x * THREADS + tid; p < m; p += (u64)gridDim.x * THREADS) {
        const u32 id = ids[p];
        const u32 b = block_of(starts, B, id);
        const u64 pos2 = (u64)id + h;
        const u64 r2 = pos2 < __ldg(starts + b + 1) ? (u64)__ldg(isa + pos2) + 1u + B : 1u + b;
        const u64 key = ((u64)(ranks[p] >> 1) << kb) | r2;
        keys_out[p] = key;
        hist_add_key(s_hist, key, 0, num_passes);
    }
    __syncthreads();
    hist_flush(s_hist, g_hist, num_passes, tid, THREADS);
}
// (block number, suffix) pairs of the interleaved suffix array, for the stable sort by block number
template <int THREADS>
__global__ void __launch_bounds__(THREADS)
k_many_blocks_of_sa(const u32* __restrict__ sa, u32 n, const u32* __restrict__ starts, u32 B, u64* __restrict__ keys_out,
                    u32* __restrict__ ids_out, u32* __restrict__ g_hist, int num_passes) {
    __shared__ u32 s_hist[kMaxPasses * kRadix];
    const int tid = threadIdx.x;
    hist_clear(s_hist, tid, THREADS);
    __syncthreads();
    for (u64 j = (u64)blockIdx.x * THREADS + tid; j < n; j += (u64)gridDim.x * THREADS) {
        const u32 id = sa[j];
        const u64 key = block_of(starts, B, id);
        keys_out[j] = key;
        ids_out[j] = id;
        hist_add_key(s_hist, key, 0, num_passes);
    }
    __syncthreads();
    hist_flush(s_hist, g_hist, num_passes, tid, THREADS);
}
// position p of the sorted list is slot p - starts[b] of block b: its BWT byte, the block's origin, its SA entry
__global__ void __launch_bounds__(256)
k_many_emit(const u64* __restrict__ blk, const u32* __restrict__ ids, u32 n, const u8* __restrict__ text, const u32* __restrict__ starts,
            u8* __restrict__ bwt, unsigned long long* __restrict__ origins, u32* __restrict__ sa_out) {
    const u64 p = (u64)blockIdx.x * 256 + threadIdx.x;
    if (p >= n) return;
    const u32 b = (u32)blk[p], id = ids[p];
    const u32 first = __ldg(starts + b);
    if (id == first) {
        bwt[p] = text[__ldg(starts + b + 1) - 1];
        origins[b] = p - first;
    } else {
        bwt[p] = text[id - 1];
    }
    if (sa_out != nullptr) sa_out[p] = id - first;
}

// ---- inverse BWT of many blocks in one pass (dark_bwt_inverse_many) ---------------------------------
// The single-block method ("inverse BWT" above) over one ROW SPACE shared by B blocks.  Block b (bytes [starts[b],
// starts[b+1]) of the concatenated BWTs, n_b of them) owns the n_b + 1 global rows [starts[b] + b, starts[b+1] + b + 1):
// its '$' row first, then its real rows.
//   psi    the real rows' last symbols under the key (b << 8) | symbol, sorted stably (one byte pass + 1-2 passes on
//          the block number): the stable partition of every block at once.  Sorted slot q of block b is row q + b + 1;
//          the row id stored there is its psi, the key's low byte its first symbol (one index for both loads, no
//          symbol bases).  psi never leaves a block, whatever the input.
//   walk   k_ibwt_walk<MODE, true>: splitters are every stride-th global row plus each block's head row (local row
//          origin_b + 1, splitter `regular + b`).  A walk finds its block once (binary search over the row offsets) and
//          stops at a stride-th row or at its own block's head; reaching the head means it came through the '$' row, so
//          that sublist ends the block's list (nil).  k_ibwt_jump then runs unchanged over the forest of lists.
//   offset a splitter's text offset is starts[b] + n_b + 1 - dist (k_ibwt_unstash<true>, k_ibwt_walk<1, true>).
//   check  every block's list covers its n_b + 1 rows: dist[regular + b] == n_b + 1 (k_ibwt_check<true>).
// (key, row) of every real row, in row order within each block (the sort is stable), and the digit histogram
template <int THREADS>
__global__ void __launch_bounds__(THREADS)
k_ibwt_many_elements(const u8* __restrict__ bwt, u32 n, const u32* __restrict__ starts, u32 B,
                     const unsigned long long* __restrict__ origins, u64* __restrict__ keys, u32* __restrict__ rows,
                     u32* __restrict__ g_hist, int num_passes) {
    __shared__ u32 s_hist[kMaxPasses * kRadix];
    const int tid = threadIdx.x;
    hist_clear(s_hist, tid, THREADS);
    __syncthreads();
    for (u64 e = (u64)blockIdx.x * THREADS + tid; e < n; e += (u64)gridDim.x * THREADS) {
        const u32 b = block_of(starts, B, (u32)e);
        const u32 first = __ldg(starts + b), origin = (u32)__ldg(origins + b);
        const u32 le = (u32)e - first;
        const u32 r = le == 0 ? 0u : (le <= origin ? le : le + 1u);  // local row, as in k_ibwt_elements
        const u32 sym = le == 0 ? bwt[first + origin] : bwt[first + r - 1];
        const u64 key = ((u64)b << 8) | sym;
        keys[e] = key;
        rows[e] = first + b + r;
        hist_add_key(s_hist, key, 0, num_passes);
    }
    __syncthreads();
    hist_flush(s_hist, g_hist, num_passes, tid, THREADS);
}

// ---- verification (independent of the construction kernels) ------------------------------------
template <int THREADS>
__global__ void __launch_bounds__(THREADS) k_verify_scatter(const u32* __restrict__ sa, u32 n, u32* __restrict__ isa, unsigned long long* bad) {
    const u64 j = (u64)blockIdx.x * THREADS + threadIdx.x;
    if (j >= n) return;
    const u32 v = sa[j];
    if (v >= n) atomicAdd(bad, 1ull);
    else isa[v] = (u32)j;
}
template <int THREADS>
__global__ void __launch_bounds__(THREADS)
k_verify_order(const u8* __restrict__ text, const u32* __restrict__ sa, u32 n, const u32* __restrict__ isa, unsigned long long* bad) {
    const u64 j = (u64)blockIdx.x * THREADS + threadIdx.x;
    if (j >= n) return;
    const u32 b = sa[j];
    if (b >= n) return;  // counted by the scatter kernel
    bool ok = isa[b] == (u32)j;  // permutation: every value hit exactly once
    if (ok && j > 0) {
        const u32 a = sa[j - 1];
        if (a >= n) return;
        const u8 ta = text[a], tb = text[b];
        if (ta > tb) ok = false;
        else if (ta == tb) {
            const long long ra = ((u64)a + 1 < n) ? (long long)isa[a + 1] : -1;
            const long long rb = ((u64)b + 1 < n) ? (long long)isa[b + 1] : -1;
            ok = ra < rb;
        }
    }
    if (!ok) atomicAdd(bad, 1ull);
}

}  // namespace dark
