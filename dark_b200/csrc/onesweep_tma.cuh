// onesweep_tma.cuh — the radix pass of radix_sort.cuh rebuilt as a software-pipelined persistent kernel:
//
//   * TMA bulk staging.  One elected thread brings the NEXT tile's keys and values (or, in the key-generating
//     first pass, its slice of the text) from HBM into a shared-memory stage with cp.async.bulk (SASS: UBLKCP),
//     completion signalled on an mbarrier, while the CTA scatters and re-orders: no thread ever waits on a
//     global load, and the pairs live in registers only from the stage to the re-order.
//   * Scanner CTAs instead of a look-back.  In round 1 every tile walked 10-25 predecessor status rows: three
//     L2 round trips of 2-3 k cycles each on its critical path and 18 % of its instructions
//     (profiles/r1_pass_trace_v4.md).  Here the first kScanners CTAs to arrive (tickets 0 .. kScanners-1 of the
//     tile counter) do not sort: scanner k owns 256 / kScanners digits, sweeps their status words in tile order
//     with three batches of 32 rows in flight per digit, and turns every published digit count [01 | count] into
//     the tile's exclusive prefix [1 | prefix] (PipeStatus below).  A worker publishes its counts after ranking tile j, goes on to
//     load and rank tile j+1 (tile j sits re-ordered in shared memory meanwhile), and then reads ONE word per
//     digit - its own row, resolved long before - and scatters tile j.  The worker CTA that shares an SM with a
//     scanner retires (its scatter stores would queue ahead of the scanner's loads in the SM's memory pipeline).
//   * Tickets.  Tiles are claimed from a counter, so only running CTAs ever own a tile and nothing can wait on a
//     CTA that is not resident.  A ticket is taken AFTER the wait for the previous tile's prefix and used for a
//     load that lands during the scatter and re-order: the scanners work in tile order, so every tile behind a
//     late one waits for it, and a wait between taking a ticket and publishing its counts would feed on itself
//     (measured: 1.16 -> 0.92 ms per 2^27-pair pass, profiles/r2_rejected.md).
//   * Leaner inner loops: 69 instructions per 32 pairs instead of 104 (8 ballots folded by four 3-input ANDs,
//     predicated leader store, values carried in registers, no debug hooks in release builds).
//
// Bound: shared-memory wavefronts.  ncu (profiles/r2_ncu_pass_tma.md): LSU data pipe 75 % busy, 4,200 wavefronts per
// 4,096-pair tile of which half are bank conflicts of the digit-indexed accesses (per-warp counters, re-order); DRAM
// traffic 1.003 x the algorithmic 24 B per pair; 4.0 TB/s = 0.61 of the measured HBM copy peak (round 1: 0.48-0.53).
//
// Same contract as k_onesweep_pass: one stable LSD pass on the byte-aligned digit at `shift`, 12 B read +
// 12 B written per pair.  The status buffer must be zeroed for (tiles + 3 * kScannerBatch) rows.
// Replaces the induced-sorting sweeps of the reference (/root/reference/src/saca.rs:99-163).
#pragma once

#include "radix_sort.cuh"

namespace dark {

template <int THREADS, int ITEMS>
struct PipeSmem {
    static constexpr int kTile = THREADS * ITEMS;
    static constexpr int kWarps = THREADS / 32;
    u64 stage_keys[kTile];  // TMA destination (GEN: text bytes at 0, code words at kGenWordsOff)
    u32 stage_vals[kTile];
    u64 keys[kTile];        // the previous tile, re-ordered by digit, waiting for its look-back
    u32 vals[kTile];
    u32 warp_hist[kWarps][kRadix];  // per-warp digit counters -> tile-local offsets
    u32 global_off[kRadix];
    u32 warp_sum[kRadix / 32];
    u32 next_tile;
    u32 pad_;
    u64 mbar;
    u8 lut[256];
};

constexpr int kScanners = 4;  // scanner CTAs per pass: each owns 256 / kScanners digits (tickets 0 .. kScanners-1)
static_assert(256 % kScanners == 0, "every digit needs a scanner: the scanner count must divide 256");
constexpr int kScannerBatch = 32;      // status rows per scanner batch (three in flight: 3 * 32 zeroed rows follow the last tile)
constexpr u32 kGenStageBytes = 4288;   // text slice of a 4,096-suffix tile: 4,096 + 64 symbols of look-ahead + alignment slack
constexpr u32 kGenWordsOff = 8192;     // byte offset of the packed code words inside stage_keys

// Status word of this pass: 0 = nothing yet, [01 | count] = the tile's digit count is published, [1 | prefix] = the
// scanner resolved the exclusive prefix.  One flag bit on a resolved word leaves 31 (63) bits for the prefix, so the
// 4-byte word serves every m <= 2^31 (k_onesweep_pass keeps its own two-flag-bit words, radix_sort.cuh).
template <typename T>
struct PipeStatus {
    static constexpr int kBits = (int)sizeof(T) * 8;
    static constexpr int kShift = kBits - 2;
    static constexpr T kPub = (T)1 << (kBits - 2);
    static constexpr T kRes = (T)1 << (kBits - 1);
    static constexpr T kPrefix = kRes - 1;
    __device__ static __forceinline__ bool resolved(T w) { return (w >> (kBits - 1)) != 0; }
};

// Lanes (of `peers`) whose 8-bit digit equals mine: 8 ballots, each complemented on the lanes whose bit is clear (one
// test for seven bits at once - ptxas turns the per-bit tests into R2P - one vote and a predicated NOT per bit), folded
// with four 3-input ANDs.  match_digit_bits (radix_sort.cuh) chains eight 2-input ANDs instead.
template <int BIT>
__device__ __forceinline__ u32 vote_digit_bit(u32 d) {
    u32 v;
    asm("{\n"
        ".reg .pred p;\n"
        ".reg .b32 t;\n"
        "and.b32 t, %1, %2;\n"
        "setp.ne.u32 p, t, 0;\n"
        "vote.sync.ballot.b32 %0, p, 0xffffffff;\n"
        "@!p not.b32 %0, %0;\n"
        "}\n"
        : "=r"(v)
        : "r"(d), "n"(1 << BIT));
    return v;
}
__device__ __forceinline__ u32 match_digit_lop3(u32 peers, u32 d) {
    const u32 v0 = vote_digit_bit<0>(d), v1 = vote_digit_bit<1>(d), v2 = vote_digit_bit<2>(d), v3 = vote_digit_bit<3>(d);
    const u32 v4 = vote_digit_bit<4>(d), v5 = vote_digit_bit<5>(d), v6 = vote_digit_bit<6>(d), v7 = vote_digit_bit<7>(d);
    u32 a, b, c;  // explicit 3-input ANDs: left to itself the compiler chains eight 2-input ones
    asm("lop3.b32 %0, %1, %2, %3, 0x80;" : "=r"(a) : "r"(peers), "r"(v0), "r"(v1));
    asm("lop3.b32 %0, %1, %2, %3, 0x80;" : "=r"(b) : "r"(v2), "r"(v3), "r"(v4));
    asm("lop3.b32 %0, %1, %2, %3, 0x80;" : "=r"(c) : "r"(v5), "r"(v6), "r"(v7));
    asm("lop3.b32 %0, %1, %2, %3, 0x80;" : "=r"(a) : "r"(a), "r"(b), "r"(c));
    return a;
}

template <bool V>
struct BoolC {
    static constexpr bool value = V;
};

template <int THREADS, int ITEMS, int MINBLOCKS, int ILP, typename StatusT, bool GEN, bool HI>
__global__ void __launch_bounds__(THREADS, MINBLOCKS)
k_onesweep_tma(const u64* __restrict__ keys_in, const u32* __restrict__ vals_in, u64* __restrict__ keys_out,
               u32* __restrict__ vals_out, const u32 m, const int shift, const u32* __restrict__ digit_base,
               StatusT* __restrict__ status, StatusT* __restrict__ status_clean, u32* __restrict__ tile_counter, const KeyGen gen,
               const u8* __restrict__ prev_text) {
    // status_clean (nullable): the status buffer the NEXT pass will use.  Every worker zeroes the row of each tile it
    // processes there, so the host need not launch a memset between passes (64 MB per 2^28 pairs and a launch gap each).
    static_assert(THREADS >= kRadix && THREADS % 32 == 0, "one thread per digit is assumed");
    static_assert(ITEMS % 2 == 0 && 32 * ITEMS < 65536, "ranks are packed two per register");
    typedef PipeSmem<THREADS, ITEMS> Smem;
    typedef PipeStatus<StatusT> ST;
    constexpr int TILE = Smem::kTile;
    static_assert(!GEN || (TILE + 64 + 48 <= (int)kGenStageBytes && 2 * TILE >= (int)kGenStageBytes + 32), "the staged text slice must cover a tile and end before the text does (tiles >= 1)");
    extern __shared__ __align__(128) unsigned char smem_pipe[];
    Smem& s = *reinterpret_cast<Smem*>(smem_pipe);
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const u32 num_tiles = (u32)(((u64)m + TILE - 1) / TILE);
    // the digit is one byte of the high (HI) or low key word: a single PRMT
    const u32 bsel = 0x4440u | ((u32)(shift & 31) >> 3);
    auto digit = [&](u64 key) -> u32 { return __byte_perm(HI ? (u32)(key >> 32) : (u32)key, 0u, bsel); };
    const u32 local0 = warp * (32 * ITEMS) + lane;  // warp-striped: element (warp, k, lane) = warp*32*ITEMS + k*32 + lane
    const u32 lt = lanemask_lt();
    u32* const whist = s.warp_hist[warp];
    const u32 whist_addr = smem_addr(whist);
    const bool digit_thread = tid < kRadix;

    if (tid == 0) {
        mbar_init(&s.mbar, 1);
        fence_mbar_init();
        s.next_tile = atomicAdd(tile_counter, 1u);
    }
    for (int i = tid; i < Smem::kWarps * kRadix; i += THREADS) (&s.warp_hist[0][0])[i] = 0;
    if (GEN && tid < 256) s.lut[tid] = gen.lut[tid];
    __syncthreads();
    // ticket 0 = the scanner; ticket t > 0 = tile t-1 (only running CTAs ever hold a ticket)
    if (s.next_tile < (u32)kScanners) {
        // Thread d owns digit d.  It walks the status rows in tile order and replaces [01 | count] by
        // [1 | exclusive prefix] (each count is added less its flag bit: one three-input add).  Three batches
        // of kScannerBatch rows are in flight per digit (registers), always starting at the first unresolved row, so
        // the scanner is never more than one round trip behind the tiles and resolves 3 * kScannerBatch rows per round
        // trip when it has fallen behind.  Rows past the last tile stay zero (never published).
        if (tid == 0) {  // tell the worker CTA that shares this SM to retire: its stores would queue ahead of the scanner's loads
            u32 smid;
            asm volatile("mov.u32 %0, %%smid;" : "=r"(smid));
            st_relaxed(tile_counter + 1 + s.next_tile, smid + 1u);
        }
        if (tid < kRadix / kScanners) {
            constexpr int B = (sizeof(StatusT) == 8 ? kScannerBatch / 2 : kScannerBatch) / (THREADS * MINBLOCKS > 512 ? 2 : 1);  // 96 registers (48 in the narrower register budget of wider CTAs)
            StatusT* row = status + s.next_tile * (kRadix / kScanners) + tid;  // this digit's word of the first unresolved tile
            u32 j = 0;
            StatusT run = 0;
            StatusT v0[B], v1[B], v2[B];
            auto load = [&](StatusT(&v)[B], int ahead) {
#pragma unroll
                for (int i = 0; i < B; ++i) v[i] = ld_relaxed(row + (size_t)(ahead * B + i) * kRadix);
            };
            // resolves the leading published rows of a batch that starts at the first unresolved row; true if all B were
            auto resolve = [&](StatusT(&v)[B]) -> bool {
                StatusT every = v[0];
#pragma unroll
                for (int i = 1; i < B; ++i) every &= v[i];
                if ((u32)(every >> ST::kShift) & 1u) {  // the usual case when behind: every row is a published count
                    StatusT acc = run;
#pragma unroll
                    for (int i = 0; i < B; ++i) {
                        st_relaxed(row + (size_t)i * kRadix, ST::kRes | (acc & ST::kPrefix));
                        acc += v[i] - ST::kPub;
                    }
                    run = acc;
                    j += B;
                    row += (size_t)B * kRadix;
                    return true;
                }
                int done = 0;
                bool ok = true;
#pragma unroll
                for (int i = 0; i < B; ++i) {
                    ok = ok && (u32)(v[i] >> ST::kShift) == 1u;
                    if (ok) {
                        DARK_ASSERT(j + i < num_tiles);
                        st_relaxed(row + (size_t)i * kRadix, ST::kRes | (run & ST::kPrefix));
                        run += v[i] - ST::kPub;
                        done = i + 1;
                    }
                }
                j += (u32)done;
                row += (size_t)done * kRadix;
                return false;
            };
            while (j < num_tiles) {
                load(v0, 0);
                load(v1, 1);
                load(v2, 2);
                for (;;) {  // each batch is resolved while the other two are in flight
                    if (!resolve(v0) || j >= num_tiles) break;
                    load(v0, 2);
                    if (!resolve(v1) || j >= num_tiles) break;
                    load(v1, 2);
                    if (!resolve(v2) || j >= num_tiles) break;
                    load(v2, 2);
                }
            }
        }
        return;
    }
    u32 tile = s.next_tile - (u32)kScanners;
    if (tile >= num_tiles) return;
    u32 claimed = 0;  // thread 0: the next ticket
    u32 scanner_sm = 0, my_sm = 0;  // thread 0: set once a scanner is seen on this SM
    bool retire = false;
    asm volatile("mov.u32 %0, %%smid;" : "=r"(my_sm));

    // A full tile other than (GEN) the first and the last is staged by TMA; the rest load with guards.
    auto staged = [&](u32 t) -> bool {
        if ((u64)(t + 1) * TILE > (u64)m) return false;
        if (GEN) return t >= 1 && t + 1 < num_tiles;
        return true;
    };
    auto issue_load = [&](u32 t) {  // thread 0 only
        fence_proxy_async();
        if (GEN) {
            const u64 i_lo = (u64)gen.n - (u64)(t + 1) * TILE;
            const u8* a0 = (const u8*)((uintptr_t)(gen.text + i_lo - 1) & ~(uintptr_t)15);
            mbar_expect_tx(&s.mbar, kGenStageBytes);
            tma_load_1d(s.stage_keys, a0, kGenStageBytes, &s.mbar);
        } else {
            mbar_expect_tx(&s.mbar, (u32)(TILE * 12));
            tma_load_1d(s.stage_keys, keys_in + (u64)t * TILE, (u32)(TILE * 8), &s.mbar);
            tma_load_1d(s.stage_vals, vals_in + (u64)t * TILE, (u32)(TILE * 4), &s.mbar);
        }
    };
    if (tid == 0 && staged(tile)) issue_load(tile);

    u32 phase = 0;
    bool have_prev = false;
    u32 prev_tile = 0, prev_nvalid = 0, prev_dstart = 0;
    StatusT my_row = 0;  // the previous tile's status word of this digit, as last read
    // ---- scatter of the tile that sits re-ordered in shared memory
    auto scatter = [&](auto full_c, const u32 nvalid) {
        constexpr bool FULL = decltype(full_c)::value;
#pragma unroll
        for (int k = 0; k < ITEMS; ++k) {
            const u32 p = k * THREADS + tid;
            if (FULL || p < nvalid) {
                const u64 kk = s.keys[p];
                const u32 idx = s.global_off[digit(kk)] + p;
                DARK_ASSERT(idx < m);
                keys_out[idx] = kk;
                vals_out[idx] = s.vals[p];
            }
        }
    };

    u64 key[ITEMS];
    u32 val[ITEMS];
    u32 rank2[ITEMS / 2];

    // ---- the tile's pairs into registers; then the stage is handed back and the next tile's load started
    auto load_tile = [&](auto full_c, const u32 nvalid) {
        constexpr bool FULL = decltype(full_c)::value;
        const bool is_staged = staged(tile);
        const u64 tile_base = (u64)tile * TILE;
        if (!GEN) {
            if (FULL) {  // every full tile of a plain pass is staged
                mbar_wait(&s.mbar, phase);
                phase ^= 1u;
#pragma unroll
                for (int k = 0; k < ITEMS; ++k) {
                    key[k] = s.stage_keys[local0 + k * 32];
                    val[k] = s.stage_vals[local0 + k * 32];
                }
            } else {
#pragma unroll
                for (int k = 0; k < ITEMS; ++k) {
                    const bool v = local0 + k * 32 < nvalid;
                    key[k] = v ? ld_stream(keys_in + tile_base + local0 + k * 32) : ~0ull;
                    val[k] = v ? ld_stream(vals_in + tile_base + local0 + k * 32) : 0u;
                }
            }
        } else {
            // Key-generating pass (round 0 of the suffix sorter): element j is suffix id = n-1-j, its key the first 64/s
            // symbols as dense s-bit codes, exactly what k_init_keys_packed would have written (suffix_kernels.cuh).
            const int lg_s = gen.lg_s, sbits = 1 << lg_s, spw = 32 >> lg_s;
            const u64 i_lo = (u64)gen.n - tile_base - nvalid;  // lowest text position of this tile
            const u32 nwords = ((u32)(TILE + (64 >> lg_s)) >> (5 - lg_s)) + 3;
            u32* words = reinterpret_cast<u32*>(reinterpret_cast<unsigned char*>(s.stage_keys) + kGenWordsOff);
            const u8* bytes = reinterpret_cast<const u8*>(s.stage_keys);
            u32 delta = 0;
            if (is_staged) {
                const u8* a0 = (const u8*)((uintptr_t)(gen.text + i_lo - 1) & ~(uintptr_t)15);
                delta = (u32)((gen.text + i_lo) - a0);  // stage byte of text position i_lo: 1..16
                mbar_wait(&s.mbar, phase);
                phase ^= 1u;
                const u32* b32 = reinterpret_cast<const u32*>(bytes);
                const u32 rot = (delta & 3u) * 8u;
                for (u32 w = tid; w < nwords; w += THREADS) {
                    const u32 q0 = delta + (w << (5 - lg_s));
                    u32 word = 0;
                    u32 lo = b32[q0 >> 2];
                    for (int c = 0; c < spw; c += 4) {
                        const u32 hi = b32[((q0 + c) >> 2) + 1];
                        const u32 b4 = __funnelshift_r(lo, hi, rot);  // text bytes q0+c .. q0+c+3, first byte lowest
                        lo = hi;
                        word = (word << sbits) | s.lut[b4 & 0xFFu];
                        word = (word << sbits) | s.lut[(b4 >> 8) & 0xFFu];
                        word = (word << sbits) | s.lut[(b4 >> 16) & 0xFFu];
                        word = (word << sbits) | s.lut[b4 >> 24];
                    }
                    words[w] = word;
                }
            } else {
                for (u32 w = tid; w < nwords; w += THREADS) {
                    u32 word = 0;
                    const u64 pos0 = i_lo + ((u64)w << (5 - lg_s));
                    for (int c = 0; c < spw; ++c) {
                        const u64 pos = pos0 + c;
                        const u32 code = pos < gen.n ? (u32)s.lut[__ldg(gen.text + pos)] : 0u;
                        word = (word << sbits) | code;
                    }
                    words[w] = word;
                }
            }
            __syncthreads();
#pragma unroll
            for (int k = 0; k < ITEMS; ++k) {
                const u32 jl = local0 + k * 32;
                key[k] = ~0ull;
                val[k] = 0u;
                if (FULL || jl < nvalid) {
                    const u32 x = nvalid - 1 - jl;
                    const u32 bit = x << lg_s;
                    const u32 wi = bit >> 5, sh = bit & 31;
                    const u32 w0 = words[wi], w1 = words[wi + 1], w2 = words[wi + 2];
                    u64 kk = ((u64)__funnelshift_l(w1, w0, sh) << 32) | __funnelshift_l(w2, w1, sh);
                    const u32 id = (u32)(i_lo + x);
                    if (prev_text != nullptr) {
                        // pruned initial sort: the BWT byte T[id-1] rides in the (unsorted) low key byte
                        const u32 pb = is_staged ? (u32)bytes[delta + x - 1] : (u32)__ldg(prev_text + (id == 0 ? gen.n - 1 : id - 1));
                        kk = (kk & ~0xFFull) | (u64)pb;
                    }
                    key[k] = kk;
                    val[k] = id;
                }
            }
        }
        __syncthreads();  // every thread has read the stage: it may be refilled
    };

    // ---- rank inside the warp.  Lanes with equal digits are found with 8 ballots (match_digit_bits, radix_sort.cuh);
    // every lane reads its digit's counter, the lowest lane of each group then bumps it (predicated store, no
    // branch).  The previous tile's status word is requested first: the scanner has had a re-order and a tile load
    // to resolve it, and the answer has the whole ranking loop to arrive.
    auto rank_tile = [&](auto full_c, const u32 nvalid) {
        constexpr bool FULL = decltype(full_c)::value;
        StatusT early_row = 0;
        if (have_prev && digit_thread) early_row = ld_relaxed(status + (size_t)prev_tile * kRadix + tid);
#pragma unroll
        for (int k = 0; k < ITEMS; ++k) {
            // a second look two thirds into the loop: a tile that was published late is resolved by then
            if (k == (ITEMS * 2) / 3 && have_prev && digit_thread) my_row = ld_relaxed(status + (size_t)prev_tile * kRadix + tid);
            const bool valid = FULL || (local0 + k * 32) < nvalid;
            u32 d = digit(key[k]);
            if (k >= ILP) asm volatile("" : "+r"(d) : "r"(rank2[(k - ILP) / 2]));  // at most ILP items in flight (registers)
            u32 peers = FULL ? 0xffffffffu : __ballot_sync(0xffffffffu, valid);
            peers = match_digit_lop3(peers, d);
            const u32 cell = whist_addr + d * 4u;
            u32 prev;
            asm volatile("ld.shared.u32 %0, [%1];" : "=r"(prev) : "r"(cell) : "memory");
            const u32 below = peers & lt;
            const u32 r = prev + __popc(below);
            const u32 nv = prev + __popc(peers);
            __syncwarp();
            if (FULL)
                asm volatile("{\n.reg .pred p;\nsetp.eq.u32 p, %0, 0;\n@p st.shared.u32 [%1], %2;\n}\n" ::"r"(below), "r"(cell), "r"(nv) : "memory");
            else
                asm volatile("{\n.reg .pred p;\nsetp.eq.u32 p, %0, 0;\n@p st.shared.u32 [%1], %2;\n}\n" ::"r"(valid ? below : 1u), "r"(cell), "r"(nv) : "memory");
            if (k & 1) rank2[k / 2] |= r << 16;
            else rank2[k / 2] = r;
            __syncwarp();
        }
        if (ST::resolved(early_row)) my_row = early_row;
    };

    // ---- re-order the tile by digit in shared memory; each warp then clears its own counters for the next tile (no
    // other warp touches them before the next barrier)
    auto reorder_tile = [&](auto full_c, const u32 nvalid) {
        constexpr bool FULL = decltype(full_c)::value;
#pragma unroll
        for (int k = 0; k < ITEMS; ++k) {
            if (FULL || (local0 + k * 32) < nvalid) {
                const u32 pos = whist[digit(key[k])] + ((rank2[k / 2] >> (16 * (k & 1))) & 0xFFFFu);
                DARK_ASSERT(pos < nvalid);
                s.keys[pos] = key[k];
                s.vals[pos] = val[k];
            }
        }
        __syncwarp();
        uint4* row = reinterpret_cast<uint4*>(whist);
#pragma unroll
        for (int i = lane; i < kRadix / 4; i += 32) row[i] = make_uint4(0u, 0u, 0u, 0u);
    };

    for (;;) {
        const u32 nvalid = (u32)min((u64)TILE, (u64)m - (u64)tile * TILE);
        const bool full = nvalid == (u32)TILE;
        if (status_clean != nullptr && digit_thread) status_clean[(size_t)tile * kRadix + tid] = 0;
        if (full) {
            load_tile(BoolC<true>(), nvalid);
            rank_tile(BoolC<true>(), nvalid);
        } else {
            load_tile(BoolC<false>(), nvalid);
            rank_tile(BoolC<false>(), nvalid);
        }
        __syncthreads();

        // ---- per digit: exclusive offsets across warps, tile total, publish the aggregate
        u32 count = 0;
        if (digit_thread) {
            u32 run = 0;
#pragma unroll
            for (int w = 0; w < Smem::kWarps; ++w) {
                const u32 c = s.warp_hist[w][tid];
                s.warp_hist[w][tid] = run;
                run += c;
            }
            count = run;
            DARK_ASSERT(tile < num_tiles && count <= nvalid);
            st_relaxed(status + (size_t)tile * kRadix + tid, ST::kPub | (StatusT)count);
        }
        u32 incl = count;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const u32 t = __shfl_up_sync(0xffffffffu, incl, o);
            if (lane >= o) incl += t;
        }
        if (digit_thread && lane == 31) s.warp_sum[warp] = incl;
        __syncthreads();
        u32 dstart = 0;
        if (digit_thread) {
            u32 wbase = 0;
            for (int w = 0; w < warp; ++w) wbase += s.warp_sum[w];
            dstart = wbase + incl - count;
#pragma unroll
            for (int w = 0; w < Smem::kWarps; ++w) s.warp_hist[w][tid] += dstart;
            if (have_prev) {
                while (!ST::resolved(my_row)) {
                    __nanosleep(32);  // the scanner is behind: do not hammer L2 with 256 polls per CTA
                    my_row = ld_relaxed(status + (size_t)prev_tile * kRadix + tid);
                }
                s.global_off[tid] = digit_base[tid] + (u32)(my_row & ST::kPrefix) - prev_dstart;
            }
        }
        __syncthreads();
        // The next ticket is taken only now, after the wait for the previous tile's prefix: tickets must be handed out
        // in (nearly) the order in which the tiles will publish their counts - the scanner works in tile order, so
        // every tile behind a late one waits for it - and a wait between ticket and counts would feed on itself.
        // The atomic's latency hides behind the scatter; the load it triggers lands during the re-order.
        if (tid == 0 && !retire) {
            claimed = atomicAdd(tile_counter, 1u);
#pragma unroll
            for (int k = 0; k < kScanners; ++k) scanner_sm |= (ld_relaxed(tile_counter + 1 + k) == my_sm + 1u) ? 1u : 0u;
        }

        if (have_prev) {
            if (prev_nvalid == (u32)TILE) scatter(BoolC<true>(), prev_nvalid);
            else scatter(BoolC<false>(), prev_nvalid);
        }
        if (tid == 0) {
            const u32 nxt = retire ? ~0u : claimed - (u32)kScanners;  // the first tickets are the scanners'
            // A worker that shares its SM with the scanner retires (its stores would queue ahead of the scanner's loads
            // in the SM's memory pipeline): the ticket it has just taken is still processed, no further one is taken.
            // Only in a grid with workers to spare: in a tiny grid every worker could sit beside a scanner.
            if (scanner_sm != 0u && gridDim.x >= 64u) retire = true;
            s.next_tile = nxt;
            if (nxt < num_tiles && staged(nxt)) issue_load(nxt);
        }
        __syncthreads();  // the re-order buffer is free
        const u32 nxt_tile = s.next_tile;

        if (full) reorder_tile(BoolC<true>(), nvalid);
        else reorder_tile(BoolC<false>(), nvalid);
        have_prev = true;
        prev_tile = tile;
        prev_nvalid = nvalid;
        prev_dstart = dstart;
        tile = nxt_tile;
        if (tile >= num_tiles) break;
    }

    // ---- drain: the last tile of this CTA
    __syncthreads();
    if (digit_thread) {
        do my_row = ld_relaxed(status + (size_t)prev_tile * kRadix + tid);
        while (!ST::resolved(my_row));
        s.global_off[tid] = digit_base[tid] + (u32)(my_row & ST::kPrefix) - prev_dstart;
    }
    __syncthreads();
    if (prev_nvalid == (u32)TILE) scatter(BoolC<true>(), prev_nvalid);
    else scatter(BoolC<false>(), prev_nvalid);
}

}  // namespace dark
