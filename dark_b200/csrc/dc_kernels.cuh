// dc_kernels.cuh — distance coding + move-to-front of a BWT block on the GPU (SURVEY.md 8(f) rank 3).
//
// Replaces `bwt::dc::encode(&output, suf, &mut self.mtf)` and the (distance, Context) items its iterator yields
// (/root/reference/src/block/dc.rs:52, 82-85).  The code being replaced is third-party (`compress::bwt::dc`,
// `compress::bwt::mtf`, Cargo.toml:18) and absent from the reference tree: PARITY UNPINNED — the kernels are checked
// against the test suite's CPU restatement of upstream rust-compress (written from memory) and by encode -> decode round trips.
//
// What is computed (n bytes of BWT in, all positions 0-based):
//   distances[i] = n (filler) unless i is the LAST position of a run of equal bytes; then with s = bwt[i], i' = the next
//   occurrence of s (start of its next run) and rank = number of distinct symbols in (i, i'):
//       distances[i] = i' - i - rank - 1;       for the last run of s: n - i - rank - 1, rank = final MTF rank of s
//   rank is exactly what mtf.encode(s) returns at i'.  init[s] = first occurrence of s (n if absent).
//   The item stream has one entry per run, in order: (run end, distance, symbol, last_rank = the MTF rank at which the
//   run began, 0 for a symbol's first run); distance_limit = n - run end.
//
// The sequential MTF list is replaced by "last occurrence" tables: the rank of s at position i' is the number of
// symbols whose last occurrence before i' is later than that of s.
//   k_dc_tables   per 4,096-byte block: last occurrence of every symbol inside the block, first occurrences, run count;
//                 fills distances[] with the filler                                   (n read, 4n written)
//   k_dc_scan_*   per symbol: running "last occurrence before block b" over the blocks, in two levels  (n/16 bytes)
//   k_dc_ranks    one warp per block walks its run starts with the last-occurrence table in registers (alphabets of up to
//                 32 symbols: one shuffle, one compare, one ballot per run) or in shared memory (8 entries per lane, one
//                 compare each, one warp reduction): rank, distance of the previous run of s, run record
//   k_dc_final    last runs and the final MTF order;   k_dc_stream   run ends + their distances, compacted
//
// MANY = true: many BWT blocks back to back (DESIGN.md §3.5).  The 4,096-byte chunks stay chunks of the concatenation and
// the scans run unchanged over global positions; a reader clamps a last occurrence against the start s_b of its own
// block (a value v <= s_b reads as "none": the symbol has not occurred in the block yet).  Every block start is a run
// start, so runs never cross a boundary.  k_dc_ranks finalises each block at its end (what k_dc_final does for one
// block) into a DcRecDev record; k_dc_final is not used.
#pragma once

#include "common.cuh"

namespace dark {

constexpr int kDcBlock = 4096;

struct DcInfoDev {  // mirrors the head of dark_bwt_dc_info
    unsigned long long init[256];
    u8 mtf_symbols[256];
    u32 num_unique;
    u32 reserved_;
    unsigned long long num_items;
};

// Per-block result of the many-block pass, expanded into dark_bwt_dc_info on the host (num_items from the item starts).
struct DcRecDev {
    u32 init[256];
    u8 mtf_symbols[256];
    u32 num_unique;
    u32 reserved_;
};
static_assert(sizeof(DcRecDev) == 1288, "include/dark_bwt.h states the record size");

// What the many-block instantiations read besides the single-block arguments (zero in the single-block ones).
struct DcMany {
    const u32* starts;      // block offsets [0..count], starts[count] = n
    u32 count;
    const u32* start_bits;  // bit p set: a block starts at position p
    DcRecDev* recs;         // [count]
    u32* item_starts;       // [0..count]: index of each block's first run; [count] = total runs
};

// the block holding position pos: the largest b < count with starts[b] <= pos
__device__ __forceinline__ u32 dc_block_of(const u32* __restrict__ starts, u32 count, u32 pos) {
    u32 lo = 0, hi = count - 1;
    while (lo < hi) {
        const u32 mid = (lo + hi + 1) >> 1;
        if (starts[mid] <= pos) lo = mid;
        else hi = mid - 1;
    }
    return lo;
}

// Block-start bitmap of the many-block pass (bits zeroed before), and item_starts[0] = 0.
__global__ void __launch_bounds__(256) k_dc_mark_starts(const u32* __restrict__ starts, u32 count, u32* __restrict__ bits,
                                                        u32* __restrict__ item_starts) {
    const u32 b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b < count) atomicOr(&bits[starts[b] >> 5], 1u << (starts[b] & 31));
    if (b == 0) item_starts[0] = 0u;
}

// first[256] must be preset to 0xFFFFFFFF, *total_runs to 0.  MANY: the filler is the length of the position's block,
// and a block start is a run start even where its byte equals the previous block's last byte.
template <bool MANY>
__global__ void __launch_bounds__(256)
k_dc_tables(const u8* __restrict__ bwt, u32 n, u32* __restrict__ tab, u32* __restrict__ first, u32* __restrict__ run_counts,
            u32* __restrict__ dist, unsigned long long* __restrict__ total_runs, DcMany many) {
    __shared__ u32 s_last[256], s_first[256];
    __shared__ u32 s_runs;
    const int tid = threadIdx.x;
    s_last[tid] = 0u;
    s_first[tid] = 0xFFFFFFFFu;
    if (tid == 0) s_runs = 0u;
    __syncthreads();
    const u64 base = (u64)blockIdx.x * kDcBlock + (u64)tid * 16;
    u32 runs = 0;
    if (base < n) {
        u32 prev = base > 0 ? (u32)bwt[base - 1] : 0x100u;
        u32 last_pos = 0;
        u32 b = 0, bs = 0, be = n;  // MANY: the block [bs, be) holding pos
        if constexpr (MANY) {
            b = dc_block_of(many.starts, many.count, (u32)base);
            bs = many.starts[b];
            be = many.starts[b + 1];
        }
#pragma unroll 4
        for (int k = 0; k < 16; ++k) {
            const u64 pos = base + k;
            if (pos < n) {
                const u32 s = bwt[pos];
                bool run_start = s != prev;
                if constexpr (MANY) {
                    if ((u32)pos == be) {  // blocks hold >= 1 byte: one step at most
                        bs = be;
                        be = many.starts[++b + 1];
                    }
                    run_start |= (u32)pos == bs;
                }
                if (run_start) {
                    ++runs;
                    atomicMin(&s_first[s], (u32)pos);
                    if (k > 0) atomicMax(&s_last[prev], (u32)pos);  // the run of prev ended at pos-1 (stored +1)
                }
                prev = s;
                last_pos = (u32)pos;
                if constexpr (MANY) dist[pos] = be - bs;
                else dist[pos] = n;
            }
        }
        atomicMax(&s_last[prev], last_pos + 1u);  // this thread's last byte (its run may go on in the next thread's bytes)
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) runs += __shfl_xor_sync(0xffffffffu, runs, o);
    if ((tid & 31) == 0 && runs) atomicAdd(&s_runs, runs);
    __syncthreads();
    tab[(size_t)blockIdx.x * 256 + tid] = s_last[tid];
    if (s_first[tid] != 0xFFFFFFFFu) atomicMin(&first[tid], s_first[tid]);
    if (tid == 0) {
        run_counts[blockIdx.x] = s_runs;
        atomicAdd(total_runs, (unsigned long long)s_runs);
    }
}

// tab[b][c] (last occurrence + 1 of c inside block b, 0 = none)  ->  last occurrence + 1 of c BEFORE block b, in two
// levels so that no thread walks more than kDcGroup + ngroups rows (one CTA walking all n / 4096 rows took 5 ms of a
// 16 ms stage on a 256 MiB block):
//   k_dc_scan_groups  CTA g, thread c: running last occurrence over the kDcGroup blocks of group g, starting from "none";
//                     group_last[g][c] = the group's own last occurrence
//   k_dc_scan_carry   one CTA: group_last[g][c] -> last occurrence before group g; final_last[c] = over the whole input
// A reader takes tab[b][c], or the carry of b's group where the group has not seen c before b.
constexpr int kDcGroup = 256;
__global__ void __launch_bounds__(256) k_dc_scan_groups(u32* __restrict__ tab, u32 nblocks, u32* __restrict__ group_last) {
    const int c = threadIdx.x;
    const u32 b0 = blockIdx.x * kDcGroup, b1 = min(nblocks, b0 + kDcGroup);
    u32 run = 0;
    u32 b = b0;
    for (; b + 8 <= b1; b += 8) {
        u32 t[8];
#pragma unroll
        for (int k = 0; k < 8; ++k) t[k] = tab[(size_t)(b + k) * 256 + c];
#pragma unroll
        for (int k = 0; k < 8; ++k) {
            tab[(size_t)(b + k) * 256 + c] = run;
            if (t[k]) run = t[k];
        }
    }
    for (; b < b1; ++b) {
        const u32 t = tab[(size_t)b * 256 + c];
        tab[(size_t)b * 256 + c] = run;
        if (t) run = t;
    }
    group_last[(size_t)blockIdx.x * 256 + c] = run;
}
__global__ void __launch_bounds__(256) k_dc_scan_carry(u32* __restrict__ group_last, u32 ngroups, u32* __restrict__ final_last) {
    const int c = threadIdx.x;
    u32 run = 0;
    for (u32 g = 0; g < ngroups; ++g) {
        const u32 t = group_last[(size_t)g * 256 + c];
        group_last[(size_t)g * 256 + c] = run;
        if (t) run = t;
    }
    final_last[c] = run;
}

// Dense codes of the symbols that occur (first[c] != ~0): alpha[0..255] = byte -> code, alpha[256..511] = code -> byte,
// alpha[512] = sigma.  One CTA of 256 threads.
__global__ void __launch_bounds__(256) k_dc_alphabet(const u32* __restrict__ first, u32* __restrict__ alpha) {
    __shared__ u32 s_warp[8];
    const int c = threadIdx.x, lane = c & 31, warp = c >> 5;
    const bool present = first[c] != 0xFFFFFFFFu;
    const u32 bal = __ballot_sync(0xffffffffu, present);
    if (lane == 0) s_warp[warp] = __popc(bal);
    __syncthreads();
    u32 base = 0;
    for (int w = 0; w < warp; ++w) base += s_warp[w];
    const u32 code = base + __popc(bal & ((1u << lane) - 1u));
    alpha[c] = present ? code : 0xFFu;
    if (present) alpha[256 + code] = (u32)c;
    if (c == 255) alpha[512] = base + __popc(bal);
}

// One warp per block.  run_offsets = exclusive scan of the blocks' run counts.
// Alphabets of up to 32 symbols (DNA, most text) keep the table in registers, one symbol per lane: the rank of a run start
// is one shuffle, one compare and one ballot.  Larger alphabets keep 256 entries in shared memory, 8 per lane.
// MANY: the warp tracks the text block [bs, be) of its position, found once by binary search.  At the run start i == be
// (or at the chunk's end when be is there) the table holds the block's final runs, and the warp finalises the block:
// last-run distances, MTF list, init of absent symbols, item_starts[b + 1].  A first run in the block records init.
template <bool MANY>
__global__ void __launch_bounds__(256, MANY ? 6 : 1)
k_dc_ranks(const u8* __restrict__ bwt, u32 n, const u32* __restrict__ tab, const u32* __restrict__ group_carry,
           const u32* __restrict__ run_offsets, u32 nblocks, const u32* __restrict__ alpha, u32* __restrict__ dist, u32* __restrict__ run_start, u8* __restrict__ run_sym,
           u8* __restrict__ run_rank, DcMany many) {
    __shared__ u32 s_tab[8][256];
    __shared__ u8 s_dense[256];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    s_dense[threadIdx.x] = (u8)alpha[threadIdx.x];
    const u32 sigma = alpha[512];
    __syncthreads();
    const u32 block = blockIdx.x * 8 + warp;
    if (block >= nblocks) return;
    const bool small = sigma <= 32u;
    u32* last = s_tab[warp];
    u32 lastreg = 0;  // small alphabets: last occurrence + 1 of the symbol with dense code `lane`
    const u32* carry_row = group_carry + (size_t)(block / kDcGroup) * 256;  // where the block's group had not met the symbol yet
    if (small) {
        if ((u32)lane < sigma) {
            const u32 c = alpha[256 + lane];
            const u32 t = tab[(size_t)block * 256 + c];
            lastreg = t ? t : carry_row[c];
        }
    } else {
#pragma unroll
        for (int k = 0; k < 8; ++k) {
            const u32 t = tab[(size_t)block * 256 + lane + 32 * k];
            last[lane + 32 * k] = t ? t : carry_row[lane + 32 * k];
        }
    }
    __syncwarp();
    u32 run_idx = run_offsets[block];
    const u64 block_base = (u64)block * kDcBlock;
    u32 tb = 0, bs = 0, be = n;  // MANY: the text block [bs, be) of the current position
    if constexpr (MANY) {
        tb = dc_block_of(many.starts, many.count, (u32)block_base);
        bs = many.starts[tb];
        be = many.starts[tb + 1];
    }
    // MANY: finalise text block tb (the table holds its final runs; next_run = index of the run after its last), step to
    // the next.  Symbols with v > bs occur in the block; a later v is in the block too, so their ranks need no clamping.
    auto finish = [&](u32 next_run) {
        DcRecDev* rec = many.recs + tb;
        const u32 nb = be - bs;
        u32 nu = 0, below;
        if (small) {
            const bool present = lastreg > bs;  // lanes >= sigma hold 0
            u32 rank = 0;
            for (int t = 0; t < 32; ++t) rank += __shfl_sync(0xffffffffu, lastreg, t) > lastreg ? 1u : 0u;
            nu = __popc(__ballot_sync(0xffffffffu, present));
            if (present) {
                dist[lastreg - 1] = be - lastreg - rank;
                rec->mtf_symbols[rank] = (u8)alpha[256 + lane];
            }
        } else {
#pragma unroll 1
            for (int k = 0; k < 8; ++k) {
                const u32 v = last[lane + 32 * k];
                if (v > bs) {
                    u32 rank = 0;
                    for (int c = 0; c < 256; ++c) rank += last[c] > v ? 1u : 0u;
                    dist[v - 1] = be - v - rank;
                    rec->mtf_symbols[rank] = (u8)(lane + 32 * k);
                    ++nu;
                }
            }
            nu = __reduce_add_sync(0xffffffffu, nu);
        }
        below = nu;  // absent symbols: the tail of the list in ascending order, init = block length
#pragma unroll 1
        for (int k = 0; k < 8; ++k) {
            const u32 c = (u32)lane + 32u * k;
            bool absent;
            if (small) {
                const u32 d = s_dense[c];
                const u32 v = __shfl_sync(0xffffffffu, lastreg, (int)(d & 31u));
                absent = d == 0xFFu || v <= bs;
            } else {
                absent = last[c] <= bs;
            }
            const u32 ab = __ballot_sync(0xffffffffu, absent);
            if (absent) {
                rec->mtf_symbols[below + __popc(ab & ((1u << lane) - 1u))] = (u8)c;
                rec->init[c] = nb;
            }
            below += __popc(ab);
        }
        if (lane == 0) {
            rec->num_unique = nu;
            rec->reserved_ = 0u;
            many.item_starts[tb + 1] = next_run;
        }
        __syncwarp();
        ++tb;
        bs = be;
        if (tb < many.count) be = many.starts[tb + 1];
    };
    (void)finish;
    u32 carry = block_base > 0 ? (u32)bwt[block_base - 1] : 0x100u;
    for (int chunk = 0; chunk < kDcBlock / 32; ++chunk) {
        const u64 pos0 = block_base + (u64)chunk * 32;
        if (pos0 >= n) break;
        const u64 pos = pos0 + lane;
        const bool valid = pos < n;
        const u32 byte = valid ? (u32)bwt[pos] : 0u;
        u32 prevb = __shfl_up_sync(0xffffffffu, byte, 1);
        if (lane == 0) prevb = carry;
        u32 mask = __ballot_sync(0xffffffffu, valid && byte != prevb);
        if constexpr (MANY) mask |= many.start_bits[pos0 >> 5];  // pos0 is a multiple of 32; no block starts at or past n
        // run records of this chunk are written together: lane q keeps the q-th run start of the chunk
        const u32 nruns = __popc(mask);
        u32 rec_start = 0, rec_sym = 0, rec_rank = 0;
        u32 q = 0;
        while (mask) {
            const int j = __ffs(mask) - 1;
            mask &= mask - 1;
            const u32 s = __shfl_sync(0xffffffffu, byte, j), ps = __shfl_sync(0xffffffffu, prevb, j);
            const u32 i = (u32)(pos0 + j);
            u32 old, rank;
            if (small) {
                if (ps < 0x100u && (u32)lane == (u32)s_dense[ps]) lastreg = i;  // the run before this one ended at i-1 (stored +1)
                if constexpr (MANY)
                    if (i == be) finish(run_idx + q);
                old = __shfl_sync(0xffffffffu, lastreg, (int)s_dense[s]);
                if constexpr (MANY)
                    if (old <= bs) old = 0u;  // last seen in an earlier block: the first run of s in this one
                rank = __popc(__ballot_sync(0xffffffffu, lastreg > old));
            } else {
                if (lane == 0 && ps < 0x100u) last[ps] = i;
                __syncwarp();
                if constexpr (MANY)
                    if (i == be) finish(run_idx + q);
                old = last[s];  // end + 1 of the previous run of s (0: this is its first)
                if constexpr (MANY)
                    if (old <= bs) old = 0u;
                u32 cnt = 0;
#pragma unroll
                for (int k = 0; k < 8; ++k) cnt += last[lane + 32 * k] > old ? 1u : 0u;
                rank = __reduce_add_sync(0xffffffffu, cnt);
                __syncwarp();
            }
            DARK_ASSERT(old <= i && (old == 0 || i >= old + rank));
            if constexpr (MANY)
                if (lane == 0 && !old) many.recs[tb].init[s] = i - bs;
            if (lane == 0 && old) dist[old - 1] = i - (old - 1u) - rank - 1u;
            if ((u32)lane == q) {
                rec_start = i;
                rec_sym = s;
                rec_rank = old ? rank : 0u;
            }
            ++q;
        }
        DARK_ASSERT((u64)run_idx + nruns <= (u64)n);
        if ((u32)lane < nruns) {
            run_start[run_idx + lane] = rec_start;
            run_sym[run_idx + lane] = (u8)rec_sym;
            run_rank[run_idx + lane] = (u8)rec_rank;
        }
        run_idx += nruns;
        carry = __shfl_sync(0xffffffffu, byte, 31);
    }
    if constexpr (MANY) {
        const u32 chunk_end = block_base + kDcBlock < (u64)n ? (u32)(block_base + kDcBlock) : n;
        if (be == chunk_end) {  // the text block ends with this chunk: its final run goes into the table first
            const u32 ps = bwt[chunk_end - 1];
            if (small) {
                if ((u32)lane == (u32)s_dense[ps]) lastreg = chunk_end;
            } else {
                if (lane == 0) last[ps] = chunk_end;
                __syncwarp();
            }
            finish(run_idx);
        }
    }
}

// Last runs + final MTF order + init.  One CTA of 256 threads.
__global__ void __launch_bounds__(256)
k_dc_final(u32 n, const u32* __restrict__ final_last, const u32* __restrict__ first, u32* __restrict__ dist,
           const unsigned long long* __restrict__ total_runs, DcInfoDev* __restrict__ info) {
    __shared__ u32 s_last[256];
    __shared__ u32 s_present;
    const int c = threadIdx.x;
    const u32 mine = final_last[c];
    s_last[c] = mine;
    if (c == 0) s_present = 0;
    __syncthreads();
    u32 rank = 0;
    for (int k = 0; k < 256; ++k) rank += s_last[k] > mine ? 1u : 0u;
    if (mine) {
        dist[mine - 1] = n - (mine - 1u) - rank - 1u;
        info->mtf_symbols[rank] = (u8)c;
        atomicAdd(&s_present, 1u);
    }
    info->init[c] = mine ? (unsigned long long)first[c] : (unsigned long long)n;
    __syncthreads();
    if (!mine) {  // absent symbols fill the tail of the list in ascending order (any order will do: they are never looked up)
        u32 below = 0;
        for (int k = 0; k < c; ++k) below += s_last[k] == 0 ? 1u : 0u;
        info->mtf_symbols[s_present + below] = (u8)c;
    }
    if (c == 0) {
        info->num_unique = s_present;
        info->reserved_ = 0;
        info->num_items = *total_runs;
    }
}

// The item stream: run r ends just before run r+1 starts (MANY: runs never cross a block; positions are block-relative).
template <bool MANY>
__global__ void __launch_bounds__(256)
k_dc_stream(const u32* __restrict__ run_start, const unsigned long long* __restrict__ total_runs, u32 n, const u32* __restrict__ dist,
            u32* __restrict__ out_pos, u32* __restrict__ out_dist, DcMany many) {
    const u64 R = *total_runs;
    const u64 stride = (u64)gridDim.x * blockDim.x;
    for (u64 r = (u64)blockIdx.x * blockDim.x + threadIdx.x; r < R; r += stride) {
        const u32 end = (r + 1 < R ? run_start[r + 1] : n) - 1u;
        u32 pos = end;
        if constexpr (MANY) pos -= many.starts[dc_block_of(many.starts, many.count, end)];
        out_pos[r] = pos;
        out_dist[r] = dist[end];
    }
}

// ---- the packed item stream (include/dark_bwt.h): per item sym, rank, varint(run length - 1), varint(dist) ----------
// The items k_dc_stream wrote, m of them, become one byte string in three launches over tiles of kPackTile items:
//   k_dc_pack_sizes   each tile's byte count                                     (reads pos, dist: 8 B per item)
//   k_dc_pack_scan    one CTA: the tile counts -> u64 tile offsets and the total (a stream can pass 2^32 bytes)
//   k_dc_pack_write   each tile again: sizes, block scan, the tile's bytes built in shared memory, then stored as one
//                     contiguous span with 16-byte stores (bytes one by one only in the span's first and last 16-byte word)
// MANY = true: the items of a many-block pass, back to back in block order (item_pos block-relative).  Each block's stream
// is what the block alone packs to: at an item that opens a block (a bit of k_dc_mark_items' bitmap) the previous run end
// is -1 again, so the streams of the blocks are simply concatenated, and the thread that codes a block's first item writes
// where it lands to stream_starts[block].  k_dc_pack_scan serves both forms.
constexpr int kPackThreads = 256;
constexpr int kPackItems = 8;  // consecutive items per thread
constexpr int kPackTile = kPackThreads * kPackItems;
constexpr int kPackMaxItemBytes = 12;  // sym + rank + two varints of at most 5 bytes

__device__ __forceinline__ u32 varint_bytes(u32 v) {
    return 1u + (v >= (1u << 7)) + (v >= (1u << 14)) + (v >= (1u << 21)) + (v >= (1u << 28));
}

// What the many-block instantiations of the pack read and write besides the single-block arguments (zero in the others).
struct PackMany {
    const u32* first_bits;   // bit k set: item k is the first item of a block
    const u32* item_starts;  // [0..count]: index of each block's first item (k_dc_ranks), [count] = all items
    u32 count;
    u64* stream_starts;      // [0..count): offset of each block's first byte in the stream
};

// The first-item bitmap of the pack (bits zeroed before): blocks hold at least one run, so item_starts[b] are distinct.
__global__ void __launch_bounds__(256) k_dc_mark_items(const u32* __restrict__ item_starts, u32 count, u32* __restrict__ bits) {
    const u32 b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b < count) atomicOr(&bits[item_starts[b] >> 5], 1u << (item_starts[b] & 31));
}

__device__ __forceinline__ bool first_item(const PackMany& many, u64 k) { return (many.first_bits[k >> 5] >> (k & 31)) & 1u; }

// run length - 1 of item k is pos[k] - pos[k-1] - 1 with pos[-1] = -1: in u32 arithmetic, prev = 0xFFFFFFFF for k = 0
// (MANY: and for the first item of every block)
template <bool MANY>
__global__ void __launch_bounds__(kPackThreads)
k_dc_pack_sizes(const u32* __restrict__ pos, const u32* __restrict__ dist, u64 m, u32* __restrict__ tile_bytes, PackMany many) {
    __shared__ u32 s_warp[kPackThreads / 32];
    const u64 k0 = (u64)blockIdx.x * kPackTile + threadIdx.x;
    u32 bytes = 0;
#pragma unroll
    for (int j = 0; j < kPackItems; ++j) {
        const u64 k = k0 + (u64)j * kPackThreads;
        if (k < m) {
            u32 prev = k ? pos[k - 1] : 0xFFFFFFFFu;
            if constexpr (MANY)
                if (first_item(many, k)) prev = 0xFFFFFFFFu;
            bytes += 2u + varint_bytes(pos[k] - prev - 1u) + varint_bytes(dist[k]);
        }
    }
    bytes = __reduce_add_sync(0xffffffffu, bytes);
    if ((threadIdx.x & 31) == 0) s_warp[threadIdx.x >> 5] = bytes;
    __syncthreads();
    if (threadIdx.x == 0) {
        u32 t = 0;
#pragma unroll
        for (int w = 0; w < kPackThreads / 32; ++w) t += s_warp[w];
        tile_bytes[blockIdx.x] = t;
    }
}

// One CTA of 1024 threads, 4 tiles per thread and step: tile_off[t] = bytes of the tiles before t; *total = all of them
// (the context's mapped mailbox: the host reads it after one synchronise).
__global__ void __launch_bounds__(1024, 1)
k_dc_pack_scan(const u32* __restrict__ tile_bytes, u32 ntiles, u64* __restrict__ tile_off, unsigned long long* __restrict__ total) {
    __shared__ u64 s_warp[32];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    u64 carry = 0;
    for (u32 base = 0; base < ntiles; base += 4096) {
        const u32 i0 = base + 4u * (u32)tid;
        u32 v[4];
        u64 sum = 0;
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            v[j] = i0 + j < ntiles ? tile_bytes[i0 + j] : 0u;
            sum += v[j];
        }
        u64 x = sum;  // inclusive scan over the warp
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const u64 y = __shfl_up_sync(0xffffffffu, x, o);
            if (lane >= o) x += y;
        }
        if (lane == 31) s_warp[warp] = x;
        __syncthreads();
        if (warp == 0) {
            u64 w = s_warp[lane];
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const u64 y = __shfl_up_sync(0xffffffffu, w, o);
                if (lane >= o) w += y;
            }
            s_warp[lane] = w;
        }
        __syncthreads();
        u64 off = carry + (warp ? s_warp[warp - 1] : 0ull) + x - sum;
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            if (i0 + j < ntiles) tile_off[i0 + j] = off;
            off += v[j];
        }
        carry += s_warp[31];
        __syncthreads();  // s_warp is rewritten by the next step
    }
    if (tid == 0) *total = carry;
}

// Thread t of a tile codes its items tile0 + 8t .. 8t+7 into s_buf at shift + (bytes of the tile's items before them),
// shift = the address of the tile's first byte mod 16, so that s_buf's 16-byte words line up with out's.
// MANY: a thread's 8 items (k0 is a multiple of 8) have their first-item bits in one bitmap word.
template <bool MANY>
__global__ void __launch_bounds__(kPackThreads)
k_dc_pack_write(const u32* __restrict__ pos, const u32* __restrict__ dist, const u8* __restrict__ sym, const u8* __restrict__ rank,
                u64 m, const u64* __restrict__ tile_off, u8* __restrict__ out, PackMany many) {
    __shared__ __align__(16) u8 s_buf[kPackTile * kPackMaxItemBytes + 16];
    __shared__ u32 s_warp[kPackThreads / 32];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const u64 k0 = (u64)blockIdx.x * kPackTile + (u64)tid * kPackItems;
    u32 p[kPackItems], d[kPackItems];
    u32 prev = k0 > 0 && k0 < m ? pos[k0 - 1] : 0xFFFFFFFFu;
    u32 firsts = 0;  // MANY: bit j set: item k0 + j is the first item of a block
    if constexpr (MANY)
        if (k0 < m) firsts = (many.first_bits[k0 >> 5] >> (k0 & 31)) & 0xFFu;
    u32 bytes = 0;
    {
        u32 q = prev;
#pragma unroll
        for (int j = 0; j < kPackItems; ++j) {
            const u64 k = k0 + j;
            p[j] = k < m ? pos[k] : 0u;
            d[j] = k < m ? dist[k] : 0u;
            if constexpr (MANY)
                if ((firsts >> j) & 1u) q = 0xFFFFFFFFu;
            if (k < m) bytes += 2u + varint_bytes(p[j] - q - 1u) + varint_bytes(d[j]);
            q = p[j];
        }
    }
    u32 x = bytes;  // exclusive block scan of the threads' byte counts
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const u32 y = __shfl_up_sync(0xffffffffu, x, o);
        if (lane >= o) x += y;
    }
    if (lane == 31) s_warp[warp] = x;
    __syncthreads();
    u32 before = 0, tile_bytes = 0;
#pragma unroll
    for (int w = 0; w < kPackThreads / 32; ++w) {
        const u32 t = s_warp[w];
        if (w < warp) before += t;
        tile_bytes += t;
    }
    const u64 base = tile_off[blockIdx.x];
    const u32 shift = (u32)(((uintptr_t)out + base) & 15u);
    u32 o = shift + before + x - bytes;
    DARK_ASSERT(o + bytes <= sizeof(s_buf));
#pragma unroll
    for (int j = 0; j < kPackItems; ++j) {
        if (k0 + j >= m) break;
        if constexpr (MANY) {
            if ((firsts >> j) & 1u) {
                prev = 0xFFFFFFFFu;
                many.stream_starts[dc_block_of(many.item_starts, many.count, (u32)(k0 + j))] = base + (o - shift);
            }
        }
        s_buf[o++] = sym[k0 + j];
        s_buf[o++] = rank[k0 + j];
        u32 v = p[j] - prev - 1u;
        prev = p[j];
        for (; v >= 0x80u; v >>= 7) s_buf[o++] = (u8)(v | 0x80u);
        s_buf[o++] = (u8)v;
        v = d[j];
        for (; v >= 0x80u; v >>= 7) s_buf[o++] = (u8)(v | 0x80u);
        s_buf[o++] = (u8)v;
    }
    __syncthreads();
    u8* const dst = (u8*)((uintptr_t)out + base - shift);  // 16-byte aligned; only [shift, end) of it is written
    const u32 end = shift + tile_bytes;
    for (u32 w = (u32)tid; w * 16u < end; w += kPackThreads) {
        const u32 lo = w * 16u, hi = lo + 16u;
        if (lo >= shift && hi <= end) {
            *(uint4*)(dst + lo) = *(const uint4*)(s_buf + lo);
        } else {
            for (u32 b = max(lo, shift); b < min(hi, end); ++b) dst[b] = s_buf[b];
        }
    }
}

}  // namespace dark
