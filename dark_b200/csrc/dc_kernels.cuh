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

// ---- decoding the packed item stream (the inverse of the pack; DESIGN.md §3.9) ---------------------------------------
// Item boundaries are sequential: sym and rank bytes are arbitrary, only the varints end on a byte with bit 7 clear.  A
// stretch of the stream is summarised for each of the four states it may be entered in (0 = at an item's sym byte, 1 = at
// its rank byte, 2 = inside the run-length varint, 3 = inside the distance varint) and the summaries compose, so the
// boundaries are found in parallel:
//   k_dc_unpack_tiles   per tile of kUnpackTile bytes: its summary (a block scan of the threads' 32-byte chunks)
//   k_dc_unpack_chain   one CTA: the tiles chained from state 0 at byte 0 -> each tile's entry state, item base and run
//                       start base; the totals and the first malformed item into the mailbox (the host checks them)
//   k_dc_unpack_items   each tile again from its entry state: every item's run start and symbol
//   k_dc_unpack_expand  per 4 KiB of output: the tile's runs by binary search, its bytes with 16-byte stores
//   k_dc_unpack_compare the first byte at which the stream differs from the decoded block's re-pack
// An item is decoded whole by the thread whose chunk holds its sym byte, which reads at most kPackMaxItemBytes bytes and
// never at or past the end of the stream; a varint of more than 5 bytes, one above 2^32 - 1, or an item cut off by the end
// is malformed.  The walks jump from item to item, so a chunk costs at most its 32 bytes whatever the bytes are.
constexpr int kUnpackThreads = 256;
constexpr int kUnpackChunk = 32;  // bytes per thread
constexpr int kUnpackTile = kUnpackThreads * kUnpackChunk;
constexpr u32 kUnpackNone = 0xFFFFFFFFu;
constexpr u64 kUnpackSumCap = 1ull << 40;  // the chain saturates run-length sums here (a valid stream sums to n < 2^32)

// A stretch of the stream, for each entry state s.  Composing stretch a, then b: b is entered in a's exit state.
struct UnpackSum {
    u64 sum[4];    // run lengths of the items whose sym byte lies in the stretch
    u32 items[4];  // those items
    u32 err[4];    // tile-relative offset of the first malformed one, kUnpackNone if none
    u32 exit;      // 2 bits per s: the state after the stretch
    u32 pad_;
};

struct UnpackBase {  // a tile as the chain enters it
    u64 item;  // index of the first item whose sym byte lies in the tile
    u64 pos;   // its run start
    u32 state;
    u32 pad_;
};

template <typename T>
__device__ __forceinline__ T unpack_pick(const T (&a)[4], u32 s) {  // a[s] without dynamic indexing (no local memory)
    return s == 0 ? a[0] : s == 1 ? a[1] : s == 2 ? a[2] : a[3];
}

__device__ __forceinline__ UnpackSum unpack_identity() {
    UnpackSum r;
#pragma unroll
    for (int s = 0; s < 4; ++s) r.sum[s] = 0, r.items[s] = 0, r.err[s] = kUnpackNone;
    r.exit = 0xE4u;  // s -> s
    r.pad_ = 0;
    return r;
}

__device__ __forceinline__ UnpackSum unpack_then(const UnpackSum& a, const UnpackSum& b) {
    UnpackSum r;
    r.exit = 0;
    r.pad_ = 0;
#pragma unroll
    for (int s = 0; s < 4; ++s) {
        const u32 t = (a.exit >> (2 * s)) & 3u;
        r.exit |= ((b.exit >> (2 * t)) & 3u) << (2 * s);
        r.items[s] = a.items[s] + unpack_pick(b.items, t);
        r.sum[s] = a.sum[s] + unpack_pick(b.sum, t);
        r.err[s] = a.err[s] != kUnpackNone ? a.err[s] : unpack_pick(b.err, t);
    }
    return r;
}

__device__ __forceinline__ UnpackSum unpack_shfl_up(const UnpackSum& v, int o) {
    UnpackSum r;
#pragma unroll
    for (int s = 0; s < 4; ++s) {
        r.sum[s] = __shfl_up_sync(0xffffffffu, v.sum[s], o);
        r.items[s] = __shfl_up_sync(0xffffffffu, v.items[s], o);
        r.err[s] = __shfl_up_sync(0xffffffffu, v.err[s], o);
    }
    r.exit = __shfl_up_sync(0xffffffffu, v.exit, o);
    r.pad_ = 0;
    return r;
}

// Exclusive block scan of the threads' summaries in thread order (blockDim.x = 32 * warps); *total = all of them.
template <int WARPS>
__device__ __forceinline__ UnpackSum unpack_block_scan(const UnpackSum& v, UnpackSum* s_warp /* [WARPS] */, UnpackSum* total) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    UnpackSum x = v;  // inclusive scan over the warp
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const UnpackSum y = unpack_shfl_up(x, o);
        if (lane >= o) x = unpack_then(y, x);
    }
    UnpackSum ex = unpack_shfl_up(x, 1);
    if (lane == 0) ex = unpack_identity();
    if (lane == 31) s_warp[warp] = x;
    __syncthreads();
    if (warp == 0) {  // the warps' totals, scanned in place
        UnpackSum w = lane < WARPS ? s_warp[lane] : unpack_identity();
#pragma unroll
        for (int o = 1; o < WARPS; o <<= 1) {
            const UnpackSum y = unpack_shfl_up(w, o);
            if (lane >= o) w = unpack_then(y, w);
        }
        if (lane < WARPS) s_warp[lane] = w;
    }
    __syncthreads();
    *total = s_warp[WARPS - 1];
    const UnpackSum r = warp ? unpack_then(s_warp[warp - 1], ex) : ex;
    __syncthreads();  // s_warp may be rewritten by the caller's next scan
    return r;
}

// One unsigned LEB128 of at most 5 bytes at buf[q], not reaching lim: the offset after it, or 0 if malformed (*val = its value).
__device__ __forceinline__ u32 unpack_varint(const u8* buf, u32 q, u32 lim, u32* val) {
    u64 v = 0;
    u32 b = 0x80u;
    int k = 0;
    for (; k < 5 && (b & 0x80u) && q < lim; ++k, ++q) {
        b = buf[q];
        v |= (u64)(b & 0x7Fu) << (7 * k);
    }
    *val = (u32)v;
    return (b & 0x80u) || v > 0xFFFFFFFFull ? 0u : q;
}

// Walks buf[c0, c1) entered in `state`; lim = the stream's bytes in buf (>= c1).  Items whose sym byte lies in the chunk
// are decoded whole (they may reach past c1, never to lim); emit(sym, run length) is called for each in order.
// *err_at = the chunk's first malformed item (kUnpackNone: none); the walk stops there.  Returns the exit state.
template <typename Emit>
__device__ __forceinline__ u32 unpack_walk(const u8* buf, u32 c0, u32 c1, u32 lim, u32 state, u32* err_at, Emit emit) {
    *err_at = kUnpackNone;
    u32 p = c0;
    while (p < c1) {
        if (state == 0) {
            u32 len1 = 0, d = 0;
            const u32 len_end = p + 1 < lim ? unpack_varint(buf, p + 2, lim, &len1) : 0u;
            const u32 q = len_end ? unpack_varint(buf, len_end, lim, &d) : 0u;
            if (!q) {
                *err_at = p;
                return 0;
            }
            emit((u32)buf[p], (u64)len1 + 1u);
            if (q <= c1) {
                p = q;
                continue;
            }
            return c1 == p + 1 ? 1u : c1 < len_end ? 2u : 3u;  // the item goes on past the chunk
        }
        const u32 b = buf[p++];
        if (state == 1) state = 2;
        else if (!(b & 0x80u)) state = state == 2 ? 3u : 0u;
    }
    return state;
}

// The tile's bytes [tile0, tile0 + kUnpackTile + 16) into shared memory (zero past the stream); returns the stream's bytes
// in it (the walks' lim) and sets *len = those of the tile proper.
__device__ __forceinline__ u32 unpack_load_tile(const u8* __restrict__ stream, u64 bytes, u64 tile0, u8* s_buf, u32* len) {
    const u64 left = bytes - tile0;
    const u32 lim = (u32)min(left, (u64)kUnpackTile + 16);
    for (u32 i = threadIdx.x; i < (u32)kUnpackTile + 16; i += blockDim.x) s_buf[i] = i < lim ? stream[tile0 + i] : (u8)0;
    *len = min(lim, (u32)kUnpackTile);
    __syncthreads();
    return lim;
}

// The summary of this thread's chunk for each entry state.
__device__ __forceinline__ UnpackSum unpack_chunk(const u8* s_buf, u32 len, u32 lim) {
    const u32 c0 = min((u32)threadIdx.x * kUnpackChunk, len), c1 = min(c0 + kUnpackChunk, len);
    UnpackSum v;
    v.exit = 0;
    v.pad_ = 0;
#pragma unroll
    for (int s = 0; s < 4; ++s) {
        u32 items = 0;
        u64 sum = 0;
        const u32 x = unpack_walk(s_buf, c0, c1, lim, (u32)s, &v.err[s], [&](u32, u64 run) {
            ++items;
            sum += run;
        });
        v.exit |= x << (2 * s);
        v.items[s] = items;
        v.sum[s] = sum;
    }
    return v;
}

__global__ void __launch_bounds__(kUnpackThreads, 1)
k_dc_unpack_tiles(const u8* __restrict__ stream, u64 bytes, UnpackSum* __restrict__ tiles) {
    __shared__ __align__(16) u8 s_buf[kUnpackTile + 16];
    __shared__ UnpackSum s_warp[kUnpackThreads / 32];
    u32 len;
    const u32 lim = unpack_load_tile(stream, bytes, (u64)blockIdx.x * kUnpackTile, s_buf, &len);
    UnpackSum total;
    unpack_block_scan<kUnpackThreads / 32>(unpack_chunk(s_buf, len, lim), s_warp, &total);
    if (threadIdx.x == 0) tiles[blockIdx.x] = total;
}

// Mailbox fields the chain writes (the context's mapped mailbox; the host reads them after one synchronise).
struct UnpackTotals {
    unsigned long long items;  // items of the whole stream
    unsigned long long sum;    // their run lengths (saturated at kUnpackSumCap)
    unsigned long long err;    // byte offset of the first malformed item, ~0 if none
    u32 state;                 // the state after the last byte (0: the stream ends at an item boundary)
    u32 pad_;
};

// One CTA of kChainThreads threads, kChainTiles tiles per thread and step: the tiles in order from state 0, item 0, run start 0.
constexpr int kChainThreads = 512, kChainTiles = 8;
__global__ void __launch_bounds__(kChainThreads, 1)
k_dc_unpack_chain(const UnpackSum* __restrict__ tiles, u32 ntiles, UnpackBase* __restrict__ bases, UnpackTotals* __restrict__ out) {
    __shared__ UnpackSum s_warp[kChainThreads / 32];
    __shared__ unsigned long long s_err;
    if (threadIdx.x == 0) s_err = ~0ull;
    u32 state = 0;
    u64 item = 0, pos = 0;
    for (u32 base = 0; base < ntiles; base += kChainThreads * kChainTiles) {
        const u32 i0 = base + (u32)kChainTiles * threadIdx.x;
        UnpackSum mine = unpack_identity();
#pragma unroll 1
        for (int j = 0; j < kChainTiles; ++j)
            if (i0 + j < ntiles) mine = unpack_then(mine, tiles[i0 + j]);
        UnpackSum total;
        const UnpackSum before = unpack_block_scan<kChainThreads / 32>(mine, s_warp, &total);
        u32 st = (before.exit >> (2 * state)) & 3u;
        u64 it = item + unpack_pick(before.items, state), ps = pos + unpack_pick(before.sum, state);
#pragma unroll 1
        for (int j = 0; j < kChainTiles; ++j) {
            if (i0 + j >= ntiles) break;
            const UnpackSum& t = tiles[i0 + j];
            bases[i0 + j] = UnpackBase{it, ps, st, 0u};
            const u32 e = unpack_pick(t.err, st);
            if (e != kUnpackNone) atomicMin(&s_err, (unsigned long long)(i0 + j) * kUnpackTile + e);
            it += unpack_pick(t.items, st);
            ps += unpack_pick(t.sum, st);
            st = (t.exit >> (2 * st)) & 3u;
        }
        item += unpack_pick(total.items, state);
        pos = min(pos + unpack_pick(total.sum, state), kUnpackSumCap);
        state = (total.exit >> (2 * state)) & 3u;
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        out->items = item;
        out->sum = pos;
        out->err = s_err;
        out->state = state;
    }
}

// Each tile from its entry state: run_start[k] and run_sym[k] of every item k whose sym byte lies in it.  The host has
// checked the chain's totals (no malformed item, the run lengths add up to n), so k < n and every start is below n; the
// bound is kept anyway.
__global__ void __launch_bounds__(kUnpackThreads, 1)
k_dc_unpack_items(const u8* __restrict__ stream, u64 bytes, const UnpackBase* __restrict__ bases, u32 n, u32* __restrict__ run_start,
                  u8* __restrict__ run_sym) {
    __shared__ __align__(16) u8 s_buf[kUnpackTile + 16];
    __shared__ UnpackSum s_warp[kUnpackThreads / 32];
    u32 len;
    const u32 lim = unpack_load_tile(stream, bytes, (u64)blockIdx.x * kUnpackTile, s_buf, &len);
    const UnpackBase tb = bases[blockIdx.x];
    UnpackSum total;
    const UnpackSum before = unpack_block_scan<kUnpackThreads / 32>(unpack_chunk(s_buf, len, lim), s_warp, &total);
    const u32 state = (before.exit >> (2 * tb.state)) & 3u;
    u64 k = tb.item + unpack_pick(before.items, tb.state);
    u64 pos = tb.pos + unpack_pick(before.sum, tb.state);
    const u32 c0 = min((u32)threadIdx.x * kUnpackChunk, len), c1 = min(c0 + kUnpackChunk, len);
    u32 err;
    unpack_walk(s_buf, c0, c1, lim, state, &err, [&](u32 sym, u64 run) {
        DARK_ASSERT(k < n && pos < n);
        if (k < n) {
            run_start[k] = (u32)pos;
            run_sym[k] = (u8)sym;
        }
        ++k;
        pos += run;
    });
}

// Output tile b covers the 16-byte words [256 b, 256 b + 256) of out's aligned address space; thread t writes word 256 b + t
// (16-byte store where all its bytes are in [0, n)).  run_start[0..m) strictly increases from 0 (the host's checks): the
// tile's runs are the lo..hi found by binary search, at most 4,096 of them, staged in shared memory.
constexpr int kExpandWords = 256;
__global__ void __launch_bounds__(kExpandWords)
k_dc_unpack_expand(const u32* __restrict__ run_start, const u8* __restrict__ run_sym, u32 m, u32 n, u8* __restrict__ out) {
    __shared__ u32 s_start[kExpandWords * 16];
    __shared__ u8 s_sym[kExpandWords * 16];
    __shared__ u32 s_run[2];
    const u32 shift = (u32)((uintptr_t)out & 15u);
    const u64 v0 = (u64)blockIdx.x * kExpandWords * 16;  // the tile's first position in the aligned space (output byte v0 - shift)
    if (threadIdx.x < 2) {  // the runs holding the tile's first (thread 0) and last (thread 1) byte: the largest r with run_start[r] <= p
        const u32 p = threadIdx.x ? (u32)min(v0 + kExpandWords * 16 - shift, (u64)n) - 1u : (u32)(v0 > shift ? v0 - shift : 0);
        u32 lo = 0, hi = m - 1;
        while (lo < hi) {
            const u32 mid = lo + (hi - lo + 1) / 2;
            if (run_start[mid] <= p) lo = mid;
            else hi = mid - 1;
        }
        s_run[threadIdx.x] = lo;
    }
    __syncthreads();
    const u32 lo = s_run[0], cnt = min(s_run[1] - lo + 1u, (u32)kExpandWords * 16);
    DARK_ASSERT(s_run[1] >= lo && s_run[1] - lo < (u32)kExpandWords * 16);
    for (u32 j = threadIdx.x; j < cnt; j += kExpandWords) {
        s_start[j] = run_start[lo + j];
        s_sym[j] = run_sym[lo + j];
    }
    __syncthreads();
    const u64 w0 = v0 + (u64)threadIdx.x * 16;  // this thread's word; its bytes are output positions w0 - shift + 0..15
    if (w0 + 16 <= shift || w0 >= (u64)n + shift) return;
    const u32 a = (u32)(w0 > shift ? w0 - shift : 0), b = (u32)min(w0 + 16 - shift, (u64)n);  // [a, b) valid
    u32 j = 0, hi = cnt - 1;  // the run holding a
    while (j < hi) {
        const u32 mid = j + (hi - j + 1) / 2;
        if (s_start[mid] <= a) j = mid;
        else hi = mid - 1;
    }
    u32 word[4] = {0u, 0u, 0u, 0u};
#pragma unroll
    for (int k = 0; k < 16; ++k) {
        const u64 p = w0 + k - shift;  // wraps below 0 for the bytes before out: those are never stored
        if (p >= a && p < b) {
            while (j + 1 < cnt && s_start[j + 1] <= (u32)p) ++j;
            word[k >> 2] |= (u32)s_sym[j] << (8 * (k & 3));
        }
    }
    if (b - a == 16) {
        *(uint4*)(out + (w0 - shift)) = make_uint4(word[0], word[1], word[2], word[3]);
    } else {
#pragma unroll
        for (int k = 0; k < 16; ++k) {
            const u64 p = w0 + k - shift;
            if (p >= a && p < b) out[p] = (u8)(word[k >> 2] >> (8 * (k & 3)));
        }
    }
}

// *first = min(*first, the first offset < bytes where a and b differ); first preset to ~0, *done to 0.  The last CTA to
// finish copies the answer into the mailbox (*out).
__global__ void __launch_bounds__(256)
k_dc_unpack_compare(const u8* __restrict__ a, const u8* __restrict__ b, u64 bytes, unsigned long long* first, u32* done,
                    unsigned long long* out) {
    __shared__ unsigned long long s_first;
    __shared__ bool s_last;
    if (threadIdx.x == 0) s_first = ~0ull;
    __syncthreads();
    unsigned long long mine = ~0ull;
    const u64 stride = (u64)gridDim.x * blockDim.x;
    for (u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x; i < bytes; i += stride)
        if (a[i] != b[i]) {
            mine = i;
            break;  // later offsets of this thread are larger
        }
    if (mine != ~0ull) atomicMin(&s_first, mine);
    __syncthreads();
    if (threadIdx.x == 0) {
        if (s_first != ~0ull) atomicMin(first, s_first);
        __threadfence();
        s_last = atomicAdd(done, 1u) == gridDim.x - 1;
    }
    __syncthreads();
    if (s_last && threadIdx.x == 0) *out = atomicMin(first, ~0ull);
}

}  // namespace dark
