/*
 * dark_bwt.h — C ABI of the B200-native forward Burrows–Wheeler transform that replaces
 * kvark/dark's `saca::Constructor::compute` + `compress::bwt::TransformIterator`.
 *
 * This is the drop-in boundary: plain pointers and sizes, no C++/torch types, nothing
 * unwinds across it.  A Rust `-sys` crate binds exactly these symbols (INTEGRATION.md
 * shows the binding and the 6-line patch to src/block/{dc,raw}.rs).
 *
 * Reference interface each entry point replaces (paths under /root/reference):
 *
 *   dark_bwt_create        saca::Constructor::new(max_n)            src/saca.rs:351-360
 *   dark_bwt_capacity      Constructor::capacity()                  src/saca.rs:363-365
 *   dark_bwt_forward       Constructor::compute(input) followed by  src/saca.rs:368-378
 *                          bwt::TransformIterator::new(input, suf)
 *                          .collect() / .get_origin()               src/block/dc.rs:45-50
 *                                                                   src/block/raw.rs:39-44
 *   dark_bwt_reuse         Constructor::reuse()                     src/saca.rs:381-383
 *   dark_bwt_destroy       Drop of Constructor
 *   dark_bwt_strerror      text of the panic the Rust wrapper raises (assert!s at
 *                          src/saca.rs:272,300,369)
 *
 * Semantics (bit-exact with the reference, SURVEY.md App. A.1):
 *   SA   = the permutation of 0..n-1 sorting the suffixes T[i..n) as byte strings,
 *          a proper prefix sorting first (virtual end-of-text below every byte);
 *   bwt[i] = T[SA[i]-1], except at the one i with SA[i]==0 where bwt[i] = T[n-1]
 *          and origin = i (known-answer test src/saca.rs:409-413).
 *   Suffix = uint32_t (src/saca.rs:20), so 2 <= n <= 2^32-2; n < 2 is an error because
 *   the reference panics there (n==0: src/saca.rs:69, n==1: src/saca.rs:300).
 *
 * Threading: a context is NOT thread-safe (the reference's `&mut self`); distinct
 * contexts are independent — one per GPU per host thread.  Every call selects the
 * context's device itself.  There is no CPU fallback: without a usable CUDA device
 * dark_bwt_create fails with DARK_BWT_E_CUDA.
 */
#ifndef DARK_BWT_H
#define DARK_BWT_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define DARK_BWT_ABI_VERSION 2

/* error codes (0 = ok) */
#define DARK_BWT_OK 0
#define DARK_BWT_E_INVALID_N 1   /* n < 2, n > capacity, or n > 2^32-2                       */
#define DARK_BWT_E_INVALID_ARG 2 /* null pointer / bad device / bad flags                    */
#define DARK_BWT_E_CUDA 3        /* a CUDA call failed; dark_bwt_last_error() has the text    */
#define DARK_BWT_E_NOMEM 4       /* device or pinned-host allocation failed at create        */
#define DARK_BWT_E_INTERNAL 5    /* invariant violated (should not happen; reported, not UB) */

/* flags for dark_bwt_create_ex */
#define DARK_BWT_F_DEFAULT 0u
/* Canonical mode of SURVEY.md §8(d): 8 raw bytes per initial key (no alphabet packing), so
 * the per-round active counts equal the oracle profiler's m_r.  Results are identical. */
#define DARK_BWT_F_NO_ALPHABET_PACKING 1u
/* Do not allocate the host-entry staging (device text/BWT/SA-out buffers, pinned memory):
 * for callers that only use dark_bwt_forward_device. */
#define DARK_BWT_F_DEVICE_ONLY 2u
/* Reserve two distance-coding output slots (dist 4N + item_pos 4N + item_dist 4N + item_sym N + item_rank N, twice:
 * 28 N bytes more, 73 N in all; 18.3 GiB for a 256 MiB block, 146 GiB for 2 GiB) for dark_bwt_forward_dc_batch.
 * Not combinable with DARK_BWT_F_DEVICE_ONLY. */
#define DARK_BWT_F_DC_BATCH 4u

#define DARK_BWT_MAX_ROUNDS 40

typedef struct dark_bwt_ctx dark_bwt_ctx;

/* Filled by the forward calls when `stats` is non-null.  Times are CUDA-event times on the
 * context's stream (milliseconds). */
typedef struct dark_bwt_stats {
    uint64_t n;
    uint32_t sigma;           /* distinct byte values in the block                        */
    uint32_t bits_per_symbol; /* s                                                        */
    uint32_t symbols_per_key; /* K: symbols packed into the initial 64-bit key            */
    uint32_t initial_symbols; /* K0 <= K: whole symbols the (pruned) initial sort ordered */
    uint32_t pair_rounds;     /* rounds handled by the pairs kernel (every group was a pair)  */
    uint32_t rounds;          /* prefix-doubling rounds after the initial sort            */
    uint32_t sort_passes;     /* radix-pass kernel launches, all rounds                   */
    uint32_t kernel_launches; /* every kernel this call launched                          */
    uint64_t active[DARK_BWT_MAX_ROUNDS]; /* [0] = n; [r] = unsettled suffixes entering round r */
    uint32_t passes[DARK_BWT_MAX_ROUNDS]; /* radix passes run in round r (0 = initial sort)     */
    uint64_t sorted_elements; /* sum over pass launches of the elements each one moved    */
    float device_ms;          /* whole forward: first kernel -> BWT + origin in HBM       */
    float init_ms;            /* alphabet scan + initial key build                        */
    float sort_ms;            /* histogram scan + radix-pass kernels (incl. host round trip) */
    float pass_ms;            /* radix-pass kernels alone (with their status memsets)     */
    float keybuild_ms;        /* (rank[i], rank[i+h]) key construction                    */
    float rerank_ms;          /* re-rank + compaction scans                               */
    float emit_ms;            /* BWT gather + origin                                      */
    float h2d_ms;             /* blocking host entries: host-clock time of all copies of the caller's buffers to the
                                 device; 0 in the pipelined batch entries and the device entries */
    float d2h_ms;             /* the same for the copies back to the caller's buffers     */
    /* the key-generating first pass (reads 1 B of text and writes 12 B per suffix instead of 12 + 12), part of the figures above */
    uint32_t gen_passes;      /* key-generating pass launches (0 or 1)                    */
    float gen_pass_ms;        /* their share of pass_ms                                   */
    uint64_t gen_elements;    /* their share of sorted_elements                           */
    uint32_t host_syncs;      /* stream synchronisations this call needed (host round trips) */
    uint32_t reserved_;
} dark_bwt_stats;

/* Constructor::new — allocates every device buffer for blocks of up to max_n bytes on
 * CUDA device `device`: one arena of dark_bwt_arena_bytes(max_n, flags) bytes of HBM, about 44.8 * max_n (40.8 * max_n with
 * DARK_BWT_F_DEVICE_ONLY, 72.8 * max_n with DARK_BWT_F_DC_BATCH; 12.0 GB for a 256 MiB block, 96.2 GB for 2^31).  Above
 * 2^31 bytes, without DARK_BWT_F_DEVICE_ONLY or DARK_BWT_F_DC_BATCH, the context keeps one host-entry staging pair instead
 * of two (about 42.8 * max_n: 183.8 GB for 2^32-2, which a 180 GB B200 holds); the batch entries then run their blocks one
 * after another.  DARK_BWT_F_DC_BATCH tops out near 2.4 GiB on a B200.  No device memory is allocated later; the pinned
 * staging lanes for pageable host buffers (12 lanes x 2 slots x 2 MiB per direction) and the `reuse` scratch are allocated
 * by the first call that needs them. */
int dark_bwt_create(uint64_t max_n, int device, dark_bwt_ctx **out);
int dark_bwt_create_ex(uint64_t max_n, int device, uint32_t flags, dark_bwt_ctx **out);

/* The exact bytes dark_bwt_create_ex(max_n, ., flags, .) allocates in its arena, or 0 for a max_n or flags it rejects.
 * Host arithmetic only: touches no device.  Lets a caller learn before create whether a block fits a card. */
uint64_t dark_bwt_arena_bytes(uint64_t max_n, uint32_t flags);

/* Constructor::capacity */
uint64_t dark_bwt_capacity(const dark_bwt_ctx *ctx);

/* compute + TransformIterator on HOST buffers: text[0..n) -> bwt_out[0..n), *origin_out,
 * and, if sa_out is non-null, the suffix array sa_out[0..n).  Pinned (cudaHostAlloc / cudaHostRegister) buffers are
 * DMA'd directly; pageable ones (a plain Vec<u8>, malloc) of 1 MiB or more go through the context's pinned staging
 * lanes: DARK_BWT_HOST_THREADS host threads (default 12, at most the host's cores less two; 0 = leave it to the driver) each copy 2 MiB chunks into their
 * own pinned chunk and send them on, so the memcpy of one lane overlaps the DMA of the others.  `stats` nullable. */
int dark_bwt_forward(dark_bwt_ctx *ctx, const uint8_t *text, uint64_t n, uint8_t *bwt_out, uint64_t *origin_out,
                     uint32_t *sa_out, dark_bwt_stats *stats);

/* `count` independent host blocks through one context, pipelined: while block k is transformed, block
 * k+1 is copied in and block k-1 is copied out (two copy streams beside the compute stream, double-
 * buffered device staging).  This is how a corpus of blocks is fed — the reference encodes one block
 * per Encoder (src/main.rs:95-113) and blocks share nothing.  Pinned host buffers overlap fully;
 * pageable ones still work.  A context above 2^31 has one staging pair (dark_bwt_create) and does not overlap
 * blocks: each is copied in, transformed and copied out before the next is copied in.  sa_outs and stats are nullable (entries of sa_outs too); stats, if
 * given, is an array of `count` records.  Results are identical to `count` dark_bwt_forward calls. */
int dark_bwt_forward_batch(dark_bwt_ctx *ctx, const uint8_t *const *texts, const uint64_t *ns, uint8_t *const *bwt_outs,
                           uint64_t *origins_out, uint32_t *const *sa_outs, uint64_t count, dark_bwt_stats *stats);

/* MANY SMALL blocks in ONE sort.  A block the size of the reference's CPU test file (768 KB) keeps a B200 busy
 * for a fraction of its 0.5 ms of launches; `count` such blocks (each >= 2 bytes, sum <= capacity, count <=
 * DARK_BWT_MAX_MANY_BLOCKS) are concatenated and their suffixes sorted together, every suffix ending at the end
 * of its own block.  Results are identical to `count` dark_bwt_forward calls: bwt_outs[k][0..ns[k]) and
 * origins_out[k].  One H2D copy per block into one device text, one device pass, one D2H copy per block (pageable blocks
 * of 1 MiB or more go through the staging lanes, as in dark_bwt_forward).
 * (src/main.rs:87-113: the reference's CLI feeds its blocks one after another through one Encoder.) */
#define DARK_BWT_MAX_MANY_BLOCKS 65536u
int dark_bwt_forward_many(dark_bwt_ctx *ctx, const uint8_t *const *texts, const uint64_t *ns, uint8_t *const *bwt_outs,
                          uint64_t *origins_out, uint64_t count, dark_bwt_stats *stats);
/* Same on device buffers: d_text holds the blocks back to back, d_starts[0..count] their offsets (d_starts[0] = 0,
 * d_starts[count] = total bytes); d_bwt_out gets the BWTs at the same offsets, d_origins_out[0..count) the origins,
 * d_sa_out (nullable) the per-block suffix arrays (block-relative indices) at the same offsets. */
int dark_bwt_forward_many_device(dark_bwt_ctx *ctx, const uint8_t *d_text, const uint32_t *d_starts, uint64_t count,
                                 uint8_t *d_bwt_out, uint64_t *d_origins_out, uint32_t *d_sa_out, dark_bwt_stats *stats);

/* Same on DEVICE buffers (d_text, d_bwt_out, d_sa_out live on the context's device;
 * d_sa_out nullable; origin_out and stats are host pointers).  No readable slack after
 * d_text[n-1] is required.  Returns after the work has completed on the stream. */
int dark_bwt_forward_device(dark_bwt_ctx *ctx, const uint8_t *d_text, uint64_t n, uint8_t *d_bwt_out,
                            uint64_t *origin_out, uint32_t *d_sa_out, dark_bwt_stats *stats);

/* Inverse transform (SURVEY.md 8f, the unpack side): text_out[0..n) from bwt[0..n) and origin — what
 * `compress::bwt::decode(&input, origin, &mut suffixes)` yields at src/block/dc.rs:154-156 and
 * src/block/raw.rs:98-100 (also saca.rs:405,424).  Host and device-buffer forms; 1 <= n <= capacity,
 * origin < n.  DARK_BWT_E_INVALID_ARG if (bwt, origin) is not the forward transform of any text. */
int dark_bwt_inverse(dark_bwt_ctx *ctx, const uint8_t *bwt, uint64_t n, uint64_t origin, uint8_t *text_out);
int dark_bwt_inverse_device(dark_bwt_ctx *ctx, const uint8_t *d_bwt, uint64_t n, uint64_t origin, uint8_t *d_text_out,
                            float *ms_out /* nullable */);

/* `count` independent host blocks, pipelined like dark_bwt_forward_batch: while block k is inverted, block k+1 is copied
 * in and block k-1 copied out (double-buffered device staging, the two copy streams, pageable buffers of 1 MiB or more
 * through the staging lanes; no overlap on a context above 2^31, as in dark_bwt_forward_batch).  Each block:
 * 1 <= ns[k] <= capacity, origins[k] < ns[k].  ms_out (nullable) = `count`
 * device times.  Results identical to `count` dark_bwt_inverse calls; DARK_BWT_E_INVALID_ARG with a device-only context. */
int dark_bwt_inverse_batch(dark_bwt_ctx *ctx, const uint8_t *const *bwts, const uint64_t *ns, const uint64_t *origins,
                           uint8_t *const *text_outs, uint64_t count, float *ms_out);

/* MANY SMALL blocks inverted in ONE pass, the unpack side of dark_bwt_forward_many: `count` BWT blocks (each >= 1 byte,
 * origins[k] < ns[k], count <= DARK_BWT_MAX_MANY_BLOCKS) give text_outs[k][0..ns[k]), what dark_bwt_inverse(bwts[k],
 * ns[k], origins[k]) gives.  The blocks share one row space of sum(ns) + count rows (one '$' row per block), which must
 * fit: sum(ns) + count <= capacity, else DARK_BWT_E_INVALID_N.  One H2D copy per block, one device pass, one D2H copy per
 * block (pageable blocks of 1 MiB or more go through the staging lanes).  ms_out (nullable) = device time of the pass.
 * DARK_BWT_E_INVALID_ARG if some (bwt, origin) is not the forward transform of any text; dark_bwt_last_error() then names
 * the first such block. */
int dark_bwt_inverse_many(dark_bwt_ctx *ctx, const uint8_t *const *bwts, const uint64_t *ns, const uint64_t *origins,
                          uint8_t *const *text_outs, uint64_t count, float *ms_out);
/* Same on device buffers, the layout dark_bwt_forward_many_device writes: d_bwt holds the blocks back to back,
 * d_starts[0..count] (u32) their offsets, d_origins[0..count) (u64) their origins, all on the device (offsets and origins
 * are read back and checked before any kernel runs); d_text_out gets the texts at the same offsets. */
int dark_bwt_inverse_many_device(dark_bwt_ctx *ctx, const uint8_t *d_bwt, const uint32_t *d_starts, const uint64_t *d_origins,
                                 uint64_t count, uint8_t *d_text_out, float *ms_out);

/* ---- distance coding + MTF (SURVEY.md 8f rank 3) ---------------------------------------------------------------
 * What `bwt::dc::encode(&output, suf, &mut self.mtf)` computes and what iterating its result yields
 * (/root/reference/src/block/dc.rs:52, 54-85).  That code is third-party (`compress::bwt::dc`, Cargo.toml:18) and absent
 * from the reference tree, and no reference test holds a known answer for it: PARITY UNPINNED (checked against a
 * CPU restatement of upstream rust-compress in the test suite and by encode -> decode round trips).
 *   dist[i]  = n (the filler) unless i is the last byte of a run; then next_occurrence - i - rank - 1, rank = the MTF rank
 *              of the symbol at its next occurrence (= distinct symbols in between); for a symbol's last run
 *              n - i - final rank - 1.  This is the `distances` slice the reference passes in as `suf` (block/dc.rs:51).
 *   items    = one (distance, Context) per run, in order: item_pos = run end (Context.distance_limit = n - item_pos),
 *              item_dist, item_sym = Context.symbol, item_rank = Context.last_rank.  */
typedef struct dark_bwt_dc_info {
    uint64_t init[256];       /* get_init(): first occurrence of each byte value, n if it does not occur */
    uint8_t mtf_symbols[256]; /* the MTF list after the block: the num_unique symbols by recency, then the absent ones */
    uint32_t num_unique;
    uint32_t reserved_;
    uint64_t num_items;       /* runs of equal bytes = (distance, Context) items */
    float device_ms;          /* CUDA-event time of the DC kernels */
    uint32_t reserved2_;
} dark_bwt_dc_info;

/* Device buffers.  d_dist_out (n words) and the four item arrays (room for n entries each) are nullable: what the caller
 * does not ask for stays in the context's arena.  1 <= n <= capacity. */
int dark_bwt_dc_encode_device(dark_bwt_ctx *ctx, const uint8_t *d_bwt, uint64_t n, uint32_t *d_dist_out, uint32_t *d_item_pos,
                              uint32_t *d_item_dist, uint8_t *d_item_sym, uint8_t *d_item_rank, dark_bwt_dc_info *info);
/* Host buffers (pageable or pinned); every output but `info` nullable.  The item arrays need room for n entries
 * (info->num_items are written). */
int dark_bwt_dc_encode(dark_bwt_ctx *ctx, const uint8_t *bwt, uint64_t n, uint32_t *dist_out, uint32_t *item_pos,
                       uint32_t *item_dist, uint8_t *item_sym, uint8_t *item_rank, dark_bwt_dc_info *info);
/* block/dc.rs:45-52 in one call: forward BWT of text[0..n), then distance coding of the BWT while it is still in HBM.
 * bwt_out and the DC outputs are nullable (a caller that codes the item stream needs neither bwt_out nor dist_out). */
int dark_bwt_forward_dc(dark_bwt_ctx *ctx, const uint8_t *text, uint64_t n, uint8_t *bwt_out, uint64_t *origin_out,
                        uint32_t *dist_out, uint32_t *item_pos, uint32_t *item_dist, uint8_t *item_sym, uint8_t *item_rank,
                        dark_bwt_dc_info *info, dark_bwt_stats *stats);
/* `count` independent host blocks through dark_bwt_forward_dc, pipelined like dark_bwt_forward_batch: while block k is
 * transformed and distance-coded, block k+1 is copied in and the outputs of block k-1 are copied out (two device BWT
 * buffers and the two DC output slots of a context created with DARK_BWT_F_DC_BATCH).  This is how the reference's
 * per-block loop (src/main.rs:87-113 -> block/dc.rs:45-85) feeds a run of large blocks.  Block k gets exactly what
 * dark_bwt_forward_dc(texts[k], ...) gives: bwt_outs[k][0..ns[k]), origins_out[k], dist_outs[k][0..ns[k]), the
 * infos[k].num_items items, and infos[k] (device_ms = that block's DC time).  Required: texts (and every entry), ns,
 * origins_out, infos (`count` records).  Nullable: every output array and every entry of one (a caller that codes the
 * item stream passes neither BWT nor distances: then only the items cross PCIe), and stats (`count` records).  Pinned
 * host buffers overlap fully; pageable ones of 1 MiB or more go through the staging lanes.  DARK_BWT_E_INVALID_ARG,
 * before any device work, for a context without DARK_BWT_F_DC_BATCH or a null required pointer; DARK_BWT_E_INVALID_N
 * for any ns[k] outside [2, capacity].  count == 0 is DARK_BWT_OK. */
int dark_bwt_forward_dc_batch(dark_bwt_ctx *ctx, const uint8_t *const *texts, const uint64_t *ns, uint64_t count,
                              uint8_t *const *bwt_outs, uint64_t *origins_out, uint32_t *const *dist_outs,
                              uint32_t *const *item_pos, uint32_t *const *item_dist, uint8_t *const *item_sym,
                              uint8_t *const *item_rank, dark_bwt_dc_info *infos, dark_bwt_stats *stats);

/* ---- the packed item stream: the items of one block as one byte string ---------------------------------------------
 * The four item arrays cost 10 bytes per run on the way out; most of those bytes are zero.  The packed entries below code
 * a block's info->num_items items, k = 0, 1, ..., as one byte string, per item in this order:
 *     item_sym[k]                                    1 byte
 *     item_rank[k]                                   1 byte
 *     varint(item_pos[k] - item_pos[k-1] - 1)        run length - 1, with item_pos[-1] = -1
 *     varint(item_dist[k])
 * varint = unsigned LEB128: 7 bits per byte, the low group first, bit 7 set on every byte but the last (a u32 takes at
 * most 5 bytes).  A consumer keeps a running run end, pos = -1 before the first item and pos += 1 + the first varint at
 * each item; that is item_pos[k], and Context.distance_limit = n - pos.  init[], the MTF list, num_unique and num_items stay in dark_bwt_dc_info.  About 4 bytes per run on DNA and
 * text blocks instead of 10.
 * Size: the run lengths add up to n, and varint(len - 1) <= len bytes, so a block of n bytes packs into at most
 * 2 + 5 bytes per item plus n, at most DARK_BWT_DC_PACKED_MAX(n) bytes: a buffer of that size never fails the capacity
 * check.  Capacity: the stream's size is always written to *stream_bytes_out (stream_bytes_out[k]); a size above the
 * buffer's capacity is DARK_BWT_E_INVALID_ARG, nothing is written to the stream buffer, dark_bwt_last_error() names the
 * bytes needed (and, in the batch, the block), and the context stays usable.  info->device_ms includes the pack kernels. */
#define DARK_BWT_DC_PACKED_MAX(n) (8ull * (uint64_t)(n))
/* Device buffers: distance coding of d_bwt[0..n), its items packed into d_stream_out (stream_capacity bytes).  The item
 * arrays stay in the context's arena.  1 <= n <= capacity.  Returns after the work has completed on the stream. */
int dark_bwt_dc_encode_packed_device(dark_bwt_ctx *ctx, const uint8_t *d_bwt, uint64_t n, uint8_t *d_stream_out,
                                     uint64_t stream_capacity, uint64_t *stream_bytes_out, dark_bwt_dc_info *info);
/* dark_bwt_forward_dc with the packed stream as the only DC output: only the stream (and the BWT, if bwt_out is non-null)
 * crosses PCIe.  Host buffers, pageable or pinned; 2 <= n <= capacity; stats nullable. */
int dark_bwt_forward_dc_packed(dark_bwt_ctx *ctx, const uint8_t *text, uint64_t n, uint8_t *bwt_out /* nullable */,
                               uint64_t *origin_out, uint8_t *stream_out, uint64_t stream_capacity,
                               uint64_t *stream_bytes_out, dark_bwt_dc_info *info, dark_bwt_stats *stats /* nullable */);
/* `count` host blocks through dark_bwt_forward_dc_packed, pipelined like dark_bwt_forward_dc_batch (a context created with
 * DARK_BWT_F_DC_BATCH; block k's stream is packed into its DC output slot).  Block k gets exactly what
 * dark_bwt_forward_dc_packed(texts[k], ...) gives.  Required: texts, ns, origins_out, stream_outs (every entry),
 * stream_capacities, stream_bytes_out, infos (`count` records each).  Nullable: bwt_outs and its entries, stats.
 * DARK_BWT_E_INVALID_ARG, before any device work, for a context without DARK_BWT_F_DC_BATCH or a null required pointer;
 * DARK_BWT_E_INVALID_N for any ns[k] outside [2, capacity].  count == 0 is DARK_BWT_OK.  A block whose stream does not fit
 * its buffer ends the call: every block before it is complete, stream_bytes_out[k] holds the size it needs. */
int dark_bwt_forward_dc_packed_batch(dark_bwt_ctx *ctx, const uint8_t *const *texts, const uint64_t *ns, uint64_t count,
                                     uint8_t *const *bwt_outs /* nullable, entries too */, uint64_t *origins_out,
                                     uint8_t *const *stream_outs, const uint64_t *stream_capacities,
                                     uint64_t *stream_bytes_out, dark_bwt_dc_info *infos, dark_bwt_stats *stats /* nullable */);

/* MANY SMALL blocks distance-coded in ONE pass.  Block k gives exactly what dark_bwt_dc_encode gives on that block alone:
 * every value is block-relative (filler and last-run distances use n_k, init[c] is the first occurrence inside the block
 * or n_k, item_pos is the run end inside the block, runs never merge across a boundary).  Outputs:
 *   infos[0..count)          host array, one record per block; device_ms is the time of the one pass (also *ms_out);
 *   dist                     the blocks' distances at their byte offsets (room for sum(ns) words);
 *   item_starts[0..count]    u32 offsets of each block's items, item_starts[count] = total runs;
 *   item_pos/dist/sym/rank   the items of all blocks in block order (room for sum(ns) entries each).
 * Every output but `infos` is nullable.  Limits: count <= DARK_BWT_MAX_MANY_BLOCKS (else DARK_BWT_E_INVALID_ARG), each
 * block >= 1 byte, sum(ns) <= capacity and <= 2^32-2, and the per-block records (1,288 bytes each) are staged in an
 * 8 * capacity + 1 KiB buffer: count * 1288 <= 8 * capacity + 1024 (blocks of about 161 bytes or more on average at full
 * capacity), else DARK_BWT_E_INVALID_N.  One H2D copy per block, one device pass, one D2H copy per output array (pageable
 * blocks and arrays of 1 MiB or more go through the staging lanes).
 * DARK_BWT_E_INVALID_ARG with a device-only context. */
int dark_bwt_dc_encode_many(dark_bwt_ctx *ctx, const uint8_t *const *bwts, const uint64_t *ns, uint64_t count, uint32_t *dist_out,
                            uint32_t *item_starts, uint32_t *item_pos, uint32_t *item_dist, uint8_t *item_sym, uint8_t *item_rank,
                            dark_bwt_dc_info *infos, float *ms_out);
/* Same on device buffers, the layout dark_bwt_forward_many_device writes: d_bwt holds the blocks back to back at the u32
 * offsets d_starts[0..count] (on the device; read back and checked before any kernel runs: d_starts[0] = 0, offsets
 * increasing).  The outputs are device buffers with the layout above; `infos` and `ms_out` are host pointers. */
int dark_bwt_dc_encode_many_device(dark_bwt_ctx *ctx, const uint8_t *d_bwt, const uint32_t *d_starts, uint64_t count,
                                   uint32_t *d_dist_out, uint32_t *d_item_starts, uint32_t *d_item_pos, uint32_t *d_item_dist,
                                   uint8_t *d_item_sym, uint8_t *d_item_rank, dark_bwt_dc_info *infos, float *ms_out);
/* block/dc.rs:45-52 for many small blocks: dark_bwt_forward_many, then the pass above over the BWTs while they are still in
 * HBM.  Each block >= 2 bytes; bwt_outs (and its entries) nullable; stats reports the sort as dark_bwt_forward_many does. */
int dark_bwt_forward_dc_many(dark_bwt_ctx *ctx, const uint8_t *const *texts, const uint64_t *ns, uint64_t count,
                             uint8_t *const *bwt_outs, uint64_t *origins_out, uint32_t *dist_out, uint32_t *item_starts,
                             uint32_t *item_pos, uint32_t *item_dist, uint8_t *item_sym, uint8_t *item_rank,
                             dark_bwt_dc_info *infos, dark_bwt_stats *stats);

/* MANY SMALL blocks with the packed item stream: the pass above, each block's items packed as the packed entries pack them.
 * Block k's bytes are exactly what dark_bwt_dc_encode_packed_device / dark_bwt_forward_dc_packed give for that block alone;
 * the blocks' streams lie back to back in block order, and count + 1 u64 offsets locate them: block k is
 * stream[stream_starts[k] .. stream_starts[k+1]), stream_starts[0] = 0, stream_starts[count] = *stream_bytes_out = the
 * total, at most DARK_BWT_DC_PACKED_MAX(sum(ns)).  Limits and errors are those of the entries above (count <=
 * DARK_BWT_MAX_MANY_BLOCKS, sum(ns) <= capacity, the record bound count * 1288 <= 8 * capacity + 1024).  The capacity rule
 * is the packed entries': the total is always written to *stream_bytes_out; a total above stream_capacity is
 * DARK_BWT_E_INVALID_ARG, neither the stream nor the offsets are written, dark_bwt_last_error() names the bytes needed, and
 * the context stays usable.  infos[k].device_ms (and *ms_out) = the time of the pass and the pack.  count == 0 is
 * DARK_BWT_OK with *stream_bytes_out = 0 (and, in the host form, stream_starts[0] = 0). */
/* Device buffers, the layout of dark_bwt_dc_encode_many_device: the blocks (each >= 1 byte) back to back in d_bwt at the u32
 * offsets d_starts[0..count]; the stream goes to d_stream_out (stream_capacity bytes), the offsets to d_stream_starts
 * (count + 1 u64, on the device).  infos (count records), stream_bytes_out and ms_out (nullable) are host pointers.  The
 * item arrays stay in the context's arena.  Returns after the work has completed on the stream. */
int dark_bwt_dc_encode_packed_many_device(dark_bwt_ctx *ctx, const uint8_t *d_bwt, const uint32_t *d_starts, uint64_t count,
                                          uint8_t *d_stream_out, uint64_t stream_capacity, uint64_t *d_stream_starts,
                                          uint64_t *stream_bytes_out, dark_bwt_dc_info *infos, float *ms_out);
/* Host buffers: dark_bwt_forward_many of texts[0..count) (each >= 2 bytes), then the pass above while the BWTs are in HBM;
 * only the stream, its offsets (stream_starts: a host array of count + 1) and the BWTs, if asked for, cross PCIe.  Pageable
 * or pinned; bwt_outs (and its entries) and stats nullable.  DARK_BWT_E_INVALID_ARG with a device-only context. */
int dark_bwt_forward_dc_packed_many(dark_bwt_ctx *ctx, const uint8_t *const *texts, const uint64_t *ns, uint64_t count,
                                    uint8_t *const *bwt_outs /* nullable, entries too */, uint64_t *origins_out,
                                    uint8_t *stream_out, uint64_t stream_capacity, uint64_t *stream_starts,
                                    uint64_t *stream_bytes_out, dark_bwt_dc_info *infos, dark_bwt_stats *stats /* nullable */);

/* ---- decoding the packed item stream: the unpack side of the packed entries ------------------------------------------
 * A stream is valid for n when it is byte for byte what dark_bwt_dc_encode_packed_device writes for some block of n bytes;
 * the symbols and run lengths fix that block, and the decoders return it.  Any other byte string is
 * DARK_BWT_E_INVALID_ARG (wrong distances or ranks, non-canonical varints such as 0x80 0x00, two adjacent items with the
 * same symbol, trailing bytes included), and the context stays usable.  The decoders are safe for any input bytes: they
 * read nothing past stream_bytes, write nothing past n output bytes, and end in bounded time. */
/* The inverse of dark_bwt_dc_encode_packed_device: d_bwt_out[0..n) gets the block whose packed item stream is
 * d_stream[0..stream_bytes) (device buffers, any alignment).  1 <= n <= capacity.  DARK_BWT_E_INVALID_ARG unless the
 * stream is exactly the packed stream of some block of n bytes (dark_bwt_last_error() says why: where the parse failed,
 * the run lengths' sum against n, or the first byte at which the stream differs from the decoded block's); d_bwt_out is
 * then unspecified.  info (nullable) gets what dark_bwt_dc_encode_packed_device gives for the decoded block, device_ms =
 * this call's device time.  Returns after the work has completed on the stream. */
int dark_bwt_dc_decode_packed_device(dark_bwt_ctx *ctx, const uint8_t *d_stream, uint64_t stream_bytes, uint64_t n,
                                     uint8_t *d_bwt_out, dark_bwt_dc_info *info);
/* The unpack side of dark_bwt_forward_dc_packed in one call: the stream (host, pageable or pinned) is decoded into the BWT,
 * which stays in HBM and is inverted with `origin` into text_out[0..n).  bwt_out and info nullable.  1 <= n <= capacity,
 * origin < n.  DARK_BWT_E_INVALID_ARG as above, or when (BWT, origin) is not the transform of any text (the inverse's own
 * check); neither text_out nor bwt_out is written then.  DARK_BWT_E_INVALID_ARG with a device-only context.
 * Both entries, before any device work: a null required pointer is DARK_BWT_E_INVALID_ARG, n outside [1, capacity]
 * DARK_BWT_E_INVALID_N, stream_bytes == 0 or above DARK_BWT_DC_PACKED_MAX(n) (no valid stream is that long) and
 * origin >= n DARK_BWT_E_INVALID_ARG. */
int dark_bwt_inverse_dc_packed(dark_bwt_ctx *ctx, const uint8_t *stream, uint64_t stream_bytes, uint64_t n, uint64_t origin,
                               uint8_t *text_out, uint8_t *bwt_out, dark_bwt_dc_info *info);

/* Constructor::reuse — lends >= capacity host u32 words of scratch (DC distances in
 * block/dc.rs:51).  Allocated on first use; owned by the context. */
int dark_bwt_reuse(dark_bwt_ctx *ctx, uint32_t **words_out, uint64_t *count_out);

void dark_bwt_destroy(dark_bwt_ctx *ctx);

const char *dark_bwt_strerror(int code);
/* Text of the last CUDA/internal failure on this context ("" if none). */
const char *dark_bwt_last_error(const dark_bwt_ctx *ctx);

/* The CUDA stream (cudaStream_t) all of this context's work is launched on, so a harness
 * can bracket calls with its own events. */
void *dark_bwt_stream(const dark_bwt_ctx *ctx);

int dark_bwt_abi_version(void);

/* ---- building blocks, exported for unit tests, verification and benches ------------------ */

/* LSD radix sort of (u64 key, u32 value) pairs on bits [begin_bit, end_bit) with the
 * context's onesweep passes.  d_keys/d_vals hold the input; d_keys_alt/d_vals_alt are
 * scratch of the same size.  *in_alt_out = 1 if the sorted data ended in the alt buffers.
 * count <= capacity. */
int dark_bwt_sort_pairs_device(dark_bwt_ctx *ctx, uint64_t *d_keys, uint32_t *d_vals, uint64_t *d_keys_alt,
                               uint32_t *d_vals_alt, uint64_t count, int begin_bit, int end_bit, int *in_alt_out,
                               float *ms_out);

/* O(n) device check that d_sa is the suffix array of d_text (permutation; then for every j:
 * T[SA[j]] < T[SA[j+1]], or equal and ISA[SA[j]+1] < ISA[SA[j+1]+1], end-of-text lowest).
 * *bad_out = number of violations (0 = correct). Independent of the construction kernels. */
int dark_bwt_verify_sa_device(dark_bwt_ctx *ctx, const uint8_t *d_text, uint64_t n, const uint32_t *d_sa,
                              uint64_t *bad_out);

/* LCP profile of a block from its suffix array (SURVEY.md 8d): m_out[r-1] = number of suffixes not unique by
 * their first 8*2^(r-1) bytes, r = 1..*rounds_out (m_out has 64 entries), and the maximum LCP.  This is the
 * data-defined round structure behind the algorithmic byte count B_alg = 243 n + (48 + 24 P) * sum(m_r). */
int dark_bwt_lcp_profile_device(dark_bwt_ctx *ctx, const uint8_t *d_text, uint64_t n, const uint32_t *d_sa, uint64_t *m_out,
                                uint32_t *rounds_out, uint64_t *max_lcp_out);

/* BWT emission alone: bwt[i] = T[SA[i]-1] / origin, from a device SA. */
int dark_bwt_emit_device(dark_bwt_ctx *ctx, const uint8_t *d_text, uint64_t n, const uint32_t *d_sa,
                         uint8_t *d_bwt_out, uint64_t *origin_out);

/* Synthetic block generators of SURVEY.md App. D on the host ("dna", "rep17", "text",
 * "mixed").  Returns DARK_BWT_E_INVALID_ARG for an unknown kind. */
int dark_bwt_synth(const char *kind, uint64_t seed, uint8_t *out, uint64_t n);

#ifdef __cplusplus
}
#endif
#endif /* DARK_BWT_H */
