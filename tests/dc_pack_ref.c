/*
 * TEST INFRASTRUCTURE ONLY: a straight sequential statement of the packed item stream of include/dark_bwt.h, which the
 * tests compare the GPU's stream against.  Built by tests/dc_pack_ref.py; dark_b200/ never uses it.
 *
 * Per item k, in order: item_sym[k], item_rank[k], varint(item_pos[k] - item_pos[k-1] - 1) with item_pos[-1] = -1,
 * varint(item_dist[k]); varint = unsigned LEB128 (7 bits per byte, low group first, bit 7 set on all bytes but the last).
 */
#include <stdint.h>

static uint8_t *put_varint(uint8_t *o, uint32_t v) {
    while (v >= 0x80u) {
        *o++ = (uint8_t)(v | 0x80u);
        v >>= 7;
    }
    *o++ = (uint8_t)v;
    return o;
}

/* The stream of m items into out (room for 12 m bytes); returns its size. */
uint64_t dc_pack_ref(const uint32_t *pos, const uint32_t *dist, const uint8_t *sym, const uint8_t *rank, uint64_t m, uint8_t *out) {
    uint8_t *o = out;
    uint32_t prev = 0xFFFFFFFFu;
    for (uint64_t k = 0; k < m; ++k) {
        *o++ = sym[k];
        *o++ = rank[k];
        o = put_varint(o, pos[k] - prev - 1u);
        o = put_varint(o, dist[k]);
        prev = pos[k];
    }
    return (uint64_t)(o - out);
}

/* One varint of at most 5 bytes whose value fits 32 bits; 0 on a truncated or over-long one. */
static int get_varint(const uint8_t **p, const uint8_t *end, uint32_t *v) {
    uint64_t x = 0;
    for (int i = 0; i < 5; ++i) {
        if (*p == end) return 0;
        const uint8_t b = *(*p)++;
        x |= (uint64_t)(b & 0x7Fu) << (7 * i);
        if (!(b & 0x80u)) {
            if (x > 0xFFFFFFFFull) return 0;
            *v = (uint32_t)x;
            return 1;
        }
    }
    return 0;
}

/* The items of a stream of `bytes` bytes, at most max_items of them; returns their count, or UINT64_MAX for a stream that
 * is malformed (truncated item, over-long varint, run end past 2^32 - 2) or holds more than max_items items. */
uint64_t dc_unpack_ref(const uint8_t *in, uint64_t bytes, uint32_t *pos, uint32_t *dist, uint8_t *sym, uint8_t *rank,
                       uint64_t max_items) {
    const uint8_t *p = in, *end = in + bytes;
    int64_t at = -1;
    uint64_t k = 0;
    while (p != end) {
        if (k == max_items || end - p < 4) return UINT64_MAX;
        const uint8_t s = *p++, r = *p++;
        uint32_t len1, d;
        if (!get_varint(&p, end, &len1) || !get_varint(&p, end, &d)) return UINT64_MAX;
        at += 1 + (int64_t)len1;
        if (at > 0xFFFFFFFELL) return UINT64_MAX;
        pos[k] = (uint32_t)at;
        dist[k] = d;
        sym[k] = s;
        rank[k] = r;
        ++k;
    }
    return k;
}
