/* tests/c/mincost_walk.c -- TEST INFRASTRUCTURE (the checker of the min-cost parse), never shipped.
 *
 * The min-cost walk over a match table, the sibling of the oracle's greedy walk
 * (oracle/sqz_oracle.c: oracle_tokens_from_table) and of tests/c/lazy_walk.c, with
 * the same arguments.  The input is cut into segments of 16384 positions at
 * offsets that are multiples of 16384 (the last one may be shorter).  In each
 * segment [s, e), backwards from e - 1, with c(j) = 0 for j >= e:
 *   c(i) = min( 8 + c(i + 1),                                   the literal
 *               cost(k, dist[i]) + c(i + k) for min_len <= k <= len[i] )
 *   cost(k, d) = 6 + len_extra[bucket(k)] + 5 + pos_extra[bucket(d)]
 * ties to the longest step (a match beats a literal of equal cost).  The walk
 * then starts at `start` and follows the chosen steps across segment ends.
 * tests/mincost_oracle.py compiles and loads it.                             */
#include <stdint.h>
#include <stdlib.h>

enum { segment = 16384, literal_cost = 8, length_symbol_cost = 6, distance_symbol_cost = 5 };

/* the bucket tables of sqz_codec.c (reference squeeze.h:29-79) */
static const uint16_t len_base[29] = {
    3, 4, 5, 6, 7, 8, 9, 10, 11, 13, 15, 17, 19, 23, 27, 31, 35, 43, 51, 59,
    67, 83, 99, 115, 131, 163, 195, 227, 258 };
static const uint8_t len_extra[29] = {
    0, 0, 0, 0, 0, 0, 0, 0, 1, 1, 1, 1, 2, 2, 2, 2, 3, 3, 3, 3,
    4, 4, 4, 4, 5, 5, 5, 5, 0 };
static const uint16_t pos_base[30] = {
    1, 2, 3, 4, 5, 7, 9, 13, 17, 25, 33, 49, 65, 97, 129, 193, 257, 385, 513,
    769, 1025, 1537, 2049, 3073, 4097, 6145, 8193, 12289, 16385, 24577 };
static const uint8_t pos_extra[30] = {
    0, 0, 0, 0, 1, 1, 2, 2, 3, 3, 4, 4, 5, 5, 6, 6, 7, 7, 8, 8,
    9, 9, 10, 10, 11, 11, 12, 12, 13, 13 };

static uint32_t extra_bits(const uint16_t* base, const uint8_t* extra, int buckets, uint32_t v) {
    int b = 0;
    while (b + 1 < buckets && base[b + 1] <= v) { b++; }
    return extra[b];
}

static uint32_t match_cost(uint32_t k, uint32_t d) {
    return length_symbol_cost + extra_bits(len_base, len_extra, 29, k) +
           distance_symbol_cost + extra_bits(pos_base, pos_extra, 30, d);
}

/* returns the token count (tokens beyond cap are not stored), or UINT64_MAX without memory */
uint64_t mincost_tokens_from_table(const uint8_t* data, uint64_t bytes,
                                   const uint16_t* len, const uint16_t* dist,
                                   uint32_t min_len, uint64_t start,
                                   uint32_t* tokens, uint64_t cap,
                                   uint64_t* end_pos) {
    uint32_t* c = malloc((bytes + 1) * sizeof(uint32_t));
    uint16_t* step = malloc((bytes + 1) * sizeof(uint16_t));   /* 0: literal, else the match length */
    if (c == NULL || step == NULL) { free(c); free(step); return UINT64_MAX; }
    for (uint64_t s = 0; s < bytes; s += segment) {
        const uint64_t e = bytes - s < segment ? bytes : s + segment;
        for (uint64_t i = e; i-- > s;) {
            uint32_t best = literal_cost + (i + 1 < e ? c[i + 1] : 0);
            uint16_t k_best = 0;
            if (len[i] >= min_len) {
                for (uint32_t k = min_len; k <= len[i]; k++) {
                    const uint32_t v = match_cost(k, dist[i]) + (i + k < e ? c[i + k] : 0);
                    if (v <= best) { best = v; k_best = (uint16_t)k; }    /* k grows: ties go to the longer */
                }
            }
            c[i] = best;
            step[i] = k_best;
        }
    }
    uint64_t i = start, n = 0;
    while (i < bytes) {
        uint32_t t;
        if (step[i] != 0) { t = ((uint32_t)step[i] << 16) | dist[i]; i += step[i]; }
        else              { t = data[i];                              i += 1; }
        if (n < cap) { tokens[n] = t; }
        n++;
    }
    if (end_pos) { *end_pos = i; }
    free(c);
    free(step);
    return n;
}
