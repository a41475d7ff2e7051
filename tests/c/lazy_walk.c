/* tests/c/lazy_walk.c -- TEST INFRASTRUCTURE (the checker of the lazy parse), never shipped.
 *
 * The lazy walk over a match table, the sibling of the oracle's greedy walk
 * (oracle/sqz_oracle.c: oracle_tokens_from_table), with the same arguments.
 * With len[bytes] = 0: at parse position i, when len[i] >= min_len and
 * len[i+1] > len[i], emit the literal data[i] and go on at i+1 (where the
 * decision is taken again); otherwise the greedy step -- the match and len[i]
 * positions on when len[i] >= min_len, else the literal and one position on.
 * tests/lazy_oracle.py compiles and loads it.                                */
#include <stdint.h>

uint64_t lazy_tokens_from_table(const uint8_t* data, uint64_t bytes,
                                const uint16_t* len, const uint16_t* dist,
                                uint32_t min_len, uint64_t start,
                                uint32_t* tokens, uint64_t cap,
                                uint64_t* end_pos) {
    uint64_t i = start, n = 0;
    while (i < bytes) {
        const uint32_t next = i + 1 < bytes ? len[i + 1] : 0;
        uint32_t t;
        if (len[i] >= min_len && next <= len[i]) { t = ((uint32_t)len[i] << 16) | dist[i]; i += len[i]; }
        else                                     { t = data[i];                             i += 1; }
        if (n < cap) { tokens[n] = t; }
        n++;
    }
    if (end_pos) { *end_pos = i; }
    return n;
}
