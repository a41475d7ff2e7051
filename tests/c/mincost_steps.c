/* tests/c/mincost_steps.c -- TEST INFRASTRUCTURE (the checker of the min-cost table rewrite), never shipped.
 *
 * The table words the min-cost rewrite leaves (sqz_gpu_mincost_steps_device, the
 * kernel mincost_steps): the same backward pass over segments of 16384 positions
 * as tests/c/mincost_walk.c, whose tables and costs it takes, but instead of
 * walking the chosen steps it stores them -- (k << 16) | dist for a match of
 * k <= len, 0 for a literal.  Segments start at offset 0 of the arrays given, so
 * a caller who passes one shard's part of a table gets shard-local segments.
 * tests/mincost_steps.py compiles and loads it.                              */
#include "mincost_walk.c"

/* returns 0, or -1 without memory */
int mincost_steps_from_table(const uint16_t* len, const uint16_t* dist, uint64_t bytes, uint32_t min_len,
                             uint32_t* words) {
    uint32_t* c = malloc((bytes + 1) * sizeof(uint32_t));
    if (c == NULL) { return -1; }
    for (uint64_t s = 0; s < bytes; s += segment) {
        const uint64_t e = bytes - s < segment ? bytes : s + segment;
        for (uint64_t i = e; i-- > s;) {
            uint32_t best = literal_cost + (i + 1 < e ? c[i + 1] : 0);
            uint32_t k_best = 0;
            if (len[i] >= min_len) {
                for (uint32_t k = min_len; k <= len[i]; k++) {
                    const uint32_t v = match_cost(k, dist[i]) + (i + k < e ? c[i + k] : 0);
                    if (v <= best) { best = v; k_best = k; }           /* k grows: ties go to the longer */
                }
            }
            c[i] = best;
            words[i] = k_best != 0 ? (k_best << 16) | dist[i] : 0;
        }
    }
    free(c);
    return 0;
}
