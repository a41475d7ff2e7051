/* tests/c/lz_execute.c -- TEST INFRASTRUCTURE (the checker of the GPU copy phase), never shipped.
 *
 * The reference decoder's copy loop (squeeze.h:533-539) over a whole token stream: a literal
 * stores its byte, a match copies len bytes from dist back one byte at a time, so that a copy
 * that overlaps its own output repeats it.  No rule set is assumed: len 1..65535, dist 1..65535.
 *
 * Returns 0 when the tokens describe exactly `bytes` bytes (all of out[0, bytes) written);
 * 1 + k when token k is the first bad one: a literal word above 0xFF, dist 0, a match that reaches
 * before byte 0, or a token that ends past `bytes` (out holds what the tokens before it wrote);
 * LZ_SHORT when every token is good but together they describe fewer than `bytes` bytes.
 * tests/lz_reference.py compiles and loads it.                                                  */
#include <stdint.h>

#define LZ_SHORT UINT64_MAX

uint64_t lz_execute(const uint32_t* tokens, uint64_t n_tokens, uint8_t* out, uint64_t bytes) {
    uint64_t i = 0;
    for (uint64_t k = 0; k < n_tokens; k++) {
        const uint32_t t = tokens[k], len = t >> 16, dist = t & 0xFFFFu;
        if (len == 0) {
            if (t > 0xFFu || i >= bytes) { return 1 + k; }
            out[i++] = (uint8_t)t;
        } else {
            if (dist == 0 || dist > i || len > bytes - i) { return 1 + k; }
            for (uint32_t b = 0; b < len; b++, i++) { out[i] = out[i - dist]; }
        }
    }
    return i == bytes ? 0 : LZ_SHORT;
}
