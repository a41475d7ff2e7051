/* sqz_codec.c -- host half of sqz-b200: header, bit I/O, the adaptive-Huffman
 * token coder and the decompressor.  Written from the behavioural description
 * in SURVEY.md Appendix A; every emitted bit has to equal what the reference
 * (/root/reference/attic/map_experiment/{squeeze,huffman,bitstream}.h) emits,
 * which tests/test_codec.py checks against oracle/_ref and tests/golden.
 *
 * The LZ77 search that feeds sqz_compress() lives on the GPU (sqz_gpu.cu).
 * This file never searches: no CPU fallback exists for that step.
 */
#include "sqz.h"
#include "sqz_gpu.h"

#include <errno.h>
#include <pthread.h>
#include <sched.h>
#include <stdatomic.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <time.h>
#include <unistd.h>

/* ---- deflate-style bucket tables (RFC 1951 3.2.5; reference squeeze.h:29-79) */
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

enum { len_symbol0 = 257 };

static double now_seconds(void) {
    struct timespec ts;
    clock_gettime(CLOCK_MONOTONIC, &ts);
    return (double)ts.tv_sec + 1e-9 * (double)ts.tv_nsec;
}

/* ======================================================================== *
 *  bit I/O  (reference bitstream.h:28-114)                                  *
 *  Bits enter b64 from the right, so the first bit written ends up as the   *
 *  MSB of a 64-bit word; values are fed least-significant bit first.        *
 * ======================================================================== */

static inline uint64_t reverse64(uint64_t v) {
    v = ((v >> 1)  & 0x5555555555555555ull) | ((v & 0x5555555555555555ull) << 1);
    v = ((v >> 2)  & 0x3333333333333333ull) | ((v & 0x3333333333333333ull) << 2);
    v = ((v >> 4)  & 0x0F0F0F0F0F0F0F0Full) | ((v & 0x0F0F0F0F0F0F0F0Full) << 4);
    return __builtin_bswap64(v);
}

static void word_out(struct sqz_bitstream* bs) {
    if (bs->data != NULL && bs->capacity > 0) {
        for (int k = 7; k >= 0 && bs->error == 0; k--) {      /* big-endian */
            if (bs->bytes == bs->capacity) { bs->error = E2BIG; }
            else { bs->data[bs->bytes++] = (uint8_t)(bs->b64 >> (k * 8)); }
        }
    } else if (bs->output != NULL) {
        bs->error = bs->output(bs);                           /* host order */
        if (bs->error == 0) { bs->bytes += 8; }
    } else {
        bs->error = EINVAL;
    }
    bs->bits = 0;
    bs->b64 = 0;
}

/* append `count` bits that are already in emission order (first bit = MSB of the field) */
static inline void put_code(struct sqz_bitstream* bs, uint64_t seq, int count) {
    if (bs->error != 0 || count <= 0) { return; }
    int room = 64 - bs->bits;
    if (count < room) {
        bs->b64 = (bs->b64 << count) | seq;
        bs->bits += count;
        return;
    }
    int rest = count - room;
    bs->b64 = (room == 64 ? 0 : bs->b64 << room) | (seq >> rest);
    word_out(bs);
    if (rest > 0 && bs->error == 0) {
        bs->b64 = seq & (((uint64_t)1 << rest) - 1);
        bs->bits = rest;
    }
}

/* append the low `count` bits of `value`, least significant first */
static inline void put_bits(struct sqz_bitstream* bs, uint64_t value, int count) {
    if (bs->error != 0 || count <= 0) { return; }
    /* in emission order the value is bit-reversed: its bit 0 goes out first */
    put_code(bs, reverse64(value) >> (64 - count), count);
}

static inline void pad_to_word(struct sqz_bitstream* bs) {     /* bitstream.h:112-114 */
    if (bs->error == 0 && bs->bits > 0) { put_bits(bs, 0, 64 - bs->bits); }
}

static void word_in(struct sqz_bitstream* bs) {
    bs->b64 = 0;
    if (bs->data != NULL && bs->bytes > 0) {
        for (int k = 7; k >= 0 && bs->error == 0; k--) {
            if (bs->read == bs->bytes) { bs->error = E2BIG; }
            else { bs->b64 |= (uint64_t)bs->data[bs->read++] << (k * 8); }
        }
    } else if (bs->input != NULL) {
        bs->error = bs->input(bs);
        if (bs->error == 0) { bs->read += 8; }
    } else {
        bs->error = EINVAL;
    }
    bs->bits = 64;
}

static inline int get_bit(struct sqz_bitstream* bs) {
    if (bs->error != 0) { return 0; }
    if (bs->bits == 0) { word_in(bs); if (bs->error != 0) { return 0; } }
    int bit = (int)(bs->b64 >> 63);
    bs->b64 <<= 1;
    bs->bits--;
    return bit;
}

static inline uint64_t get_bits(struct sqz_bitstream* bs, int count) {
    uint64_t v = 0;
    if (bs->error == 0 && bs->bits >= count && count > 0 && count < 64) {
        /* whole field is in the register: top `count` bits, first bit = LSB */
        uint64_t top = bs->b64 >> (64 - count);
        bs->b64 <<= count;
        bs->bits -= count;
        return reverse64(top) >> (64 - count);
    }
    for (int k = 0; k < count && bs->error == 0; k++) {
        v |= (uint64_t)get_bit(bs) << k;
    }
    return v;
}

/* ======================================================================== *
 *  adaptive Huffman tree  (reference huffman.h:36-269, SURVEY.md App. A)    *
 *  Leaves are 0..n-1 (index == symbol); the root is 2n-2; further internal  *
 *  nodes are allocated downward from 2n-3.                                  *
 *                                                                           *
 *  Stored as a structure of arrays (16-bit links) so that the per-symbol    *
 *  walk stays in L1.  Two kinds of walk exist:                              *
 *   - the exact one (weight_changed), the reference's algorithm step by     *
 *     step, which may reorder the tree;                                     *
 *   - the quick one (quick_count), which only adds 1 to every weight on the *
 *     path and is taken when no reordering can happen.  Whether one can is  *
 *     known per node: a walk through node i does something other than add 1 *
 *     only if i, after its increment, outweighs one fixed other node --     *
 *     its right sibling when i is a left child (the two would trade places, *
 *     huffman.h:64-86), its parent's sibling when i is a right child (i     *
 *     would be promoted, huffman.h:98-128).  That comparator is a function  *
 *     of the tree's shape, which changes about once per 2700 symbols on the *
 *     bench corpus.  Every leaf therefore keeps a plan: the (node,          *
 *     comparator) pairs from itself to the root, one cache line, so the     *
 *     quick walk is a loop over independent loads instead of a pointer      *
 *     chase.  A plan is dropped when the shape above or beside its leaf     *
 *     changes (relabel, forget_plans) and rebuilt on the leaf's next use.   *
 * ======================================================================== */

enum { none = -1, no_node = 0xFFFF,
       lit_lut_bits = 10, pos_lut_bits = 6,     /* sizes of sqz.h's lit_lut / pos_lut */
       lut_node_bits = 10 };                    /* a table entry: node (< 1023) | bits to consume << 10 */

static void note_change(struct sqz_tree* t, int32_t leaf);
struct code_tables;
struct duo;
struct segment;
/* who is told when a leaf's code changes: the one-thread coder's tables, the two-thread coder's ring
 * of changes, or the segment the model of the several-thread coder is working on.  `now` is the
 * stamp a change gets: index (within the stream or chunk) of the token being modelled, + 1 = the
 * first token the new code applies to; `k_now` that token's index within the chunk.              */
struct watch { struct code_tables* tables; struct duo* d; struct segment* seg; uint64_t now, k_now; int error; };

static inline int32_t tree_root(const struct sqz_tree* t) { return 2 * t->n - 2; }
static inline uint32_t always_node(const struct sqz_tree* t) { return 2 * (uint32_t)t->n - 1; } /* weight 0 */
static inline uint32_t never_node(const struct sqz_tree* t) { return 2 * (uint32_t)t->n; }       /* weight 2^63-1 */
static inline uint32_t spare_node(const struct sqz_tree* t, int k) { return 2 * (uint32_t)t->n + 1 + ((uint32_t)k & 7); }

#define SQZ_BIND_TREE(t, store, leaves) do {                                      \
    (t)->freq = (store).freq; (t)->path = (store).path; (t)->code = (store).code; \
    (t)->up = (store).up; (t)->lo = (store).lo; (t)->hi = (store).hi;             \
    (t)->plan = &(store).plan[0][0]; (t)->steps = (store).steps;                  \
    (t)->bits = (store).bits; (t)->n = (leaves); (t)->lut = NULL; (t)->watcher = NULL; \
    (t)->lut_bits = (leaves) == sqz_lit_symbols ? lit_lut_bits : pos_lut_bits; } while (0)

static void tree_init(struct sqz_tree* t) {
    const int32_t nodes = 2 * t->n - 1;
    t->next = 2 * t->n - 2;
    t->depth = 0;
    t->complete = 0;
    t->lazy = t->lazy_start = t->eager = 0;
    for (int32_t k = 0; k < nodes; k++) {
        t->freq[k] = 0; t->path[k] = 0; t->bits[k] = 0;
        t->up[k] = none; t->lo[k] = none; t->hi[k] = none;
    }
    for (int32_t k = 0; k < t->n; k++) { t->code[k] = 0; t->steps[k] = 0; }
    t->freq[always_node(t)] = 0;
    t->freq[never_node(t)] = (uint64_t)INT64_MAX;
    for (int k = 0; k < 8; k++) { t->freq[spare_node(t, k)] = 0; }
}

/* Re-derive code length and code of everything below `top` from top's own.
 * A relabel that starts at the root restarts the depth high-water mark
 * (huffman.h:41-62).  Iterative: the order of visits does not matter.       */
#ifdef SQZ_SELFCHECK
static _Thread_local uint64_t selfcheck_relabels;    /* how often this thread changed a tree's shape */
uint64_t sqz_selfcheck_spans, sqz_selfcheck_span_tokens;   /* spans replayed one by one, for the tests to see */
#endif

static void relabel(struct sqz_tree* t, int32_t top) {
    int16_t stack[2 * sqz_lit_symbols];
#ifdef SQZ_SELFCHECK
    selfcheck_relabels++;
#endif
    int sp = 0;
    int32_t depth = (top == tree_root(t)) ? 0 : t->depth;
    stack[sp++] = (int16_t)top;
    while (sp > 0) {
        const int32_t i = stack[--sp];
        const int32_t bits = t->bits[i];
        const uint64_t path = t->path[i];
        if (bits > depth) { depth = bits; }
        const int32_t lo = t->lo[i], hi = t->hi[i];
        if (lo >= 0) { t->bits[lo] = (uint8_t)(bits + 1); t->path[lo] = path; stack[sp++] = (int16_t)lo; }
        if (hi >= 0) { t->bits[hi] = (uint8_t)(bits + 1); t->path[hi] = path | ((uint64_t)1 << bits); stack[sp++] = (int16_t)hi; }
        if (i < t->n) {
            if (bits > 0) {
                t->code[i] = reverse64(path) >> (64 - bits);
                if (t->watcher != NULL) { note_change(t, i); }      /* the emitter's tables follow */
            }
            t->steps[i] = 0;            /* the shape above this leaf changed: its plan is void */
        }
        /* decoder only: every lut_bits-bit look-ahead that starts with this node's code leads here */
        if (t->lut != NULL && bits > 0 && bits <= t->lut_bits && (i < t->n || bits == t->lut_bits)) {
            const int32_t spread = t->lut_bits - bits;
            const uint64_t first = (reverse64(path) >> (64 - bits)) << spread;
            const uint16_t entry = (uint16_t)(i | (bits << lut_node_bits));   /* the node and the bits its code takes */
            for (uint64_t k = 0; k < ((uint64_t)1 << spread); k++) { t->lut[first + k] = entry; }
        }
    }
    t->depth = depth;
}

/* drop the plans of every leaf below `top` */
static void forget_plans(struct sqz_tree* t, int32_t top) {
    int16_t stack[2 * sqz_lit_symbols];
    int sp = 0;
    stack[sp++] = (int16_t)top;
    while (sp > 0) {
        const int32_t i = stack[--sp];
        if (i < t->n) { t->steps[i] = 0; continue; }
        if (t->lo[i] >= 0) { stack[sp++] = t->lo[i]; }
        if (t->hi[i] >= 0) { stack[sp++] = t->hi[i]; }
    }
}

static inline uint64_t weight_or_zero(const struct sqz_tree* t, int32_t i) {
    return i >= 0 ? t->freq[i] : 0;
}

static inline void sum_children(struct sqz_tree* t, int32_t i) {
    t->freq[i] = weight_or_zero(t, t->lo[i]) + weight_or_zero(t, t->hi[i]);
}

/* Keep the lighter child on the left.  When the children trade places the
 * caller continues with the node that now sits where `i` used to be, i.e.
 * i's sibling (huffman.h:64-86).                                            */
static int32_t order_siblings(struct sqz_tree* t, int32_t i) {
    if (i == tree_root(t)) { return i; }
    const int32_t p = t->up[i];
    const int32_t lo = t->lo[p], hi = t->hi[p];
    if (lo >= 0 && hi >= 0 && t->freq[lo] > t->freq[hi]) {
        t->lo[p] = (int16_t)hi;
        t->hi[p] = (int16_t)lo;
        relabel(t, p);
        return i == lo ? hi : lo;
    }
    return i;
}

static void weight_changed(struct sqz_tree* t, int32_t i);

/* `x` is the right child of p; if it outweighs p's sibling u the two trade
 * places: x moves up next to p, u moves down under p (huffman.h:98-128).    */
static void promote(struct sqz_tree* t, int32_t x) {
    const int32_t p = t->up[x];
    const int32_t g = t->up[p];
    const int p_left = t->lo[g] == p;
    const int32_t u = p_left ? t->hi[g] : t->lo[g];
    if (u >= 0 && t->freq[x] > t->freq[u]) {
        t->up[x] = (int16_t)g;
        if (p_left) { t->hi[g] = (int16_t)x; } else { t->lo[g] = (int16_t)x; }
        t->hi[p] = (int16_t)u;
        t->up[u] = (int16_t)p;
        sum_children(t, p);
        sum_children(t, g);
        (void)order_siblings(t, x);
        (void)order_siblings(t, u);
        (void)order_siblings(t, p);
        relabel(t, g);
        weight_changed(t, g);
    }
}

/* The exact walk.  Propagate a weight change from `i` to the root, re-ordering
 * siblings on the way up and, on the way back down, promoting right children
 * that outgrew their uncle (huffman.h:130-147).  The reference recurses; this
 * is the same sequence of steps with the recursion unrolled: first every level
 * from the leaf to the root refreshes its parent's weight and orders the two
 * children (continuing, after a swap, with the node that took the old slot),
 * then the levels are revisited from the root down for the promotion test,
 * each with the (node, parent) pair it captured on the way up.              */
static void weight_changed(struct sqz_tree* t, int32_t i) {
    int16_t node_at[2 * sqz_lit_symbols], parent_at[2 * sqz_lit_symbols];
    int levels = 0;
    for (;;) {
        const int32_t p = t->up[i];
        if (p < 0) {                    /* the root: refresh its own weight, nothing to order */
            sum_children(t, i);
            break;
        }
        const int32_t lo = t->lo[p], hi = t->hi[p];
        const uint64_t wl = weight_or_zero(t, lo), wh = weight_or_zero(t, hi);
        t->freq[p] = wl + wh;
        if (lo >= 0 && hi >= 0 && wl > wh) { /* heavier child goes right */
            t->lo[p] = (int16_t)hi;
            t->hi[p] = (int16_t)lo;
            relabel(t, p);
            i = (i == lo) ? hi : lo;
        }
        node_at[levels] = (int16_t)i;
        parent_at[levels] = (int16_t)p;
        levels++;
        i = p;
    }
    while (levels > 0) {
        levels--;
        const int32_t p = parent_at[levels];
        if (t->up[p] >= 0 && t->hi[p] == node_at[levels]) { promote(t, node_at[levels]); }
    }
}

/* The node whose weight `i` may not exceed without the tree being reordered.
 * A parent that is not in the state the quick walk relies on (children out of
 * order, a weight that is not the sum of its children) yields the weight-0
 * comparator, which sends every walk through `i` to the exact path.          */
static uint32_t comparator(const struct sqz_tree* t, int32_t i) {
    const int32_t p = t->up[i];
    if (p < 0) { return never_node(t); }
    const int32_t lo = t->lo[p], hi = t->hi[p];
    /* (the root's own weight is exempt: nothing compares against it, quick walks leave it alone
     * and every exact walk recomputes it from its children before anything reads it) */
    if ((t->up[p] >= 0 && t->freq[p] != weight_or_zero(t, lo) + weight_or_zero(t, hi)) ||
        (lo >= 0 && hi >= 0 && t->freq[lo] > t->freq[hi])) {
        return always_node(t);
    }
    if (i == lo) { return hi >= 0 ? (uint32_t)hi : never_node(t); }
    const int32_t g = t->up[p];
    if (g < 0) { return never_node(t); }
    const int32_t u = t->lo[g] == p ? t->hi[g] : t->lo[g];
    return u >= 0 ? (uint32_t)u : always_node(t);
}

#ifndef SQZ_TOP_LEVELS
#define SQZ_TOP_LEVELS 3
#endif
enum { plan_levels = 16, plan_too_deep = 0xFF,
       lit_plan = 9, pos_plan = 6,     /* covers 98 % / 97 % of the symbols of the bench corpus */
       top_levels = SQZ_TOP_LEVELS,                 /* internal nodes this close to the root are kept up to date lazily */
       lazy_least = 32,                /* a lazy stretch shorter than this is not worth its bookkeeping */
       eager_run = 32 };               /* symbols coded with full walks before the top is looked at again */

/* plan of leaf `s`: one cache line, plan[0..15] the nodes from the leaf up to
 * the root's child, plan[16..31] their comparators, padded with spare nodes
 * nobody reads to the tree's usual plan length (so that the common walk is
 * straight-line code), or to 16 when deeper.  The walk compares weights as
 * signed numbers; a path that already carries 2^61 gets no plan.             */
static int plan_for(const struct sqz_tree* t, int32_t s, uint16_t* plan) {
    const int usual = t->n == sqz_lit_symbols ? lit_plan : pos_plan;
    int32_t chain[plan_levels] = { s };              /* chain[0] = the leaf ... chain[d-1] = the root's child */
    int d = 0;
    for (int32_t i = s; t->up[i] >= 0; i = t->up[i]) {
        if (d == plan_levels || t->freq[i] >> 61 != 0) { return plan_too_deep; }
        chain[d++] = i;
    }
    /* order: [0] the leaf, [1..3] its ancestors at depth 1, 2, 3 -- the entries the lazy walk
     * leaves out --, [4..] the ancestors at depth 4 and below; spare nodes where there is none */
    int k = 0, pad = 0;
#define SQZ_PLAN_PUT(node_) do { plan[k] = (uint16_t)(node_);                                   \
                                 plan[plan_levels + k] = (uint16_t)comparator(t, (int32_t)(node_)); k++; } while (0)
#define SQZ_PLAN_PAD() do { plan[k] = (uint16_t)spare_node(t, pad++);                            \
                            plan[plan_levels + k] = (uint16_t)never_node(t); k++; } while (0)
    SQZ_PLAN_PUT(chain[0]);
    for (int depth = 1; depth <= top_levels; depth++) {
        if (d - depth >= 1) { SQZ_PLAN_PUT(chain[d - depth]); } else { SQZ_PLAN_PAD(); }
    }
    for (int depth = top_levels + 1; depth <= d - 1; depth++) { SQZ_PLAN_PUT(chain[d - depth]); }
    const int padded = k <= usual ? usual : plan_levels;
    while (k < padded) { SQZ_PLAN_PAD(); }
#undef SQZ_PLAN_PUT
#undef SQZ_PLAN_PAD
    return padded;
}

static void make_plan(struct sqz_tree* t, int32_t s) {
    t->steps[s] = (uint8_t)plan_for(t, s, t->plan + (size_t)s * 2 * plan_levels);
}

static void settle(struct sqz_tree* t);

#ifdef SQZ_SELFCHECK
/* Test builds only (tests/test_codec.py): after every symbol, every plan that
 * is held valid must equal a freshly made one, and the state the quick walk
 * relies on must hold everywhere: weights are the sums of their children,
 * the lighter child is on the left.                                          */
#include <stdio.h>
#include <stdlib.h>
static void selfcheck(struct sqz_tree* t) {
    const int32_t root = tree_root(t);
    settle(t);                          /* the checks below are about exact weights */
    for (int32_t s = 0; s < t->n; s++) {
        if (t->up[s] < 0 || t->steps[s] == 0) { continue; }
        uint16_t fresh[2 * plan_levels];
        const uint16_t* held = t->plan + (size_t)s * 2 * plan_levels;
        const int steps = plan_for(t, s, fresh);
        if (steps != t->steps[s] ||
            (steps != plan_too_deep && (memcmp(fresh, held, 2 * (size_t)steps) != 0 ||
                                        memcmp(fresh + plan_levels, held + plan_levels, 2 * (size_t)steps) != 0))) {
            fprintf(stderr, "sqz selfcheck: stale plan of leaf %d\n", s);
            abort();
        }
    }
    for (uint32_t look = 0; t->lut != NULL && look < (1u << t->lut_bits); look++) {
        int32_t i = root;
        for (int b = t->lut_bits - 1; b >= 0 && i >= t->n; b--) { i = (look >> b) & 1 ? t->hi[i] : t->lo[i]; }
        if (t->lut[look] != (i >= 0 ? (uint16_t)(i | (t->bits[i] << lut_node_bits)) : (uint16_t)no_node)) {
            fprintf(stderr, "sqz selfcheck: stale decode table entry %u\n", look);
            abort();
        }
    }
    for (int32_t p = t->next; p < root; p++) {
        const int32_t lo = t->lo[p], hi = t->hi[p];
        if (t->freq[p] != weight_or_zero(t, lo) + weight_or_zero(t, hi) || lo < 0 || hi < 0 ||
            t->freq[lo] > t->freq[hi]) {
            fprintf(stderr, "sqz selfcheck: node %d is not in the state the quick walk relies on\n", p);
            abort();
        }
    }
}
#define SQZ_CHECK(t) selfcheck(t)
#else
#define SQZ_CHECK(t) ((void)0)
#endif

/* The quick walk: add 1 to every weight from leaf `s` to the root's child,
 * provided no node on the way comes to outweigh its comparator.  Returns 0
 * with all weights as they were when one would: the exact walk has to decide
 * then.  `usual` is the tree's usual plan length (a constant at every call).  */
#define SQZ_PLAN_STEP(k_) do {                                                   \
        const int64_t w_ = (int64_t)freq[plan[k_]] + 1;                          \
        fires |= (int64_t)freq[plan[plan_levels + (k_)]] - w_;   /* negative: outweighs */ \
        freq[plan[k_]] = (uint64_t)w_; } while (0)

/* The weights of the internal nodes at depth 1..top_levels, from their children.  Only when
 * lazy walks went by since they were last exact: then every one of them was in order and the
 * sum of its children (lazy_budget checks), so the sums are what full walks would have left. */
static void settle(struct sqz_tree* t) {
    if (t->lazy == t->lazy_start) { return; }
    int32_t level[top_levels][1 << top_levels];
    int count[top_levels];
    int32_t above[1] = { tree_root(t) };
    const int32_t* from = above;
    int from_count = 1;
    for (int l = 0; l < top_levels; l++) {
        count[l] = 0;
        for (int k = 0; k < from_count; k++) {
            const int32_t lo = t->lo[from[k]], hi = t->hi[from[k]];
            if (lo >= t->n) { level[l][count[l]++] = lo; }
            if (hi >= t->n) { level[l][count[l]++] = hi; }
        }
        from = level[l];
        from_count = count[l];
    }
    for (int l = top_levels - 1; l >= 0; l--) {
        for (int k = 0; k < count[l]; k++) { sum_children(t, level[l][k]); }
    }
    t->lazy_start = t->lazy;
}

/* How many symbols can be coded without looking at the internal nodes at depth 1..top_levels:
 * each symbol moves each of their weights by at most one, so none of them can outweigh its
 * comparator before the smallest margin among them is used up.  0 when one of them is not in
 * the state the quick walk relies on.  Call with the top exact (settle).                     */
static int32_t lazy_budget(const struct sqz_tree* t) {
    int64_t least = 1 << 20;
    int32_t frontier[1 << top_levels], next[1 << top_levels];
    int n_frontier = 1;
    frontier[0] = tree_root(t);
    for (int l = 0; l < top_levels; l++) {
        int n_next = 0;
        for (int k = 0; k < n_frontier; k++) {
            const int32_t kids[2] = { t->lo[frontier[k]], t->hi[frontier[k]] };
            for (int c = 0; c < 2; c++) {
                const int32_t i = kids[c];
                if (i < t->n) { continue; }              /* a leaf (or no child): leaves are always walked */
                const int32_t lo = t->lo[i], hi = t->hi[i];
                if (t->freq[i] != weight_or_zero(t, lo) + weight_or_zero(t, hi) || lo < 0 || hi < 0 ||
                    t->freq[lo] > t->freq[hi]) {
                    return 0;
                }
                const uint32_t cmp = comparator(t, i);
                if (cmp == always_node(t)) { return 0; }
                if (cmp != never_node(t)) {
                    const int64_t margin = (int64_t)t->freq[cmp] - (int64_t)t->freq[i];
                    if (margin < least) { least = margin; }
                }
                next[n_next++] = i;
            }
        }
        memcpy(frontier, next, sizeof(int32_t) * (size_t)n_next);
        n_frontier = n_next;
    }
    return least < lazy_least ? 0 : (int32_t)least;
}

static inline __attribute__((always_inline))
int quick_count(struct sqz_tree* t, int32_t s, const int usual, const int lazily) {
    uint64_t* const freq = t->freq;
    if (t->steps[s] == 0) { settle(t); make_plan(t, s); }              /* plans are made from exact weights */
    const int steps = t->steps[s];
    const uint16_t* const plan = t->plan + (size_t)s * 2 * plan_levels;
    int64_t fires = 0;
    if (steps == usual) {
        SQZ_PLAN_STEP(0);
#pragma GCC unroll 16
        for (int k = lazily ? top_levels + 1 : 1; k < usual; k++) { SQZ_PLAN_STEP(k); }   /* usual is a constant here */
    } else if (steps == plan_levels) {
        SQZ_PLAN_STEP(0);
#pragma GCC unroll 16
        for (int k = lazily ? top_levels + 1 : 1; k < plan_levels; k++) { SQZ_PLAN_STEP(k); }
    } else {
        return 0;                                                       /* deeper than a plan */
    }
    if (fires >= 0) { return 1; }
    freq[plan[0]]--;
    for (int k = lazily ? top_levels + 1 : 1; k < steps; k++) { freq[plan[k]]--; }
    return 0;
}

/* First occurrence of symbol `s` (huffman.h:149-216): walk from the root,
 * always to the left, to the first free child slot (right slot preferred) or
 * to a leaf, which is then split by a fresh internal node.                  */
static int tree_insert(struct sqz_tree* t, int32_t s) {
    int ok = 1;
    int32_t at = tree_root(t);
    settle(t);                          /* what follows reads and reorders exact weights */
    t->lazy = t->lazy_start = t->eager = 0;
    t->freq[s] = 1;
    while (at >= t->n) {
        if (t->hi[at] < 0)      { t->hi[at] = (int16_t)s; t->up[s] = (int16_t)at; break; }
        else if (t->lo[at] < 0) { t->lo[at] = (int16_t)s; t->up[s] = (int16_t)at; break; }
        else                    { at = t->lo[at]; }
    }
    if (at >= t->n) {
        t->freq[at]++;
        s = order_siblings(t, s);
    } else if (t->next == t->n) {
        ok = 0;
        t->complete = 1;
    } else {
        const int32_t leaf = at;
        const int32_t x = --t->next;
        t->freq[x] = t->freq[leaf];
        t->path[x] = t->path[leaf];
        t->bits[x] = t->bits[leaf];
        t->up[x]   = t->up[leaf];
        t->lo[x]   = (int16_t)leaf;
        t->hi[x]   = (int16_t)s;
        if (t->up[x] >= 0) {
            const int32_t above = t->up[x];
            if (t->lo[above] == leaf) { t->lo[above] = (int16_t)x; } else { t->hi[above] = (int16_t)x; }
        }
        t->up[leaf] = (int16_t)x;
        t->bits[leaf] = (uint8_t)(t->bits[x] + 1);   /* left edge: same code, one longer */
        t->up[s] = (int16_t)x;
        t->bits[s] = (uint8_t)(t->bits[x] + 1);
        t->path[s] = t->path[x] | ((uint64_t)1 << t->bits[x]);
        sum_children(t, x);
        at = x;
        /* x took the leaf's place: it is now the comparator of the leaf's old neighbours */
        forget_plans(t, t->up[x] >= 0 ? t->up[x] : x);
    }
    weight_changed(t, s);
    relabel(t, at);
    return ok;
}

static inline __attribute__((always_inline))
void tree_count_as(struct sqz_tree* t, int32_t s, const int usual) {   /* huffman.h:218-235 */
    /* the common case first: a lazy stretch is on (which implies the tree is neither complete nor
     * 63 deep: both only change where `lazy` is reset) and the leaf has a plan of the usual length */
    if (t->lazy > 0 && t->steps[s] == usual) {
        uint64_t* const freq = t->freq;
        const uint16_t* const plan = t->plan + (size_t)s * 2 * plan_levels;
        int64_t fires = 0;
        SQZ_PLAN_STEP(0);
#pragma GCC unroll 16
        for (int k = top_levels + 1; k < usual; k++) { SQZ_PLAN_STEP(k); }
        if (fires >= 0) { t->lazy--; return; }
        freq[plan[0]]--;
        for (int k = top_levels + 1; k < usual; k++) { freq[plan[k]]--; }
    }
    if (t->up[s] < 0) {
        (void)tree_insert(t, s);
    } else if (!t->complete && t->depth < 63 && t->freq[s] < UINT64_MAX - 1) {
        if (t->lazy == 0 && t->eager == 0) {            /* decide how the next stretch is walked */
            settle(t);
            t->lazy = t->lazy_start = lazy_budget(t);
            if (t->lazy == 0) { t->eager = eager_run; }
        }
        if (t->lazy > 0) {
            if (quick_count(t, s, usual, 1)) { t->lazy--; return; }
            /* something may outweigh its comparator -- possibly only because the comparator's weight
             * is behind: make the top exact and let the full walk decide */
            settle(t);
            t->lazy = t->lazy_start = 0;
            t->eager = eager_run;
        }
        if (quick_count(t, s, usual, 0)) { t->eager--; return; }
        t->eager = 0;
        t->freq[s]++;
        weight_changed(t, s);
    } else {
        t->complete = 1;
    }
}

/* What tree_count_as does first thing when no stretch is on, done ahead of the tree's next symbol:
 * the decision only depends on the tree as it stands, and that does not change until then.       */
static void renew_stretch(struct sqz_tree* t) {
    if (!t->complete && t->depth < 63 && t->lazy == 0 && t->eager == 0) {
        settle(t);
        t->lazy = t->lazy_start = lazy_budget(t);
        if (t->lazy == 0) { t->eager = eager_run; }
    }
}

static void tree_count(struct sqz_tree* t, int32_t s) {
    if (t->n == sqz_lit_symbols) { tree_count_as(t, s, lit_plan); } else { tree_count_as(t, s, pos_plan); }
    SQZ_CHECK(t);
}

/* ======================================================================== *
 *  counting a block of symbols at once                                      *
 *  A reordering happens about once per 3600 symbols on the bench corpus; in *
 *  between the model only adds 1 along a path per symbol, and additions     *
 *  commute.  So a block of symbols (4096 tokens) is tallied per leaf and    *
 *  every distinct leaf walks its plan once, adding its count -- provided no *
 *  walk of the block, taken one by one, could have reordered anything.      *
 *  First test, for every node walked: all weights only grow during the      *
 *  block, so a node whose weight at the END of the block does not exceed    *
 *  its comparator's weight at the START of the block exceeded it at no      *
 *  moment in between, whatever the order of the symbols.  The few nodes     *
 *  that fail it (the culprits; two near-equal siblings as a rule) get the   *
 *  exact answer: the words are walked in order with just those nodes' and   *
 *  their comparators' weights, counting who lies below which -- and only    *
 *  the rows of the block's tallies in which a culprit could catch up at     *
 *  all.  No word at which one does: the block stands.  Else everything      *
 *  before that word is one span (it passes by construction), the word goes  *
 *  through the one-by-one path -- it may reorder the tree --, and the rest  *
 *  of the block goes on from its tallies.  Exact, not approximate: what is  *
 *  not proven harmless takes the reference's walk.                          *
 * ======================================================================== */

#ifndef SQZ_PART_TOKENS
#define SQZ_PART_TOKENS 256
#endif
enum { part_tokens = SQZ_PART_TOKENS,              /* tokens per part: the unit a block is tallied in and falls back to */
       parts_most = 16,
       block_most = part_tokens * parts_most,       /* tokens per block when all goes well */
       mini_tokens = 32,               /* a part that does not pass is tallied again in four minis */
       block_least = 32 };             /* below this a block is not worth its snapshot */

/* A block is tallied once, part by part; the counts of a span of parts are the sums of the parts'.
 * When the whole block does not pass, its quarters are tried, then their parts, each from the
 * tallies already made; only a part that does not pass is walked one by one.                    */
struct tally {
    /* rows of 16-bit counters, 8-byte aligned: a span's counts are added four symbols at a time (no
     * count reaches 2^16, so nothing carries from one into the next) */
    _Alignas(8) uint16_t lit_part[parts_most][sqz_lit_symbols];
    _Alignas(8) uint16_t pos_part[parts_most][sqz_pos_symbols + 8];   /* + slots a literal's "no distance" goes to, in turn */
    _Alignas(8) uint16_t lit_count[sqz_lit_symbols];           /* the span being tried */
    _Alignas(8) uint16_t pos_count[sqz_pos_symbols + 8];
    uint16_t lit_seen[sqz_lit_symbols];            /* its distinct symbols */
    uint16_t pos_seen[sqz_pos_symbols];
    uint8_t lit_suspect[sqz_lit_symbols], pos_suspect[sqz_pos_symbols];   /* span_apply's verdict per seen leaf */
    uint8_t lit_below[sqz_lit_symbols], lit_beside[sqz_lit_symbols];      /* culprit_leaves */
    uint8_t pos_below[sqz_pos_symbols], pos_beside[sqz_pos_symbols];
    uint64_t lit_start[2 * sqz_lit_symbols + 1];   /* weights as they were when the span began, and */
    uint64_t pos_start[2 * sqz_pos_symbols + 1];   /* the comparators "always" (0) and "never" (2^63-1) */
    /* Where reorderings come every few hundred tokens -- the first 100,000 tokens of any stream, bytes
     * that are close to uniform throughout -- a block is cut so often that the one-by-one path is the
     * faster one: after such a block the next `rest` tokens go one by one, twice as many each time it
     * happens again (up to rest_most), and blocks are tried again after that.                        */
    uint32_t rest, rest_next;
};

enum { rest_least = block_most, rest_most = 16 * block_most,
       cut_every = block_most / 8 };    /* tokens per cut below which blocks do not pay */

static void tally_init(struct tally* y) {
    memset(y->lit_part, 0, sizeof(y->lit_part));
    memset(y->pos_part, 0, sizeof(y->pos_part));
    y->rest = y->rest_next = 0;
    y->lit_start[2 * sqz_lit_symbols - 1] = 0;  y->lit_start[2 * sqz_lit_symbols] = (uint64_t)INT64_MAX;
    y->pos_start[2 * sqz_pos_symbols - 1] = 0;  y->pos_start[2 * sqz_pos_symbols] = (uint64_t)INT64_MAX;
}

static inline void keep_weights(const struct sqz_tree* t, uint64_t* start) {
    memcpy(start, t->freq, sizeof(uint64_t) * (size_t)t->n);                         /* the leaves */
    memcpy(start + t->next, t->freq + t->next, sizeof(uint64_t) * (size_t)(2 * t->n - 1 - t->next));
}

static inline void restore_weights(struct sqz_tree* t, const uint64_t* start) {
    memcpy(t->freq, start, sizeof(uint64_t) * (size_t)t->n);
    memcpy(t->freq + t->next, start + t->next, sizeof(uint64_t) * (size_t)(2 * t->n - 1 - t->next));
}

/* A span on one tree, in steps.  `kinds` distinct leaves `seen[]`, leaf s occurring count[s] times,
 * `total` occurrences in all.
 * span_ready: 0 when the span cannot be counted at once on this tree (a symbol not yet in the tree
 *   or not a symbol at all, the lazy stretch too short, a path deeper than a plan); makes the plans.
 * span_apply: keeps the weights in `start`, adds the counts along the plans; 1 when no node's end
 *   weight exceeds its comparator's start weight (then nothing can have reordered, whatever the order
 *   of the symbols), 0 when some do -- the culprits.
 * span_culprits: which (node, comparator) pairs those are.
 * restore_weights undoes span_apply; span_done closes a span that stands.                          */
enum { span_lazily = 1, span_fully = 2 };

static inline int span_ready(struct sqz_tree* t, const uint16_t* seen, uint32_t kinds, uint32_t total,
                             const int32_t nyt) {
    int how = span_lazily;
    renew_stretch(t);                   /* between two stretches: decide the next one, as the next symbol would */
    if (t->lazy < (int32_t)total) {
        /* no lazy stretch that long: the span walks the top of the tree as well, from exact weights */
        if (t->complete || t->depth >= 63) { return 0; }
        settle(t);
        t->lazy = t->lazy_start = 0;
        how = span_fully;
    }
    for (uint32_t j = 0; j < kinds; j++) {
        const int32_t s = seen[j];
        if (t->up[s] < 0 || s == nyt) { return 0; }
        if (t->steps[s] == 0) { settle(t); make_plan(t, s); }
        if (t->steps[s] == plan_too_deep) { return 0; }
    }
    return how;
}

static inline __attribute__((always_inline))
int span_apply(struct sqz_tree* t, const uint16_t* seen, uint32_t kinds, const uint16_t* count,
               uint64_t* start, uint8_t* suspect, const int usual, const int how) {
    keep_weights(t, start);
    uint64_t* const freq = t->freq;
    int64_t any = 0;
#define SQZ_BLOCK_STEP(k_) do {                                                              \
        const int64_t w_ = (int64_t)freq[plan[k_]] + c;                                      \
        fires |= (int64_t)start[plan[plan_levels + (k_)]] - w_;                              \
        freq[plan[k_]] = (uint64_t)w_; } while (0)
    for (uint32_t j = 0; j < kinds; j++) {
        const int32_t s = seen[j];
        const int64_t c = count[s];
        const uint16_t* const plan = t->plan + (size_t)s * 2 * plan_levels;
        int64_t fires = 0;
        SQZ_BLOCK_STEP(0);
        if (how == span_fully) {
            for (int k = 1; k <= top_levels; k++) { SQZ_BLOCK_STEP(k); }
        }
#pragma GCC unroll 16
        for (int k = top_levels + 1; k < usual; k++) { SQZ_BLOCK_STEP(k); }
        if (t->steps[s] != usual) {
            for (int k = usual; k < plan_levels; k++) { SQZ_BLOCK_STEP(k); }
        }
        suspect[j] = (uint8_t)((uint64_t)fires >> 63);   /* some node on this leaf's walk, as far as it got */
        any |= fires;
    }
#undef SQZ_BLOCK_STEP
    return any >= 0;
}

enum { culprits_most = 8 };
struct culprits {                       /* nodes that may have outgrown their comparators during a span */
    int32_t count;                      /* -1: more than culprits_most */
    uint16_t node[culprits_most], over[culprits_most];
};

/* after a span_apply that returned 0, before the weights are restored */
static void span_culprits(const struct sqz_tree* t, const uint16_t* seen, uint32_t kinds,
                          const uint64_t* start, const uint8_t* suspect, const int how, struct culprits* who) {
    const uint64_t* const freq = t->freq;
    who->count = 0;
    for (uint32_t j = 0; j < kinds; j++) {
        /* a node outgrows its comparator at the latest when the last leaf below it has walked, so it
         * shows in that leaf's verdict */
        if (!suspect[j]) { continue; }
        const int32_t s = seen[j];
        const uint16_t* const plan = t->plan + (size_t)s * 2 * plan_levels;
        const int steps = t->steps[s];
        for (int k = 0; k < steps; k++) {
            if (how == span_lazily && k >= 1 && k <= top_levels) { continue; }   /* not walked, not judged */
            const uint16_t node = plan[k], over = plan[plan_levels + k];
            if ((int64_t)start[over] - (int64_t)freq[node] >= 0) { continue; }
            int known = 0;
            for (int32_t q = 0; q < who->count; q++) { known |= who->node[q] == node; }
            if (known) { continue; }
            if (who->count == culprits_most) { who->count = -1; return; }
            who->node[who->count] = node;
            who->over[who->count] = over;
            who->count++;
        }
    }
}

static inline void span_done(struct sqz_tree* t, uint32_t total, const int how) {
    if (how == span_lazily) { t->lazy -= (int32_t)total; }
    else { t->eager = t->eager > (int32_t)total ? t->eager - (int32_t)total : 0; }
}

/* Which leaves lie below a culprit (bit q of below[s]) or below its comparator (bit q of beside[s]),
 * by walking the two subtrees (small ones as a rule: what reorders is deep in the tree); and the
 * same as lists: crowd[edge[2q] .. edge[2q+1]) the leaves below culprit q, crowd[edge[2q+1] ..
 * edge[2q+2]) those below its comparator.  0 when the lists do not fit.                          */
enum { crowd_most = 512 };

static int mark_below(const struct sqz_tree* t, int32_t top, uint8_t bit, uint8_t* mark,
                      uint16_t* crowd, uint32_t* filled) {
    int16_t stack[2 * sqz_lit_symbols];
    int sp = 0;
    if (top >= 2 * t->n - 1) { return 1; }           /* the comparators "always" and "never": no leaves */
    stack[sp++] = (int16_t)top;
    while (sp > 0) {
        const int32_t i = stack[--sp];
        if (i < t->n) {
            mark[i] |= bit;
            if (*filled == crowd_most) { return 0; }
            crowd[(*filled)++] = (uint16_t)i;
            continue;
        }
        if (t->lo[i] >= 0) { stack[sp++] = t->lo[i]; }
        if (t->hi[i] >= 0) { stack[sp++] = t->hi[i]; }
    }
    return 1;
}

static int culprit_leaves(const struct sqz_tree* t, const struct culprits* who, uint8_t* below, uint8_t* beside,
                          uint16_t* crowd, uint32_t* edge) {
    uint32_t filled = 0;
    int fits = 1;
    memset(below, 0, (size_t)t->n);
    memset(beside, 0, (size_t)t->n);
    for (int32_t q = 0; q < who->count; q++) {
        edge[2 * q] = filled;
        fits &= mark_below(t, who->node[q], (uint8_t)(1u << q), below, crowd, &filled);
        edge[2 * q + 1] = filled;
        fits &= mark_below(t, who->over[q], (uint8_t)(1u << q), beside, crowd, &filled);
    }
    edge[2 * who->count] = filled;
    return fits;
}

/* count the symbols of the words [0, n) into one part's tallies (n <= part_tokens) */
static __attribute__((noinline))
void tally_words(uint16_t* lit_count, uint16_t* pos_count, const uint32_t* words, uint32_t n) {
    /* whether a token is a match cannot be predicted: no branch on it -- every token stores its
     * distance field, the position only moves on behind a match (bit 8 of the symbol) */
    uint8_t far[part_tokens + 1];
    uint32_t matches = 0;
    for (uint32_t k = 0; k < n; k++) {
        const uint32_t w = words[k];
        lit_count[w & 0x1FF]++;
        far[matches] = (uint8_t)((w >> 14) & 31);
        matches += (w >> 8) & 1;
    }
    for (uint32_t k = 0; k < matches; k++) { pos_count[far[k]]++; }
}

/* The symbol words [0, n) -- parts [first, first + parts) of the block tallied in y -- on both trees
 * as one span; words[0] is word `offset` of that block.  Returns n: done.  -1: nothing changed and the span cannot go as one (a symbol without
 * a leaf, no lazy stretch, too many culprits).  0 <= t < n: nothing changed; the words before t can
 * go as one span and word t is the first at which a node may outgrow its comparator -- found by
 * walking the words with the start weights of the culprits and their comparators, counting who is
 * below which (exact for those pairs; every other pair passed the end-against-start test).  When no
 * word is one, the span stands although that test failed.  Words that are no symbol words never
 * pass (their symbol is not in the tree, or is the escape) except for flaws the model does not look
 * at -- the emitter reports those.                                                              */
static int32_t count_span(struct sqz* s, struct tally* y, const uint32_t* words, uint32_t offset, uint32_t n,
                          uint32_t first, uint32_t parts, uint64_t* matches_) {
    struct sqz_tree* const lit = &s->lit;
    struct sqz_tree* const pos = &s->pos;
    uint32_t lit_kinds = 0, pos_kinds = 0, matches = 0, strays = 0;
    /* four 16-bit counters per addition; the symbols in use end at the escape, the rest of a row only
     * ever holds strays (symbols no tree has) */
    enum { lit_quads = sqz_lit_symbols / 4, pos_quads = sqz_pos_symbols / 4 };
    {
        /* four counters at a time: a type that may alias the 16-bit ones it is laid over */
        typedef uint64_t __attribute__((may_alias)) four_counts;
        four_counts* const ls = (four_counts*)(void*)y->lit_count;
        four_counts* const ps = (four_counts*)(void*)y->pos_count;
        memcpy(ls, y->lit_part[first], sizeof(y->lit_count));
        memcpy(ps, y->pos_part[first], sizeof(uint16_t) * sqz_pos_symbols);
        for (uint32_t q = first + 1; q < first + parts; q++) {
            const four_counts* const lp = (const four_counts*)(const void*)y->lit_part[q];
            const four_counts* const pp = (const four_counts*)(const void*)y->pos_part[q];
            for (uint32_t k = 0; k < lit_quads; k++) { ls[k] += lp[k]; }
            for (uint32_t k = 0; k < pos_quads; k++) { ps[k] += pp[k]; }
        }
    }
    for (uint32_t k = 0; k <= sqz_lit_nyt; k++) {
        y->lit_seen[lit_kinds] = (uint16_t)k;
        lit_kinds += y->lit_count[k] != 0;
    }
    for (uint32_t k = sqz_lit_nyt + 1; k < sqz_lit_symbols; k++) { strays |= y->lit_count[k]; }
    if (strays != 0) { return -1; }                  /* symbols no tree has */
    for (uint32_t pb = 0; pb < sqz_pos_symbols; pb++) {
        y->pos_seen[pos_kinds] = (uint16_t)pb;
        pos_kinds += y->pos_count[pb] != 0;
        matches += y->pos_count[pb];
    }
    const int lit_how = span_ready(lit, y->lit_seen, lit_kinds, n, sqz_lit_nyt);
    const int pos_how = lit_how == 0 ? 0 : span_ready(pos, y->pos_seen, pos_kinds, matches, sqz_pos_nyt);
    if (lit_how == 0 || pos_how == 0) {
        return -1;
    }
#ifdef SQZ_SELFCHECK
    settle(lit); settle(pos);           /* so that the replay below starts from the very same weights */
#endif
    const int pos_fine = span_apply(pos, y->pos_seen, pos_kinds, y->pos_count, y->pos_start, y->pos_suspect, pos_plan, pos_how);
    const int lit_fine = span_apply(lit, y->lit_seen, lit_kinds, y->lit_count, y->lit_start, y->lit_suspect, lit_plan, lit_how);
    int32_t reach = (int32_t)n;
    if (!pos_fine || !lit_fine) {
        struct culprits lit_who = { 0, { 0 }, { 0 } }, pos_who = { 0, { 0 }, { 0 } };
        if (!lit_fine) { span_culprits(lit, y->lit_seen, lit_kinds, y->lit_start, y->lit_suspect, lit_how, &lit_who); }
        if (!pos_fine) { span_culprits(pos, y->pos_seen, pos_kinds, y->pos_start, y->pos_suspect, pos_how, &pos_who); }
        if (lit_who.count < 0 || pos_who.count < 0) {
            reach = -1;
        } else {
            int64_t lit_lead[culprits_most], pos_lead[culprits_most];   /* comparator's weight - culprit's */
            for (int32_t q = 0; q < lit_who.count; q++) {
                lit_lead[q] = (int64_t)y->lit_start[lit_who.over[q]] - (int64_t)y->lit_start[lit_who.node[q]];
            }
            for (int32_t q = 0; q < pos_who.count; q++) {
                pos_lead[q] = (int64_t)y->pos_start[pos_who.over[q]] - (int64_t)y->pos_start[pos_who.node[q]];
            }
            uint16_t lit_crowd[crowd_most], pos_crowd[crowd_most];
            uint32_t lit_edge[2 * culprits_most + 1], pos_edge[2 * culprits_most + 1];
            const int listed = culprit_leaves(lit, &lit_who, y->lit_below, y->lit_beside, lit_crowd, lit_edge) &
                               culprit_leaves(pos, &pos_who, y->pos_below, y->pos_beside, pos_crowd, pos_edge);
            /* Row by row: a row in which a culprit cannot catch up with its comparator even if all its
             * own symbols came first only moves the leads; the others are walked word by word. */
            for (uint32_t r = first; r < first + parts && reach == (int32_t)n; r++) {
                const uint32_t from = r * part_tokens > offset ? r * part_tokens - offset : 0;
                const uint32_t to = (r + 1) * part_tokens - offset < n ? (r + 1) * part_tokens - offset : n;
                int walk = !listed;
                int64_t lit_gain[culprits_most], pos_gain[culprits_most];
                for (int32_t q = 0; q < lit_who.count && !walk; q++) {
                    int64_t own = 0, other = 0;
                    for (uint32_t j = lit_edge[2 * q]; j < lit_edge[2 * q + 1]; j++) { own += y->lit_part[r][lit_crowd[j]]; }
                    for (uint32_t j = lit_edge[2 * q + 1]; j < lit_edge[2 * q + 2]; j++) { other += y->lit_part[r][lit_crowd[j]]; }
                    walk = lit_lead[q] - own < 0;
                    lit_gain[q] = other - own;
                }
                for (int32_t q = 0; q < pos_who.count && !walk; q++) {
                    int64_t own = 0, other = 0;
                    for (uint32_t j = pos_edge[2 * q]; j < pos_edge[2 * q + 1]; j++) { own += y->pos_part[r][pos_crowd[j]]; }
                    for (uint32_t j = pos_edge[2 * q + 1]; j < pos_edge[2 * q + 2]; j++) { other += y->pos_part[r][pos_crowd[j]]; }
                    walk = pos_lead[q] - own < 0;
                    pos_gain[q] = other - own;
                }
                if (!walk) {
                    for (int32_t q = 0; q < lit_who.count; q++) { lit_lead[q] += lit_gain[q]; }
                    for (int32_t q = 0; q < pos_who.count; q++) { pos_lead[q] += pos_gain[q]; }
                    continue;
                }
                for (uint32_t k = from; k < to && reach == (int32_t)n; k++) {
                    const uint32_t w = words[k], sym = w & 0x1FF;
                    /* a symbol's walk adds 1 to every node above it, then each is compared with its
                     * comparator; the comparator is never on the same walk */
                    for (uint32_t x = y->lit_below[sym]; x != 0; x &= x - 1) {
                        if (--lit_lead[__builtin_ctz(x)] < 0) { reach = (int32_t)k; }
                    }
                    for (uint32_t c = y->lit_beside[sym]; c != 0; c &= c - 1) { lit_lead[__builtin_ctz(c)]++; }
                    if (sym >= len_symbol0 && pos_who.count != 0) {
                        const uint32_t pb = (w >> 14) & 31;
                        for (uint32_t x = y->pos_below[pb]; x != 0; x &= x - 1) {
                            if (--pos_lead[__builtin_ctz(x)] < 0) { reach = (int32_t)k; }
                        }
                        for (uint32_t c = y->pos_beside[pb]; c != 0; c &= c - 1) { pos_lead[__builtin_ctz(c)]++; }
                    }
                }
            }
        }
        if (reach != (int32_t)n) {
            restore_weights(lit, y->lit_start);
            restore_weights(pos, y->pos_start);
            return reach;
        }
    }
    span_done(lit, n, lit_how);
    span_done(pos, matches, pos_how);
    *matches_ += matches;
#ifdef SQZ_SELFCHECK
    {
        /* the same symbols one by one from the same start: no reordering, the same weights */
        static _Thread_local uint64_t lit_after[2 * sqz_lit_symbols - 1], pos_after[2 * sqz_pos_symbols - 1];
        settle(lit); settle(pos);
        memcpy(lit_after, lit->freq, sizeof(lit_after));
        memcpy(pos_after, pos->freq, sizeof(pos_after));
        restore_weights(lit, y->lit_start);
        restore_weights(pos, y->pos_start);
        lit->lazy = lit->lazy_start = lit->eager = 0;       /* the top is exact, nothing is decided */
        pos->lazy = pos->lazy_start = pos->eager = 0;
        const uint64_t shape = selfcheck_relabels;
        __atomic_fetch_add(&sqz_selfcheck_spans, 1, __ATOMIC_RELAXED);
        __atomic_fetch_add(&sqz_selfcheck_span_tokens, n, __ATOMIC_RELAXED);
        for (uint32_t k = 0; k < n; k++) {
            const uint32_t w = words[k], sym = w & 0x1FF;
            tree_count_as(lit, (int32_t)sym, lit_plan);
            if (sym >= len_symbol0) { tree_count_as(pos, (int32_t)((w >> 14) & 31), pos_plan); }
        }
        settle(lit); settle(pos);
        if (shape != selfcheck_relabels ||
            memcmp(lit_after, lit->freq, sizeof(uint64_t) * (size_t)(2 * lit->n - 2)) != 0 ||
            memcmp(pos_after, pos->freq, sizeof(uint64_t) * (size_t)(2 * pos->n - 2)) != 0) {
            fprintf(stderr, "sqz selfcheck: a span of %u symbols differs from the same symbols one by one\n", n);
            abort();
        }
        selfcheck(lit); selfcheck(pos);
    }
#endif
    return (int32_t)n;
}

/* ======================================================================== *
 *  token coder  (reference squeeze.h:151-172, 239-315)                      *
 * ======================================================================== */

static void bucket_tables(struct sqz* s) {
    /* len -> bucket: 258 would be bucket 28 in deflate, but symbol 257+28 is
     * the NYT escape here, so 227..258 all stay in bucket 27 (squeeze.h:151-161) */
    memset(s->len_index, 0, sizeof(s->len_index));
    for (int len = 3; len < (int)sizeof(s->len_index); len++) {
        int b = 0;
        while (b + 1 < 28 && len_base[b + 1] <= len) { b++; }
        s->len_index[len] = (uint8_t)b;
    }
}

/* dist -> distance bucket (squeeze.h:162-171 builds a 32 KiB table for this;
 * the buckets are deflate's: two per power of two above 4)                  */
static inline uint32_t pos_bucket(uint32_t dist) {
    if (dist <= 4) { return dist - 1; }
    const uint32_t m = dist - 1;
    const uint32_t k = 31u - (uint32_t)__builtin_clz(m);
    return 2 * k + ((m >> (k - 1)) & 1);
}

void sqz_init(struct sqz* s) {
    memset(s, 0, sizeof(*s));
    s->device = -1;                       /* the caller's current CUDA device */
    SQZ_BIND_TREE(&s->lit, s->lit_store, sqz_lit_symbols);
    SQZ_BIND_TREE(&s->pos, s->pos_store, sqz_pos_symbols);
    tree_init(&s->lit);
    tree_init(&s->pos);
}

static void coder_begin(struct sqz* s, struct sqz_bitstream* bs) {
    s->bs = bs;
    /* both escape symbols exist from the start, so the first code ever
     * written is the single bit 1 (squeeze.h:333-334) */
    if (!tree_insert(&s->lit, sqz_lit_nyt)) { s->error = EINVAL; }
    if (!tree_insert(&s->pos, sqz_pos_nyt)) { s->error = EINVAL; }
    bucket_tables(s);
}

static inline void s_put(struct sqz* s, uint64_t v, int count) {
    if (s->error == 0) { put_bits(s->bs, v, count); s->error = s->bs->error; }
}

/* current code of `sym`, then bump its weight (squeeze.h:239-246) */
static inline void emit_symbol(struct sqz* s, struct sqz_tree* t, int32_t sym) {
    if (s->error == 0) { put_code(s->bs, t->code[sym], t->bits[sym]); s->error = s->bs->error; }
    tree_count(t, sym);
}

static inline void code_lit(struct sqz* s, uint32_t sym) {     /* squeeze.h:278-288 */
    if (s->lit.bits[sym] == 0) {
        emit_symbol(s, &s->lit, sqz_lit_nyt);
        s_put(s, sym, 9);
        if (!tree_insert(&s->lit, (int32_t)sym)) { s->error = E2BIG; }
    } else {
        emit_symbol(s, &s->lit, (int32_t)sym);
    }
}

/* ---- symbol words ---------------------------------------------------------
 * What the coder consumes is one 32-bit word per token with the bucket
 * arithmetic of squeeze.h:290-315 already done (sqz_gpu.h: the GPU emits these
 * words directly, `symbols` mode of the stream; for a caller's plain tokens
 * symbols_of_token() below makes them):
 *   bits  0..8   symbol of the literal/length tree: byte, or 257 + length bucket
 *   bits  9..13  the length's extra bits, in emission order
 *   bits 14..18  symbol of the distance tree (distance bucket)
 *   bits 19..31  the distance's extra bits, in emission order
 * "In emission order" = bit-reversed within its field width, since values go
 * out least significant bit first (bitstream.h:49-63).                       */

static inline uint32_t reverse_field(uint32_t v, uint32_t width) {   /* width <= 16 */
    static const uint8_t rev4[16] = { 0, 8, 4, 12, 2, 10, 6, 14, 1, 9, 5, 13, 3, 11, 7, 15 };
    const uint32_t r = (uint32_t)rev4[v & 15] << 12 | (uint32_t)rev4[(v >> 4) & 15] << 8 |
                       (uint32_t)rev4[(v >> 8) & 15] << 4 | (uint32_t)rev4[(v >> 12) & 15];
    return r >> (16 - width);
}

static inline int token_is_valid(uint32_t t) {          /* the decoder's limits: squeeze.h:529-545 */
    const uint32_t len = t >> 16, dist = t & 0xFFFF;
    return len == 0 ? t <= 0xFF : (len >= sqz_min_len && len <= sqz_max_len && dist >= 1 && dist <= 0x7FFF);
}

static inline uint32_t symbols_of_token(const struct sqz* s, uint32_t t) {
    const uint32_t len = t >> 16;
    if (len == 0) { return t; }
    const uint32_t dist = t & 0xFFFF;
    const uint32_t lb = s->len_index[len], pb = pos_bucket(dist);
    return (len_symbol0 + lb) | reverse_field(len - len_base[lb], len_extra[lb]) << 9 |
           pb << 14 | reverse_field(dist - pos_base[pb], pos_extra[pb]) << 19;
}

static inline int word_is_valid(uint32_t w) {
    const uint32_t sym = w & 0x1FF;
    /* bucket 27 with all five extra bits set would be length 258, which no decoder accepts
     * (squeeze.h:529-545) */
    return sym <= 0xFF || (sym >= len_symbol0 && sym <= len_symbol0 + 27 && ((w >> 14) & 31) <= 29 &&
                           !(sym == len_symbol0 + 27 && ((w >> 9) & 31) == 31));
}

/* Append `count_` bits `seq_` (first bit out = most significant) to the register acc/fill; a full
 * word goes straight to memory when the sink is a buffer with room, else through word_out.      */
#define SQZ_APPEND(seq_, count_) do {                                            \
        const uint64_t q_ = (seq_); const uint32_t c_ = (count_);                \
        const uint32_t f_ = fill + c_;                                           \
        if (f_ < 64) { acc = (acc << c_) | q_; fill = f_; }                      \
        else {                                                                   \
            const uint32_t rest_ = f_ - 64;                                      \
            const uint64_t word_ = (fill == 0 ? 0 : acc << (64 - fill)) | (q_ >> rest_); \
            if (bs->data != NULL && bs->capacity - bs->bytes >= 8 && bs->capacity >= bs->bytes) { \
                const uint64_t be_ = __builtin_bswap64(word_);                   \
                memcpy(bs->data + bs->bytes, &be_, 8);                           \
                bs->bytes += 8;                                                  \
            } else {                                                             \
                bs->b64 = word_; bs->bits = 64;                                  \
                word_out(bs);                                                    \
                if (bs->error != 0) { *err = bs->error; goto done; }             \
            }                                                                    \
            acc = rest_ == 0 ? 0 : (q_ & (((uint64_t)1 << rest_) - 1));          \
            fill = rest_;                                                        \
        } } while (0)

/* What a 9-bit symbol of the literal/length tree is: 0 = nothing a word may carry (256, the
 * escape, anything above), 0x40 = a byte, 0x80 | extra bits = a length bucket.                 */
static const uint8_t symbol_kind[sqz_lit_symbols] = {
    [0 ... 255] = 0x40,
    [257 ... 264] = 0x80, [265 ... 268] = 0x81, [269 ... 272] = 0x82, [273 ... 276] = 0x83,
    [277 ... 280] = 0x84, [281 ... 284] = 0x85 };

/* What the emitter reads: the codes of both trees as they stand for the token being emitted --
 * plain, and as *words*: (code << extra bits) << 8 | code length + extra bits, ready to take the
 * extra bits in with one OR; 0 where a symbol has to go the general way (no code yet, not a symbol
 * a word may carry, more than word_lit_most / word_pos_most bits -- together 56, what one store of
 * the byte-wise emitter takes).  pos_word[32..63] stay 0: that is where a literal looks.        */
enum { word_lit_most = 30, word_pos_most = 26 };

struct code_tables {
    uint64_t lit_word[sqz_lit_symbols];
    uint64_t pos_word[2 * sqz_pos_symbols];
    uint64_t lit_code[sqz_lit_symbols];
    uint64_t pos_code[sqz_pos_symbols];
    uint8_t lit_bits[sqz_lit_symbols];
    uint8_t pos_bits[sqz_pos_symbols];
};

static inline void tables_set(struct code_tables* ct, int distance_tree, uint32_t leaf, uint64_t code, uint32_t bits) {
    if (distance_tree) {
        const uint32_t more = leaf < 30 ? pos_extra[leaf] : 0;
        ct->pos_code[leaf] = code;
        ct->pos_bits[leaf] = (uint8_t)bits;
        ct->pos_word[leaf] = (leaf < 30 && bits != 0 && bits + more <= word_pos_most)
                           ? (code << more) << 8 | (bits + more) : 0;
    } else {
        const uint32_t kind = symbol_kind[leaf], more = kind & 7;
        ct->lit_code[leaf] = code;
        ct->lit_bits[leaf] = (uint8_t)bits;
        ct->lit_word[leaf] = (kind != 0 && bits != 0 && bits + more <= word_lit_most)
                           ? (code << more) << 8 | (bits + more) : 0;
    }
}

static void tables_from_trees(struct code_tables* ct, const struct sqz* s) {
    memset(ct->pos_word, 0, sizeof(ct->pos_word));
    for (uint32_t k = 0; k < sqz_lit_symbols; k++) { tables_set(ct, 0, k, s->lit.code[k], s->lit.bits[k]); }
    for (uint32_t k = 0; k < sqz_pos_symbols; k++) { tables_set(ct, 1, k, s->pos.code[k], s->pos.bits[k]); }
}

/* Emit the words [from, until) with code tables that do not change on the way (a block the model
 * took as a whole, or the stretch between two changes of a code in the two-thread coder).  A
 * symbol without a code yet goes out as the escape plus its raw bits (squeeze.h:278-288, 300-315:
 * only the coders on several threads get here with one, their model inserts the symbol).  On an
 * error *err is set and the rest is not emitted.                                                */
static void emit_run_anywhere(int32_t* err, struct sqz_bitstream* bs, const uint32_t* words,
                              uint64_t from, uint64_t until, const struct code_tables* ct) {
    uint64_t acc = bs->b64;
    uint32_t fill = (uint32_t)bs->bits;
    for (uint64_t k = from; k < until; k++) {
        const uint32_t w = words[k];
        const uint32_t sym = w & 0x1FF;
        if (!word_is_valid(w)) {                     /* not a symbol word: the decoder would reject it */
            *err = EINVAL;
            goto done;
        }
        if (ct->lit_bits[sym] == 0) {
            SQZ_APPEND(ct->lit_code[sqz_lit_nyt], ct->lit_bits[sqz_lit_nyt]);
            SQZ_APPEND(reverse_field(sym, 9), 9);
        } else {
            SQZ_APPEND(ct->lit_code[sym], ct->lit_bits[sym]);
        }
        if (sym >= len_symbol0) {                    /* length first, then distance: squeeze.h:379-380 */
            const uint32_t pb = (w >> 14) & 31;
            SQZ_APPEND((w >> 9) & 31, len_extra[sym - len_symbol0]);
            if (ct->pos_bits[pb] == 0) {
                SQZ_APPEND(ct->pos_code[sqz_pos_nyt], ct->pos_bits[sqz_pos_nyt]);
                SQZ_APPEND(reverse_field(pb, 5), 5);
            } else {
                SQZ_APPEND(ct->pos_code[pb], ct->pos_bits[pb]);
            }
            SQZ_APPEND(w >> 19, pos_extra[pb]);
        }
    }
done:
    bs->b64 = acc;
    bs->bits = (int32_t)fill;
}

/* The same into a memory sink with room for the worst case (8 bytes a token).  The stream is
 * big-endian 64-bit words of bits entered first-bit-highest (bitstream.h:28-47), i.e. a byte
 * stream with the first bit in the top of the first byte: the bits of a whole token -- code,
 * length bits, distance code, distance bits, at most 56 -- are put together from the two table
 * words, joined to the pending bits, stored as eight bytes, and the write position moves on by
 * the whole bytes among them.  No branch depends on the data except the rare one to the general
 * way.  Returns the index it stopped at (`until`, or the token that has to go the general way);
 * *pending / *pending_bits: the bits not yet part of a whole byte, at the top of the register.
 * A function of its own so that its few loop variables stay in registers.                      */
static __attribute__((noinline))
uint64_t emit_bytes(const uint32_t* words, uint64_t from, uint64_t until, const struct code_tables* ct,
                    uint8_t** at_, uint64_t* pending, uint32_t* pending_bits) {
    const uint64_t* const lit_word = ct->lit_word;
    const uint64_t* const pos_word = ct->pos_word;
    uint8_t* at = *at_;
    uint64_t acc = *pending;
    uint32_t fill = *pending_bits;
    uint64_t k = from;
    for (; k < until; k++) {
        const uint32_t w = words[k];
        const uint32_t match = (w >> 8) & 1;                     /* bit 8 of the symbol: a length */
        const uint64_t e = lit_word[w & 0x1FF];
        const uint64_t p = pos_word[((w >> 14) & 31) | ((~w >> 3) & 32)];
        /* general way: no table word; bucket 27 with all extra bits set (length 258, squeeze.h:529-545) */
        if (__builtin_expect((e == 0) | (match & (p == 0)) | ((w & 0x3FFF) == (len_symbol0 + 27 + (31u << 9))), 0)) {
            break;
        }
        const uint32_t n = ((uint32_t)e & 0xFF) + ((uint32_t)p & 0xFF);
        uint64_t v = (e >> 8) | ((w >> 9) & 31);
        v = (v << (p & 0xFF)) | (p >> 8) | (w >> 19);
        fill += n;
        acc |= v << (64 - fill);
        const uint64_t be = __builtin_bswap64(acc);
        memcpy(at, &be, 8);
        at += fill >> 3;
        acc <<= fill & 56;
        fill &= 7;
    }
    *at_ = at;
    *pending = acc;
    *pending_bits = fill;
    return k;
}

static void emit_run(int32_t* err, struct sqz_bitstream* bs, const uint32_t* words, uint64_t from, uint64_t until,
                     const struct code_tables* ct) {
    while (from < until && *err == 0) {
        if (bs->data == NULL || bs->capacity < bs->bytes || bs->bits < 0 || bs->bits > 63 ||
            (bs->capacity - bs->bytes) / 8 < until - from + 3) {
            emit_run_anywhere(err, bs, words, from, until, ct);
            return;
        }
        uint8_t* const start = bs->data + bs->bytes;
        uint8_t* at = start;
        uint32_t fill = (uint32_t)bs->bits;                      /* pending bits, kept at the top of acc */
        uint64_t acc = fill == 0 ? 0 : bs->b64 << (64 - fill);
        const uint64_t be = __builtin_bswap64(acc);
        memcpy(at, &be, 8);
        at += fill >> 3;
        acc <<= fill & 56;
        fill &= 7;
        from = emit_bytes(words, from, until, ct, &at, &acc, &fill);
        /* back to whole words in memory + the rest in the register */
        const size_t bytes_out = (size_t)(at - start);
        const size_t whole = bytes_out & ~(size_t)7;
        uint64_t rest = 0;
        for (size_t j = whole; j < bytes_out; j++) { rest = rest << 8 | start[j]; }
        bs->bytes += whole;
        bs->b64 = fill == 0 ? rest : (rest << fill) | (acc >> (64 - fill));
        bs->bits = (int32_t)(8 * (bytes_out - whole) + fill);
        if (from < until) {
            emit_run_anywhere(err, bs, words, from, from + 1, ct);
            from++;
        }
    }
}

/* The words [from, until) one by one: emit with the current code, count, next (the reference's
 * order, squeeze.h:239-246); everything unusual (first occurrence of a symbol, callback sinks, a
 * full buffer) goes through the general functions above with the register synced.              */
static uint64_t code_one_by_one(struct sqz* s, const uint32_t* words, uint64_t from, uint64_t until) {
    struct sqz_bitstream* const bs = s->bs;
    struct sqz_tree* const lit = &s->lit;
    struct sqz_tree* const pos = &s->pos;
    int32_t* const err = &s->error;
    uint64_t acc = bs->b64;
    uint32_t fill = (uint32_t)bs->bits;
    uint64_t matches = 0;
#define SQZ_SYNC_OUT()  do { bs->b64 = acc; bs->bits = (int32_t)fill; } while (0)
#define SQZ_SYNC_IN()   do { acc = bs->b64; fill = (uint32_t)bs->bits; } while (0)
    for (uint64_t k = from; k < until; k++) {
        const uint32_t w = words[k];
        const uint32_t sym = w & 0x1FF;
        if (!word_is_valid(w)) {
            s->error = EINVAL;
            goto done;
        }
        if (lit->bits[sym] == 0) {                   /* first occurrence: escape + raw symbol */
            SQZ_SYNC_OUT();
            code_lit(s, sym);
            SQZ_SYNC_IN();
            if (s->error != 0) { goto done; }
        } else {
            SQZ_APPEND(lit->code[sym], lit->bits[sym]);
            tree_count_as(lit, (int32_t)sym, lit_plan);
            SQZ_CHECK(lit);
        }
        if (sym >= len_symbol0) {
            const uint32_t pb = (w >> 14) & 31;
            SQZ_APPEND((w >> 9) & 31, len_extra[sym - len_symbol0]);
            if (pos->bits[pb] == 0) {
                SQZ_SYNC_OUT();
                emit_symbol(s, pos, sqz_pos_nyt);
                s_put(s, pb, 5);
                if (!tree_insert(pos, (int32_t)pb)) { s->error = E2BIG; }
                SQZ_SYNC_IN();
                if (s->error != 0) { goto done; }
            } else {
                SQZ_APPEND(pos->code[pb], pos->bits[pb]);
                tree_count_as(pos, (int32_t)pb, pos_plan);
                SQZ_CHECK(pos);
            }
            SQZ_APPEND(w >> 19, pos_extra[pb]);
            matches++;
        }
    }
done:
    SQZ_SYNC_OUT();
    return matches;
#undef SQZ_SYNC_IN
#undef SQZ_SYNC_OUT
}

/* One pass over a chunk of symbol words, by one thread: model and emit (`ct` set: the one-thread
 * coder), or model only (the model thread of the coders on several threads).                     */
struct pass {
    struct sqz* s;
    struct tally* y;
    struct watch* eyes;
    const uint32_t* words;              /* the chunk */
    uint64_t base;                      /* stamp of words[0] */
    struct code_tables* ct;             /* NULL: model only */
    uint64_t matches;
    int flaw;                           /* model only: stopped at a word that is no symbol word */
};

/* the model alone over [k, until), one by one; returns where it stopped (`until`; or earlier with
 * p->flaw at a word that is no symbol word, not modelled, or with eyes->error set) */
static uint64_t model_one_by_one(struct pass* p, uint64_t k, uint64_t until) {
    struct sqz_tree* const lit = &p->s->lit;
    struct sqz_tree* const pos = &p->s->pos;
    struct watch* const eyes = p->eyes;
    for (; k < until; k++) {
        const uint32_t w = p->words[k];
        const uint32_t sym = w & 0x1FF;
        eyes->k_now = k;
        eyes->now = p->base + k + 1;
        if (!word_is_valid(w)) {
            p->flaw = 1;
            return k;
        }
        if (lit->bits[sym] == 0) {               /* squeeze.h:278-288: escape, then the new symbol */
            tree_count(lit, sqz_lit_nyt);
            if (!tree_insert(lit, (int32_t)sym)) { eyes->error = E2BIG; }
        } else {
            tree_count_as(lit, (int32_t)sym, lit_plan);
            SQZ_CHECK(lit);
        }
        if (sym >= len_symbol0 && eyes->error == 0) {
            const uint32_t pb = (w >> 14) & 31;
            if (pos->bits[pb] == 0) {            /* squeeze.h:300-315 */
                tree_count(pos, sqz_pos_nyt);
                if (!tree_insert(pos, (int32_t)pb)) { eyes->error = E2BIG; }
            } else {
                tree_count_as(pos, (int32_t)pb, pos_plan);
                SQZ_CHECK(pos);
            }
            p->matches++;
        }
        if (eyes->error != 0) { return k; }
    }
    return k;
}

/* [k, until) one by one; 1 = go on, 0 = stop (an error, a flaw) */
static int pass_one_by_one(struct pass* p, uint64_t k, uint64_t until) {
    if (p->ct != NULL) {
        p->matches += code_one_by_one(p->s, p->words, k, until);
        return p->s->error == 0;
    }
    return model_one_by_one(p, k, until) == until;
}

/* The rows of tallies of a block are aligned to the block: row r holds tokens [r * part_tokens,
 * (r + 1) * part_tokens) of it -- or, at either end of what is left of the block, the part of that
 * range that is left (pass_block tallies such a row again).                                     */
static void tally_row(struct pass* p, uint64_t block, uint32_t row, uint32_t lo, uint32_t hi) {
    struct tally* const y = p->y;
    const uint32_t from = lo > row * part_tokens ? lo : row * part_tokens;
    const uint32_t to = hi < (row + 1) * part_tokens ? hi : (row + 1) * part_tokens;
    memset(y->lit_part[row], 0, sizeof(y->lit_part[row]));
    memset(y->pos_part[row], 0, sizeof(y->pos_part[row]));
    if (from < to) { tally_words(y->lit_part[row], y->pos_part[row], p->words + block + from, to - from); }
}

static int pass_emit(struct pass* p, uint64_t from, uint64_t until) {
    if (p->ct == NULL) { return 1; }
    /* no code changed while the span was counted: its bits are those of the codes as they are */
    emit_run(&p->s->error, p->s->bs, p->words, from, until, p->ct);
    return p->s->error == 0;
}

/* The tokens [lo, hi) of the block that starts at word `block`, tallied in rows [row, row + rows):
 * as one span if that passes, else by groups of four rows, else row by row, else one by one -- the
 * way for spans that cannot be helped by finding the one word that matters.  1 = go on, 0 = stop. */
static int pass_rows(struct pass* p, uint64_t block, uint32_t lo, uint32_t hi, uint32_t row, uint32_t rows) {
    if (count_span(p->s, p->y, p->words + block + lo, lo, hi - lo, row, rows, &p->matches) == (int32_t)(hi - lo)) {
        return pass_emit(p, block + lo, block + hi);
    }
    if (rows == 1) { return pass_one_by_one(p, block + lo, block + hi); }
    const uint32_t step = rows > 4 ? 4 : 1;
    for (uint32_t q = 0; q < rows; q += step) {
        const uint32_t some = rows - q < step ? rows - q : step;
        const uint32_t from = lo > (row + q) * part_tokens ? lo : (row + q) * part_tokens;
        const uint32_t to = hi < (row + q + some) * part_tokens ? hi : (row + q + some) * part_tokens;
        if (from < to && !pass_rows(p, block, from, to, row + q, some)) { return 0; }
    }
    return 1;
}

/* the next block of the chunk, at most up to `until`; returns the tokens dealt with (fewer than it
 * took on when something stopped the pass: p->flaw, p->eyes->error, p->s->error) */
static uint64_t pass_block(struct pass* p, uint64_t k, uint64_t until) {
    const struct sqz_tree* const lit = &p->s->lit;
    uint64_t most = until - k < block_most ? until - k : block_most;
    if ((int64_t)most > lit->lazy) { most = lit->lazy > 0 ? (uint64_t)lit->lazy : 0; }
    if (most < block_least) {           /* no lazy stretch is on (or it ends): the one-by-one path renews it */
        most = until - k < block_least ? until - k : block_least;
        if (p->ct != NULL) {
            p->matches += code_one_by_one(p->s, p->words, k, k + most);
            return most;
        }
        return model_one_by_one(p, k, k + most) - k;
    }
    if (p->y->rest > 0) {               /* blocks did not pay a moment ago */
        if (most > p->y->rest) { most = p->y->rest; }
        p->y->rest -= (uint32_t)most;
        if (p->ct != NULL) {
            p->matches += code_one_by_one(p->s, p->words, k, k + most);
            return most;
        }
        return model_one_by_one(p, k, k + most) - k;
    }
    const uint32_t n = (uint32_t)most;
    const uint32_t rows = (n + part_tokens - 1) / part_tokens;
    for (uint32_t r = 0; r < rows; r++) { tally_row(p, k, r, 0, n); }
    uint32_t lo = 0, cuts = 0;
    int went = 1;
    while (lo < n && went) {
        const uint32_t row = lo / part_tokens;
        const int32_t reach = count_span(p->s, p->y, p->words + k + lo, lo, n - lo, row, rows - row, &p->matches);
        if (reach == (int32_t)(n - lo)) {
            went = pass_emit(p, k + lo, k + n);
            lo = n;
        } else if (reach < 0) {
            /* a symbol without a leaf yet, a tree between two lazy stretches, a crowd of culprits: up to
             * the end of the row one by one (that settles the first two as a rule), then the rest again */
            const uint32_t to = (row + 1) * part_tokens < n ? (row + 1) * part_tokens : n;
            cuts++;
            went = pass_one_by_one(p, k + lo, k + to);
            lo = to;
            if (went) {
                renew_stretch(&p->s->lit);
                renew_stretch(&p->s->pos);
            }
            if (went && lo < n && p->s->lit.lazy < (int32_t)(n - lo)) {
                for (uint32_t r = 0; r < rows; r++) { tally_row(p, k, r, 0, 0); }
                if (cuts * cut_every > lo) { p->y->rest = p->y->rest_next = rest_least; }
                return lo;
            }
        } else {
            /* everything before word `at` as one span (it passes: the words that matter were walked),
             * that word by itself -- it may reorder the tree --, then what is left of the block */
            const uint32_t at = lo + (uint32_t)reach;
            cuts++;
            if (at - lo >= block_least) {
                const uint32_t last = (at - 1) / part_tokens;
                tally_row(p, k, last, lo, at);
                went = pass_rows(p, k, lo, at, row, last - row + 1);
            } else if (at > lo) {
                went = pass_one_by_one(p, k + lo, k + at);
            }
            if (went) { went = pass_one_by_one(p, k + at, k + at + 1); }
            lo = at + 1;
            if (went) {                 /* a reordering ends the lazy stretch of its tree */
                renew_stretch(&p->s->lit);
                renew_stretch(&p->s->pos);
            }
            if (went && lo < n && p->s->lit.lazy < (int32_t)(n - lo)) {
                /* no stretch long enough for what is left: it is another block's */
                for (uint32_t r = 0; r < rows; r++) { tally_row(p, k, r, 0, 0); }
                if (cuts * cut_every > lo) { p->y->rest = p->y->rest_next = rest_least; }
                return lo;
            }
            if (went && lo < n && cuts * cut_every > lo + cut_every) {
                /* cut after cut: what is left of the block one by one, and no blocks for a while */
                went = pass_one_by_one(p, k + lo, k + n);
                lo = n;
            }
            if (lo < n) { tally_row(p, k, lo / part_tokens, lo, n); }
        }
    }
    for (uint32_t r = 0; r < rows; r++) {
        memset(p->y->lit_part[r], 0, sizeof(p->y->lit_part[r]));
        memset(p->y->pos_part[r], 0, sizeof(p->y->pos_part[r]));
    }
    if (cuts * cut_every > n) {
        p->y->rest_next = p->y->rest_next == 0 ? rest_least : (p->y->rest_next < rest_most ? 2 * p->y->rest_next : rest_most);
        p->y->rest = p->y->rest_next;
    } else {
        p->y->rest_next = 0;
    }
    if (!went && p->flaw) {             /* where the model stopped is what its caller wants to know */
        return p->eyes->k_now - k;
    }
    return n;
}

/* The coder proper, one thread. */
static void code_symbols(struct sqz* s, const uint32_t* words, uint64_t count) {
    struct tally y;
    struct code_tables ct;              /* kept current by relabel through the trees' watcher */
    struct watch eyes = { &ct, NULL, NULL, 0, 0, 0 };
    struct pass p = { s, &y, &eyes, words, 0, &ct, 0, 0 };
    uint64_t k = 0;
    if (s->error != 0) { return; }
    tally_init(&y);
    tables_from_trees(&ct, s);
    s->lit.watcher = s->pos.watcher = &eyes;
    while (k < count && s->error == 0) { k += pass_block(&p, k, count); }
    s->lit.watcher = s->pos.watcher = NULL;
    s->matches += p.matches;
    s->tokens += count;
}

/* plain tokens (literal byte or (len << 16) | dist): checked, turned into symbol
 * words a block at a time, coded                                             */
static void code_tokens(struct sqz* s, const uint32_t* tokens, uint64_t count) {
    enum { portion = 8 * block_most };   /* several blocks per call of the coder */
    uint32_t words[portion];
    for (uint64_t at = 0; at < count && s->error == 0; at += portion) {
        const uint64_t n = count - at < portion ? count - at : portion;
        uint64_t good = 0;
        while (good < n && token_is_valid(tokens[at + good])) {
            words[good] = symbols_of_token(s, tokens[at + good]);
            good++;
        }
        code_symbols(s, words, good);
        if (good < n && s->error == 0) { s->error = EINVAL; }
    }
}

/* ======================================================================== *
 *  the coder on two threads                                                 *
 *  What is serial about the adaptive coder is the model: every symbol       *
 *  changes the weights the next one is judged by.  Turning a symbol into    *
 *  bits only needs the code tables, and those change about once per 2700    *
 *  symbols.  So the model of both trees runs ahead on a thread of its own   *
 *  (blocks, walks, exact reorderings, insertions -- no output) and notes    *
 *  every change of a code in a log, stamped with the index of the first     *
 *  token it applies to; the calling thread follows, keeps its own copy of   *
 *  the code tables current from the log and packs the bits, from one change *
 *  of a code to the next in one go.  Same bytes as code_symbols, by         *
 *  construction: token k is emitted with the codes as they were when the    *
 *  model reached token k.                                                   *
 * ======================================================================== */

struct change { uint64_t at; uint64_t code; uint16_t leaf; uint8_t bits; };   /* leaf | pos_leaf: the distance tree's */

#ifndef SQZ_LOG_SIZE
#define SQZ_LOG_SIZE (1 << 16)        /* a power of two; tests build with a tiny one */
#endif
enum { log_size = SQZ_LOG_SIZE, duo_least = 1 << 16, pos_leaf = 0x8000 };

struct duo {                            /* one cache line per writer: the two threads never share a dirty line */
    struct sqz* s;
    /* written by the emitter, read by the model */
    _Alignas(64) const uint32_t* words; /* the current chunk */
    uint64_t count;
    uint64_t base;                      /* index of its first token in the whole stream */
    _Atomic uint64_t chunks;            /* chunks handed over so far */
    _Atomic int finish;                 /* no more chunks */
    _Alignas(64) _Atomic uint64_t log_head;   /* changes consumed */
    /* written by the model (after every block or one-by-one stretch), read by the emitter */
    _Alignas(64) _Atomic uint64_t modelled;   /* tokens of the current chunk the model is done with */
    _Atomic uint64_t log_tail;          /* changes written */
    int model_error;
    uint64_t model_matches;             /* read after the model thread was joined */
    /* either side gives up (written once) */
    _Alignas(64) _Atomic int stop;
    /* model thread only (written for every token) */
    _Alignas(64) struct watch eyes;
    /* emitter only: changes taken out of the log before they were due (so that the model never waits
     * for room while the emitter waits for the model), and the code tables as of the token being emitted */
    _Alignas(64) struct change* early;
    size_t early_count, early_room, early_next;

    _Alignas(64) struct code_tables tables;
    struct change log[log_size];
};

/* Waiting for the other thread: a short spin (the usual wait is a few hundred nanoseconds), then
 * yields, then sleeps of 20 and finally 200 microseconds -- the model thread waits tens of
 * milliseconds for the GPU search of the next chunk and must not keep a core busy meanwhile. */
static inline void spin_wait(unsigned* spins) {
    const unsigned n = ++*spins;
    if (n <= 2000) {
#if defined(__x86_64__) || defined(__i386__)
        __builtin_ia32_pause();
#endif
    } else if (n <= 2064) {
        sched_yield();
    } else {
        const struct timespec nap = { 0, n <= 2564 ? 20000 : 200000 };
        nanosleep(&nap, NULL);
        if (n > (1u << 30)) { *spins = 2565; }
    }
}

static void segment_note(struct watch* eyes, uint16_t leaf, uint64_t code, uint8_t bits);

static void note_change(struct sqz_tree* t, int32_t leaf) {
    struct watch* const eyes = (struct watch*)t->watcher;
    const uint16_t tagged = (uint16_t)(t->n == sqz_pos_symbols ? leaf | pos_leaf : leaf);
    if (eyes->tables != NULL) {
        tables_set(eyes->tables, t->n == sqz_pos_symbols, (uint32_t)leaf, t->code[leaf], t->bits[leaf]);
        return;
    }
    if (eyes->seg != NULL) {
        segment_note(eyes, tagged, t->code[leaf], t->bits[leaf]);
        return;
    }
    struct duo* d = eyes->d;
    const uint64_t tail = atomic_load_explicit(&d->log_tail, memory_order_relaxed);
    unsigned spins = 0;
    while (tail - atomic_load_explicit(&d->log_head, memory_order_acquire) >= log_size) {
        /* let the emitter come up to this token; once it waits for the model it empties the log */
        atomic_store_explicit(&d->modelled, eyes->k_now, memory_order_release);
        if (atomic_load_explicit(&d->stop, memory_order_relaxed)) { return; }
        spin_wait(&spins);
    }
    struct change* c = &d->log[tail & (log_size - 1)];
    c->at = eyes->now;
    c->code = t->code[leaf];
    c->leaf = tagged;
    c->bits = t->bits[leaf];
    atomic_store_explicit(&d->log_tail, tail + 1, memory_order_release);
}

/* The model's walk over the words [k, until) of a chunk whose first token has the stamp `base`: as
 * blocks where that works, one by one elsewhere (code_symbols without the output).  Returns where
 * it stopped: `until`; or earlier with *flaw = 1 at a word that is no symbol word (not modelled;
 * the emitter reports it when it gets there) or with eyes->error set.                            */
static uint64_t model_words(struct sqz* s, struct tally* y, struct watch* eyes, const uint32_t* words,
                            uint64_t k, uint64_t until, uint64_t base, int* flaw, uint64_t* matches) {
    struct pass p = { s, y, eyes, words, base, NULL, 0, 0 };
    while (k < until && !p.flaw && eyes->error == 0) { k += pass_block(&p, k, until); }
    *flaw = p.flaw;
    *matches += p.matches;
    return k;
}

static void* model_main(void* arg) {
    struct duo* d = (struct duo*)arg;
    struct sqz* const s = d->s;
    struct tally y;
    uint64_t seen = 0;
    unsigned spins = 0;
    tally_init(&y);
    for (;;) {
        while (atomic_load_explicit(&d->chunks, memory_order_acquire) == seen) {
            if (atomic_load_explicit(&d->finish, memory_order_acquire) ||
                atomic_load_explicit(&d->stop, memory_order_relaxed)) { return NULL; }
            spin_wait(&spins);
        }
        seen++;
        spins = 0;
        const uint32_t* const words = d->words;
        const uint64_t count = d->count;
        const uint64_t base = d->base;
        uint64_t k = 0;
        while (k < count) {
            atomic_store_explicit(&d->modelled, k, memory_order_release);
            if (atomic_load_explicit(&d->stop, memory_order_relaxed)) { return NULL; }
            int flaw = 0;
            const uint64_t until = count - k < block_most ? count : k + block_most;
            k = model_words(s, &y, &d->eyes, words, k, until, base, &flaw, &d->model_matches);
            if (flaw) {                                  /* the emitter reports it when it gets there */
                atomic_store_explicit(&d->modelled, k + 1, memory_order_release);
                return NULL;
            }
            if (d->eyes.error != 0) {
                d->model_error = d->eyes.error;
                atomic_store_explicit(&d->stop, 1, memory_order_release);
                return NULL;
            }
        }
        atomic_store_explicit(&d->modelled, count, memory_order_release);
    }
}

static inline void take_change(struct duo* d, const struct change* c) {
    tables_set(&d->tables, (c->leaf & pos_leaf) != 0, c->leaf & (pos_leaf - 1u), c->code, c->bits);
}

/* the emitter's half of one chunk */
static void duo_emit(struct sqz* s, struct duo* d, const uint32_t* words, uint64_t count) {
    struct sqz_bitstream* const bs = s->bs;
    uint64_t head = atomic_load_explicit(&d->log_head, memory_order_relaxed);
    uint64_t tail = atomic_load_explicit(&d->log_tail, memory_order_acquire);
    uint64_t avail = 0;
    unsigned spins = 0;
    const uint64_t base = d->base;
    d->words = words;
    d->count = count;
    atomic_store_explicit(&d->modelled, 0, memory_order_relaxed);
    atomic_fetch_add_explicit(&d->chunks, 1, memory_order_release);

    uint64_t k = 0;
    while (k < count) {
        if (k >= avail) {                            /* wait for the model to be past this token */
            for (;;) {
                avail = atomic_load_explicit(&d->modelled, memory_order_acquire);
                if (avail > k) { break; }
                if (atomic_load_explicit(&d->stop, memory_order_acquire)) {
                    s->error = d->model_error != 0 ? d->model_error : EIO;
                    goto done;
                }
                /* The model may be waiting for room in the log.  Nothing in there is due yet (this token
                 * has not been modelled), so set it aside: the log empties and the model goes on. */
                tail = atomic_load_explicit(&d->log_tail, memory_order_acquire);
                if (head != tail) {
                    if (d->early_next == d->early_count) { d->early_next = d->early_count = 0; }
                    if (d->early_count + (tail - head) > d->early_room) {
                        const size_t room = 2 * (d->early_count + (size_t)(tail - head)) + 1024;
                        struct change* grown = (struct change*)realloc(d->early, room * sizeof(struct change));
                        if (grown == NULL) { s->error = ENOMEM; goto done; }
                        d->early = grown;
                        d->early_room = room;
                    }
                    while (head != tail) { d->early[d->early_count++] = d->log[head++ & (log_size - 1)]; }
                }
                atomic_store_explicit(&d->log_head, head, memory_order_release);   /* everything is taken */
                spin_wait(&spins);
            }
            spins = 0;
            /* everything the model logged for tokens below `avail` is visible from here on */
            tail = atomic_load_explicit(&d->log_tail, memory_order_acquire);
        }
        /* code changes made by tokens before this one: those set aside first, they are older */
        const uint64_t stamp = base + k;
        while (d->early_next != d->early_count && d->early[d->early_next].at <= stamp) {
            take_change(d, &d->early[d->early_next++]);
        }
        while (d->early_next == d->early_count && head != tail && d->log[head & (log_size - 1)].at <= stamp) {
            take_change(d, &d->log[head & (log_size - 1)]);
            head++;
            if ((head & 1023) == 0) { atomic_store_explicit(&d->log_head, head, memory_order_release); }
        }
        /* the tables hold until the next change is due (it applies from token `at - base` on) or the
         * model's progress ends */
        uint64_t until = avail < count ? avail : count;
        if (d->early_next != d->early_count) {
            if (d->early[d->early_next].at - base < until) { until = d->early[d->early_next].at - base; }
        } else if (head != tail) {
            if (d->log[head & (log_size - 1)].at - base < until) { until = d->log[head & (log_size - 1)].at - base; }
        }
        emit_run(&s->error, bs, words, k, until, &d->tables);
        if (s->error != 0) { goto done; }
        k = until;
    }
done:
    atomic_store_explicit(&d->log_head, head, memory_order_release);
    if (s->error != 0) { atomic_store_explicit(&d->stop, 1, memory_order_release); }
    d->base = base + count;
    s->tokens += count;
}

struct duo_run { struct duo* d; pthread_t model; };

/* after coder_begin: start the model thread; 0 when that cannot be had */
static int duo_start(struct sqz* s, struct duo_run* run) {
    run->d = NULL;
    struct duo* d = (struct duo*)aligned_alloc(64, (sizeof(struct duo) + 63) & ~(size_t)63);
    if (d == NULL) { return 0; }                    /* no memory for the log: one thread will do */
    memset(d, 0, sizeof(struct duo));
    d->s = s;
    tables_from_trees(&d->tables, s);
    d->eyes.d = d;
    s->lit.watcher = s->pos.watcher = &d->eyes;
    if (pthread_create(&run->model, NULL, model_main, d) != 0) {
        s->lit.watcher = s->pos.watcher = NULL;
        free(d);
        return 0;
    }
    run->d = d;
    return 1;
}

static void duo_finish(struct sqz* s, struct duo_run* run) {
    if (run->d == NULL) { return; }
    atomic_store_explicit(&run->d->finish, 1, memory_order_release);
    pthread_join(run->model, NULL);
    s->matches += run->d->model_matches;
    s->lit.watcher = s->pos.watcher = NULL;
    free(run->d->early);
    free(run->d);
    run->d = NULL;
}

/* ======================================================================== *
 *  the coder on several threads                                             *
 *  With blocks the model needs less time per token than the emitter, and    *
 *  emitting is only serial in where the bits go.  So for coder_threads >= 3 *
 *  the model cuts the stream into segments (seg_tokens tokens; shorter at a *
 *  chunk's end or when a segment's changes pile up), gives each the code    *
 *  tables as they stand at its first token and the list of changes made     *
 *  while it modelled the segment, and publishes it; coder_threads - 1       *
 *  emitter threads take segments in turn and emit each into a buffer of its *
 *  own, starting at bit 0; the calling thread appends the buffers in order  *
 *  to the caller's bitstream, shifted to where the bits belong.  Same bytes *
 *  by construction: a token's bits are those of the codes the model had     *
 *  when it reached the token, and they land behind the previous token's.    *
 * ======================================================================== */

enum { seg_tokens = 1 << 14,
       seg_out_room = 24 * seg_tokens + 64,  /* a token is at most 63 + 9 + 5 + 63 + 5 + 13 bits */
       seg_changes_most = 1 << 18,           /* a segment ends early beyond this many changes */
       crew_most = 7,                        /* emitter threads */
       crew_least = 1 << 20 };               /* tokens from which the automatic choice takes a crew */

struct segment {
    /* the model's, until `modelled` passes the segment; then read by one emitter */
    const uint32_t* words;              /* the chunk */
    uint64_t from, until;               /* the segment's tokens within it */
    struct change* log;                 /* `at` = index within the chunk of the first token a change applies to */
    size_t log_count, log_room;
    uint64_t lit_code[sqz_lit_symbols]; /* the codes as they stand at `from` */
    uint64_t pos_code[sqz_pos_symbols];
    uint8_t lit_bits[sqz_lit_symbols];
    uint8_t pos_bits[sqz_pos_symbols];
    /* the emitter's, until `emitted` names the segment; then read by the calling thread */
    uint8_t* out;                       /* whole 64-bit words, big-endian */
    uint64_t out_bytes;
    uint64_t tail;                      /* and the bits that did not fill a word */
    int32_t tail_bits;
    int32_t error;
    _Alignas(64) _Atomic uint64_t emitted;   /* number of the segment + 1 */
};

struct crew {
    struct sqz* s;
    int emitters, ring, threads_up;
    pthread_t model;
    pthread_t emitter[crew_most];
    struct segment* seg;                /* [ring] */
    struct watch eyes;                  /* the model's */
    int model_error;
    uint64_t model_matches;             /* read after the model thread was joined */
    /* the calling thread -> the model */
    _Alignas(64) const uint32_t* words;
    uint64_t count;
    _Atomic uint64_t chunks;
    _Atomic int finish;
    _Alignas(64) _Atomic uint64_t merged;     /* segments appended to the bitstream: their slots are free */
    /* the model -> the emitters */
    _Alignas(64) _Atomic uint64_t modelled;   /* segments published */
    /* the emitters among themselves */
    _Alignas(64) _Atomic uint64_t next;       /* the next segment to take */
    /* anybody gives up (written once) */
    _Alignas(64) _Atomic int stop;
};

static void segment_note(struct watch* eyes, uint16_t leaf, uint64_t code, uint8_t bits) {
    struct segment* const g = eyes->seg;
    if (g->log_count == g->log_room) {
        const size_t room = g->log_room == 0 ? 1024 : 2 * g->log_room;
        struct change* grown = (struct change*)realloc(g->log, room * sizeof(struct change));
        if (grown == NULL) { eyes->error = ENOMEM; return; }
        g->log = grown;
        g->log_room = room;
    }
    struct change* c = &g->log[g->log_count++];
    c->at = eyes->now;
    c->code = code;
    c->leaf = leaf;
    c->bits = bits;
}

static void* crew_model_main(void* arg) {
    struct crew* c = (struct crew*)arg;
    struct sqz* const s = c->s;
    struct tally y;
    uint64_t seen = 0, published = 0;
    unsigned spins = 0;
    tally_init(&y);
    for (;;) {
        while (atomic_load_explicit(&c->chunks, memory_order_acquire) == seen) {
            if (atomic_load_explicit(&c->finish, memory_order_acquire) ||
                atomic_load_explicit(&c->stop, memory_order_relaxed)) { return NULL; }
            spin_wait(&spins);
        }
        seen++;
        spins = 0;
        const uint32_t* const words = c->words;
        const uint64_t count = c->count;
        uint64_t k = 0;
        while (k < count) {
            while (published - atomic_load_explicit(&c->merged, memory_order_acquire) >= (uint64_t)c->ring) {
                if (atomic_load_explicit(&c->stop, memory_order_relaxed)) { return NULL; }
                spin_wait(&spins);                   /* every slot holds a segment on its way */
            }
            spins = 0;
            struct segment* const g = &c->seg[published % (uint64_t)c->ring];
            g->words = words;
            g->from = k;
            g->log_count = 0;
            memcpy(g->lit_code, s->lit.code, sizeof(g->lit_code));
            memcpy(g->pos_code, s->pos.code, sizeof(g->pos_code));
            memcpy(g->lit_bits, s->lit.bits, sizeof(g->lit_bits));
            memcpy(g->pos_bits, s->pos.bits, sizeof(g->pos_bits));
            c->eyes.seg = g;
            const uint64_t end = count - k < seg_tokens ? count : k + seg_tokens;
            int flaw = 0;
            while (k < end && !flaw && g->log_count <= seg_changes_most) {
                const uint64_t until = end - k < block_most ? end : k + block_most;
                k = model_words(s, &y, &c->eyes, words, k, until, 0, &flaw, &c->model_matches);
                if (c->eyes.error != 0) {
                    c->model_error = c->eyes.error;
                    atomic_store_explicit(&c->stop, 1, memory_order_release);
                    return NULL;
                }
            }
            g->until = flaw ? k + 1 : k;             /* a word that is no symbol word: its emitter reports it */
            published++;
            atomic_store_explicit(&c->modelled, published, memory_order_release);
            if (flaw) { return NULL; }
        }
    }
}

/* one segment into its buffer: the codes as they were at its start, each change from the token on
 * that it applies to */
static void emit_segment(struct segment* g, struct code_tables* ct) {
    struct sqz_bitstream bs;
    memset(&bs, 0, sizeof(bs));
    bs.data = g->out;
    bs.capacity = seg_out_room;
    memset(ct->pos_word, 0, sizeof(ct->pos_word));
    for (uint32_t k = 0; k < sqz_lit_symbols; k++) { tables_set(ct, 0, k, g->lit_code[k], g->lit_bits[k]); }
    for (uint32_t k = 0; k < sqz_pos_symbols; k++) { tables_set(ct, 1, k, g->pos_code[k], g->pos_bits[k]); }
    g->error = 0;
    size_t next = 0;
    uint64_t k = g->from;
    while (k < g->until && g->error == 0) {
        while (next < g->log_count && g->log[next].at <= k) {
            const struct change* ch = &g->log[next++];
            tables_set(ct, (ch->leaf & pos_leaf) != 0, ch->leaf & (pos_leaf - 1u), ch->code, ch->bits);
        }
        const uint64_t until = next < g->log_count && g->log[next].at < g->until ? g->log[next].at : g->until;
        emit_run(&g->error, &bs, g->words, k, until, ct);
        k = until;
    }
    g->out_bytes = bs.bytes;
    g->tail = bs.b64;
    g->tail_bits = bs.bits;
}

static void* crew_emitter_main(void* arg) {
    struct crew* c = (struct crew*)arg;
    struct code_tables* ct = (struct code_tables*)malloc(sizeof(struct code_tables));
    unsigned spins = 0;
    for (;;) {
        const uint64_t j = atomic_fetch_add_explicit(&c->next, 1, memory_order_relaxed);
        while (atomic_load_explicit(&c->modelled, memory_order_acquire) <= j) {
            if (atomic_load_explicit(&c->finish, memory_order_acquire) ||
                atomic_load_explicit(&c->stop, memory_order_relaxed)) { free(ct); return NULL; }
            spin_wait(&spins);
        }
        spins = 0;
        struct segment* const g = &c->seg[j % (uint64_t)c->ring];
        if (ct == NULL) { g->error = ENOMEM; } else { emit_segment(g, ct); }
        atomic_store_explicit(&g->emitted, j + 1, memory_order_release);
    }
}

/* the calling thread's part of one chunk: hand it to the model, append its segments as they come */
static void crew_emit(struct sqz* s, struct crew* c, const uint32_t* words, uint64_t count) {
    struct sqz_bitstream* const bs = s->bs;
    int32_t* const err = &s->error;
    uint64_t acc = bs->b64;
    uint32_t fill = (uint32_t)bs->bits;
    uint64_t merged = atomic_load_explicit(&c->merged, memory_order_relaxed);
    uint64_t done_tokens = 0;
    unsigned spins = 0;
    if (count == 0 || s->error != 0) { return; }
    c->words = words;
    c->count = count;
    atomic_fetch_add_explicit(&c->chunks, 1, memory_order_release);
    while (done_tokens < count) {
        struct segment* const g = &c->seg[merged % (uint64_t)c->ring];
        while (atomic_load_explicit(&g->emitted, memory_order_acquire) != merged + 1) {
            if (atomic_load_explicit(&c->stop, memory_order_acquire)) {
                s->error = c->model_error != 0 ? c->model_error : EIO;
                goto done;
            }
            spin_wait(&spins);
        }
        spins = 0;
        if (g->error != 0) { s->error = g->error; goto done; }
        for (uint64_t at = 0; at < g->out_bytes; at += 8) {
            uint64_t be;
            memcpy(&be, g->out + at, 8);
            const uint64_t word = __builtin_bswap64(be);
            SQZ_APPEND(word >> 32, 32);
            SQZ_APPEND(word & 0xFFFFFFFFu, 32);
        }
        if (g->tail_bits > 0) { SQZ_APPEND(g->tail, (uint32_t)g->tail_bits); }
        done_tokens += g->until - g->from;
        merged++;
        atomic_store_explicit(&c->merged, merged, memory_order_release);
    }
done:
    if (s->error != 0) { atomic_store_explicit(&c->stop, 1, memory_order_release); }
    bs->b64 = acc;
    bs->bits = (int32_t)fill;
    s->tokens += count;
}

static void crew_free(struct crew* c) {
    if (c->seg != NULL) {
        for (int k = 0; k < c->ring; k++) { free(c->seg[k].log); free(c->seg[k].out); }
        free(c->seg);
    }
    free(c);
}

static struct crew* crew_start(struct sqz* s, int emitters) {
    struct crew* c = (struct crew*)aligned_alloc(64, (sizeof(struct crew) + 63) & ~(size_t)63);
    if (c == NULL) { return NULL; }
    memset(c, 0, sizeof(struct crew));
    c->s = s;
    c->emitters = emitters < 1 ? 1 : (emitters > crew_most ? crew_most : emitters);
    c->ring = 4 * c->emitters;
    c->seg = (struct segment*)aligned_alloc(64, sizeof(struct segment) * (size_t)c->ring);
    if (c->seg == NULL) { crew_free(c); return NULL; }
    memset(c->seg, 0, sizeof(struct segment) * (size_t)c->ring);
    for (int k = 0; k < c->ring; k++) {
        c->seg[k].out = (uint8_t*)malloc(seg_out_room);
        if (c->seg[k].out == NULL) { crew_free(c); return NULL; }
    }
    s->lit.watcher = s->pos.watcher = &c->eyes;
    if (pthread_create(&c->model, NULL, crew_model_main, c) != 0) {
        s->lit.watcher = s->pos.watcher = NULL;
        crew_free(c);
        return NULL;
    }
    for (int k = 0; k < c->emitters; k++) {
        if (pthread_create(&c->emitter[k], NULL, crew_emitter_main, c) != 0) { break; }
        c->threads_up++;
    }
    if (c->threads_up == 0) {                        /* nobody to emit: not a crew */
        atomic_store_explicit(&c->stop, 1, memory_order_release);
        pthread_join(c->model, NULL);
        s->lit.watcher = s->pos.watcher = NULL;
        crew_free(c);
        return NULL;
    }
    return c;
}

static void crew_finish(struct sqz* s, struct crew* c) {
    atomic_store_explicit(&c->finish, 1, memory_order_release);
    pthread_join(c->model, NULL);
    for (int k = 0; k < c->threads_up; k++) { pthread_join(c->emitter[k], NULL); }
    s->matches += c->model_matches;
    s->lit.watcher = s->pos.watcher = NULL;
    crew_free(c);
}

/* ---- one front for the coders on more than one thread ---- */

struct team { struct duo_run two; struct crew* crew; };

static int host_cores(void) {
    const long n = sysconf(_SC_NPROCESSORS_ONLN);
    return n < 1 ? 1 : (int)n;
}

/* after coder_begin: start the threads coder_threads asks for (0: by the stream's length and the
 * host's cores); 0 = none were started (not wanted, or not to be had), one thread will do */
static int team_size(const struct sqz* s, uint64_t expected_tokens) {
    int threads = s->coder_threads;
    if (threads <= 0) {
        const int cores = host_cores();
        threads = expected_tokens < duo_least || cores < 2 ? 1 :
                  expected_tokens < crew_least || cores < 8 ? 2 : 4;
    }
    return threads;
}

static int team_start(struct sqz* s, struct team* t, uint64_t expected_tokens) {
    t->two.d = NULL;
    t->crew = NULL;
    int threads = team_size(s, expected_tokens);
    if (threads >= 3) {
        t->crew = crew_start(s, threads - 1);
        if (t->crew != NULL) { return 1; }
        threads = 2;
    }
    return threads == 2 ? duo_start(s, &t->two) : 0;
}

static void team_emit(struct sqz* s, struct team* t, const uint32_t* words, uint64_t count) {
    if (t->crew != NULL) { crew_emit(s, t->crew, words, count); } else { duo_emit(s, t->two.d, words, count); }
}

static void team_finish(struct sqz* s, struct team* t) {
    if (t->crew != NULL) { crew_finish(s, t->crew); t->crew = NULL; }
    duo_finish(s, &t->two);
}

void sqz_write_header(struct sqz_bitstream* bs, uint64_t bytes, uint8_t win_bits) {
    if (win_bits < sqz_min_win_bits || win_bits > sqz_max_win_bits) {
        bs->error = EINVAL;
        return;
    }
    put_bits(bs, bytes, 64);
    put_bits(bs, win_bits, 8);
}

void sqz_read_header(struct sqz_bitstream* bs, uint64_t* bytes, uint8_t* win_bits) {
    uint64_t b = get_bits(bs, 64);
    uint64_t w = get_bits(bs, 8);
    if (bs->error != 0) { return; }
    if (w < sqz_min_win_bits || w > sqz_max_win_bits) { bs->error = EINVAL; return; }
    *bytes = b;
    *win_bits = (uint8_t)w;
}

void sqz_encode_tokens(struct sqz* s, struct sqz_bitstream* bs,
                       const uint32_t* tokens, uint64_t count) {
    coder_begin(s, bs);
    double t0 = now_seconds();
    code_tokens(s, tokens, count);
    if (s->error == 0) { pad_to_word(bs); s->error = bs->error; }
    s->entropy_seconds += now_seconds() - t0;
}

void sqz_symbols_of_tokens(const uint32_t* tokens, uint64_t count, uint32_t* words) {
    struct sqz s;                       /* only the length table is used */
    bucket_tables(&s);
    for (uint64_t k = 0; k < count; k++) {
        words[k] = token_is_valid(tokens[k]) ? symbols_of_token(&s, tokens[k]) : 0xFFFFFFFFu;
    }
}

void sqz_encode_symbols(struct sqz* s, struct sqz_bitstream* bs,
                        const uint32_t* words, uint64_t count) {
    coder_begin(s, bs);
    double t0 = now_seconds();
    struct team run;
    if (s->error == 0 && team_start(s, &run, count)) {
        team_emit(s, &run, words, count);
        team_finish(s, &run);
    } else {
        code_symbols(s, words, count);
    }
    if (s->error == 0) { pad_to_word(bs); s->error = bs->error; }
    s->entropy_seconds += now_seconds() - t0;
}

void sqz_encode_symbols_chunked(struct sqz* s, struct sqz_bitstream* bs,
                                const uint32_t* words, uint64_t count, uint64_t chunk) {
    coder_begin(s, bs);
    struct team run;
    const int two = s->error == 0 && team_start(s, &run, count);
    if (chunk == 0) { chunk = count; }
    for (uint64_t at = 0; at < count && s->error == 0; at += chunk) {
        const uint64_t n = count - at < chunk ? count - at : chunk;
        if (two) { team_emit(s, &run, words + at, n); } else { code_symbols(s, words + at, n); }
    }
    if (two) { team_finish(s, &run); }
    if (s->error == 0) { pad_to_word(bs); s->error = bs->error; }
}

void sqz_compress(struct sqz* s, struct sqz_bitstream* bs,
                  const uint8_t* data, uint64_t bytes, uint32_t window) {
    if (window < (1u << sqz_min_win_bits) || window > (1u << sqz_max_win_bits) ||
        (window & (window - 1)) != 0 || (s->lazy != 0 && s->lazy != 1) ||
        (s->mincost != 0 && s->mincost != 1) || (s->lazy == 1 && s->mincost == 1)) {
        s->error = EINVAL;
        return;
    }
    coder_begin(s, bs);
    if (s->error != 0) { return; }
    /* The GPU produces the token stream (greedy, lazy or min-cost) chunk by chunk, as symbol words;
     * while the host entropy-codes chunk k the device already searches chunk k+1. */
    sqz_gpu_stream* st = NULL;
    double t_search = 0, t_code = 0, t0 = now_seconds();
    /* The stream's own chunking (2, 4, 8, 16, then 32 MiB) suits a coder that is slower than the search:
     * it starts after milliseconds.  A crew is faster than the search; then what counts is that the
     * device works on chunks of a size it is efficient at: a quarter of the input each, between 4 and
     * 32 MiB, the first two shorter (the coder's first tokens are its slowest: every symbol is new). */
    size_t chunk = 0;
    if (team_size(s, bytes / 2) >= 3) {
        const uint64_t quarter = ((bytes / 4) | 0xFFFFF) + 1;
        chunk = (size_t)(quarter < ((uint64_t)4 << 20) ? (uint64_t)4 << 20 :
                         quarter > ((uint64_t)32 << 20) ? (uint64_t)32 << 20 : quarter);
    }
    int r = sqz_gpu_stream_open(&st, s->device, data, (size_t)bytes, window,
                                sqz_min_len, sqz_max_len, window - 1, chunk,
                                SQZ_GPU_STREAM_SYMBOLS | (chunk != 0 ? SQZ_GPU_STREAM_SHORT_START : 0) |
                                (s->lazy == 1 ? SQZ_GPU_STREAM_LAZY : 0) |
                                (s->mincost == 1 ? SQZ_GPU_STREAM_MINCOST : 0));
    t_search += now_seconds() - t0;
    if (r != 0) { s->error = r; return; }
    struct team run;
    const int two = team_start(s, &run, bytes / 2);    /* about 0.6 tokens per byte on mixed data */
    const int trace = getenv("SQZ_TRACE") != NULL;     /* per-chunk times on stderr */
    const double t_begin = t0;
    if (trace) { fprintf(stderr, "sqz_compress: open + team %.1f ms\n", 1e3 * (now_seconds() - t_begin)); }
    for (;;) {
        const uint32_t* words = NULL;
        size_t count = 0;
        t0 = now_seconds();
        r = sqz_gpu_stream_next(st, &words, &count);
        const double t1 = now_seconds();
        t_search += t1 - t0;
        if (r != 0) { s->error = r; break; }
        if (count == 0) { break; }
        if (two) { team_emit(s, &run, words, count); } else { code_symbols(s, words, count); }
        const double t2 = now_seconds();
        t_code += t2 - t1;
        if (trace) {
            fprintf(stderr, "sqz_compress: at %.1f ms: waited %.1f ms, coded %zu tokens in %.1f ms\n",
                    1e3 * (t0 - t_begin), 1e3 * (t1 - t0), count, 1e3 * (t2 - t1));
        }
        if (s->error != 0) { break; }
    }
    t0 = now_seconds();
    if (two) { team_finish(s, &run); }
    sqz_gpu_stream_close(st);
    if (trace) { fprintf(stderr, "sqz_compress: close %.1f ms, all %.1f ms\n", 1e3 * (now_seconds() - t0), 1e3 * (now_seconds() - t_begin)); }
    if (s->error == 0) { pad_to_word(bs); s->error = bs->error; }
    s->search_seconds = t_search;
    s->entropy_seconds = t_code;
}

/* ======================================================================== *
 *  decompressor  (reference squeeze.h:411-551); never touches the GPU       *
 * ======================================================================== */

/* The decoder reads through a window of its own: `acc` holds the next `have`
 * bits of the stream left-aligned, topped up from `pend`, the unread rest of
 * the last 64-bit word taken from the bitstream.  A word is taken when fewer
 * than 32 bits are at hand, i.e. up to 31 bits before the reference would
 * take it (bitstream.h:65-95); running dry there is only an error once bits
 * that are not there are consumed.                                           */
struct window {
    struct sqz_bitstream* bs;
    uint64_t acc, pend;
    int32_t have, pend_bits;
    int32_t dry;                        /* errno met while reading ahead */
    int32_t bad;                        /* errno of the stream: bits consumed that are not there, a code that leads nowhere */
};

static inline void window_fill(struct window* w) {
    if (w->have >= 32) { return; }
    if (w->pend_bits == 0 && w->dry == 0) {
        struct sqz_bitstream* const bs = w->bs;
        if (bs->data != NULL && bs->bytes >= 8 && bs->read <= bs->bytes - 8) {    /* memory source: one big-endian load */
            uint64_t be;
            memcpy(&be, bs->data + bs->read, 8);
            bs->read += 8;
            w->pend = __builtin_bswap64(be);
            w->pend_bits = 64;
        } else {
            word_in(bs);
            if (bs->error != 0) { w->dry = bs->error; bs->error = 0; }
            else { w->pend = bs->b64; w->pend_bits = 64; }
        }
        bs->bits = 0;
    }
    if (w->pend_bits > 0) {
        const int32_t room = 64 - w->have;
        const int32_t take = room < w->pend_bits ? room : w->pend_bits;
        w->acc |= w->pend >> w->have;
        w->pend = take == 64 ? 0 : w->pend << take;
        w->pend_bits -= take;
        w->have += take;
    }
}

/* drop `count` bits; 0 when they were not all there.  The window keeps the error to itself (`bad`):
 * the decode loop looks at it once per token instead of reading s->error back after every field. */
static inline int window_skip(struct window* w, int32_t count) {
    if (count > w->have) { w->bad = w->dry != 0 ? w->dry : E2BIG; return 0; }
    w->acc <<= count;
    w->have -= count;
    return 1;
}

/* `count` <= 16 raw bits, first bit = least significant (bitstream.h:97-110) */
static inline uint32_t window_bits(struct window* w, int32_t count) {
    window_fill(w);
    const uint32_t top = (uint32_t)(w->acc >> 48);          /* the next 16 bits */
    const uint32_t v = reverse_field(top, 16) & ((1u << count) - 1);
    return window_skip(w, count) ? v : 0;
}

static inline int32_t window_symbol(struct window* w, struct sqz_tree* t,
                                    const int lut_bits, const int usual) {  /* squeeze.h:429-442 */
    window_fill(w);
    const uint32_t entry = t->lut[w->acc >> (64 - lut_bits)];   /* one lookup walks lut_bits levels */
    if (entry == no_node) { w->bad = EINVAL; return -1; }
    int32_t i = (int32_t)(entry & ((1u << lut_node_bits) - 1));
    if (!window_skip(w, (int32_t)(entry >> lut_node_bits))) { return -1; }
    while (i >= t->n) {                              /* a longer code: leaves are the nodes below n */
        window_fill(w);
        const int bit = (int)(w->acc >> 63);
        if (!window_skip(w, 1)) { return -1; }
        i = bit ? t->hi[i] : t->lo[i];
        if (i < 0) { w->bad = EINVAL; return -1; }
    }
    tree_count_as(t, i, usual);
    SQZ_CHECK(t);
    return i;
}

/* the 57 bits (at least) that follow bit `bit` of a memory source, at the top of the result */
static inline uint64_t peek_bits(const uint8_t* src, uint64_t bit) {
    uint64_t be;
    memcpy(&be, src + (bit >> 3), 8);
    return __builtin_bswap64(be) << (bit & 7);
}

/* data != NULL: execute the tokens (squeeze.h:502-551); tokens != NULL: hand them out */
static void decode_stream(struct sqz* s, struct sqz_bitstream* bs, uint8_t* data, uint64_t bytes,
                          uint32_t* tokens, uint64_t cap, uint64_t* count) {
    uint64_t n_tokens = 0;
    s->lit.lut = s->lit_lut;
    s->pos.lut = s->pos_lut;
    memset(s->lit_lut, 0xFF, sizeof(s->lit_lut));
    memset(s->pos_lut, 0xFF, sizeof(s->pos_lut));
    coder_begin(s, bs);
    if (bs->error != 0) { s->error = bs->error; }
    struct window w = { bs, bs->bits > 0 ? bs->b64 : 0, 0, bs->bits, 0, 0, 0 };
    struct sqz_tree* const lit = &s->lit;
    struct sqz_tree* const pos = &s->pos;
    uint64_t i = 0;
    int err = s->error;
    while (i < bytes && err == 0) {
        /* Memory sources, away from the end of the stream: tokens of symbols seen before are read
         * straight from the bytes -- the stream is big-endian words of first-bit-highest bits, so
         * the next 57 bits are one unaligned load and one shift, and where a token ends is a bit
         * count, no reader state.  Anything else (an escape, a code that leads nowhere, a token that
         * does not fit, the last bytes of the stream) is left to the window reader below, token by
         * token, which reports it the reference's way; nothing of such a token is counted here.   */
        if (bs->data != NULL && w.dry == 0 && bs->bytes >= 64) {
            const uint8_t* const src = bs->data;
            const uint64_t last_start = 8 * (bs->bytes - 24);          /* two 8-byte loads per token at most */
            uint64_t at = 8 * bs->read - (uint64_t)(w.have + w.pend_bits);
            const uint64_t at_first = at;
#define SQZ_PEEK(bit_) peek_bits(src, (bit_))
            while (i < bytes && at <= last_start) {
                uint64_t peek = SQZ_PEEK(at);
                const uint32_t entry = lit->lut[peek >> (64 - lit_lut_bits)];
                if (entry == no_node) { break; }
                int32_t node = (int32_t)(entry & ((1u << lut_node_bits) - 1));
                uint32_t nb = entry >> lut_node_bits;
                while (node >= lit->n && nb < 48) {                     /* a longer code */
                    node = (peek << nb) >> 63 ? lit->hi[node] : lit->lo[node];
                    nb++;
                    if (node < 0) { break; }
                }
                if (node < 0 || node >= lit->n) { break; }
                if (node <= 0xFF) {                                     /* a literal seen before: the common case */
                    at += nb;
                    tree_count_as(lit, node, lit_plan);
                    SQZ_CHECK(lit);
                    if (data != NULL) { data[i] = (uint8_t)node; }
                    if (n_tokens < cap) { tokens[n_tokens] = (uint32_t)node; }
                    n_tokens++;
                    i++;
                    continue;
                }
                const int32_t b = node - len_symbol0;
                if (b < 0 || b >= 28) { break; }                        /* 256, the escape */
                const uint64_t rest = at + nb;
                peek = SQZ_PEEK(rest);
                uint32_t used = len_extra[b];
                const uint32_t len = len_base[b] + (used > 0 ? reverse_field((uint32_t)(peek >> (64 - used)), used) : 0);
                if (len > sqz_max_len) { break; }
                const uint32_t far_entry = pos->lut[(peek << used) >> (64 - pos_lut_bits)];
                if (far_entry == no_node) { break; }
                int32_t far = (int32_t)(far_entry & ((1u << lut_node_bits) - 1));
                used += far_entry >> lut_node_bits;
                while (far >= pos->n && used < 44) {
                    far = (peek << used) >> 63 ? pos->hi[far] : pos->lo[far];
                    used++;
                    if (far < 0) { break; }
                }
                if (far < 0 || far >= 30) { break; }                    /* the escape, no symbol */
                const uint32_t more = pos_extra[far];
                const uint32_t dist = pos_base[far] +
                                      (more > 0 ? reverse_field((uint32_t)((peek << used) >> (64 - more)), more) : 0);
                used += more;
                if (dist > 0x7FFF || dist > i || len > bytes - i) { break; }
                at = rest + used;
                tree_count_as(lit, node, lit_plan);
                SQZ_CHECK(lit);
                tree_count_as(pos, far, pos_plan);
                SQZ_CHECK(pos);
                if (data != NULL) {
                    uint8_t* to = data + i;
                    const uint8_t* from = to - dist;
                    if (dist >= len)    { memcpy(to, from, len); }
                    else if (dist == 1) { memset(to, from[0], len); }
                    else                { for (uint32_t k = 0; k < len; k++) { to[k] = from[k]; } }
                }
                if (n_tokens < cap) { tokens[n_tokens] = len << 16 | dist; }
                n_tokens++;
                i += len;
            }
#undef SQZ_PEEK
            if (at != at_first) {                                       /* the window reader goes on from bit `at` */
                bs->read = 8 * (at / 64);
                w.acc = w.pend = 0;
                w.have = w.pend_bits = 0;
                for (uint32_t skip = (uint32_t)(at % 64); skip > 0; ) {
                    window_fill(&w);
                    const int32_t take = skip < 16 ? (int32_t)skip : 16;   /* like every field: window_fill relies on it */
                    if (!window_skip(&w, take)) { break; }
                    skip -= (uint32_t)take;
                }
            }
            if (i >= bytes) { break; }
        }
        int32_t sym = window_symbol(&w, lit, lit_lut_bits, lit_plan);
        if (sym <= 0xFF && sym >= 0) {                              /* a literal seen before: the common case */
            if (data != NULL) { data[i] = (uint8_t)sym; }
            if (n_tokens < cap) { tokens[n_tokens] = (uint32_t)sym; }
            n_tokens++;
            i++;
            continue;
        }
        if (w.bad != 0) { err = w.bad; break; }
        if (sym == sqz_lit_nyt) {
            sym = (int32_t)window_bits(&w, 9);
            if (w.bad != 0) { err = w.bad; break; }
            if (lit->up[sym] >= 0) { err = EINVAL; break; }         /* already known */
            if (!tree_insert(lit, sym)) { err = E2BIG; break; }
            SQZ_CHECK(lit);
            if (sym <= 0xFF) {
                if (data != NULL) { data[i] = (uint8_t)sym; }
                if (n_tokens < cap) { tokens[n_tokens] = (uint32_t)sym; }
                n_tokens++;
                i++;
                continue;
            }
        }
        const int32_t b = sym - len_symbol0;
        if (b < 0 || b >= 28) { err = EINVAL; break; }
        uint32_t len = len_base[b];
        if (len_extra[b] > 0) { len += window_bits(&w, len_extra[b]); }
        if (len < sqz_min_len || len > sqz_max_len) { err = w.bad != 0 ? w.bad : EINVAL; break; }
        int32_t pb = window_symbol(&w, pos, pos_lut_bits, pos_plan);
        if (w.bad != 0) { err = w.bad; break; }
        if (pb == sqz_pos_nyt) {
            pb = (int32_t)window_bits(&w, 5);
            if (w.bad != 0) { err = w.bad; break; }
            if (pb >= 30 || pos->up[pb] >= 0) { err = EINVAL; break; }
            if (!tree_insert(pos, pb)) { err = E2BIG; break; }
            SQZ_CHECK(pos);
        }
        if (pb >= 30) { err = EINVAL; break; }
        uint32_t dist = pos_base[pb];
        if (pos_extra[pb] > 0) { dist += window_bits(&w, pos_extra[pb]); }
        if (w.bad != 0) { err = w.bad; break; }
        if (dist == 0 || dist > 0x7FFF || dist > i || len > bytes - i) { err = EINVAL; break; }
        /* squeeze.h:533-539 copies byte by byte because the source may overlap the
         * destination; the result is the same as these three cases */
        if (data != NULL) {
            uint8_t* to = data + i;
            const uint8_t* from = to - dist;
            if (dist >= len)    { memcpy(to, from, len); }
            else if (dist == 1) { memset(to, from[0], len); }
            else                { for (uint32_t k = 0; k < len; k++) { to[k] = from[k]; } }
        }
        if (n_tokens < cap) { tokens[n_tokens] = len << 16 | dist; }
        n_tokens++;
        i += len;
    }
    if (err != 0 && s->error == 0) { s->error = err; }
    if (count != NULL) { *count = n_tokens; }
    if (tokens != NULL && n_tokens > cap && s->error == 0) { s->error = E2BIG; }
    /* Leave the bitstream where the reference's bit-at-a-time reader would stand
     * (bitstream.h:65-95): it has taken ceil(consumed / 64) words, and the rest of the last one
     * is in b64.  The window reads ahead, so up to one whole word may have to go back: in memory
     * mode `read` is rewound; a callback source cannot take a word back, there the bits of that
     * word are lost to a caller who keeps reading from the same bitstream (see sqz.h). */
    {
        const int32_t unread = w.have + w.pend_bits;            /* < 96 */
        const int32_t rest = unread & 63;                       /* bits of the word the reference is in */
        if (unread >= 64) {
            bs->b64 = rest > 0 ? w.acc & ~(~(uint64_t)0 >> rest) : 0;
            bs->bits = rest;
            if (bs->data != NULL && bs->read >= 8) { bs->read -= 8; }
        } else {
            bs->b64 = w.acc | (w.have < 64 ? w.pend >> w.have : 0);
            bs->bits = unread;
        }
    }
    if (s->error != 0 && bs->error == 0) { bs->error = s->error; }
}

void sqz_decompress(struct sqz* s, struct sqz_bitstream* bs,
                    uint8_t* data, uint64_t bytes) {
    decode_stream(s, bs, data, bytes, NULL, 0, NULL);
}

void sqz_decode_tokens(struct sqz* s, struct sqz_bitstream* bs, uint64_t bytes,
                       uint32_t* tokens, uint64_t cap, uint64_t* count) {
    decode_stream(s, bs, NULL, bytes, tokens, tokens != NULL ? cap : 0, count);
}

/* ---- whole-buffer conveniences ----------------------------------------- */

#include <stdlib.h>

void sqz_decompress_gpu(struct sqz* s, struct sqz_bitstream* bs,
                        uint8_t* data, uint64_t bytes) {
    if (bytes >= ((uint64_t)1 << 31)) { s->error = EINVAL; return; }
    uint32_t* tokens = (uint32_t*)malloc((size_t)(bytes > 0 ? bytes : 1) * 4);   /* at most one token per byte */
    if (tokens == NULL) { s->error = ENOMEM; return; }
    uint64_t count = 0;
    double t0 = now_seconds();
    sqz_decode_tokens(s, bs, bytes, tokens, bytes, &count);
    s->entropy_seconds = now_seconds() - t0;
    if (s->error == 0) {
        t0 = now_seconds();
        s->error = sqz_gpu_expand_tokens(tokens, (size_t)count, data, (size_t)bytes);
        s->search_seconds = now_seconds() - t0;
    }
    s->tokens = count;
    free(tokens);
}

static struct sqz* state_new(void);
static void state_free(struct sqz* s);
static struct sqz* state_new(void) { return (struct sqz*)malloc(sizeof(struct sqz)); }
static void state_free(struct sqz* s) { free(s); }

int sqz_compress_buffer(const uint8_t* data, uint64_t bytes, uint8_t win_bits,
                        uint8_t* out, uint64_t capacity, uint64_t* written) {
    struct sqz_bitstream bs;
    memset(&bs, 0, sizeof(bs));
    bs.data = out;
    bs.capacity = capacity;
    sqz_write_header(&bs, bytes, win_bits);
    if (bs.error != 0) { return bs.error; }
    struct sqz* s = state_new();
    if (s == NULL) { return ENOMEM; }
    sqz_init(s);
    sqz_compress(s, &bs, data, bytes, 1u << win_bits);
    int r = s->error;
    if (written != NULL) { *written = bs.bytes; }
    state_free(s);
    return r;
}

int sqz_decompress_buffer(const uint8_t* comp, uint64_t comp_bytes,
                          uint8_t* out, uint64_t capacity, uint64_t* bytes) {
    struct sqz_bitstream bs;
    memset(&bs, 0, sizeof(bs));
    bs.data = (uint8_t*)comp;
    bs.capacity = comp_bytes;
    bs.bytes = comp_bytes;
    uint64_t n = 0;
    uint8_t wb = 0;
    sqz_read_header(&bs, &n, &wb);
    if (bs.error != 0) { return bs.error; }
    if (n > capacity) { return E2BIG; }
    struct sqz* s = state_new();
    if (s == NULL) { return ENOMEM; }
    sqz_init(s);
    sqz_decompress(s, &bs, out, n);
    int r = s->error;
    if (bytes != NULL) { *bytes = n; }
    state_free(s);
    return r;
}
