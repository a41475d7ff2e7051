/* include/sqz.h -- host codec API of sqz-b200 (C99, callable from C and C++).
 *
 * Drop-in for the reference's Huffman + LZ77 codec
 * (/root/reference/attic/map_experiment/squeeze.h:109-125,557-565, the
 * `squeeze_interface squeeze` vtable; names follow the sqz_* spelling of
 * /root/reference/shl/README.md:31-63).  Same bitstream, same header, same
 * sticky-errno error model, caller-owned buffers.  The one thing that changed:
 * sqz_compress() obtains the LZ77 token stream from the GPU
 * (include/sqz_gpu.h: sqz_gpu_tokens) instead of running the brute-force loop
 * of squeeze.h:338-358 on the CPU.  There is no CPU fallback for the search:
 * without a CUDA device sqz_compress() sets s->error = ENODEV.
 *
 *   reference                                  this library
 *   squeeze.write_header(bs, bytes, win_bits)  sqz_write_header   squeeze.h:255-265
 *   squeeze.alloc(0) / init_with / free        sqz_init (caller-owned struct, no heap)
 *   squeeze.compress(s, bs, data, bytes, win)  sqz_compress       squeeze.h:319-409
 *   squeeze.read_header(bs, &bytes, &win_bits) sqz_read_header    squeeze.h:444-456
 *   squeeze.decompress(s, bs, data, bytes)     sqz_decompress     squeeze.h:502-551
 *   struct bitstream                           struct sqz_bitstream  bitstream.h:7-18
 */
#ifndef SQZ_H_INCLUDED
#define SQZ_H_INCLUDED

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

enum {
    sqz_min_win_bits = 10,   /* squeeze.h:19 */
    sqz_max_win_bits = 15,   /* squeeze.h:20 */
    sqz_min_len      = 3,    /* squeeze.h:13 */
    sqz_max_len      = 257,  /* squeeze.h:15 */
    sqz_lit_symbols  = 512,  /* squeeze.h:204: 0..255 bytes, 257..284 lengths, 285 NYT */
    sqz_pos_symbols  = 32,   /* squeeze.h:205: 0..29 distance buckets, 30 NYT */
    sqz_lit_nyt      = 285,  /* squeeze.h:23 */
    sqz_pos_nyt      = 30    /* squeeze.h:24 */
};

/* Bit sink / source.  Either memory mode {data, capacity} (words stored
 * big-endian, bitstream.h:36-42) or callback mode {stream, output/input}: the
 * callback moves the 8 bytes at &b64 in host byte order (bitstream.h:44-47,
 * attic/map_experiment/test.c:39-42).  A memory-mode READER must set `bytes`
 * to the number of valid bytes in `data` (bitstream.h:70-74).                */
struct sqz_bitstream {
    void*    stream;
    uint8_t* data;
    uint64_t capacity;
    uint64_t bytes;     /* bytes written */
    uint64_t read;      /* bytes read */
    uint64_t b64;       /* shift register */
    int32_t  bits;      /* bits held in b64 */
    int32_t  error;     /* sticky errno */
    int    (*output)(struct sqz_bitstream* bs);
    int    (*input)(struct sqz_bitstream* bs);
};

/* One adaptive-Huffman tree (huffman.h:13-34) as a structure of arrays with
 * 16-bit links.  Node k: leaves 0..n-1 (index == symbol), root 2n-2, internal
 * nodes handed out downward from 2n-3.  freq[] has ten extra entries:
 * freq[2n-1] = 0 and freq[2n] = 2^63-1, the comparators "always" and "never"
 * of the plans, and eight spare slots that pad a plan (sqz_codec.c).  The
 * root's own weight is only kept up to date by the exact walk.              */
struct sqz_tree {
    uint64_t* freq;     /* weights */
    uint64_t* path;     /* code, emitted LSB first (huffman.h:16) */
    uint64_t* code;     /* leaves only: the same code in emission order */
    int16_t*  up;       /* parent, -1 = none */
    int16_t*  lo;       /* left child  (bit 0) */
    int16_t*  hi;       /* right child (bit 1) */
    uint16_t* plan;     /* per leaf 16 nodes (leaf to root) + their 16 comparators: one cache line */
    uint8_t*  steps;    /* per leaf: plan length; 0 = no plan yet, 255 = deeper than a plan */
    uint8_t*  bits;     /* code length; 0 = root or unseen leaf */
    void*     watcher;  /* two-thread coder only: where the model thread logs code changes */
    uint16_t* lut;      /* decoder only: node reached by the next lut_bits bits of the stream */
    int32_t lut_bits;
    int32_t n;          /* leaves; nodes = 2n-1 */
    int32_t next;       /* internal nodes are handed out downward from here */
    int32_t depth;      /* high-water mark, reset by a root-level relabel */
    int32_t complete;   /* frozen: no more frequency updates */
    int32_t lazy;       /* symbols that may still be coded without touching the top internal nodes */
    int32_t lazy_start; /* value of `lazy` when the top internal nodes were last exact */
    int32_t eager;      /* symbols left to code with full walks before the top is looked at again */
};

#define SQZ_TREE_STORE(N) struct {                                          \
    uint16_t plan[N][32];                                                     \
    uint64_t freq[2 * (N) + 9]; uint64_t path[2 * (N) - 1]; uint64_t code[N]; \
    int16_t up[2 * (N) - 1]; int16_t lo[2 * (N) - 1]; int16_t hi[2 * (N) - 1]; \
    uint8_t steps[N]; uint8_t bits[2 * (N) - 1]; }

struct sqz {
    int32_t error;      /* sticky errno: E2BIG, EINVAL, ENODEV, ENOMEM, EIO */
    int32_t device;     /* CUDA device for the match search; -1 (default) = the current one */
    struct sqz_bitstream* bs;
    /* statistics of the last sqz_compress (zero until then) */
    uint64_t tokens;
    uint64_t matches;
    double   search_seconds;            /* GPU search + parse + copies */
    double   entropy_seconds;           /* host adaptive-Huffman stage */
    int32_t  coder_threads;             /* 1 = one thread; 2 = the model of both trees on a thread of its own, the
                                           caller's thread packs the bits; n >= 3 = model thread + n - 1 emitter
                                           threads working on segments + the caller's thread appending them in
                                           order; 0 = automatic (1 below 64 Ki tokens, 2 below 1 Mi tokens or on
                                           fewer than 8 cores, else 4); same bytes in every case (sqz_codec.c) */
    int32_t  lazy;                      /* sqz_compress's parse: 0 (sqz_init) = greedy, the reference's exact
                                           stream; 1 = lazy matching (SQZ_GPU_STREAM_LAZY in sqz_gpu.h): about
                                           2 % smaller on text and code, slightly larger on data that does not
                                           compress, read by every decoder; other values: EINVAL */
    struct sqz_tree lit;
    uint8_t len_index[sqz_max_len + 2]; /* len -> length bucket, squeeze.h:151-161.  Also keeps the two tree
                                           headers on different cache lines: with two coder threads each
                                           tree's counters are written by another thread for every token */
    int32_t mincost;                    /* sqz_compress's parse: 0 (sqz_init) = as `lazy` says; 1 = the min-cost
                                           parse (SQZ_GPU_STREAM_MINCOST in sqz_gpu.h): 3-5 % smaller than greedy
                                           on text and code, the same on data that does not compress, read by
                                           every decoder; other values, and 1 with lazy = 1: EINVAL.  (It takes
                                           the first four bytes of what was apart[64]: same size and offsets.) */
    uint8_t apart[60];
    struct sqz_tree pos;
    SQZ_TREE_STORE(sqz_lit_symbols) lit_store;
    SQZ_TREE_STORE(sqz_pos_symbols) pos_store;
    uint16_t lit_lut[1 << 10];          /* decoder look-ahead tables (sqz_codec.c: lit_lut_bits, pos_lut_bits) */
    uint16_t pos_lut[1 << 6];
};

/* 64 raw bits of `bytes` then 8 raw bits of `win_bits`, each LSB first.
 * win_bits outside [10,15] sets bs->error = EINVAL.                          */
void sqz_write_header(struct sqz_bitstream* bs, uint64_t bytes, uint8_t win_bits);
void sqz_read_header(struct sqz_bitstream* bs, uint64_t* bytes, uint8_t* win_bits);

/* Fresh state; must be called before every sqz_compress / sqz_decompress
 * (a state is single use, like the reference's squeeze_type).               */
void sqz_init(struct sqz* s);

/* LZ77 (GPU) + adaptive Huffman (host).  window must be a power of two in
 * [2^10, 2^15].  The parse is greedy unless s->lazy or s->mincost is 1.  Errors are
 * reported in s->error.                                                      */
void sqz_compress(struct sqz* s, struct sqz_bitstream* bs,
                  const uint8_t* data, uint64_t bytes, uint32_t window);

/* The host half of sqz_compress alone: entropy-code an LZ77 token stream
 * (token = literal byte, or (len << 16) | dist) exactly as
 * squeeze.h:377-396 would.                                                  */
void sqz_encode_tokens(struct sqz* s, struct sqz_bitstream* bs,
                       const uint32_t* tokens, uint64_t count);

/* The same for symbol words -- tokens with the bucket arithmetic of
 * squeeze.h:290-315 already done, which is what the GPU parse emits in
 * `symbols` mode (include/sqz_gpu.h has the layout).  A word whose symbols are
 * out of range sets s->error = EINVAL; extra-bit fields are taken as they are. */
void sqz_encode_symbols(struct sqz* s, struct sqz_bitstream* bs,
                        const uint32_t* words, uint64_t count);
/* The same, handing the words to the coder `chunk` at a time -- the way
 * sqz_compress receives them from the GPU stream (0 = all at once).         */
void sqz_encode_symbols_chunked(struct sqz* s, struct sqz_bitstream* bs,
                                const uint32_t* words, uint64_t count, uint64_t chunk);
/* token -> symbol word on the host (0xFFFFFFFF for a token the decoder would
 * reject); the reference for what the GPU emits.                             */
void sqz_symbols_of_tokens(const uint32_t* tokens, uint64_t count, uint32_t* words);

/* squeeze.decompress (squeeze.h:502-551).  On return the bitstream stands where
 * the reference's bit-at-a-time reader would (bitstream.h:65-95): `read` at the
 * end of the last word the stream used, the unused bits of that word in b64/bits.
 * The decoder reads ahead; in memory mode a word it pulled too early is given
 * back, so that data stored behind the stream can be read from the same
 * sqz_bitstream.  A callback source cannot take a word back: there up to one
 * 64-bit word more than the reference would have asked for has been consumed. */
void sqz_decompress(struct sqz* s, struct sqz_bitstream* bs,
                    uint8_t* data, uint64_t bytes);

/* The serial half of sqz_decompress alone: read the tokens of a stream that
 * expands to `bytes` bytes (literal byte, or (len << 16) | dist) without
 * executing them.  *count receives the number of tokens even when it exceeds
 * `cap` (then s->error = E2BIG).  Same checks as sqz_decompress.              */
void sqz_decode_tokens(struct sqz* s, struct sqz_bitstream* bs, uint64_t bytes,
                       uint32_t* tokens, uint64_t cap, uint64_t* count);

/* sqz_decompress with the copy phase on the GPU (SURVEY 8f N4): tokens are
 * read on the host, then sqz_gpu_expand_tokens executes them.  bytes < 2 GiB.
 * Host memory for the tokens is allocated inside (4 bytes per token).         */
void sqz_decompress_gpu(struct sqz* s, struct sqz_bitstream* bs,
                        uint8_t* data, uint64_t bytes);

/* Convenience: whole buffers, memory mode, header included.  Return errno. */
int sqz_compress_buffer(const uint8_t* data, uint64_t bytes, uint8_t win_bits,
                        uint8_t* out, uint64_t capacity, uint64_t* written);
int sqz_decompress_buffer(const uint8_t* comp, uint64_t comp_bytes,
                          uint8_t* out, uint64_t capacity, uint64_t* bytes);

#ifdef __cplusplus
}
#endif
#endif /* SQZ_H_INCLUDED */
