/* include/sqz_gpu.h -- C-ABI of the B200 (sm_100a) LZ77 match search of sqz-b200.
 *
 * The reference (leok7v/sqz) has no FFI or plugin interface: its longest-match
 * search is an inline loop inside squeeze_compress
 * (/root/reference/attic/map_experiment/squeeze.h:338-358) followed by the
 * greedy token dispatch (squeeze.h:377-394).  These entry points are what a
 * maintainer would call at exactly that place (see INTEGRATION.md): plain
 * pointers and sizes, int errno return values, callable from C99.  No call
 * changes the calling thread's current CUDA device.  State that outlives a call
 * is limited to staging buffers kept for the next call -- per device at most 8
 * sets and 12 GiB of device + pinned memory, oldest out first; sqz_gpu_release
 * frees them -- and the measurement aids at the end of this file, which are off
 * unless switched on.
 *
 * Rule parameters (SURVEY.md section 8a, row A1):
 *   window    the LZ window the stream header announces (power of two)
 *   min_len   shortest match worth a back-reference     (reference G1: 3)
 *   max_len   longest match                              (reference G1: 257)
 *   max_dist  farthest candidate                         (reference G1: window-1)
 * For every position i the result is the candidate with the longest common
 * prefix (capped by max_len and by bytes-i), the nearest one among equals --
 * what the reference's "nearest first, strictly longer wins" scan selects.
 *
 * Token word (shared with sqz.h): literal = byte value (bits 31..16 zero);
 * match = (len << 16) | dist.  A match-table word uses the same packing, with
 * 0 meaning "no match of at least min_len here".
 *
 * Symbol word (what the host coder of sqz.h consumes directly, sqz_encode_symbols): the same
 * token with the bucket arithmetic of squeeze_encode_len / squeeze_encode_pos
 * (squeeze.h:290-315, tables squeeze.h:29-79,151-172) already done on the GPU:
 *   bits  0..8   symbol of the literal/length tree: byte value, or 257 + length bucket
 *   bits  9..13  the length's extra bits      (len - len_base[bucket])
 *   bits 14..18  symbol of the distance tree  (distance bucket)
 *   bits 19..31  the distance's extra bits    (dist - pos_base[bucket])
 * Extra bits are stored in emission order, i.e. bit-reversed within their field
 * width, because the bitstream takes values least significant bit first
 * (bitstream.h:49-63).  Symbol words exist only within the bitstream's own
 * limits: min_len >= 3, max_len <= 257 (what the decoders accept, squeeze.h:529-545),
 * max_dist <= 32767.
 *
 * Errors: 0, EINVAL (bad rule parameters), E2BIG (output capacity), ENOMEM,
 * ENODEV (no CUDA device / driver: there is NO CPU fallback), EIO (CUDA error;
 * sqz_gpu_last_error() has the text).
 */
#ifndef SQZ_GPU_H_INCLUDED
#define SQZ_GPU_H_INCLUDED

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SQZ_GPU_ABI_VERSION 3

enum {
    sqz_gpu_max_len_limit  = 512,     /* parse hand-off tables are sized for this */
    sqz_gpu_max_dist_limit = 65535    /* distances are reported in 16 bits */
};

/* ---- host-buffer entry points (replace squeeze.h:338-358 / 377-394) ------ *
 * They run on the calling thread's current CUDA device (device 0 unless the
 * caller selected another one); sqz_gpu_stream_open takes the device explicitly
 * (-1 = current).                                                            */

/* Full match table: for every i in [0, bytes) len_out[i] in {0} U
 * [min_len, max_len] and dist_out[i] in [1, max_dist] (0 when len is 0).
 * Replaces the search loop squeeze.h:340-358 evaluated at every position.   */
int sqz_gpu_match_table(const uint8_t* data, size_t bytes,
                        uint32_t window, uint32_t min_len, uint32_t max_len,
                        uint32_t max_dist,
                        uint16_t* len_out, uint16_t* dist_out);

/* Greedy token stream in parse order (squeeze.h:337,377-394): search + parse
 * on the GPU, tokens copied to the caller.  *n_tokens receives the count even
 * when it exceeds tokens_cap (then E2BIG is returned).                       */
int sqz_gpu_tokens(const uint8_t* data, size_t bytes,
                   uint32_t window, uint32_t min_len, uint32_t max_len,
                   uint32_t max_dist,
                   uint32_t* tokens_out, size_t tokens_cap, size_t* n_tokens);

/* sqz_gpu_tokens with flags: 0 (the call above), SQZ_GPU_STREAM_LAZY or
 * SQZ_GPU_STREAM_MINCOST, the lazy or min-cost parse of the token stream
 * below, identical to what the stream delivers with that flag.  Any other bit
 * or combination is EINVAL.                                                  */
int sqz_gpu_tokens_ex(const uint8_t* data, size_t bytes,
                      uint32_t window, uint32_t min_len, uint32_t max_len,
                      uint32_t max_dist, uint32_t flags,
                      uint32_t* tokens_out, size_t tokens_cap, size_t* n_tokens);

/* The same token stream computed on several devices at once (SURVEY.md section 8e;
 * squeeze.h:345,377-394 is where the seam dependency comes from).  The input is cut
 * into n_devices contiguous shards (sizes differ by at most one byte), each uploaded
 * with a look-back halo of max_dist bytes and a look-ahead halo of max_len bytes, so
 * the match tables are independent.  The parse depends on one number per seam -- where
 * the previous shard's last token ends -- which every device prepares for as a 1 KiB
 * exit map and the host chains with one lookup per seam.  The token arrays are then
 * concatenated in shard order by copies sized by their counts: device -> host when
 * tokens_out is host memory (pinned memory takes them by DMA from all devices at
 * once), peer-to-peer over NVLink when tokens_out is device memory.  No collective
 * library is involved.  The result is identical to sqz_gpu_tokens() for every
 * n_devices.  A device may be listed more than once (its shards then share it).
 * shard_tokens (optional, n_devices entries) receives the per-shard counts.       */
int sqz_gpu_tokens_multi(const int* devices, int n_devices,
                         const uint8_t* data, size_t bytes,
                         uint32_t window, uint32_t min_len, uint32_t max_len,
                         uint32_t max_dist,
                         uint32_t* tokens_out, size_t tokens_cap, size_t* n_tokens,
                         size_t* shard_tokens);

/* sqz_gpu_tokens_multi with flags: 0 (the call above) or SQZ_GPU_STREAM_LAZY.
 * The lazy step at a shard's last position reads the best match at the next
 * shard's first position; every shard searches that one position itself from
 * its look-ahead halo, so the seams still exchange nothing but the exit maps.
 * The result is identical to sqz_gpu_tokens_ex() with the same flags for every
 * n_devices.  Any other bit is EINVAL.                                       */
int sqz_gpu_tokens_multi_ex(const int* devices, int n_devices,
                            const uint8_t* data, size_t bytes,
                            uint32_t window, uint32_t min_len, uint32_t max_len,
                            uint32_t max_dist, uint32_t flags,
                            uint32_t* tokens_out, size_t tokens_cap, size_t* n_tokens,
                            size_t* shard_tokens);

/* sqz_gpu_tokens_multi_ex at shard boundaries of the caller's choice, and with
 * the min-cost parse.  flags: 0, SQZ_GPU_STREAM_LAZY or SQZ_GPU_STREAM_MINCOST
 * (within the bitstream's limits); any other bit or combination is EINVAL.
 * cuts: n_devices - 1 non-decreasing global offsets, each <= bytes (shards may
 * be empty); shard g is [cuts[g-1], cuts[g]) with cuts[-1] = 0 and
 * cuts[n_devices-1] = bytes.  With SQZ_GPU_STREAM_MINCOST every cut is a
 * multiple of 16384 or equal to bytes, so that every shard starts at a segment
 * and all but the last hold whole segments; each shard then rewrites its own
 * table into min-cost steps and nothing more crosses the seams than for the
 * greedy parse.  cuts = NULL: the even cut, ceil(bytes / u) units of u bytes
 * shared out as evenly as they go (the first ones one unit more), u = 1 without
 * MINCOST (the cut of sqz_gpu_tokens_multi_ex), u = 16384 with it (the partial
 * last segment in the last non-empty shard, shards past the segment count
 * empty).  Every argument is checked before any device is touched; on EINVAL
 * *n_tokens is 0.  The result is identical to sqz_gpu_tokens_ex() with the
 * same flags for every valid cut list.                                       */
int sqz_gpu_tokens_multi_cuts(const int* devices, int n_devices, const size_t* cuts /* n_devices - 1, or NULL */,
                              const uint8_t* data, size_t bytes,
                              uint32_t window, uint32_t min_len, uint32_t max_len,
                              uint32_t max_dist, uint32_t flags,
                              uint32_t* tokens_out, size_t tokens_cap, size_t* n_tokens,
                              size_t* shard_tokens);

/* Streaming form used by sqz_compress(): tokens arrive chunk by chunk, in
 * parse order, from double-buffered pinned memory while the device already
 * works on the next chunk.  *tokens stays valid until the next call.  *count
 * is 0 only when every token has been delivered; later calls return 0 again.
 * A chunk that lies inside the previous chunk's last match (possible when
 * chunk_bytes < max_len) is delivered together with the next one.  A chunk
 * larger than the input is the input: the staging is sized by the input.
 * chunk_bytes = 0: chunks of 2, 4, 8, 16, then 32 MiB -- a consumer slower
 * than the search starts after milliseconds.  chunk_bytes > 0: chunks of that
 * size -- for a consumer faster than the search, which only has to keep the
 * device on chunks it is efficient at; with SQZ_GPU_STREAM_SHORT_START the
 * first two are a quarter and a half of it.  The searches of consecutive
 * chunks run one after the other (a consumer wants them in order, not both
 * late), a chunk's parse and copy at the highest stream priority beside the
 * next chunk's search.
 * SQZ_GPU_STREAM_LAZY parses with lazy matching instead of the greedy rule:
 * at a position whose match reaches min_len, the literal is emitted instead
 * when the next position has a strictly longer match, and the decision is
 * taken again there (len at the end of the input counts as 0).  About 2 %
 * smaller streams of text and code, slightly larger ones of data that does
 * not compress; any decoder reads them.  The same flag selects the lazy parse
 * in sqz_gpu_tokens_ex, sqz_gpu_tokens_multi_ex and the _ex device-buffer
 * parse entry points below; without it every entry point is greedy.
 * SQZ_GPU_STREAM_MINCOST parses by cost instead: 3-5 % smaller streams than
 * greedy on text and code (about twice what lazy gains), in the same format.
 * The input is cut into segments of 16384 positions at offsets that are
 * multiples of 16384 (the last one may be shorter).  Costs are fixed integers:
 * a literal 8, a match (k, d) 6 + len_extra[bucket(k)] + 5 + pos_extra[bucket(d)]
 * (the buckets of the symbol words).  In a segment [s, e), backwards from
 * e - 1, with c(j) = 0 for j >= e and len, dist the best match at i:
 *   c(i) = min(8 + c(i + 1), cost(k, dist) + c(i + k) for min_len <= k <= len)
 * with ties to the longest step (a match beats a literal of equal cost).  The
 * parse starts at 0 and follows the chosen steps -- the literal, or the match
 * (k, dist), a prefix of the best match -- across segment ends.  Every step
 * depends on its own segment only, so the stream is the same for every
 * chunking.  Only within the bitstream's limits (min_len >= 3, max_len <= 257,
 * max_dist <= 32767) and not together with SQZ_GPU_STREAM_LAZY: EINVAL
 * otherwise.  Every chunk but the last holds whole segments: the default
 * chunks already do, an explicit chunk_bytes (and its SHORT_START quarter) is
 * rounded up to a multiple of 16384.  sqz_gpu_tokens_ex takes the flag as
 * well, and so do the two calls made for shards: sqz_gpu_tokens_multi_cuts,
 * which cuts at segment offsets, and sqz_gpu_mincost_steps_device, which
 * rewrites one shard's table once before the flag-0 device-buffer parse.
 * sqz_gpu_tokens_multi_ex keeps refusing it (EINVAL): its cut, sizes that
 * differ by at most one byte, is not at segment offsets.  The device-buffer
 * _ex calls refuse it too: they read the table without changing it, and the
 * rewrite must run exactly once per table.                                   */
typedef struct sqz_gpu_stream sqz_gpu_stream;
#define SQZ_GPU_STREAM_SYMBOLS 1u       /* deliver symbol words instead of plain tokens */
#define SQZ_GPU_STREAM_SHORT_START 2u   /* explicit chunk_bytes: start with chunk_bytes / 4, then / 2 */
#define SQZ_GPU_STREAM_LAZY 8u          /* lazy matching instead of the greedy parse (combines with the others) */
#define SQZ_GPU_STREAM_MINCOST 32u      /* min-cost parse instead of the greedy one (not with LAZY) */
int  sqz_gpu_stream_open(sqz_gpu_stream** st, int device,
                         const uint8_t* data, size_t bytes,
                         uint32_t window, uint32_t min_len, uint32_t max_len,
                         uint32_t max_dist, size_t chunk_bytes /* 0 = default */,
                         uint32_t flags /* SQZ_GPU_STREAM_* */);
int  sqz_gpu_stream_next(sqz_gpu_stream* st, const uint32_t** tokens, size_t* count);
void sqz_gpu_stream_close(sqz_gpu_stream* st);

/* ---- device-buffer entry points (shards, benchmarks, multi-GPU) ---------- *
 * A shard is `n` positions starting at d_shard, with `back` valid bytes
 * before it (look-back halo, min(global offset, max_dist) is enough) and
 * `ahead` valid bytes after it (look-ahead halo, min(bytes to the global end,
 * max_len) is enough).  All pointers are device pointers on the current
 * device; `stream` is a cudaStream_t (NULL = default stream).  Asynchronous. */

/* table[i] for the n positions of the shard, packed (len << 16) | dist.
 * The kernels need sqz_gpu_match_workspace(n) bytes of scratch device memory (the
 * work list the first kernel leaves for the second): the _ws form takes it from the
 * caller, the plain form borrows it from a per-device pool of the library.   */
size_t sqz_gpu_match_workspace(size_t n);
int sqz_gpu_match_table_device_ws(const uint8_t* d_shard, size_t back, size_t n,
                                  size_t ahead, uint32_t min_len, uint32_t max_len,
                                  uint32_t max_dist, uint32_t* d_table, void* d_work,
                                  void* stream);
int sqz_gpu_match_table_device(const uint8_t* d_shard, size_t back, size_t n,
                               size_t ahead, uint32_t min_len, uint32_t max_len,
                               uint32_t max_dist, uint32_t* d_table, void* stream);

/* The seam word of a lazy parse: d_table[n] = the packed best match at the
 * first position after the shard (position n, searched with the shard as
 * look-back and `ahead` - 1 bytes of look-ahead), 0 when ahead is 0 (the end
 * of the input).  A caller who searched the shard's n positions with
 * sqz_gpu_match_table_device gets the (n+1)-th word the lazy parse reads,
 * from the same halos; no byte beyond them is read.                          */
int sqz_gpu_match_seam_device(const uint8_t* d_shard, size_t back, size_t n,
                              size_t ahead, uint32_t min_len, uint32_t max_len,
                              uint32_t max_dist, uint32_t* d_table, void* stream);

/* Split a packed table into the two 16-bit arrays of sqz_gpu_match_table.   */
int sqz_gpu_unpack_table_device(const uint32_t* d_table, size_t n,
                                uint16_t* d_len, uint16_t* d_dist, void* stream);

/* Greedy parse of one shard.  `entry` is the offset of the first parse
 * position inside the shard (0 for the first shard; otherwise the overshoot
 * of the previous shard's last token).  d_work must hold
 * sqz_gpu_parse_workspace(n) bytes.  After the stream is synchronised,
 * h_result[0] = token count, h_result[1] = overshoot into the next shard
 * (h_result: 2 x uint64 in pinned or pageable host memory, or device memory
 * when result_on_device != 0).  Tokens beyond tokens_cap are not stored.     */
size_t sqz_gpu_parse_workspace(size_t n);
int sqz_gpu_parse_device(const uint8_t* d_shard, const uint32_t* d_table, size_t n,
                         uint32_t entry, uint32_t min_len, uint32_t max_len,
                         uint32_t* d_tokens, size_t tokens_cap,
                         void* d_work, uint64_t* d_result /* 2 x u64, device */,
                         void* stream);

/* The same parse, emitting symbol words (see above) instead of plain tokens:
 * replaces squeeze.h:377-394 together with the table lookups and subtractions
 * of squeeze.h:290-315.                                                      */
int sqz_gpu_parse_symbols_device(const uint8_t* d_shard, const uint32_t* d_table, size_t n,
                                 uint32_t entry, uint32_t min_len, uint32_t max_len,
                                 uint32_t* d_words, size_t words_cap,
                                 void* d_work, uint64_t* d_result /* 2 x u64, device */,
                                 void* stream);

/* Seam hand-off without waiting for the previous shard: exit_map[e] is the
 * overshoot this shard produces when entered at offset e, for every
 * e < max_len.  d_exit_map: max_len x uint16 on the device.                  */
int sqz_gpu_parse_exit_map_device(const uint32_t* d_table, size_t n,
                                  uint32_t min_len, uint32_t max_len,
                                  void* d_work, uint16_t* d_exit_map, void* stream);

/* The three calls above with flags.  sqz_gpu_parse_device_ex takes
 * SQZ_GPU_STREAM_SYMBOLS (symbol words, the limits of sqz_gpu_parse_symbols_device)
 * and SQZ_GPU_STREAM_LAZY; sqz_gpu_parse_exit_map_device_ex takes
 * SQZ_GPU_STREAM_LAZY.  Any other bit is EINVAL.  With SQZ_GPU_STREAM_LAZY
 * d_table holds n + 1 words, the last one from sqz_gpu_match_seam_device; the
 * entry and the overshoot stay below max_len, so the exit maps chain across
 * shards exactly as for the greedy parse.  flags = 0 (and SYMBOLS) give the
 * calls above.                                                               */
int sqz_gpu_parse_device_ex(const uint8_t* d_shard, const uint32_t* d_table, size_t n,
                            uint32_t entry, uint32_t min_len, uint32_t max_len,
                            uint32_t flags, uint32_t* d_out, size_t out_cap,
                            void* d_work, uint64_t* d_result /* 2 x u64, device */,
                            void* stream);
int sqz_gpu_parse_exit_map_device_ex(const uint32_t* d_table, size_t n,
                                     uint32_t min_len, uint32_t max_len, uint32_t flags,
                                     void* d_work, uint16_t* d_exit_map, void* stream);

/* The min-cost parse of a shard (SQZ_GPU_STREAM_MINCOST above): rewrites the
 * n words of d_table, as sqz_gpu_match_table_device left them with the same
 * rules, in place into min-cost steps -- (k << 16) | dist, or 0 for a literal.
 * `first` is the shard's global offset, `bytes` the size of the whole input.
 * After it, the flag-0 calls sqz_gpu_parse_exit_map_device(_ex) and
 * sqz_gpu_parse_device(_ex) give the min-cost exit map and token stream (with
 * SQZ_GPU_STREAM_SYMBOLS its symbol words), and the exit maps chain across
 * shards as for the greedy parse.  Call it once per table: what it leaves are
 * steps, not best matches, and a second rewrite would price those.  EINVAL
 * unless first % 16384 == 0, first + n <= bytes, n % 16384 == 0 or
 * first + n == bytes, and the rules are within the bitstream's limits
 * (min_len >= 3, max_len <= 257, max_dist <= 32767).  n == 0 does nothing.   */
int sqz_gpu_mincost_steps_device(uint32_t* d_table, size_t first, size_t n, size_t bytes,
                                 uint32_t min_len, uint32_t max_len, uint32_t max_dist, void* stream);

/* ---- one process per device ------------------------------------------------ *
 * Jobs that run one process per GPU (torchrun and the like) concatenate their
 * shards' tokens the same way as sqz_gpu_tokens_multi, except that the destination
 * buffer lives in one process and has to be mapped into the others: CUDA IPC, no
 * collective.  The owner allocates and exports, the others open; every process then
 * puts its tokens at its offset (the sum of the earlier shards' counts).       */
#define SQZ_GPU_IPC_HANDLE_BYTES 64
int  sqz_gpu_device_alloc(void** d_ptr, size_t bytes);
void sqz_gpu_device_free(void* d_ptr);
int  sqz_gpu_ipc_export(const void* d_ptr, uint8_t handle[SQZ_GPU_IPC_HANDLE_BYTES]);
int  sqz_gpu_ipc_open(const uint8_t handle[SQZ_GPU_IPC_HANDLE_BYTES], void** d_ptr);
int  sqz_gpu_ipc_close(void* d_ptr);
int  sqz_gpu_put_tokens(uint32_t* d_dst, size_t at, const uint32_t* d_tokens, size_t count, void* stream);

/* ---- decoder side: the LZ copy phase (replaces squeeze.h:533-539) --------- *
 * The reference's decoder executes every token as it reads it: a literal is
 * stored, a match copies len bytes from dist back, one byte at a time because
 * the ranges may overlap.  With the tokens at hand (sqz_decode_tokens in sqz.h
 * reads them from the bitstream on the host, which is the serial part) the
 * copies are a parallel problem: a scan of the token lengths places every
 * token, every output byte starts with a hop of `dist` to its source, and
 * pointer doubling shortens all chains to one hop onto a literal.  Plain
 * tokens (not symbol words): len 1..65535, dist 1..65535, whatever rules made
 * them; bytes < 2 GiB per call.  EINVAL when bytes >= 2 GiB, when the tokens
 * do not describe exactly `bytes` bytes, when a match reaches before the start
 * or has dist 0, and when a literal word is not a byte value (above 0xFF, as
 * the symbol word of a match with dist 1..4 is).  sqz_gpu_expand_tokens checks
 * the sizes before it allocates anything.                                    */
int sqz_gpu_expand_tokens(const uint32_t* tokens, size_t n_tokens, uint8_t* out, size_t bytes);
/* device pointers; d_work holds sqz_gpu_expand_workspace(n_tokens, bytes) bytes.
 * Waits for the stream twice: once for the scan of the token lengths (a stream
 * that does not describe `bytes` bytes is refused before anything is placed),
 * once at the end for the verdict on the distances.  The rounds of pointer
 * doubling in between end themselves on the device.                           */
size_t sqz_gpu_expand_workspace(size_t n_tokens, size_t bytes);
int sqz_gpu_expand_tokens_device(const uint32_t* d_tokens, size_t n_tokens, uint8_t* d_out,
                                 size_t bytes, void* d_work, void* stream);

/* ---- utilities ----------------------------------------------------------- */
int         sqz_gpu_abi_version(void);
int         sqz_gpu_device_count(void);          /* 0 when no driver / device */
const char* sqz_gpu_last_error(void);            /* thread-local text */
void*       sqz_gpu_host_alloc(size_t bytes);    /* pinned host memory (NULL on failure) */
void        sqz_gpu_host_free(void* p);
/* The host-buffer entry points and sqz_gpu_match_table_device keep their device
 * and pinned staging buffers for the next call: one set per shard or pipeline
 * slot, per device at most 8 sets and 12 GiB of device + pinned memory, oldest
 * out first.  This frees them all.                                           */
void        sqz_gpu_release(void);
/* Which match-table kernel serves sqz_gpu_match_table_device: 0 = automatic
 * (bit-sliced kernel for min_len 2 or 3, thread-per-position kernel otherwise),
 * 1 = thread-per-position, 2 = bit-sliced where applicable.  Both are exact;
 * the switch exists for A/B measurements and tests and applies to the calling
 * thread only.                                                               */
int         sqz_gpu_select_kernel(int which);
/* Debugging aid: when d_buf (device, one u64 per tile of 16256 positions) is not
 * NULL the bit-sliced kernel stores every tile's duration in SM cycles.      */
void        sqz_gpu_debug_tile_cycles(unsigned long long* d_buf);
/* kernels launched by this library in this process so far (for bench.py)    */
uint64_t    sqz_gpu_launch_count(void);
/* average device time of the match-table kernel over the launches since the
 * last call with reset != 0, measured with CUDA events on the launching
 * stream; enable with sqz_gpu_set_timing(1).  Seconds.                       */
void        sqz_gpu_set_timing(int on);
double      sqz_gpu_match_kernel_seconds(int reset, uint64_t* launches);
/* the same for the kernel of the min-cost parse (one launch per chunk)       */
double      sqz_gpu_mincost_kernel_seconds(int reset, uint64_t* launches);

#ifdef __cplusplus
}
#endif
#endif /* SQZ_GPU_H_INCLUDED */
