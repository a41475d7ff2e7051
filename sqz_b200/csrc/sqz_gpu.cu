// sqz_gpu.cu -- B200 (sm_100a) LZ77 longest-match search + greedy parse of
// sqz-b200, and the C-ABI declared in include/sqz_gpu.h.
//
// What it replaces in the reference (leok7v/sqz, generation G1):
//   /root/reference/attic/map_experiment/squeeze.h:338-358  brute-force search
//   /root/reference/attic/map_experiment/squeeze.h:337,377-394  greedy parse
// Results are bit-exact: for every position the longest common prefix with a
// candidate at distance 1..max_dist (capped by max_len and the end of data),
// the nearest candidate among equals; then the orbit of position 0 under
// next[i] = i + (len[i] >= min_len ? len[i] : 1) as the token stream.  Every token entry
// point can parse with lazy matching instead (SQZ_GPU_STREAM_LAZY, namespace parse); the token
// stream and the one-shot call can parse by cost (SQZ_GPU_STREAM_MINCOST, namespace mincost).
//
// There is no CPU fallback in this file: without a device every entry point
// returns ENODEV.
#include "sqz_gpu.h"

#include <cuda_runtime.h>

#include "match_bitsliced.cuh"
#include "lz_expand.cuh"

#include <atomic>
#include <cerrno>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <mutex>
#include <vector>

// ---------------------------------------------------------------------------
// error plumbing
// ---------------------------------------------------------------------------
static thread_local char g_err[256] = "";
static std::atomic<uint64_t> g_launches{0};

static int fail(int code, const char* what, cudaError_t ce = cudaSuccess) {
    if (ce != cudaSuccess) {
        snprintf(g_err, sizeof(g_err), "%s: %s", what, cudaGetErrorString(ce));
    } else {
        snprintf(g_err, sizeof(g_err), "%s", what);
    }
    return code;
}

static int cuda_code(cudaError_t ce) {
    switch (ce) {
        case cudaErrorMemoryAllocation: return ENOMEM;
        case cudaErrorNoDevice:
        case cudaErrorInsufficientDriver:
        case cudaErrorInvalidDevice: return ENODEV;
        default: return EIO;
    }
}

#define CU(call)                                                         \
    do {                                                                 \
        cudaError_t ce_ = (call);                                        \
        if (ce_ != cudaSuccess) { return fail(cuda_code(ce_), #call, ce_); } \
    } while (0)

#define LAUNCHED(name)                                                   \
    do {                                                                 \
        g_launches.fetch_add(1, std::memory_order_relaxed);              \
        cudaError_t ce_ = cudaGetLastError();                            \
        if (ce_ != cudaSuccess) { return fail(cuda_code(ce_), name, ce_); } \
    } while (0)

// ---------------------------------------------------------------------------
// kernel 1: match table, one position per thread, window staged in shared
// memory.  (First correct path; the tuned kernel replaces it behind the same
// launcher.)
//
// Shared-memory image: bytes [lo, hi) of the shard, where lo reaches back
// max_dist bytes before the tile and hi runs max_len bytes past it, shifted so
// that 16-byte global chunks land on 16-byte shared chunks.
//
// Scan order and acceptance are the reference's: distance 1 first, a candidate
// replaces the best only when strictly longer.  The filter that keeps the scan
// cheap is exact: to beat `best` a candidate must agree on the bytes
// [need-4, need) with need = max(best+1, min_len) (or on the first `need`
// bytes while need < 4); only candidates that pass are measured in full.
// ---------------------------------------------------------------------------
namespace v1 {

constexpr int kThreads = 512;

__device__ __forceinline__ uint32_t load_u32_unaligned(const uint8_t* S, int x) {
    const uint32_t* W = reinterpret_cast<const uint32_t*>(S);
    const int w = x >> 2;
    const uint32_t lo = W[w], hi = W[w + 1];
    return __funnelshift_r(lo, hi, (x & 3) * 8);
}

__global__ void __launch_bounds__(kThreads)
match_table(const uint8_t* __restrict__ shard, long long back, long long n,
            long long ahead, uint32_t min_len, uint32_t max_len,
            uint32_t max_dist, uint32_t* __restrict__ table) {
    extern __shared__ __align__(16) uint8_t S[];
    const long long tile0 = (long long)blockIdx.x * kThreads;
    const long long behind = min((long long)max_dist, tile0 + back);
    const long long lo = tile0 - behind;                        // first byte staged (shard-relative)
    const long long hi = min(tile0 + kThreads + (long long)max_len, n + ahead);
    const uint8_t* g = shard + lo;
    const int a = (int)(reinterpret_cast<uintptr_t>(g) & 15);   // S[a] holds byte `lo`
    const int span = a + (int)(hi - lo);                        // bytes of S in use
    const int chunks = (span + 8 + 15) >> 4;                    // + zero padding for word reads
    for (int c = threadIdx.x; c < chunks; c += kThreads) {
        const int s0 = c << 4;
        uint4 v;
        if (s0 >= a && s0 + 16 <= span) {
            v = __ldg(reinterpret_cast<const uint4*>(g - a + s0));
        } else {
            uint8_t b[16];
#pragma unroll
            for (int k = 0; k < 16; k++) {
                const int s = s0 + k;
                b[k] = (s >= a && s < span) ? __ldg(g - a + s) : (uint8_t)0;
            }
            memcpy(&v, b, 16);
        }
        reinterpret_cast<uint4*>(S)[c] = v;
    }
    __syncthreads();

    const long long p = tile0 + threadIdx.x;
    if (p >= n) { return; }
    const int xi = a + (int)(p - lo);                           // S index of position p
    const uint32_t room = (uint32_t)min((long long)max_len, n + ahead - p);
    const uint32_t reach = (uint32_t)min((long long)max_dist, p + back);
    const uint32_t* W = reinterpret_cast<const uint32_t*>(S);

    uint32_t best = 0, bdist = 0;
    uint32_t d = 1;
    while (d <= reach) {
        const uint32_t need = max(best + 1, min_len);
        if (need > room) { break; }
        const uint32_t o = need >= 4 ? need - 4 : 0;
        const uint32_t mask = need >= 4 ? 0xFFFFFFFFu : (0xFFFFFFFFu >> (8 * (4 - need)));
        const uint32_t key = load_u32_unaligned(S, xi + (int)o) & mask;
        int c = xi + (int)o - (int)d;                           // candidate word starts here
        const int c_end = xi + (int)o - (int)reach;             // farthest candidate
        int w = c >> 2;
        uint32_t hiw = W[w + 1], low = W[w];
        int kmax = c & 3;
        int found = -1;
        for (;;) {
            const uint32_t t3 = (__byte_perm(low, hiw, 0x6543) ^ key) & mask;
            const uint32_t t2 = (__byte_perm(low, hiw, 0x5432) ^ key) & mask;
            const uint32_t t1 = (__byte_perm(low, hiw, 0x4321) ^ key) & mask;
            const uint32_t t0 = (low ^ key) & mask;
            if (min(min(t0, t1), min(t2, t3)) == 0) {
                uint32_t hb = (t0 == 0 ? 1u : 0u) | (t1 == 0 ? 2u : 0u) |
                              (t2 == 0 ? 4u : 0u) | (t3 == 0 ? 8u : 0u);
                const int kmin = max(0, c_end - (w << 2));
                hb &= (2u << kmax) - 1u;
                hb &= ~((1u << kmin) - 1u);
                if (hb != 0) { found = (w << 2) + (31 - __clz(hb)); break; }
            }
            w--;
            if ((w << 2) + 3 < c_end) { break; }
            hiw = low;
            low = W[w];
            kmax = 3;
        }
        if (found < 0) { break; }
        const uint32_t dh = (uint32_t)(xi + (int)o - found);
        const uint8_t* A = S + xi;
        const uint8_t* B = S + xi - (int)dh;
        uint32_t m = 0;
        while (m < room && A[m] == B[m]) { m++; }
        if (m >= need) {
            best = m;
            bdist = dh;
            if (best >= room) { break; }
        }
        d = dh + 1;
    }
    table[p] = best >= min_len ? ((best << 16) | bdist) : 0u;
}

static size_t smem_bytes(uint32_t max_len, uint32_t max_dist) {
    size_t b = 16 + (size_t)max_dist + kThreads + max_len + 16 + 16;
    return (b + 15) & ~(size_t)15;
}

}  // namespace v1

// ---------------------------------------------------------------------------
// kernel 2: split packed table words into the two u16 arrays of the host ABI
// ---------------------------------------------------------------------------
__global__ void unpack_table(const uint32_t* __restrict__ table, size_t n,
                             uint16_t* __restrict__ len, uint16_t* __restrict__ dist) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    const size_t stride = (size_t)gridDim.x * blockDim.x;
    for (; i < n; i += stride) {
        const uint32_t w = table[i];
        len[i] = (uint16_t)(w >> 16);
        dist[i] = (uint16_t)(w & 0xFFFF);
    }
}

// ---------------------------------------------------------------------------
// greedy parse (squeeze.h:337,377-394) as block-wise pointer jumping.
//
// The shard is cut into parse blocks of kPB positions.  A token never jumps
// more than max_len, so a block can only be entered at an offset < max_len
// ("entry") and leaves with an overshoot < max_len into the next block.
//   parse_exit_map   per block: overshoot for every possible entry, by pointer
//                    doubling over next[] in shared memory
//   chain_groups     compose the maps of kGroup consecutive blocks
//   chain_top        serial walk over the groups -> entry of every group,
//                    overshoot of the whole shard
//   chain_expand     entry of every block
//   parse_walk<0>    per block (one warp, steps staged in shared memory): number of tokens on the real path
//   scan_counts      exclusive prefix sum -> output offsets, total
//   parse_walk<1>    per block: the same walk, then all lanes write the tokens (or symbol words)
// The lazy parse (kLazy) is the same machinery with another step, which also reads table[i + 1]: its
// steps are still 1 or len <= max_len, so entries, overshoots and maps keep their bounds.
// ---------------------------------------------------------------------------
namespace parse {

constexpr int kPBLarge = 4096;   // positions per parse block
constexpr int kPBSmall = 1024;   // ... of a small shard: the walks of a block are serial, shorter ones finish sooner
constexpr size_t kSmallShard = (size_t)8 << 20;
constexpr int kMapStride = 512;  // = sqz_gpu_max_len_limit entries per exit map
constexpr int kGroupMax = 128;   // blocks per chain group (large shards; small ones use about sqrt(blocks))

static int parse_block(size_t n) { return n <= kSmallShard ? kPBSmall : kPBLarge; }

static int group_size(size_t blocks) {
    int g = 8;
    while (g < kGroupMax && (size_t)g * g < blocks) { g <<= 1; }
    return g;
}

struct Work {                    // carved out of the caller's d_work
    uint16_t* exit_map;          // [blocks][kMapStride]
    uint16_t* group_map;         // [groups][kMapStride]
    uint32_t* group_entry;       // [groups + 1]
    uint32_t* block_entry;       // [blocks]
    uint32_t* count;             // [blocks]
    uint64_t* offset;            // [blocks]
    size_t blocks, groups;
    int pb, group;               // positions per block, blocks per group
};

static size_t align_up(size_t x) { return (x + 255) & ~(size_t)255; }

static size_t workspace_for(size_t n, int pb) {
    const size_t blocks = (n + pb - 1) / pb + 1;
    const size_t groups = (blocks + 8 - 1) / 8 + 1;            // the smallest group size: an upper bound
    return align_up(blocks * kMapStride * 2) + align_up(groups * kMapStride * 2) +
           align_up((groups + 1) * 4) + align_up(blocks * 4) + align_up(blocks * 4) +
           align_up(blocks * 8) + 256;
}

// enough for every shard of at most n positions (small shards use smaller blocks)
static size_t workspace(size_t n) {
    return std::max(workspace_for(n, parse_block(n)), workspace_for(std::min(n, kSmallShard), kPBSmall));
}

static Work carve(void* d_work, size_t n) {
    Work w;
    w.pb = parse_block(n);
    w.blocks = (n + w.pb - 1) / w.pb;
    w.group = group_size(w.blocks);
    w.groups = (w.blocks + w.group - 1) / w.group;
    const size_t blocks = w.blocks + 1, groups = w.groups + 1;
    uint8_t* p = (uint8_t*)d_work;
    p = (uint8_t*)(((uintptr_t)p + 255) & ~(uintptr_t)255);
    w.exit_map = (uint16_t*)p;    p += align_up(blocks * kMapStride * 2);
    w.group_map = (uint16_t*)p;   p += align_up(groups * kMapStride * 2);
    w.group_entry = (uint32_t*)p; p += align_up((groups + 1) * 4);
    w.block_entry = (uint32_t*)p; p += align_up(blocks * 4);
    w.count = (uint32_t*)p;       p += align_up(blocks * 4);
    w.offset = (uint64_t*)p;
    return w;
}

// The decision at a parse position i, from its table word and, for the lazy parse, table[i + 1] (at
// the shard's last position table[n], which the caller provides).  Greedy: the match when it reaches
// min_len.  Lazy: not when the next position has a strictly longer one -- then the literal, and the
// decision is taken again at i + 1.  Either way the step is 1 or len <= max_len, which is all the
// exit maps and the walk rely on.
template <bool kLazy>
__device__ __forceinline__ uint32_t next_word(const uint32_t* __restrict__ table, size_t i) {
    return kLazy ? table[i + 1] : 0u;
}

template <bool kLazy>
__device__ __forceinline__ bool takes_match(uint32_t word, uint32_t next, uint32_t min_len) {
    const uint32_t len = word >> 16;
    return len >= min_len && !(kLazy && (next >> 16) > len);
}

template <bool kLazy>
__device__ __forceinline__ uint32_t step_of(uint32_t word, uint32_t next, uint32_t min_len) {
    return takes_match<kLazy>(word, next, min_len) ? word >> 16 : 1u;
}

template <int kPB, bool kLazy>
__global__ void __launch_bounds__(256)
parse_exit_map(const uint32_t* __restrict__ table, size_t n, uint32_t min_len,
               uint32_t max_len, uint16_t* __restrict__ exit_map) {
    __shared__ uint16_t jump[kPB];
    const size_t b0 = (size_t)blockIdx.x * kPB;
    const int size = (int)min((size_t)kPB, n - b0);            // positions in this block
    for (int p = threadIdx.x; p < size; p += blockDim.x) {
        jump[p] = (uint16_t)(p + step_of<kLazy>(table[b0 + p], next_word<kLazy>(table, b0 + p), min_len));
    }
    __syncthreads();
    // asynchronous pointer doubling: every value stored is a point on p's own
    // path, so reading a neighbour's half-updated entry is still correct
    for (;;) {
        int changed = 0;
        for (int p = threadIdx.x; p < size; p += blockDim.x) {
            const int j = jump[p];
            if (j < size) {
                jump[p] = jump[j];
                changed = 1;
            }
        }
        if (!__syncthreads_or(changed)) { break; }
    }
    uint16_t* out = exit_map + (size_t)blockIdx.x * kMapStride;
    for (int e = threadIdx.x; e < (int)max_len; e += blockDim.x) {
        out[e] = (uint16_t)(e < size ? jump[e] - size : e - size);
    }
}

__global__ void chain_groups(const uint16_t* __restrict__ exit_map, size_t blocks, int group,
                             uint32_t max_len, uint16_t* __restrict__ group_map) {
    const size_t g = blockIdx.x;
    const size_t first = g * (size_t)group;
    const size_t last = min(first + (size_t)group, blocks);
    for (uint32_t e = threadIdx.x; e < max_len; e += blockDim.x) {
        uint32_t x = e;
        for (size_t b = first; b < last; b++) { x = exit_map[b * kMapStride + x]; }
        group_map[g * kMapStride + e] = (uint16_t)x;
    }
}

// one thread: entries of all groups, then the shard's overshoot and (later,
// from scan_counts) the token total
__global__ void chain_top(const uint16_t* __restrict__ group_map, size_t groups,
                          const uint32_t* __restrict__ entry_in, uint32_t entry_imm,
                          uint32_t* __restrict__ group_entry, uint64_t* __restrict__ result) {
    uint32_t x = entry_in != nullptr ? *entry_in : entry_imm;
    for (size_t g = 0; g < groups; g++) {
        group_entry[g] = x;
        x = group_map[g * kMapStride + x];
    }
    group_entry[groups] = x;
    result[1] = x;
}

// composed map of the whole shard, for seam hand-off between GPUs
__global__ void chain_total(const uint16_t* __restrict__ group_map, size_t groups,
                            uint32_t max_len, uint16_t* __restrict__ out) {
    for (uint32_t e = threadIdx.x; e < max_len; e += blockDim.x) {
        uint32_t x = e;
        for (size_t g = 0; g < groups; g++) { x = group_map[g * kMapStride + x]; }
        out[e] = (uint16_t)x;
    }
}

__global__ void chain_expand(const uint16_t* __restrict__ exit_map, size_t blocks, int group,
                             size_t groups, const uint32_t* __restrict__ group_entry,
                             uint32_t* __restrict__ block_entry) {
    const size_t g = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (g >= groups) { return; }
    const size_t first = g * (size_t)group;
    const size_t last = min(first + (size_t)group, blocks);
    uint32_t x = group_entry[g];
    for (size_t b = first; b < last; b++) {
        block_entry[b] = x;
        x = exit_map[b * kMapStride + x];
    }
}

__global__ void __launch_bounds__(1024)
scan_counts(const uint32_t* __restrict__ count, size_t blocks,
            uint64_t* __restrict__ offset, uint64_t* __restrict__ result) {
    __shared__ uint64_t warp_sum[32];
    __shared__ uint64_t carry_s;
    if (threadIdx.x == 0) { carry_s = 0; }
    __syncthreads();
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    for (size_t base = 0; base < blocks; base += 1024) {
        const size_t i = base + threadIdx.x;
        const uint64_t v = i < blocks ? count[i] : 0;
        uint64_t s = v;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            const uint64_t t = __shfl_up_sync(0xFFFFFFFFu, s, d);
            if (lane >= d) { s += t; }
        }
        if (lane == 31) { warp_sum[wid] = s; }
        __syncthreads();
        if (wid == 0) {
            uint64_t ws = warp_sum[lane];
#pragma unroll
            for (int d = 1; d < 32; d <<= 1) {
                const uint64_t t = __shfl_up_sync(0xFFFFFFFFu, ws, d);
                if (lane >= d) { ws += t; }
            }
            warp_sum[lane] = ws;
        }
        __syncthreads();
        const uint64_t carry = carry_s;
        const uint64_t before = carry + (wid > 0 ? warp_sum[wid - 1] : 0) + s - v;
        if (i < blocks) { offset[i] = before; }
        __syncthreads();
        if (threadIdx.x == 1023) { carry_s = before + v; }
        __syncthreads();
    }
    if (threadIdx.x == 0) { result[0] = carry_s; }
}

// Symbol word of a match token (include/sqz_gpu.h): the bucket arithmetic of the reference's
// squeeze_encode_len / squeeze_encode_pos (squeeze.h:290-315, tables squeeze.h:29-79) done here,
// extra bits already in emission order (bit-reversed within their field).
//   lengths   3..10 -> buckets 0..7, no extra bits; above that four buckets per power of two of
//             len-3, with 258 kept in bucket 27 (squeeze.h:151-161)
//   distances 1..4 -> buckets 0..3; above that two buckets per power of two of dist-1
__device__ __forceinline__ uint32_t symbols_of_match(uint32_t len, uint32_t dist) {
    const uint32_t m = len - 3;
    uint32_t lb = m, lxb = 0;
    if (m >= 8) {
        const uint32_t k = 31u - (uint32_t)__clz((int)m);
        lxb = k - 2;
        lb = 4 * (k - 1) + ((m >> lxb) & 3);
    }
    const uint32_t lx = lxb ? __brev(m & ((1u << lxb) - 1)) >> (32 - lxb) : 0;
    const uint32_t q = dist - 1;
    uint32_t pb = q, pxb = 0;
    if (q >= 4) {
        const uint32_t k = 31u - (uint32_t)__clz((int)q);
        pxb = k - 1;
        pb = 2 * k + ((q >> pxb) & 1);
    }
    const uint32_t px = pxb ? __brev(q & ((1u << pxb) - 1)) >> (32 - pxb) : 0;
    return (257 + lb) | lx << 9 | pb << 14 | px << 19;
}

// The walk itself, one warp per block of kPB positions.  The warp stages the block's steps
// (len, or 1 for a literal) in shared memory with coalesced loads, lane 0 walks them from the
// block's entry offset -- about 30 cycles per token instead of a dependent global load -- and
// notes the positions it visits; then all lanes turn those positions into tokens (table word
// or literal byte, optionally as the coder's symbol word) and store them side by side.
// kEmit = false: count only (first pass, feeds the scan that places every block's tokens).
// The emit pass takes the same decision as the step (takes_match): under the lazy rule a literal
// can sit where the table word is a match.
constexpr int kParseWarps = 2;

template <bool kEmit, bool kSymbols, int kPB, bool kLazy>
__global__ void __launch_bounds__(32 * kParseWarps)
parse_walk(const uint8_t* __restrict__ shard, const uint32_t* __restrict__ table, size_t n,
           size_t blocks, uint32_t min_len, const uint32_t* __restrict__ block_entry,
           uint32_t* __restrict__ count, const uint64_t* __restrict__ offset,
           uint32_t* __restrict__ tokens, size_t cap) {
    __shared__ uint16_t step_s[kParseWarps][kPB];
    __shared__ uint16_t seen_s[kEmit ? kParseWarps : 1][kEmit ? kPB : 1];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const size_t b = (size_t)blockIdx.x * kParseWarps + warp;
    if (b >= blocks) { return; }                               // the whole warp leaves together
    const size_t b0 = b * kPB;
    const uint32_t size = (uint32_t)min((size_t)kPB, n - b0);
    for (uint32_t p = lane; p < size; p += 32) {
        step_s[warp][p] = (uint16_t)step_of<kLazy>(table[b0 + p], next_word<kLazy>(table, b0 + p), min_len);
    }
    __syncwarp();
    uint32_t c = 0;
    if (lane == 0) {
        uint32_t p = block_entry[b];
        while (p < size) {
            if (kEmit) { seen_s[warp][c] = (uint16_t)p; }
            p += step_s[warp][p];
            c++;
        }
    }
    c = __shfl_sync(0xFFFFFFFFu, c, 0);
    if (!kEmit) {
        if (lane == 0) { count[b] = c; }
        return;
    }
    __syncwarp();
    const uint64_t first = offset[b];
    for (uint32_t j = lane; j < c; j += 32) {
        const uint32_t p = seen_s[warp][j];
        const uint32_t w = table[b0 + p];
        const uint32_t len = w >> 16;
        uint32_t t;
        if (takes_match<kLazy>(w, next_word<kLazy>(table, b0 + p), min_len)) {
            t = kSymbols ? symbols_of_match(len, w & 0xFFFF) : w;
        } else {
            t = shard[b0 + p];
        }
        if (first + j < cap) { tokens[first + j] = t; }
    }
}

}  // namespace parse

// ---------------------------------------------------------------------------
// min-cost parse (SQZ_GPU_STREAM_MINCOST, include/sqz_gpu.h): the table is rewritten so that every
// word holds the chosen step -- (k << 16) | dist for a match of k <= len, 0 for a literal -- and the
// greedy parse above then walks exactly the min-cost path.  Segments of kSegment positions at global
// offsets that are multiples of kSegment; within one, backwards from its end e with c(j) = 0 for
// j >= e,
//   c(i) = min(8 + c(i + 1),  11 + len_extra(k) + pos_extra(dist) + c(i + k) for min_len <= k <= len)
// ties to the longest step.  The extra-bit counts are those of symbols_of_match.
// One warp per segment.  c(i) reads at most max_len <= 257 ahead, so the warp keeps the last
// kRing costs in a shared ring, which starts as zeros: c beyond the segment's end.  At a match the
// lanes share the lengths k and one redux.sync takes the minimum of (cost << 9) | (511 - k), which
// breaks ties towards the larger k and ranks the literal (k = 1) after every match of equal cost;
// costs stay below 2^18 (8 x 16384 for a segment of literals).  The table words of 32 positions come
// in with one coalesced load and leave, rewritten, with one store; each position reads only its own.
// ---------------------------------------------------------------------------
namespace mincost {

constexpr int kSegment = 16384;
constexpr int kRing = 512;
constexpr int kWarps = 4;        // segments per CTA

__device__ __forceinline__ uint32_t len_extra_bits(uint32_t len) {     // 3 <= len <= 257
    const uint32_t m = len - 3;
    return m >= 8 ? 29u - (uint32_t)__clz((int)m) : 0u;
}

__device__ __forceinline__ uint32_t dist_extra_bits(uint32_t dist) {   // 1 <= dist <= 32767
    const uint32_t q = dist - 1;
    return q >= 4 ? 30u - (uint32_t)__clz((int)q) : 0u;
}

__global__ void __launch_bounds__(32 * kWarps)
mincost_steps(uint32_t* __restrict__ table, size_t n, uint32_t min_len) {
    __shared__ uint32_t ring_s[kWarps][kRing];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const size_t s0 = ((size_t)blockIdx.x * kWarps + warp) * kSegment;
    if (s0 >= n) { return; }                                   // the whole warp leaves together
    const int size = (int)min((size_t)kSegment, n - s0);
    uint32_t* ring = ring_s[warp];
    for (int j = lane; j < kRing; j += 32) { ring[j] = 0; }
    __syncwarp();
    uint32_t after = 0;                                        // c(i + 1), the same in every lane
    for (int base = (size - 1) & ~31; base >= 0; base -= 32) {
        const int p = base + lane;
        const uint32_t mine = p < size ? table[s0 + p] : 0u;
        uint32_t out = 0;
        for (int l = min(31, size - 1 - base); l >= 0; l--) {
            const int i = base + l;
            const uint32_t w = __shfl_sync(0xFFFFFFFFu, mine, l);
            const uint32_t len = w >> 16;
            uint32_t best = (after + 8) << 9 | (511u - 1u);    // the literal
            if (len >= min_len) {
                const uint32_t fixed = 11u + dist_extra_bits(w & 0xFFFF);
                for (uint32_t k = min_len + lane; k <= len; k += 32) {
                    const uint32_t c = fixed + len_extra_bits(k) + ring[(i + k) & (kRing - 1)];
                    best = min(best, c << 9 | (511u - k));
                }
                best = __reduce_min_sync(0xFFFFFFFFu, best);
            }
            after = best >> 9;
            const uint32_t k = 511u - (best & 511u);
            if (lane == 0) { ring[i & (kRing - 1)] = after; }
            if (lane == l) { out = k == 1 ? 0u : (k << 16 | (w & 0xFFFF)); }
            __syncwarp();
        }
        if (p < size) { table[s0 + p] = out; }
    }
}

}  // namespace mincost

// ---------------------------------------------------------------------------
// launchers (device-buffer ABI)
// ---------------------------------------------------------------------------
static int check_rules(uint32_t min_len, uint32_t max_len, uint32_t max_dist) {
    if (min_len < 1 || max_len < min_len || max_len > sqz_gpu_max_len_limit ||
        max_dist < 1 || max_dist > sqz_gpu_max_dist_limit) {
        return fail(EINVAL, "rule parameters out of range (1 <= min_len <= max_len <= 512, 1 <= max_dist <= 65535)");
    }
    return 0;
}

// --- optional CUDA-event timing of the match kernel (bench.py roofline leg) and of the min-cost steps ---
static std::mutex g_time_mu;
static bool g_timing = false;

struct KernelTimes {
    std::vector<std::pair<cudaEvent_t, cudaEvent_t>> pending;
    double seconds = 0;
    uint64_t launches = 0;
};
static KernelTimes g_match_times, g_mincost_times;

static void timing_drain_locked(KernelTimes& t) {
    for (auto& pr : t.pending) {
        float ms = 0;
        if (cudaEventSynchronize(pr.second) == cudaSuccess &&
            cudaEventElapsedTime(&ms, pr.first, pr.second) == cudaSuccess) {
            t.seconds += 1e-3 * (double)ms;
            t.launches++;
        }
        cudaEventDestroy(pr.first);
        cudaEventDestroy(pr.second);
    }
    t.pending.clear();
}

// Events around one launcher call on stream s when timing is on: begin() records the start, end(ok)
// the stop, and the pair waits in t.pending until the next query.  With timing off both do nothing.
struct TimedLaunch {
    KernelTimes& t;
    cudaStream_t s;
    cudaEvent_t e0 = nullptr, e1 = nullptr;
    TimedLaunch(KernelTimes& times, cudaStream_t stream) : t(times), s(stream) {}
    cudaError_t begin() {
        {
            std::lock_guard<std::mutex> lk(g_time_mu);
            if (!g_timing) { return cudaSuccess; }
            if (t.pending.size() > 4096) { timing_drain_locked(t); }
        }
        cudaError_t e = cudaEventCreate(&e0);
        if (e == cudaSuccess) { e = cudaEventCreate(&e1); }
        if (e == cudaSuccess) { e = cudaEventRecord(e0, s); }
        return e;
    }
    void end(bool ok) {
        if (ok && e0 != nullptr && e1 != nullptr && cudaEventRecord(e1, s) == cudaSuccess) {
            std::lock_guard<std::mutex> lk(g_time_mu);
            t.pending.emplace_back(e0, e1);
        } else {
            if (e0 != nullptr) { cudaEventDestroy(e0); }
            if (e1 != nullptr) { cudaEventDestroy(e1); }
        }
        e0 = e1 = nullptr;
    }
    ~TimedLaunch() { end(false); }
};

static double kernel_seconds(KernelTimes& t, int reset, uint64_t* launches) {
    std::lock_guard<std::mutex> lk(g_time_mu);
    timing_drain_locked(t);
    const double avg = t.launches ? t.seconds / (double)t.launches : 0.0;
    if (launches != nullptr) { *launches = t.launches; }
    if (reset) { t.seconds = 0; t.launches = 0; }
    return avg;
}

extern "C" void sqz_gpu_set_timing(int on) {
    std::lock_guard<std::mutex> lk(g_time_mu);
    g_timing = on != 0;
}

extern "C" double sqz_gpu_match_kernel_seconds(int reset, uint64_t* launches) {
    return kernel_seconds(g_match_times, reset, launches);
}

extern "C" double sqz_gpu_mincost_kernel_seconds(int reset, uint64_t* launches) {
    return kernel_seconds(g_mincost_times, reset, launches);
}

static unsigned long long* g_tile_cycles = nullptr;   // debugging aid, see sqz_gpu_debug_tile_cycles

extern "C" void sqz_gpu_debug_tile_cycles(unsigned long long* d_buf) { g_tile_cycles = d_buf; }

// A/B switch for tests and measurements; per calling thread, so that it is no process-wide state
static thread_local int g_kernel_choice = 0;   // 0 auto, 1 thread-per-position (v1), 2 bit-sliced (v2)

extern "C" int sqz_gpu_select_kernel(int which) {
    if (which < 0 || which > 2) { return fail(EINVAL, "kernel choice must be 0, 1 or 2"); }
    g_kernel_choice = which;
    return 0;
}

// ---------------------------------------------------------------------------
// per-device set-up: function attributes, the two side streams of the edge tiles, SM count
// ---------------------------------------------------------------------------
constexpr int kMaxDevices = 64;

struct DeviceState {
    std::once_flag once;
    cudaError_t err = cudaSuccess;
    cudaStream_t side = nullptr, side2 = nullptr;
    int sms = 0;
};
static DeviceState g_dev[kMaxDevices];

template <typename K>
static cudaError_t allow_smem(K kernel, int bytes) {
    cudaError_t e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes);
    // several CTAs per SM only fit when the L1/shared split favours shared memory
    if (e == cudaSuccess) {
        e = cudaFuncSetAttribute(kernel, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared);
    }
    return e;
}

static int device_state(DeviceState** out) {
    int dev = 0;
    CU(cudaGetDevice(&dev));
    if (dev < 0 || dev >= kMaxDevices) { return fail(ENODEV, "device index out of range"); }
    DeviceState& d = g_dev[dev];
    std::call_once(d.once, [&d, dev] {
        const int big4 = v2::geometry(sqz_gpu_max_len_limit, sqz_gpu_max_dist_limit, true, true, 4).smem_bytes;
        const int big1 = v2::geometry(sqz_gpu_max_len_limit, sqz_gpu_max_dist_limit, true, true, 1).smem_bytes;
        cudaError_t e = allow_smem(v2::match_table<3, false, 4>, big4);
        if (e == cudaSuccess) { e = allow_smem(v2::match_table<3, true, 4>, big4); }
        if (e == cudaSuccess) { e = allow_smem(v2::match_table<2, false, 4>, big4); }
        if (e == cudaSuccess) { e = allow_smem(v2::match_table<2, true, 4>, big4); }
        if (e == cudaSuccess) { e = allow_smem(v2::match_table<3, false, 1>, big1); }
        if (e == cudaSuccess) { e = allow_smem(v2::match_table<3, true, 1>, big1); }
        if (e == cudaSuccess) { e = allow_smem(v2::match_table<2, false, 1>, big1); }
        if (e == cudaSuccess) { e = allow_smem(v2::match_table<2, true, 1>, big1); }
        if (e == cudaSuccess) {
            e = cudaFuncSetAttribute(v1::match_table, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                     (int)v1::smem_bytes(sqz_gpu_max_len_limit, sqz_gpu_max_dist_limit));
        }
        if (e == cudaSuccess) {
            e = allow_smem(v2::finish_marked, v2::finish_shape(1LL << 30, sqz_gpu_max_len_limit, sqz_gpu_max_dist_limit, 148).smem_bytes);
        }
        if (e == cudaSuccess) { e = cudaDeviceGetAttribute(&d.sms, cudaDevAttrMultiProcessorCount, dev); }
        if (e == cudaSuccess) { e = cudaStreamCreateWithFlags(&d.side, cudaStreamNonBlocking); }
        if (e == cudaSuccess) { e = cudaStreamCreateWithFlags(&d.side2, cudaStreamNonBlocking); }
        d.err = e;
    });
    if (d.err != cudaSuccess) { return fail(cuda_code(d.err), "per-device set-up", d.err); }
    *out = &d;
    return 0;
}

static int sm_count() {
    DeviceState* d = nullptr;
    return device_state(&d) == 0 ? d->sms : 148;
}

// an event that lives as long as one launcher call, whatever way the call ends
struct ScopedEvent {
    cudaEvent_t e = nullptr;
    ~ScopedEvent() { if (e != nullptr) { cudaEventDestroy(e); } }
    cudaError_t create() { return cudaEventCreateWithFlags(&e, cudaEventDisableTiming); }
};

// ---------------------------------------------------------------------------
// workspace of the match table: the segment cursor of phase 2 and phase 1's work list
// (one bit per position).  Callers of the _ws entry point own it; the plain entry point
// borrows a parked one (a kWorkspace stage, below) and gives it back on the caller's stream.
// ---------------------------------------------------------------------------
constexpr size_t kCursorBytes = 256;

struct SlicePlan { int q; int slices; int slice_words; size_t stride; };

// How a shard is cut (match_bitsliced.cuh).  From a wave of throughput tiles on (444 resident CTAs of
// 16,256 positions: 148 SMs x 3) it is tiles only, four blocks per thread.  Below that the latency
// shape takes over -- one block per thread, 3,968 positions per CTA, five CTAs per SM -- and the
// distance range is split into as many slices as it takes to give the device about two waves of
// CTAs (a power of two, at most 32).  Fixed numbers, so that the workspace size depends on n only.
constexpr size_t kWaveQ4 = 148 * 3, kWaveQ1 = 148 * 5;

static SlicePlan slice_plan(size_t n, uint32_t max_dist) {
    SlicePlan sp{4, 1, 0, 0};
    const size_t tiles4 = (n + v2::tile_pos(4) - 1) / v2::tile_pos(4);
    int force_q = 0, force_s = 0;
#ifdef SQZ_TUNING
    if (const char* e = getenv("SQZ_Q")) { force_q = atoi(e); }
    if (const char* e = getenv("SQZ_SLICES")) { force_s = atoi(e); }
#endif
    if (n == 0 || (force_q == 0 && tiles4 > kWaveQ4) || force_q == 4) {
        if (force_s <= 1) { return sp; }
    } else {
        sp.q = 1;
    }
    const size_t tiles = (n + v2::tile_pos(sp.q) - 1) / v2::tile_pos(sp.q);
    const size_t want = force_s > 0 ? (size_t)force_s : (2 * (sp.q == 1 ? kWaveQ1 : kWaveQ4) + tiles - 1) / tiles;
    int slices = 1;
    while ((size_t)slices < want && slices < 32) { slices <<= 1; }
    const int words = (int)((max_dist + 31) / 32);                 // word distances of a full scan
    int per = (words + slices - 1) / slices;
    per = (per + 31) / 32 * 32;                                    // whole units of the resume tag (1024 distances)
    slices = (words + per - 1) / per;
    if (slices <= 1) { return sp; }
    sp.slices = slices;
    sp.slice_words = per;
    sp.stride = (n + 63) / 64 * 64;
    return sp;
}

static size_t mask_bytes(size_t n) { return (((n + 31) / 32 + 8) * 4 + 255) / 256 * 256; }

static size_t slice_bytes(const SlicePlan& sp) { return sp.slices > 1 ? (size_t)(sp.slices - 1) * sp.stride * 4 : 0; }

// A workspace sized for n serves every shard of at most n positions (the pipeline's slots are
// sized once and see chunks of many sizes): the slice tables are what a smaller shard may need
// more of, so their part is the largest any n' <= n asks for.
extern "C" size_t sqz_gpu_match_workspace(size_t n) {
    size_t tables = slice_bytes(slice_plan(n, sqz_gpu_max_dist_limit));
    const size_t tp = v2::tile_pos(1);
    const size_t tiles = std::min<size_t>((n + tp - 1) / tp, 2 * kWaveQ1 + 1);
    for (size_t t = 1; t <= tiles; t++) {
        tables = std::max(tables, slice_bytes(slice_plan(std::min(n, t * tp), sqz_gpu_max_dist_limit)));
    }
#ifdef SQZ_TUNING
    tables = std::max(tables, (size_t)31 * ((std::min<size_t>(n, (size_t)64 << 20) + 63) / 64 * 64) * 4);   // whatever SQZ_SLICES asks for
#endif
    return kCursorBytes + mask_bytes(n) + tables;
}

// ---------------------------------------------------------------------------
// staging buffers, kept between calls
// ---------------------------------------------------------------------------

// the calling thread's current device is the caller's business: every entry point that has to
// switch (an explicit stream device, the multi-device call) puts it back on the way out
struct DeviceScope {
    int saved = -1;
    DeviceScope() { if (cudaGetDevice(&saved) != cudaSuccess) { saved = -1; cudaGetLastError(); } }
    ~DeviceScope() { if (saved >= 0) { cudaSetDevice(saved); } }
};

// What a stage holds depends on what its user needs:
//   kWorkspace  the match workspace only: sqz_gpu_match_table_device borrows it on the caller's stream.
//   the others  the workspace, a stream of their own, the shard with its halos (sized for the library's
//               limits), its match table, the parse result (device and pinned) and the events, and
//     kTable    the table's two 16-bit halves (sqz_gpu_match_table);
//     kTokens   the tokens, the parse workspace and the exit map (sqz_gpu_tokens, sqz_gpu_tokens_multi);
//     kConsumer kTokens plus pinned tokens and a stream of the highest priority (sqz_gpu_stream_*).
enum { kWorkspace, kTable, kTokens, kConsumer };

// the buffers and streams for one shard of at most `cap` positions on one device
struct Stage {
    int device = -1, kind = kWorkspace;
    size_t cap = 0;
    size_t bytes = 0;                 // device + pinned memory it holds
    cudaEvent_t idle = nullptr;       // all its work is over (recorded when it is given back)
    void* d_mwork = nullptr;          // match workspace (cursor + work list of phase 2)
    cudaStream_t stream = nullptr;
    cudaStream_t ahead_of_all = nullptr;   // highest priority: a consumer's parse and token copy
    cudaEvent_t done = nullptr;       // everything of the chunk has been issued and finished
    cudaEvent_t parsed = nullptr;     // the chunk's token count and overshoot are in h_result
    cudaEvent_t tabled = nullptr;     // the match table is complete (multi-device call: its exit map is in h_map)
    uint8_t* d_data = nullptr;        // back halo + shard + ahead halo
    uint32_t* d_table = nullptr;
    uint64_t* d_result = nullptr;     // [0] tokens, [1] overshoot (next shard's entry)
    uint64_t* h_result = nullptr;     // pinned
    uint16_t* d_len = nullptr;
    uint16_t* d_dist = nullptr;
    uint32_t* d_tokens = nullptr;
    void* d_work = nullptr;           // parse workspace
    uint16_t* d_map = nullptr;        // exit map
    uint16_t* h_map = nullptr;        // pinned
    uint32_t* h_tokens = nullptr;     // pinned
    size_t first = 0, n = 0, back = 0;     // the shard it holds: [first, first + n) of the input
    bool busy = false;
};

// on the current device, which is s.device
static int stage_alloc(Stage& s) {
    auto dev = [&s](auto** p, size_t b) { s.bytes += b; return cudaMalloc(p, b); };
    auto pin = [&s](auto** p, size_t b) { s.bytes += b; return cudaHostAlloc(p, b, cudaHostAllocDefault); };
    CU(cudaEventCreateWithFlags(&s.idle, cudaEventDisableTiming));
    CU(dev(&s.d_mwork, sqz_gpu_match_workspace(s.cap)));
    if (s.kind == kWorkspace) { return 0; }
    CU(cudaStreamCreateWithFlags(&s.stream, cudaStreamNonBlocking));
    CU(cudaEventCreateWithFlags(&s.done, cudaEventDisableTiming));
    CU(cudaEventCreateWithFlags(&s.parsed, cudaEventDisableTiming));
    CU(cudaEventCreateWithFlags(&s.tabled, cudaEventDisableTiming));
    CU(dev(&s.d_data, (size_t)sqz_gpu_max_dist_limit + s.cap + sqz_gpu_max_len_limit + 64));
    CU(dev(&s.d_table, s.cap * 4 + 4));   // + the seam word a lazy parse reads after a full shard
    CU(dev(&s.d_result, 16));
    CU(pin(&s.h_result, 16));
    if (s.kind == kTable) {
        CU(dev(&s.d_len, s.cap * 2));
        CU(dev(&s.d_dist, s.cap * 2));
        return 0;
    }
    CU(dev(&s.d_tokens, s.cap * 4 + 16));
    CU(dev(&s.d_work, parse::workspace(s.cap)));
    CU(dev(&s.d_map, parse::kMapStride * 2));
    CU(pin(&s.h_map, parse::kMapStride * 2));
    if (s.kind == kConsumer) {
        CU(pin(&s.h_tokens, s.cap * 4 + 16));
        int least = 0, greatest = 0;
        CU(cudaDeviceGetStreamPriorityRange(&least, &greatest));
        CU(cudaStreamCreateWithPriority(&s.ahead_of_all, cudaStreamNonBlocking, greatest));
    }
    return 0;
}

static void stage_free(Stage& s) {
    DeviceScope keep;
    cudaSetDevice(s.device);
    if (s.idle) { cudaEventSynchronize(s.idle); }
    if (s.stream) { cudaStreamSynchronize(s.stream); }
    if (s.ahead_of_all) { cudaStreamSynchronize(s.ahead_of_all); }
    cudaFree(s.d_mwork); cudaFree(s.d_data); cudaFree(s.d_table); cudaFree(s.d_result); cudaFree(s.d_len);
    cudaFree(s.d_dist); cudaFree(s.d_tokens); cudaFree(s.d_work); cudaFree(s.d_map);
    cudaFreeHost(s.h_result); cudaFreeHost(s.h_map); cudaFreeHost(s.h_tokens);
    for (cudaEvent_t e : {s.idle, s.done, s.parsed, s.tabled}) { if (e) { cudaEventDestroy(e); } }
    for (cudaStream_t q : {s.stream, s.ahead_of_all}) { if (q) { cudaStreamDestroy(q); } }
    s = Stage();
}

// Allocating and freeing gigabytes of device and pinned memory per call costs more than the search of
// a small input and stalls the device: finished calls park their stages here, and a later call takes
// back one of the same device and kind that is large enough and at most four times too large.  Per
// device at most kParkStages stages and kParkBytes of device + pinned memory stay parked, oldest out
// first (a 512 MiB shard of sqz_gpu_tokens_multi holds about 4.7 GiB); sqz_gpu_release() frees them.
static std::mutex g_park_mu;
static std::vector<Stage> g_park;                 // oldest first
constexpr size_t kParkStages = 8;
constexpr size_t kParkBytes = (size_t)12 << 30;

// a stage of this kind for n positions on `device`, which is the current device
static int stage_take(Stage& s, int device, int kind, size_t n) {
    // no device holds 2^60 positions, and beyond them the power of two below and the stage's byte counts
    // (several bytes per position) would overflow
    if (n > ((size_t)1 << 60)) { return fail(ENOMEM, "staging for more than 2^60 positions"); }
    size_t cap = (size_t)1 << 20;            // a power of two (>= 1 Mi) so that calls of similar size share stages
    while (cap < n) { cap <<= 1; }
    {
        std::lock_guard<std::mutex> lk(g_park_mu);
        for (size_t k = 0; k < g_park.size(); k++) {
            const Stage& c = g_park[k];
            if (c.device == device && c.kind == kind && c.cap >= cap && c.cap <= 4 * cap &&
                cudaEventQuery(c.idle) == cudaSuccess) {
                s = c;
                s.busy = false;
                g_park.erase(g_park.begin() + (long)k);
                return 0;
            }
        }
        cudaGetLastError();                  // cudaErrorNotReady of a stage still in use is not an error
    }
    s = Stage();
    s.device = device;
    s.kind = kind;
    s.cap = cap;
    const int r = stage_alloc(s);
    if (r != 0) { stage_free(s); }
    return r;
}

// parks a stage whose work so far is all joined into `q`
static void stage_give_back(Stage& s, cudaStream_t q) {
    if (s.idle == nullptr) { return; }       // never allocated
    cudaError_t ce;
    {
        DeviceScope keep;
        cudaSetDevice(s.device);
        ce = cudaEventRecord(s.idle, q);
    }
    // not kept: a stage without its idle mark, and one above the bound on its own (it would only push
    // the others out)
    std::vector<Stage> victims;
    if (ce != cudaSuccess || s.bytes > kParkBytes) {
        victims.push_back(s);
    } else {
        std::lock_guard<std::mutex> lk(g_park_mu);
        g_park.push_back(s);
        size_t count = 0, bytes = 0;
        for (const Stage& c : g_park) {
            if (c.device == s.device) { count++; bytes += c.bytes; }
        }
        for (size_t k = 0; k < g_park.size() && (count > kParkStages || bytes > kParkBytes);) {
            if (g_park[k].device != s.device) { k++; continue; }
            count--;
            bytes -= g_park[k].bytes;
            victims.push_back(g_park[k]);
            g_park.erase(g_park.begin() + (long)k);
        }
    }
    s = Stage();
    for (Stage& v : victims) { stage_free(v); }
}

// waits for the stage's stream and parks the stage; returns rc, or the wait's error when rc is 0
static int stage_finish(Stage& s, int rc) {
    if (s.stream != nullptr) {
        const cudaError_t ce = cudaStreamSynchronize(s.stream);
        if (ce != cudaSuccess && rc == 0) { rc = fail(cuda_code(ce), "cudaStreamSynchronize", ce); }
    }
    stage_give_back(s, s.stream);
    return rc;
}

extern "C" void sqz_gpu_release(void) {
    std::vector<Stage> all;
    {
        std::lock_guard<std::mutex> lk(g_park_mu);
        all.swap(g_park);
    }
    for (Stage& s : all) { stage_free(s); }
}

static int launch_v1(const uint8_t* d_shard, size_t back, size_t n, size_t ahead, uint32_t min_len,
                     uint32_t max_len, uint32_t max_dist, uint32_t* d_table, cudaStream_t s) {
    DeviceState* dv = nullptr;
    if (int r = device_state(&dv)) { return r; }
    const size_t tiles = (n + v1::kThreads - 1) / v1::kThreads;
    if (tiles > 0x7FFFFFFFull) { return fail(EINVAL, "shard too large for one launch"); }
    v1::match_table<<<(unsigned)tiles, v1::kThreads, v1::smem_bytes(max_len, max_dist), s>>>(
        d_shard, (long long)back, (long long)n, (long long)ahead, min_len, max_len, max_dist, d_table);
    LAUNCHED("match_table_v1");
    return 0;
}

// The seam word of a lazy parse: the lazy step at a shard's last position reads table[n], the best match
// at the first position after the shard, which belongs to the next shard (or chunk) and is searched there
// only later, if at all.  That one position is searched here on its own, by the exact thread-per-position
// kernel.  Its look-back is the shard and the halo before it; its look-ahead is the shard's own halo, which
// holds every byte a match there can reach (min(rest, max_len) bytes).  At the end of the input
// (ahead = 0) table[n] is 0: len(bytes) = 0.  The same halos as the shard's table search, nothing more.
static int seam_word(const uint8_t* d_shard, size_t back, size_t n, size_t ahead, uint32_t min_len,
                     uint32_t max_len, uint32_t max_dist, uint32_t* d_table, cudaStream_t s) {
    if (ahead == 0) {
        CU(cudaMemsetAsync(d_table + n, 0, 4, s));
        return 0;
    }
    return launch_v1(d_shard + n, back + n, 1, ahead - 1, min_len, max_len, max_dist, d_table + n, s);
}

template <int kMinLen, int kQ>
static int launch_tiles(const SlicePlan& sp, const uint8_t* d_shard, size_t back, size_t n, size_t ahead, uint32_t max_len,
                        uint32_t max_dist, uint32_t* d_table, void* d_work, cudaStream_t s) {
    DeviceState* dv = nullptr;
    if (int r = device_state(&dv)) { return r; }
    // Tiles whose every position sees the full max_dist window and max_len of
    // look-ahead run the plain variant; the rest (start of the first shard, end
    // of the last one, a partial last tile) run the variant with a validity plane.
    const long long tp = v2::tile_pos(kQ);
    const long long tiles = ((long long)n + tp - 1) / tp;
    if (tiles > 0x7FFFFFFFll) { return fail(EINVAL, "shard too large for one launch"); }
    long long t_lo = back >= max_dist ? 0 : ((long long)max_dist - (long long)back + tp - 1) / tp;
    long long tail = (long long)n + (long long)std::min<size_t>(ahead, max_len) - (long long)max_len;
    long long t_hi = tail <= 0 ? 0 : tail / tp;
    t_lo = std::min(t_lo, tiles);
    t_hi = std::max(std::min(t_hi, tiles), t_lo);
    if ((unsigned long long)n > 0xFFFFFFFFull) { return fail(EINVAL, "shard too large for one launch"); }
    unsigned int* d_counters = static_cast<unsigned int*>(d_work);
    uint32_t* d_open = reinterpret_cast<uint32_t*>(static_cast<uint8_t*>(d_work) + kCursorBytes);
    CU(cudaMemsetAsync(d_counters, 0, 16, s));
    const int smem_main = v2::geometry(max_len, max_dist, false, false, kQ).smem_bytes;
    const int smem_edge = v2::geometry(max_len, max_dist, true, false, kQ).smem_bytes;
    // small shards: the distance range is split across CTAs as well, the slices' tables sit behind
    // the work list and are folded into d_table afterwards
    uint32_t* d_slices = sp.slices > 1 ? reinterpret_cast<uint32_t*>(static_cast<uint8_t*>(d_work) + kCursorBytes + mask_bytes(n)) : nullptr;
    // The few edge tiles run concurrently with the interior tiles: leading and trailing edge
    // tiles each on a side stream of the device, forked from and joined back into `s`.
    const bool lead = t_lo > 0, trail = tiles > t_hi;
    ScopedEvent fork, join1, join2;
    if (lead || trail) {
        CU(fork.create());
        CU(cudaEventRecord(fork.e, s));
    }
    // sliced: the nearest slice first (into d_table), then the others seeded with its result
    const int smem_main_seeded = v2::geometry(max_len, max_dist, false, true, kQ).smem_bytes;
    const int smem_edge_seeded = v2::geometry(max_len, max_dist, true, true, kQ).smem_bytes;
    auto launch = [&](auto kernel, long long first, long long count, bool edge, cudaStream_t on, int slices,
                      int slice_words, long long stride, uint32_t* slice_tables) -> cudaError_t {
        kernel<<<dim3((unsigned)count, 1), v2::kThreads, edge ? smem_edge : smem_main, on>>>(
            d_shard, (long long)back, (long long)n, (long long)ahead, max_len, max_dist, d_table, slice_tables,
            slices > 1 ? nullptr : d_open, (int)first, slice_words, stride, 0, nullptr, g_tile_cycles);
        g_launches.fetch_add(1, std::memory_order_relaxed);
        cudaError_t e = cudaGetLastError();
        if (e != cudaSuccess || slices <= 1) { return e; }
        kernel<<<dim3((unsigned)count, (unsigned)(slices - 1)), v2::kThreads, edge ? smem_edge_seeded : smem_main_seeded, on>>>(
            d_shard, (long long)back, (long long)n, (long long)ahead, max_len, max_dist, d_table, slice_tables,
            nullptr, (int)first, slice_words, stride, 1, d_table, g_tile_cycles);
        g_launches.fetch_add(1, std::memory_order_relaxed);
        return cudaGetLastError();
    };
    cudaError_t le = cudaSuccess;
    if (lead) {
        CU(cudaStreamWaitEvent(dv->side, fork.e, 0));
        le = launch(v2::match_table<kMinLen, true, kQ>, 0, t_lo, true, dv->side, sp.slices, sp.slice_words, (long long)sp.stride, d_slices);
        if (le != cudaSuccess) { return fail(cuda_code(le), "match_table_v2_edge", le); }
        CU(join1.create());
        CU(cudaEventRecord(join1.e, dv->side));
    }
    if (trail) {
        CU(cudaStreamWaitEvent(dv->side2, fork.e, 0));
        le = launch(v2::match_table<kMinLen, true, kQ>, t_hi, tiles - t_hi, true, dv->side2, sp.slices, sp.slice_words, (long long)sp.stride, d_slices);
        if (le != cudaSuccess) { return fail(cuda_code(le), "match_table_v2_edge", le); }
        CU(join2.create());
        CU(cudaEventRecord(join2.e, dv->side2));
    }
    if (t_hi > t_lo) {
        le = launch(v2::match_table<kMinLen, false, kQ>, t_lo, t_hi - t_lo, false, s, sp.slices, sp.slice_words, (long long)sp.stride, d_slices);
        if (le != cudaSuccess) { return fail(cuda_code(le), "match_table_v2", le); }
    }
    if (join1.e != nullptr) { CU(cudaStreamWaitEvent(s, join1.e, 0)); }
    if (join2.e != nullptr) { CU(cudaStreamWaitEvent(s, join2.e, 0)); }
    if (sp.slices > 1) {
        const unsigned grid = (unsigned)std::min<size_t>((n + 255) / 256, (size_t)dv->sms * 8);
        v2::combine_slices<<<grid, 256, 0, s>>>(d_table, d_slices, 0LL, (long long)n, (long long)sp.stride, sp.slices, d_open);
        LAUNCHED("combine_slices");
    }
    const v2::FinishShape fs = v2::finish_shape((long long)n, max_len, max_dist, dv->sms);
    const long long chunks = ((long long)n + fs.chunk - 1) / fs.chunk;
    const unsigned finish_ctas = (unsigned)std::min<long long>(chunks, (long long)dv->sms * v2::kFinishCtasPerSm);
    v2::finish_marked<<<finish_ctas, v2::kThreads, fs.smem_bytes, s>>>(
        d_shard, (long long)back, (long long)n, (long long)ahead, (uint32_t)kMinLen, max_len, max_dist, d_table, d_open,
        d_counters, g_tile_cycles ? g_tile_cycles + (1 << 20) : nullptr, fs.chunk, fs.sub);
    LAUNCHED("match_finish_marked");
    return 0;
}

template <int kMinLen>
static int launch_v2(const uint8_t* d_shard, size_t back, size_t n, size_t ahead, uint32_t max_len,
                     uint32_t max_dist, uint32_t* d_table, void* d_work, cudaStream_t s) {
    const SlicePlan sp = slice_plan(n, max_dist);
    return sp.q == 1 ? launch_tiles<kMinLen, 1>(sp, d_shard, back, n, ahead, max_len, max_dist, d_table, d_work, s)
                     : launch_tiles<kMinLen, 4>(sp, d_shard, back, n, ahead, max_len, max_dist, d_table, d_work, s);
}

extern "C" int sqz_gpu_match_table_device_ws(const uint8_t* d_shard, size_t back, size_t n,
                                             size_t ahead, uint32_t min_len, uint32_t max_len,
                                             uint32_t max_dist, uint32_t* d_table, void* d_work, void* stream) {
    if (int r = check_rules(min_len, max_len, max_dist)) { return r; }
    if (n == 0) { return 0; }
    if (d_work == nullptr) { return fail(EINVAL, "null workspace"); }
    cudaStream_t s = (cudaStream_t)stream;
    TimedLaunch timed(g_match_times, s);
    CU(timed.begin());
    const int choice = g_kernel_choice;
    int r;
    const bool v2_ok = max_len > 32;      // the bit-sliced kernel measures runs in a 32-bit window
    if (choice != 1 && v2_ok && min_len == 3)      { r = launch_v2<3>(d_shard, back, n, ahead, max_len, max_dist, d_table, d_work, s); }
    else if (choice != 1 && v2_ok && min_len == 2) { r = launch_v2<2>(d_shard, back, n, ahead, max_len, max_dist, d_table, d_work, s); }
    else { r = launch_v1(d_shard, back, n, ahead, min_len, max_len, max_dist, d_table, s); }
    timed.end(r == 0);
    return r;
}

extern "C" int sqz_gpu_match_table_device(const uint8_t* d_shard, size_t back, size_t n,
                                          size_t ahead, uint32_t min_len, uint32_t max_len,
                                          uint32_t max_dist, uint32_t* d_table, void* stream) {
    if (int r = check_rules(min_len, max_len, max_dist)) { return r; }
    if (n == 0) { return 0; }
    int dev = 0;
    CU(cudaGetDevice(&dev));
    Stage w;
    if (int r = stage_take(w, dev, kWorkspace, n)) { return r; }
    const int r = sqz_gpu_match_table_device_ws(d_shard, back, n, ahead, min_len, max_len, max_dist, d_table, w.d_mwork, stream);
    stage_give_back(w, (cudaStream_t)stream);
    return r;
}

extern "C" int sqz_gpu_match_seam_device(const uint8_t* d_shard, size_t back, size_t n, size_t ahead,
                                         uint32_t min_len, uint32_t max_len, uint32_t max_dist,
                                         uint32_t* d_table, void* stream) {
    if (int r = check_rules(min_len, max_len, max_dist)) { return r; }
    return seam_word(d_shard, back, n, ahead, min_len, max_len, max_dist, d_table, (cudaStream_t)stream);
}

extern "C" int sqz_gpu_unpack_table_device(const uint32_t* d_table, size_t n,
                                           uint16_t* d_len, uint16_t* d_dist, void* stream) {
    if (n == 0) { return 0; }
    const unsigned blocks = (unsigned)std::min<size_t>((n + 255) / 256, (size_t)sm_count() * 16);
    unpack_table<<<blocks, 256, 0, (cudaStream_t)stream>>>(d_table, n, d_len, d_dist);
    LAUNCHED("unpack_table");
    return 0;
}

extern "C" size_t sqz_gpu_parse_workspace(size_t n) { return parse::workspace(n); }

// lazy: the lazy rule, which reads d_table[n] as well
static int parse_maps(const uint32_t* d_table, size_t n, uint32_t min_len, uint32_t max_len,
                      const parse::Work& w, cudaStream_t s, bool lazy) {
#define SQZ_MAP(PB, LAZY) parse::parse_exit_map<PB, LAZY><<<(unsigned)w.blocks, 256, 0, s>>>(d_table, n, min_len, max_len, \
                                                                                             w.exit_map)
    if (lazy) { if (w.pb == parse::kPBSmall) { SQZ_MAP(parse::kPBSmall, true); } else { SQZ_MAP(parse::kPBLarge, true); } }
    else      { if (w.pb == parse::kPBSmall) { SQZ_MAP(parse::kPBSmall, false); } else { SQZ_MAP(parse::kPBLarge, false); } }
#undef SQZ_MAP
    LAUNCHED("parse_exit_map");
    parse::chain_groups<<<(unsigned)w.groups, 256, 0, s>>>(w.exit_map, w.blocks, w.group, max_len, w.group_map);
    LAUNCHED("chain_groups");
    return 0;
}

// the two walks of the parse (count, then emit) with the scan that places every block's tokens between them
template <int kPB, bool kLazy>
static int parse_walks(const uint8_t* d_shard, const uint32_t* d_table, size_t n, uint32_t min_len,
                       const parse::Work& w, uint32_t* d_tokens, size_t cap, uint64_t* d_result,
                       cudaStream_t s, bool symbols) {
    const unsigned wb = (unsigned)((w.blocks + parse::kParseWarps - 1) / parse::kParseWarps);
    const unsigned wt = 32 * parse::kParseWarps;
    parse::parse_walk<false, false, kPB, kLazy><<<wb, wt, 0, s>>>(d_shard, d_table, n, w.blocks, min_len, w.block_entry,
                                                                  w.count, nullptr, nullptr, 0);
    LAUNCHED("parse_count");
    parse::scan_counts<<<1, 1024, 0, s>>>(w.count, w.blocks, w.offset, d_result);
    LAUNCHED("scan_counts");
#define SQZ_EMIT(SYM) parse::parse_walk<true, SYM, kPB, kLazy><<<wb, wt, 0, s>>>(d_shard, d_table, n, w.blocks, min_len, \
                                                                                 w.block_entry, nullptr, w.offset, d_tokens, cap)
    if (symbols) { SQZ_EMIT(true); } else { SQZ_EMIT(false); }
#undef SQZ_EMIT
    LAUNCHED("parse_emit");
    return 0;
}

// entry either from device memory (d_entry != null) or immediate; lazy: the lazy rule, for which
// d_table holds n + 1 words (the last one the best match at the first position after the shard, 0
// at the end of the input)
static int parse_launch(const uint8_t* d_shard, const uint32_t* d_table, size_t n,
                        const uint32_t* d_entry, uint32_t entry, uint32_t min_len,
                        uint32_t max_len, uint32_t* d_tokens, size_t cap, void* d_work,
                        uint64_t* d_result, cudaStream_t s, bool symbols = false, bool lazy = false) {
    if (n == 0) {
        // nothing to parse: count 0, overshoot = entry
        CU(cudaMemsetAsync(d_result, 0, 16, s));
        if (d_entry != nullptr) {
            CU(cudaMemcpyAsync(d_result + 1, d_entry, 4, cudaMemcpyDeviceToDevice, s));
        } else if (entry != 0) {
            return fail(EINVAL, "entry into an empty shard");
        }
        return 0;
    }
    parse::Work w = parse::carve(d_work, n);
    if (w.blocks > 0x7FFFFFFFull) { return fail(EINVAL, "shard too large for one launch"); }
    if (int r = parse_maps(d_table, n, min_len, max_len, w, s, lazy)) { return r; }
    parse::chain_top<<<1, 1, 0, s>>>(w.group_map, w.groups, d_entry, entry, w.group_entry, d_result);
    LAUNCHED("chain_top");
    parse::chain_expand<<<(unsigned)((w.groups + 127) / 128), 128, 0, s>>>(
        w.exit_map, w.blocks, w.group, w.groups, w.group_entry, w.block_entry);
    LAUNCHED("chain_expand");
    const bool small = w.pb == parse::kPBSmall;
    if (lazy) {
        return small ? parse_walks<parse::kPBSmall, true>(d_shard, d_table, n, min_len, w, d_tokens, cap, d_result, s, symbols)
                     : parse_walks<parse::kPBLarge, true>(d_shard, d_table, n, min_len, w, d_tokens, cap, d_result, s, symbols);
    }
    return small ? parse_walks<parse::kPBSmall, false>(d_shard, d_table, n, min_len, w, d_tokens, cap, d_result, s, symbols)
                 : parse_walks<parse::kPBLarge, false>(d_shard, d_table, n, min_len, w, d_tokens, cap, d_result, s, symbols);
}

// symbol words only exist for the bitstream's own limits (squeeze.h:13-15, 529-545)
static int check_symbol_rules(uint32_t min_len, uint32_t max_len, uint32_t max_dist) {
    // 258 has a bucket (27, extra bits 31) but no decoder accepts it: squeeze.h:529-545 and
    // sqz_decompress reject every length above 257 with EINVAL
    if (min_len < 3 || max_len > 257 || max_dist > 0x7FFF) {
        return fail(EINVAL, "symbol words need min_len >= 3, max_len <= 257, max_dist <= 32767");
    }
    return 0;
}

// the flag bits an entry point takes (SQZ_GPU_STREAM_*); any other bit is EINVAL
static int check_flags(uint32_t flags, uint32_t allowed) {
    if ((flags & ~allowed) != 0) { return fail(EINVAL, "flag bits this entry point does not take"); }
    return 0;
}

// The min-cost parse prices matches with the buckets of the symbol words, so it exists within their
// limits only, and it is a parse of its own: not together with the lazy rule.
static int check_mincost(uint32_t flags, uint32_t min_len, uint32_t max_len, uint32_t max_dist) {
    if ((flags & SQZ_GPU_STREAM_MINCOST) == 0) { return 0; }
    if ((flags & SQZ_GPU_STREAM_LAZY) != 0) { return fail(EINVAL, "the min-cost and the lazy parse exclude each other"); }
    return check_symbol_rules(min_len, max_len, max_dist);
}

// Rewrites d_table[0, n) into min-cost steps; the shard starts at a global offset that is a multiple
// of mincost::kSegment.
static int mincost_launch(uint32_t* d_table, size_t n, uint32_t min_len, cudaStream_t s) {
    if (n == 0) { return 0; }
    const size_t segments = (n + mincost::kSegment - 1) / mincost::kSegment;
    const size_t ctas = (segments + mincost::kWarps - 1) / mincost::kWarps;
    if (ctas > 0x7FFFFFFFull) { return fail(EINVAL, "shard too large for one launch"); }
    TimedLaunch timed(g_mincost_times, s);
    CU(timed.begin());
    mincost::mincost_steps<<<(unsigned)ctas, 32 * mincost::kWarps, 0, s>>>(d_table, n, min_len);
    LAUNCHED("mincost_steps");
    timed.end(true);
    return 0;
}

extern "C" int sqz_gpu_parse_device_ex(const uint8_t* d_shard, const uint32_t* d_table, size_t n,
                                       uint32_t entry, uint32_t min_len, uint32_t max_len, uint32_t flags,
                                       uint32_t* d_out, size_t out_cap, void* d_work,
                                       uint64_t* d_result, void* stream) {
    if (int r = check_flags(flags, SQZ_GPU_STREAM_LAZY | SQZ_GPU_STREAM_SYMBOLS)) { return r; }
    const bool symbols = (flags & SQZ_GPU_STREAM_SYMBOLS) != 0;
    if (int r = check_rules(min_len, max_len, 1)) { return r; }
    if (symbols) {
        if (int r = check_symbol_rules(min_len, max_len, 1)) { return r; }
    }
    if (entry >= max_len) { return fail(EINVAL, "entry must be < max_len"); }
    return parse_launch(d_shard, d_table, n, nullptr, entry, min_len, max_len, d_out, out_cap, d_work, d_result,
                        (cudaStream_t)stream, symbols, (flags & SQZ_GPU_STREAM_LAZY) != 0);
}

extern "C" int sqz_gpu_parse_device(const uint8_t* d_shard, const uint32_t* d_table, size_t n,
                                    uint32_t entry, uint32_t min_len, uint32_t max_len,
                                    uint32_t* d_tokens, size_t tokens_cap, void* d_work,
                                    uint64_t* d_result, void* stream) {
    return sqz_gpu_parse_device_ex(d_shard, d_table, n, entry, min_len, max_len, 0, d_tokens, tokens_cap, d_work,
                                   d_result, stream);
}

extern "C" int sqz_gpu_parse_symbols_device(const uint8_t* d_shard, const uint32_t* d_table, size_t n,
                                            uint32_t entry, uint32_t min_len, uint32_t max_len,
                                            uint32_t* d_words, size_t words_cap, void* d_work,
                                            uint64_t* d_result, void* stream) {
    return sqz_gpu_parse_device_ex(d_shard, d_table, n, entry, min_len, max_len, SQZ_GPU_STREAM_SYMBOLS, d_words,
                                   words_cap, d_work, d_result, stream);
}

extern "C" int sqz_gpu_parse_exit_map_device_ex(const uint32_t* d_table, size_t n, uint32_t min_len,
                                                uint32_t max_len, uint32_t flags, void* d_work,
                                                uint16_t* d_exit_map, void* stream) {
    if (int r = check_flags(flags, SQZ_GPU_STREAM_LAZY)) { return r; }
    if (int r = check_rules(min_len, max_len, 1)) { return r; }
    if (n == 0) { return fail(EINVAL, "empty shard"); }
    cudaStream_t s = (cudaStream_t)stream;
    parse::Work w = parse::carve(d_work, n);
    if (int r = parse_maps(d_table, n, min_len, max_len, w, s, (flags & SQZ_GPU_STREAM_LAZY) != 0)) { return r; }
    parse::chain_total<<<1, 512, 0, s>>>(w.group_map, w.groups, max_len, d_exit_map);
    LAUNCHED("chain_total");
    return 0;
}

extern "C" int sqz_gpu_parse_exit_map_device(const uint32_t* d_table, size_t n,
                                             uint32_t min_len, uint32_t max_len, void* d_work,
                                             uint16_t* d_exit_map, void* stream) {
    return sqz_gpu_parse_exit_map_device_ex(d_table, n, min_len, max_len, 0, d_work, d_exit_map, stream);
}

// A shard's segments are the input's when it starts at a multiple of the segment and holds whole
// segments, or runs to the end of the input.
extern "C" int sqz_gpu_mincost_steps_device(uint32_t* d_table, size_t first, size_t n, size_t bytes,
                                            uint32_t min_len, uint32_t max_len, uint32_t max_dist, void* stream) {
    if (int r = check_rules(min_len, max_len, max_dist)) { return r; }
    if (int r = check_symbol_rules(min_len, max_len, max_dist)) { return r; }
    if (first % mincost::kSegment != 0 || first > bytes || n > bytes - first ||
        (n % mincost::kSegment != 0 && first + n != bytes)) {
        return fail(EINVAL, "a min-cost shard starts at a multiple of 16384 and holds whole segments or ends at bytes");
    }
    return mincost_launch(d_table, n, min_len, (cudaStream_t)stream);
}

// ---------------------------------------------------------------------------
// host-buffer ABI: chunked, double-buffered pipeline
// ---------------------------------------------------------------------------

// Tokens leave the device sized by their count, which only the device knows when the copy is
// queued: this kernel reads the count the parse left in result[0] and stores exactly that many
// words into pinned host memory (mapped into the device's address space by cudaHostAlloc) with
// 16-byte stores.  No host round trip, no copy of unused slots.
__global__ void __launch_bounds__(256)
tokens_to_host(const uint32_t* __restrict__ d_tokens, const uint64_t* __restrict__ d_result,
               uint32_t* __restrict__ h_tokens) {
    const size_t count = (size_t)d_result[0];
    const size_t quads = (count + 3) / 4;               // both buffers are 16-byte aligned and padded
    const uint4* src = reinterpret_cast<const uint4*>(d_tokens);
    uint4* dst = reinterpret_cast<uint4*>(h_tokens);
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < quads; i += (size_t)gridDim.x * blockDim.x) {
        dst[i] = src[i];
    }
}

struct sqz_gpu_stream {
    int device = 0;
    const uint8_t* data = nullptr;
    size_t bytes = 0;
    uint32_t min_len = 0, max_len = 0, max_dist = 0;
    size_t chunk = 0;
    size_t ramp = 0;                  // size of the next chunk while it is still below `chunk`
    size_t launched = 0;              // input bytes handed to the device so far
    size_t delivered = 0;             // input bytes whose tokens were returned
    int next_slot = 0, read_slot = 0;
    int kind = kConsumer;             // of its two stages: kTable, kTokens or kConsumer
    bool symbols = false;             // emit symbol words instead of plain tokens
    bool lazy = false;                // parse with the lazy rule
    bool mincost = false;             // rewrite the table into min-cost steps before the parse
    Stage slot[2];
    const uint64_t* prev_result = nullptr;   // device: previous chunk's result (entry hand-off)
    cudaEvent_t prev_parsed = nullptr;
    cudaEvent_t prev_tabled = nullptr;
};

// device < 0 = the calling thread's current device
static int ensure_device(int& device) {
    int count = 0;
    cudaError_t ce = cudaGetDeviceCount(&count);
    if (ce != cudaSuccess || count == 0) {
        return fail(ENODEV, "no CUDA device: the match search has no CPU fallback", ce);
    }
    if (device < 0) { CU(cudaGetDevice(&device)); }
    if (device >= count) { return fail(ENODEV, "no such CUDA device"); }
    CU(cudaSetDevice(device));
    return 0;
}

// the arguments every host-buffer entry point checks, in this order: rules, window, input, device
// (which ensure_device makes current)
static int check_call(int& device, uint32_t window, uint32_t min_len, uint32_t max_len, uint32_t max_dist,
                      const uint8_t* data, size_t bytes) {
    if (int r = check_rules(min_len, max_len, max_dist)) { return r; }
    if (window == 0 || (window & (window - 1)) != 0 || max_dist > window) {
        return fail(EINVAL, "window must be a power of two and max_dist <= window");
    }
    if (data == nullptr && bytes != 0) { return fail(EINVAL, "null input"); }
    return ensure_device(device);
}

// Uploads positions [first, first + n) of `data` with their halos and searches them on the stage's
// stream; the search, not the upload, waits for `after` when there is one.
static int stage_search(Stage& s, const uint8_t* data, size_t first, size_t n, size_t back, size_t ahead,
                        uint32_t min_len, uint32_t max_len, uint32_t max_dist, cudaEvent_t after) {
    s.first = first;
    s.n = n;
    s.back = back;
    CU(cudaMemcpyAsync(s.d_data, data + first - back, back + n + ahead, cudaMemcpyHostToDevice, s.stream));
    if (after != nullptr) { CU(cudaStreamWaitEvent(s.stream, after, 0)); }
    return sqz_gpu_match_table_device_ws(s.d_data + back, back, n, ahead, min_len, max_len, max_dist,
                                         s.d_table, s.d_mwork, s.stream);
}

// issue everything for the next chunk on its slot; returns without waiting
static int stream_launch_next(sqz_gpu_stream* st, uint16_t* len_out, uint16_t* dist_out) {
    Stage& s = st->slot[st->next_slot];
    const size_t first = st->launched;
    size_t n = std::min(st->chunk, st->bytes - first);
    if (st->ramp != 0) {               // short chunks first: the consumer starts after milliseconds
        n = std::min(n, st->ramp);
        st->ramp = st->ramp * 2 >= st->chunk ? 0 : st->ramp * 2;
    }
    const size_t back = std::min<size_t>(first, st->max_dist);
    const size_t ahead = std::min<size_t>(st->bytes - (first + n), st->max_len);
    const bool consumer = st->kind == kConsumer;
    // A consumer waits for the chunks in order: two searches sharing the device would both be ready
    // late.  This chunk's search starts when the one before has its table; only that one's parse and
    // copy run beside it.
    if (int r = stage_search(s, st->data, first, n, back, ahead, st->min_len, st->max_len, st->max_dist,
                             consumer ? st->prev_tabled : nullptr)) { return r; }
    if (st->lazy) {                     // table[n]: the next chunk is not searched yet
        if (int r = seam_word(s.d_data + back, back, n, ahead, st->min_len, st->max_len, st->max_dist,
                              s.d_table, s.stream)) { return r; }
    }
    CU(cudaEventRecord(s.tabled, s.stream));
    st->prev_tabled = s.tabled;
    const uint8_t* d_shard = s.d_data + back;
    // A consumer's parse and token copy go on a stream of the highest priority: the next chunk's search
    // is queued behind this one's and fills the device as soon as it may -- at equal priority the few
    // small kernels that finish this chunk would wait for free CTA slots until that search is over.
    cudaStream_t late = consumer ? s.ahead_of_all : s.stream;
    if (late != s.stream) { CU(cudaStreamWaitEvent(late, s.tabled, 0)); }
    if (st->kind != kTable) {
        const uint32_t* d_entry = nullptr;
        // every chunk but the last holds whole segments (stream_open), so the chunk's segments are the
        // input's, and the greedy parse of the rewritten table is the min-cost parse
        if (st->mincost) {
            if (int r = mincost_launch(s.d_table, n, st->min_len, late)) { return r; }
        }
        if (st->prev_result != nullptr) {
            CU(cudaStreamWaitEvent(late, st->prev_parsed, 0));
            d_entry = reinterpret_cast<const uint32_t*>(st->prev_result + 1);  // low half of overshoot
        }
        if (int r = parse_launch(d_shard, s.d_table, n, d_entry, 0, st->min_len, st->max_len,
                                 s.d_tokens, n, s.d_work, s.d_result, late, st->symbols, st->lazy)) { return r; }
        CU(cudaMemcpyAsync(s.h_result, s.d_result, 16, cudaMemcpyDeviceToHost, late));
        CU(cudaEventRecord(s.parsed, late));
        st->prev_parsed = s.parsed;
        st->prev_result = s.d_result;
        if (consumer) {
            // the tokens follow right away, exactly as many as there are: the consumer finds them
            // in pinned memory when it asks
            const unsigned grid = (unsigned)std::min<size_t>((n / 4 + 255) / 256 + 1, (size_t)sm_count() * 4);
            tokens_to_host<<<grid, 256, 0, late>>>(s.d_tokens, s.d_result, s.h_tokens);
            LAUNCHED("tokens_to_host");
        }
        // kTokens: the caller copies count x 4 bytes to their final place once it knows the count
    } else {
        if (int r = sqz_gpu_unpack_table_device(s.d_table, n, s.d_len, s.d_dist, s.stream)) { return r; }
        CU(cudaMemcpyAsync(len_out + first, s.d_len, n * 2, cudaMemcpyDeviceToHost, s.stream));
        CU(cudaMemcpyAsync(dist_out + first, s.d_dist, n * 2, cudaMemcpyDeviceToHost, s.stream));
    }
    if (late != s.stream) {             // the slot is free when both streams are through
        CU(cudaEventRecord(s.done, late));
        CU(cudaStreamWaitEvent(s.stream, s.done, 0));
    }
    CU(cudaEventRecord(s.done, s.stream));
    s.busy = true;
    st->launched = first + n;
    st->next_slot ^= 1;
    return 0;
}

// Token mode feeds a host consumer chunk by chunk: smaller chunks overlap better.
// Table mode only streams: larger chunks waste less on the last wave of tiles.
static size_t default_chunk(size_t bytes, bool consumer) {
    const size_t kDefault = consumer ? (size_t)32 << 20 : (size_t)128 << 20;
    return std::max<size_t>(std::min(bytes, kDefault), 1);
}

static int stream_open(sqz_gpu_stream** out, int device, const uint8_t* data, size_t bytes,
                       uint32_t window, uint32_t min_len, uint32_t max_len, uint32_t max_dist,
                       size_t chunk, int kind, bool short_start = false, bool mincost = false) {
    *out = nullptr;
    if (int r = check_call(device, window, min_len, max_len, max_dist, data, bytes)) { return r; }
    sqz_gpu_stream* st = new (std::nothrow) sqz_gpu_stream();
    if (st == nullptr) { return fail(ENOMEM, "out of host memory"); }
    st->device = device;
    st->data = data;
    st->bytes = bytes;
    st->min_len = min_len; st->max_len = max_len; st->max_dist = max_dist;
    st->mincost = mincost;
    // The min-cost parse needs every chunk but the last to be whole segments.  The default chunks
    // (2-32 MiB, 128 MiB) are; an explicit size and its short start are rounded up to them (a size
    // too close to SIZE_MAX to round exceeds any input: its one chunk is the last).
    auto whole_segments = [mincost](size_t b) {
        const size_t seg = mincost::kSegment;
        return mincost && b <= SIZE_MAX - seg ? (b + seg - 1) / seg * seg : b;
    };
    chunk = whole_segments(chunk);
    st->chunk = chunk ? chunk : default_chunk(bytes, kind == kConsumer);
    st->kind = kind;
    // token streams with the default chunking start with short chunks: 2, 4, 8, 16 MiB, then 32 MiB
    if (kind == kConsumer && chunk == 0 && st->chunk > ((size_t)2 << 20)) { st->ramp = (size_t)2 << 20; }
    if (short_start && chunk >= ((size_t)4 << 20)) { st->ramp = whole_segments(chunk / 4); }
    const int slots = bytes > (st->ramp ? st->ramp : st->chunk) ? 2 : 1;
    // no chunk is larger than the input, however large the size asked for
    for (int k = 0; k < slots && bytes > 0; k++) {
        if (int r = stage_take(st->slot[k], device, kind, std::min(st->chunk, bytes))) {
            sqz_gpu_stream_close(st);
            return r;
        }
    }
    *out = st;
    return 0;
}

// Waits for both slots, parks them and deletes the stream; returns rc, or the first error of the
// waits when rc is 0.
static int stream_finish(sqz_gpu_stream* st, int rc) {
    for (Stage& s : st->slot) { rc = stage_finish(s, rc); }
    delete st;
    return rc;
}

extern "C" int sqz_gpu_stream_open(sqz_gpu_stream** st, int device, const uint8_t* data,
                                   size_t bytes, uint32_t window, uint32_t min_len,
                                   uint32_t max_len, uint32_t max_dist, size_t chunk_bytes,
                                   uint32_t flags) {
    if (st == nullptr) { return fail(EINVAL, "null stream handle"); }
    if ((flags & ~(uint32_t)(SQZ_GPU_STREAM_SYMBOLS | SQZ_GPU_STREAM_SHORT_START | SQZ_GPU_STREAM_LAZY |
                             SQZ_GPU_STREAM_MINCOST)) != 0) {
        return fail(EINVAL, "unknown stream flags");
    }
    if (flags & SQZ_GPU_STREAM_SYMBOLS) {
        if (int r = check_symbol_rules(min_len, max_len, max_dist)) { return r; }
    }
    if (int r = check_mincost(flags, min_len, max_len, max_dist)) { return r; }
    DeviceScope keep;
    if (int r = stream_open(st, device, data, bytes, window, min_len, max_len, max_dist,
                            chunk_bytes, kConsumer, (flags & SQZ_GPU_STREAM_SHORT_START) != 0,
                            (flags & SQZ_GPU_STREAM_MINCOST) != 0)) { return r; }
    (*st)->symbols = (flags & SQZ_GPU_STREAM_SYMBOLS) != 0;
    (*st)->lazy = (flags & SQZ_GPU_STREAM_LAZY) != 0;
    if (bytes > 0) {
        if (int r = stream_launch_next(*st, nullptr, nullptr)) {
            sqz_gpu_stream_close(*st);
            *st = nullptr;
            return r;
        }
    }
    return 0;
}

extern "C" int sqz_gpu_stream_next(sqz_gpu_stream* st, const uint32_t** tokens, size_t* count) {
    if (st == nullptr || tokens == nullptr || count == nullptr) { return fail(EINVAL, "null argument"); }
    *tokens = nullptr;
    *count = 0;
    if (st->delivered >= st->bytes) { return 0; }
    DeviceScope keep;
    CU(cudaSetDevice(st->device));
    // keep the device busy: the slot the caller has just finished reading is free now
    static const bool trace = getenv("SQZ_TRACE") != nullptr;
    // A chunk that lies inside the previous chunk's last match (chunk_bytes < max_len) has no tokens:
    // it is consumed here and the next one read, so that a count of 0 only ever means the end.
    for (;;) {
        const auto t0 = std::chrono::steady_clock::now();
        if (st->launched < st->bytes) {
            if (int r = stream_launch_next(st, nullptr, nullptr)) { return r; }
        }
        const auto t1 = std::chrono::steady_clock::now();
        Stage& s = st->slot[st->read_slot];
        CU(cudaEventSynchronize(s.done));
        if (trace) {
            const auto t2 = std::chrono::steady_clock::now();
            fprintf(stderr, "sqz_gpu_stream_next: queued the next chunk in %.1f ms, waited %.1f ms for this one\n",
                    std::chrono::duration<double, std::milli>(t1 - t0).count(),
                    std::chrono::duration<double, std::milli>(t2 - t1).count());
        }
        const uint64_t n_tok = s.h_result[0];
        if (n_tok > s.n) { return fail(EIO, "parse produced more tokens than positions"); }
        s.busy = false;
        st->delivered = s.first + s.n;
        st->read_slot ^= 1;
        if (n_tok != 0 || st->delivered >= st->bytes) {
            *tokens = s.h_tokens;
            *count = (size_t)n_tok;
            return 0;
        }
    }
}

extern "C" void sqz_gpu_stream_close(sqz_gpu_stream* st) {
    if (st == nullptr) { return; }
    DeviceScope keep;
    cudaSetDevice(st->device);
    stream_finish(st, 0);
}

// One-shot token call: the chunks' tokens go straight from device memory to their final place in
// the caller's buffer, count x 4 bytes each (a pinned destination takes them by DMA while the next
// chunk is searched; a pageable one through the driver's staging).  Nothing consumes the chunks
// on the way, so the larger streaming chunk is used.  The lazy parse crosses its chunk seams as in the
// token stream: every chunk searches its seam word.  The min-cost parse needs nothing across seams:
// the 128 MiB chunks are whole segments.
extern "C" int sqz_gpu_tokens_ex(const uint8_t* data, size_t bytes, uint32_t window,
                                 uint32_t min_len, uint32_t max_len, uint32_t max_dist, uint32_t flags,
                                 uint32_t* tokens_out, size_t tokens_cap, size_t* n_tokens) {
    if (n_tokens == nullptr) { return fail(EINVAL, "null n_tokens"); }
    *n_tokens = 0;
    if (int r = check_flags(flags, SQZ_GPU_STREAM_LAZY | SQZ_GPU_STREAM_MINCOST)) { return r; }
    if (int r = check_mincost(flags, min_len, max_len, max_dist)) { return r; }
    sqz_gpu_stream* st = nullptr;
    DeviceScope keep;
    if (int r = stream_open(&st, -1, data, bytes, window, min_len, max_len, max_dist, 0, kTokens, false,
                            (flags & SQZ_GPU_STREAM_MINCOST) != 0)) {
        return r;
    }
    st->lazy = (flags & SQZ_GPU_STREAM_LAZY) != 0;
    size_t total = 0;
    int rc = 0;
    if (bytes > 0) { rc = stream_launch_next(st, nullptr, nullptr); }
    while (rc == 0 && st->delivered < st->bytes) {
        Stage& s = st->slot[st->read_slot];
        // the other slot is free (its copy was queued before its `done`): keep the device busy
        if (st->launched < st->bytes) {
            Stage& o = st->slot[st->next_slot];
            if (o.busy) {
                cudaError_t ce = cudaEventSynchronize(o.done);
                if (ce != cudaSuccess) { rc = fail(cuda_code(ce), "cudaEventSynchronize", ce); break; }
                o.busy = false;
            }
            rc = stream_launch_next(st, nullptr, nullptr);
            if (rc != 0) { break; }
        }
        cudaError_t ce = cudaEventSynchronize(s.parsed);
        if (ce != cudaSuccess) { rc = fail(cuda_code(ce), "cudaEventSynchronize", ce); break; }
        const size_t c = (size_t)s.h_result[0];
        if (c > s.n) { rc = fail(EIO, "parse produced more tokens than positions"); break; }
        if (tokens_out != nullptr && total < tokens_cap) {
            ce = cudaMemcpyAsync(tokens_out + total, s.d_tokens, std::min(c, tokens_cap - total) * 4,
                                 cudaMemcpyDeviceToHost, s.stream);
            if (ce != cudaSuccess) { rc = fail(cuda_code(ce), "cudaMemcpyAsync", ce); break; }
        }
        ce = cudaEventRecord(s.done, s.stream);      // the slot is free again once the copy has landed
        if (ce != cudaSuccess) { rc = fail(cuda_code(ce), "cudaEventRecord", ce); break; }
        total += c;
        st->delivered = s.first + s.n;
        st->read_slot ^= 1;
    }
    rc = stream_finish(st, rc);
    *n_tokens = total;
    if (rc == 0 && total > tokens_cap) { rc = fail(E2BIG, "token buffer too small"); }
    return rc;
}

extern "C" int sqz_gpu_tokens(const uint8_t* data, size_t bytes, uint32_t window,
                              uint32_t min_len, uint32_t max_len, uint32_t max_dist,
                              uint32_t* tokens_out, size_t tokens_cap, size_t* n_tokens) {
    return sqz_gpu_tokens_ex(data, bytes, window, min_len, max_len, max_dist, 0, tokens_out, tokens_cap, n_tokens);
}

extern "C" int sqz_gpu_match_table(const uint8_t* data, size_t bytes, uint32_t window,
                                   uint32_t min_len, uint32_t max_len, uint32_t max_dist,
                                   uint16_t* len_out, uint16_t* dist_out) {
    if (bytes != 0 && (len_out == nullptr || dist_out == nullptr)) {
        return fail(EINVAL, "null output");
    }
    sqz_gpu_stream* st = nullptr;
    DeviceScope keep;
    if (int r = stream_open(&st, -1, data, bytes, window, min_len, max_len, max_dist, 0, kTable)) {
        return r;
    }
    int rc = 0;
    while (rc == 0 && st->launched < st->bytes) {
        Stage& s = st->slot[st->next_slot];
        if (s.busy) {                      // reuse only after its copies have landed
            cudaError_t ce = cudaEventSynchronize(s.done);
            if (ce != cudaSuccess) { rc = fail(cuda_code(ce), "cudaEventSynchronize", ce); break; }
            s.busy = false;
        }
        rc = stream_launch_next(st, len_out, dist_out);
    }
    return stream_finish(st, rc);
}

// ---------------------------------------------------------------------------
// several devices, one call (SURVEY.md section 8e).  The input is cut into contiguous shards,
// one per device, each uploaded with its look-back and look-ahead halo, so the match tables need
// no exchange at all.  The greedy parse has one scalar dependency per seam -- where the previous
// shard's last token ends (squeeze.h:377-394: i += len) -- which is resolved without a
// collective: every device composes its shard's exit map (overshoot for every possible entry,
// 1 KiB), the host chains the maps (one lookup per seam), every device then emits its tokens from
// its true entry, and the token arrays are concatenated in shard order by plain copies sized by
// their counts: device -> host when tokens_out is host memory, peer-to-peer (cudaMemcpyPeerAsync
// over NVLink) when it is device memory.  The lazy parse adds one dependency per seam, the best match
// at the next shard's first position (table[n]), which every shard searches from its own halos: no
// exchange beyond the exit maps.  The min-cost parse adds none: with every shard starting at a multiple
// of mincost::kSegment and holding whole segments (all but the last), a shard's segments are the input's,
// and each shard rewrites its own table before its exit map.
// ---------------------------------------------------------------------------

// The shard boundaries of [0, bytes) cut into n shards of whole units: ceil(bytes / unit) units shared
// out as evenly as they go, the first (units % n) shards one unit more, every boundary clamped to bytes
// (so the partial last unit lives in the last non-empty shard, and shards past the units are empty).
// Returns n + 1 offsets, from 0 to bytes.  unit = 1 gives shards whose sizes differ by at most one byte.
static std::vector<size_t> even_cuts(size_t bytes, size_t n, size_t unit) {
    const size_t units = (bytes + unit - 1) / unit, base = units / n, extra = units % n;
    std::vector<size_t> at(n + 1, 0);
    for (size_t g = 0; g < n; g++) {
        at[g + 1] = std::min(bytes, at[g] + (base + (g < extra ? 1 : 0)) * unit);
    }
    return at;
}

// `at`: parts.size() + 1 non-decreasing shard boundaries from 0 to bytes.  `mincost` needs every
// boundary at a multiple of mincost::kSegment or at bytes.
static int multi_run(std::vector<Stage>& parts, const int* devices, const std::vector<size_t>& at,
                     const uint8_t* data, size_t bytes, uint32_t min_len, uint32_t max_len, uint32_t max_dist,
                     bool lazy, bool mincost, uint32_t* tokens_out, size_t tokens_cap, bool out_on_device,
                     int out_device, size_t* n_tokens, size_t* shard_tokens) {
    // phase A on every device at once: upload, match table (and the seam word or the min-cost steps),
    // composed exit map
    for (size_t g = 0; g < parts.size(); g++) {
        const size_t first = at[g], n = at[g + 1] - at[g];
        if (n > 0) {
            Stage& p = parts[g];
            CU(cudaSetDevice(devices[g]));
            if (int r = stage_take(p, devices[g], kTokens, n)) { return r; }
            const size_t back = std::min<size_t>(first, max_dist), ahead = std::min<size_t>(bytes - (first + n), max_len);
            if (int r = stage_search(p, data, first, n, back, ahead, min_len, max_len, max_dist, nullptr)) { return r; }
            if (lazy) {
                if (int r = seam_word(p.d_data + back, back, n, ahead, min_len, max_len, max_dist, p.d_table,
                                      p.stream)) { return r; }
            }
            if (mincost) {
                if (int r = mincost_launch(p.d_table, n, min_len, p.stream)) { return r; }
            }
            if (int r = sqz_gpu_parse_exit_map_device_ex(p.d_table, n, min_len, max_len, lazy ? SQZ_GPU_STREAM_LAZY : 0,
                                                         p.d_work, p.d_map, p.stream)) { return r; }
            CU(cudaMemcpyAsync(p.h_map, p.d_map, (size_t)max_len * 2, cudaMemcpyDeviceToHost, p.stream));
            CU(cudaEventRecord(p.tabled, p.stream));
        }
    }
    // seams: shard g+1 is entered where shard g's last token ends
    uint32_t entry = 0;
    for (Stage& p : parts) {
        if (p.n == 0) { continue; }
        CU(cudaSetDevice(p.device));
        CU(cudaEventSynchronize(p.tabled));
        if (entry >= max_len) { return fail(EIO, "seam entry out of range"); }
        const uint32_t next_entry = p.h_map[entry];
        if (int r = parse_launch(p.d_data + p.back, p.d_table, p.n, nullptr, entry, min_len, max_len, p.d_tokens,
                                 p.n, p.d_work, p.d_result, p.stream, false, lazy)) { return r; }
        CU(cudaMemcpyAsync(p.h_result, p.d_result, 16, cudaMemcpyDeviceToHost, p.stream));
        CU(cudaEventRecord(p.parsed, p.stream));
        entry = next_entry;
    }
    // concatenation in shard order, every copy sized by its shard's count
    size_t total = 0;
    for (size_t g = 0; g < parts.size(); g++) {
        Stage& p = parts[g];
        size_t c = 0;
        if (p.n != 0) {
            CU(cudaSetDevice(p.device));
            CU(cudaEventSynchronize(p.parsed));
            c = (size_t)p.h_result[0];
            if (c > p.n) { return fail(EIO, "parse produced more tokens than positions"); }
            if (tokens_out != nullptr && total < tokens_cap) {
                const size_t take = std::min(c, tokens_cap - total);
                if (out_on_device) {
                    CU(cudaMemcpyPeerAsync(tokens_out + total, out_device, p.d_tokens, p.device, take * 4, p.stream));
                } else {
                    CU(cudaMemcpyAsync(tokens_out + total, p.d_tokens, take * 4, cudaMemcpyDeviceToHost, p.stream));
                }
            }
        }
        if (shard_tokens != nullptr) { shard_tokens[g] = c; }
        total += c;
    }
    *n_tokens = total;
    if (entry != 0) { return fail(EIO, "the parse does not end at the end of the input"); }
    return total > tokens_cap ? fail(E2BIG, "token buffer too small") : 0;
}

// The multi-device calls after their own argument checks: `at` holds the shard boundaries, flags are
// 0, LAZY or MINCOST.
static int multi_call(const int* devices, int n_devices, const std::vector<size_t>& at, const uint8_t* data,
                      size_t bytes, uint32_t window, uint32_t min_len, uint32_t max_len, uint32_t max_dist,
                      uint32_t flags, uint32_t* tokens_out, size_t tokens_cap, size_t* n_tokens,
                      size_t* shard_tokens) {
    DeviceScope keep;
    int device = devices[0];
    if (int r = check_call(device, window, min_len, max_len, max_dist, data, bytes)) { return r; }
    const int count = sqz_gpu_device_count();
    for (int g = 0; g < n_devices; g++) {
        // (a device may be listed more than once: its shards then share it, each on its own stream)
        if (devices[g] < 0 || devices[g] >= count) { return fail(ENODEV, "no such CUDA device"); }
    }
    // where do the tokens go: host memory, or device memory (then peer copies gather them there)
    bool out_on_device = false;
    int out_device = devices[0];
    if (tokens_out != nullptr) {
        cudaPointerAttributes at;
        if (cudaPointerGetAttributes(&at, tokens_out) == cudaSuccess && at.type == cudaMemoryTypeDevice) {
            out_on_device = true;
            out_device = at.device;
        }
        cudaGetLastError();
    }
    if (out_on_device) {
        for (int g = 0; g < n_devices; g++) {
            if (devices[g] == out_device) { continue; }
            int can = 0;
            CU(cudaDeviceCanAccessPeer(&can, devices[g], out_device));
            if (can) {
                CU(cudaSetDevice(devices[g]));
                cudaError_t ce = cudaDeviceEnablePeerAccess(out_device, 0);
                if (ce != cudaSuccess && ce != cudaErrorPeerAccessAlreadyEnabled) { return fail(cuda_code(ce), "cudaDeviceEnablePeerAccess", ce); }
                cudaGetLastError();
            }   // without peer access cudaMemcpyPeerAsync still works, staged through the host
        }
    }
    std::vector<Stage> parts((size_t)n_devices);
    int rc = multi_run(parts, devices, at, data, bytes, min_len, max_len, max_dist, (flags & SQZ_GPU_STREAM_LAZY) != 0,
                       (flags & SQZ_GPU_STREAM_MINCOST) != 0, tokens_out, tokens_cap, out_on_device, out_device,
                       n_tokens, shard_tokens);
    for (Stage& p : parts) { rc = stage_finish(p, rc); }
    return rc;
}

static int check_device_list(const int* devices, int n_devices) {
    if (devices == nullptr || n_devices < 1 || n_devices > kMaxDevices) { return fail(EINVAL, "bad device list"); }
    return 0;
}

extern "C" int sqz_gpu_tokens_multi_ex(const int* devices, int n_devices, const uint8_t* data, size_t bytes,
                                       uint32_t window, uint32_t min_len, uint32_t max_len, uint32_t max_dist,
                                       uint32_t flags, uint32_t* tokens_out, size_t tokens_cap, size_t* n_tokens,
                                       size_t* shard_tokens) {
    if (n_tokens == nullptr) { return fail(EINVAL, "null n_tokens"); }
    *n_tokens = 0;
    if (int r = check_flags(flags, SQZ_GPU_STREAM_LAZY)) { return r; }
    if (int r = check_device_list(devices, n_devices)) { return r; }
    return multi_call(devices, n_devices, even_cuts(bytes, (size_t)n_devices, 1), data, bytes, window, min_len,
                      max_len, max_dist, flags, tokens_out, tokens_cap, n_tokens, shard_tokens);
}

extern "C" int sqz_gpu_tokens_multi_cuts(const int* devices, int n_devices, const size_t* cuts,
                                         const uint8_t* data, size_t bytes, uint32_t window, uint32_t min_len,
                                         uint32_t max_len, uint32_t max_dist, uint32_t flags,
                                         uint32_t* tokens_out, size_t tokens_cap, size_t* n_tokens,
                                         size_t* shard_tokens) {
    if (n_tokens == nullptr) { return fail(EINVAL, "null n_tokens"); }
    *n_tokens = 0;
    if (int r = check_flags(flags, SQZ_GPU_STREAM_LAZY | SQZ_GPU_STREAM_MINCOST)) { return r; }
    if (int r = check_mincost(flags, min_len, max_len, max_dist)) { return r; }
    if (int r = check_device_list(devices, n_devices)) { return r; }
    const bool mincost = (flags & SQZ_GPU_STREAM_MINCOST) != 0;
    const size_t unit = mincost ? (size_t)mincost::kSegment : 1;
    std::vector<size_t> at = even_cuts(bytes, (size_t)n_devices, unit);
    if (cuts != nullptr) {
        for (int g = 1; g < n_devices; g++) {
            const size_t c = cuts[g - 1];
            if (c < at[g - 1] || c > bytes) { return fail(EINVAL, "cuts must be non-decreasing and <= bytes"); }
            if (c % unit != 0 && c != bytes) {
                return fail(EINVAL, "the min-cost parse needs every cut at a multiple of 16384 or at bytes");
            }
            at[g] = c;
        }
    }
    return multi_call(devices, n_devices, at, data, bytes, window, min_len, max_len, max_dist, flags, tokens_out,
                      tokens_cap, n_tokens, shard_tokens);
}

extern "C" int sqz_gpu_tokens_multi(const int* devices, int n_devices, const uint8_t* data, size_t bytes,
                                    uint32_t window, uint32_t min_len, uint32_t max_len, uint32_t max_dist,
                                    uint32_t* tokens_out, size_t tokens_cap, size_t* n_tokens,
                                    size_t* shard_tokens) {
    return sqz_gpu_tokens_multi_ex(devices, n_devices, data, bytes, window, min_len, max_len, max_dist, 0, tokens_out,
                                   tokens_cap, n_tokens, shard_tokens);
}

// ---------------------------------------------------------------------------
// one process per device (torchrun-style jobs): the same gather needs the destination buffer of
// one process mapped into the others.  Plain CUDA IPC, no collective library.
// ---------------------------------------------------------------------------
extern "C" int sqz_gpu_device_alloc(void** d_ptr, size_t bytes) {
    if (d_ptr == nullptr) { return fail(EINVAL, "null argument"); }
    *d_ptr = nullptr;
    CU(cudaMalloc(d_ptr, bytes ? bytes : 1));
    return 0;
}

extern "C" void sqz_gpu_device_free(void* d_ptr) {
    if (d_ptr != nullptr) { cudaFree(d_ptr); }
}

extern "C" int sqz_gpu_ipc_export(const void* d_ptr, uint8_t handle[SQZ_GPU_IPC_HANDLE_BYTES]) {
    static_assert(sizeof(cudaIpcMemHandle_t) == SQZ_GPU_IPC_HANDLE_BYTES, "IPC handle size");
    if (d_ptr == nullptr || handle == nullptr) { return fail(EINVAL, "null argument"); }
    cudaIpcMemHandle_t h;
    CU(cudaIpcGetMemHandle(&h, const_cast<void*>(d_ptr)));
    memcpy(handle, &h, sizeof(h));
    return 0;
}

extern "C" int sqz_gpu_ipc_open(const uint8_t handle[SQZ_GPU_IPC_HANDLE_BYTES], void** d_ptr) {
    if (d_ptr == nullptr || handle == nullptr) { return fail(EINVAL, "null argument"); }
    *d_ptr = nullptr;
    cudaIpcMemHandle_t h;
    memcpy(&h, handle, sizeof(h));
    CU(cudaIpcOpenMemHandle(d_ptr, h, cudaIpcMemLazyEnablePeerAccess));
    return 0;
}

extern "C" int sqz_gpu_ipc_close(void* d_ptr) {
    if (d_ptr == nullptr) { return 0; }
    CU(cudaIpcCloseMemHandle(d_ptr));
    return 0;
}

// copy `count` tokens of this process's device into a (possibly IPC-mapped, possibly remote)
// device buffer at token offset `at`: the per-shard step of the gather
extern "C" int sqz_gpu_put_tokens(uint32_t* d_dst, size_t at, const uint32_t* d_tokens, size_t count, void* stream) {
    if (count == 0) { return 0; }
    if (d_dst == nullptr || d_tokens == nullptr) { return fail(EINVAL, "null argument"); }
    CU(cudaMemcpyAsync(d_dst + at, d_tokens, count * 4, cudaMemcpyDefault, (cudaStream_t)stream));
    return 0;
}

// ---------------------------------------------------------------------------
// decoder side: the LZ copy phase on the GPU (lz_expand.cuh; SURVEY.md 8f N4)
// ---------------------------------------------------------------------------
static size_t expand_blocks(size_t n_tokens) { return (n_tokens + expand::kScanBlock - 1) / expand::kScanBlock; }

extern "C" size_t sqz_gpu_expand_workspace(size_t n_tokens, size_t bytes) {
    // block offsets + {total, bad, changed} + one 32-bit hop per output byte
    return parse::align_up(expand_blocks(n_tokens) * 8 + 8) + 256 + parse::align_up(bytes * 4 + 4);
}

// the sizes both expand entry points refuse before they touch the device
static int expand_check(size_t n_tokens, size_t bytes) {
    if (bytes >= ((size_t)1 << 31)) { return fail(EINVAL, "one expand call handles less than 2 GiB"); }
    if (n_tokens > bytes) { return fail(EINVAL, "more tokens than bytes"); }
    if (n_tokens == 0 && bytes > 0) { return fail(EINVAL, "tokens describe fewer bytes than announced"); }
    return 0;
}

extern "C" int sqz_gpu_expand_tokens_device(const uint32_t* d_tokens, size_t n_tokens, uint8_t* d_out,
                                            size_t bytes, void* d_work, void* stream) {
    if (int r = expand_check(n_tokens, bytes)) { return r; }
    if (bytes == 0) { return 0; }
    cudaStream_t s = (cudaStream_t)stream;
    const size_t blocks = expand_blocks(n_tokens);
    if (blocks > 0x7FFFFFFFull) { return fail(EINVAL, "too many tokens for one launch"); }
    uint8_t* w = static_cast<uint8_t*>(d_work);
    uint64_t* block_off = reinterpret_cast<uint64_t*>(w);
    uint8_t* flags = w + parse::align_up(blocks * 8 + 8);
    uint64_t* d_total = reinterpret_cast<uint64_t*>(flags);
    int* d_bad = reinterpret_cast<int*>(flags + 8);
    int* d_rounds = reinterpret_cast<int*>(flags + 16);          // three flags of the doubling rounds
    uint32_t* hop = reinterpret_cast<uint32_t*>(flags + 256);
    CU(cudaMemsetAsync(flags, 0, 256, s));
    expand::block_lengths<<<(unsigned)blocks, 256, 0, s>>>(d_tokens, n_tokens, block_off);
    LAUNCHED("expand_block_lengths");
    expand::scan_blocks<<<1, 1024, 0, s>>>(block_off, blocks, d_total);
    LAUNCHED("expand_scan_blocks");
    struct { uint64_t total; int bad; int pad; int changed; } h = { 0, 0, 0, 0 };
    CU(cudaMemcpyAsync(&h, flags, 8, cudaMemcpyDeviceToHost, s));
    CU(cudaStreamSynchronize(s));
    if (h.total != bytes) { return fail(EINVAL, "tokens do not describe the announced number of bytes"); }
    expand::place_tokens<<<(unsigned)blocks, 256, 0, s>>>(d_tokens, n_tokens, block_off, d_out, hop,
                                                        (uint64_t)bytes, d_bad);
    LAUNCHED("expand_place_tokens");
    const unsigned grid = (unsigned)sm_count() * 8;
    // a chain halves its hop count every round: 32 rounds cover 31-bit hops; rounds after the last
    // useful one return at once (the device decides, the host does not wait in between)
    for (int round = 0; round < 32; round++) {
        expand::double_hops<<<grid, 256, 0, s>>>(hop, (uint64_t)bytes, d_rounds, round);
        LAUNCHED("expand_double_hops");
    }
    expand::fetch_bytes<<<grid, 256, 0, s>>>(hop, d_out, (uint64_t)bytes);
    LAUNCHED("expand_fetch_bytes");
    // one wait for the whole copy phase: was a token out of range?  (The bytes of such a stream are
    // garbage but in bounds: place_tokens cut every bad hop to 0.)
    CU(cudaMemcpyAsync(&h, flags, 16, cudaMemcpyDeviceToHost, s));
    CU(cudaStreamSynchronize(s));
    if (h.bad != 0) {
        return fail(EINVAL, "a bad token: a match from before the start of the output or at distance 0, "
                            "or a literal word above 0xFF");
    }
    return 0;
}

extern "C" int sqz_gpu_expand_tokens(const uint32_t* tokens, size_t n_tokens, uint8_t* out, size_t bytes) {
    // refused before a stream or a buffer is made: the buffers below take 5 device bytes per output byte
    if (int r = expand_check(n_tokens, bytes)) { return r; }
    if (bytes == 0) { return 0; }
    if (tokens == nullptr || out == nullptr) { return fail(EINVAL, "null argument"); }
    int device = -1;
    if (int r = ensure_device(device)) { return r; }
    uint32_t* d_tokens = nullptr;
    uint8_t* d_out = nullptr;
    void* d_work = nullptr;
    cudaStream_t s = nullptr;
    int rc = 0;
    cudaError_t ce = cudaStreamCreateWithFlags(&s, cudaStreamNonBlocking);
    if (ce == cudaSuccess) { ce = cudaMalloc(&d_tokens, n_tokens * 4 + 4); }
    if (ce == cudaSuccess) { ce = cudaMalloc(&d_out, bytes); }
    if (ce == cudaSuccess) { ce = cudaMalloc(&d_work, sqz_gpu_expand_workspace(n_tokens, bytes)); }
    if (ce == cudaSuccess) { ce = cudaMemcpyAsync(d_tokens, tokens, n_tokens * 4, cudaMemcpyHostToDevice, s); }
    if (ce != cudaSuccess) { rc = fail(cuda_code(ce), "expand: allocation or upload", ce); }
    if (rc == 0) { rc = sqz_gpu_expand_tokens_device(d_tokens, n_tokens, d_out, bytes, d_work, s); }
    if (rc == 0) {
        ce = cudaMemcpyAsync(out, d_out, bytes, cudaMemcpyDeviceToHost, s);
        if (ce == cudaSuccess) { ce = cudaStreamSynchronize(s); }
        if (ce != cudaSuccess) { rc = fail(cuda_code(ce), "expand: download", ce); }
    }
    cudaFree(d_tokens); cudaFree(d_out); cudaFree(d_work);
    if (s != nullptr) { cudaStreamDestroy(s); }
    return rc;
}

// ---------------------------------------------------------------------------
// utilities
// ---------------------------------------------------------------------------
extern "C" int sqz_gpu_abi_version(void) { return SQZ_GPU_ABI_VERSION; }

extern "C" int sqz_gpu_device_count(void) {
    int count = 0;
    if (cudaGetDeviceCount(&count) != cudaSuccess) { cudaGetLastError(); return 0; }
    return count;
}

extern "C" const char* sqz_gpu_last_error(void) { return g_err; }

extern "C" void* sqz_gpu_host_alloc(size_t bytes) {
    void* p = nullptr;
    if (cudaHostAlloc(&p, bytes ? bytes : 1, cudaHostAllocDefault) != cudaSuccess) {
        cudaGetLastError();
        return nullptr;
    }
    return p;
}

extern "C" void sqz_gpu_host_free(void* p) {
    if (p != nullptr) { cudaFreeHost(p); }
}

extern "C" uint64_t sqz_gpu_launch_count(void) { return g_launches.load(); }
