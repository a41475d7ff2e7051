// lz_expand.cuh -- the copy phase of the decoder on the GPU (SURVEY.md section 8f, N4).
//
// The reference's decoder (/root/reference/attic/map_experiment/squeeze.h:502-551) interleaves two
// things: reading a token from the adaptive-Huffman stream (serial, host) and executing it --
// storing a literal or copying `len` bytes from `dist` back, byte by byte because source and
// destination may overlap (squeeze.h:533-539).  Once the tokens are known the second part is a
// parallel problem:
//
//   1. an exclusive scan of the token lengths gives every token its output offset;
//   2. every output byte learns how far back its value comes from: 0 for a literal, `dist` for a
//      byte of a match (`hop`);
//   3. pointer doubling: hop[j] += hop[j - hop[j]] until the byte j - hop[j] is a literal.  A chain
//      only ever walks towards the start, so in-place updates are safe: whatever a thread reads
//      from a neighbour is a valid (possibly already longer) hop of the same chain.  A hop that
//      has reached its literal is marked (bit 31) and never looked at again, and whoever lands
//      on a marked hop is done as well: after two or three rounds most bytes cost one read;
//   4. out[j] = out[j - hop[j]].
//
// Distances accumulate along a chain, so hops are 31-bit and one call handles < 2 GiB.
#pragma once

#include <cstdint>
#include <cuda_runtime.h>

namespace expand {

constexpr int kScanBlock = 2048;          // tokens per block of the length scan (256 threads x 8)
constexpr uint32_t kLanded = 0x80000000u; // hop mark: the byte this hop points at is a literal

__device__ __forceinline__ uint32_t token_len(uint32_t t) { return (t >> 16) != 0 ? (t >> 16) : 1u; }

// per block of kScanBlock tokens: total output length
__global__ void __launch_bounds__(256)
block_lengths(const uint32_t* __restrict__ tokens, size_t n_tokens, uint64_t* __restrict__ block_sum) {
    __shared__ uint32_t warp_sum[8];
    const size_t base = (size_t)blockIdx.x * kScanBlock;
    uint32_t mine = 0;
#pragma unroll
    for (int k = 0; k < kScanBlock / 256; k++) {
        const size_t i = base + (size_t)k * 256 + threadIdx.x;
        if (i < n_tokens) { mine += token_len(tokens[i]); }
    }
#pragma unroll
    for (int s = 16; s > 0; s >>= 1) { mine += __shfl_xor_sync(0xFFFFFFFFu, mine, s); }
    if ((threadIdx.x & 31) == 0) { warp_sum[threadIdx.x >> 5] = mine; }
    __syncthreads();
    if (threadIdx.x == 0) {
        uint64_t total = 0;
        for (int w = 0; w < 8; w++) { total += warp_sum[w]; }
        block_sum[blockIdx.x] = total;
    }
}

// exclusive scan of the block sums, one CTA (the array is n_tokens / 2048 long); total -> *result
__global__ void __launch_bounds__(1024)
scan_blocks(uint64_t* __restrict__ block_sum, size_t blocks, uint64_t* __restrict__ result) {
    __shared__ uint64_t part[1024];
    const size_t per = (blocks + 1023) / 1024;
    const size_t lo = (size_t)threadIdx.x * per, hi = min(lo + per, blocks);
    uint64_t mine = 0;
    for (size_t k = lo; k < hi; k++) { mine += block_sum[k]; }
    part[threadIdx.x] = mine;
    __syncthreads();
    for (int s = 1; s < 1024; s <<= 1) {
        const uint64_t add = threadIdx.x >= s ? part[threadIdx.x - s] : 0;
        __syncthreads();
        part[threadIdx.x] += add;
        __syncthreads();
    }
    uint64_t run = part[threadIdx.x] - mine;             // exclusive prefix of this thread's range
    for (size_t k = lo; k < hi; k++) {
        const uint64_t v = block_sum[k];
        block_sum[k] = run;
        run += v;
    }
    if (threadIdx.x == 1023) { *result = part[1023]; }
}

// Every token writes its bytes' hops (and a literal its value).  One warp per 32 tokens: the
// lanes scan their lengths, then the warp walks the 32 tokens' output range together so that
// the stores are coalesced.  A bad token (a literal word above 0xFF, dist 0, a match reaching
// before byte 0) raises *bad and leaves hop 0 and byte 0: garbage, but every later read is in bounds.
__global__ void __launch_bounds__(256)
place_tokens(const uint32_t* __restrict__ tokens, size_t n_tokens, const uint64_t* __restrict__ block_off,
             uint8_t* __restrict__ out, uint32_t* __restrict__ hop, uint64_t bytes, int* __restrict__ bad) {
    __shared__ uint32_t warp_sum[8];
    __shared__ uint32_t tok_s[8][32], off_s[8][33];
    const size_t base = (size_t)blockIdx.x * kScanBlock;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    // warp w owns tokens [base + 256 w, base + 256 (w+1)): first its total, then the warp prefix
    uint32_t lens[8], total = 0;
#pragma unroll
    for (int k = 0; k < 8; k++) {
        const size_t i = base + (size_t)warp * 256 + (size_t)k * 32 + lane;
        lens[k] = i < n_tokens ? token_len(tokens[i]) : 0u;
        total += lens[k];
    }
    uint32_t wt = total;
#pragma unroll
    for (int s = 16; s > 0; s >>= 1) { wt += __shfl_xor_sync(0xFFFFFFFFu, wt, s); }
    if (lane == 0) { warp_sum[warp] = wt; }
    __syncthreads();
    uint64_t at = block_off[blockIdx.x];
    for (int w = 0; w < warp; w++) { at += warp_sum[w]; }
#pragma unroll 1
    for (int k = 0; k < 8; k++) {
        const size_t i = base + (size_t)warp * 256 + (size_t)k * 32 + lane;
        // inclusive scan of the 32 lengths of this row
        uint32_t inc = lens[k];
#pragma unroll
        for (int s = 1; s < 32; s <<= 1) {
            const uint32_t up = __shfl_up_sync(0xFFFFFFFFu, inc, s);
            if (lane >= s) { inc += up; }
        }
        const uint32_t row = __shfl_sync(0xFFFFFFFFu, inc, 31);
        tok_s[warp][lane] = i < n_tokens ? tokens[i] : 0u;
        off_s[warp][lane] = inc - lens[k];
        if (lane == 31) { off_s[warp][32] = row; }
        __syncwarp();
        // the row's output range [at, at + row): lane j handles bytes at + j, at + j + 32, ...
        int t = 0;
        for (uint32_t b = lane; b < row; b += 32) {
            while (off_s[warp][t + 1] <= b) { t++; }            // token that owns byte b (offsets ascend)
            const uint32_t tk = tok_s[warp][t];
            const uint64_t j = at + b;
            if (j < bytes) {
                const uint32_t len = tk >> 16, dist = tk & 0xFFFFu;
                if (len == 0) {
                    // a literal is a byte value: a word such as a symbol word (bits 8..15 set) is refused
                    if (tk > 0xFFu) { *bad = 1; out[j] = 0; }
                    else { out[j] = (uint8_t)tk; }
                    hop[j] = 0;
                } else {
                    // a match may not reach before the start of the output (squeeze.h:529-545)
                    const uint64_t first = at + off_s[warp][t];
                    if (dist == 0 || dist > first) { *bad = 1; hop[j] = 0; out[j] = 0; }
                    else { hop[j] = dist; }
                }
            } else {
                *bad = 1;                                       // tokens describe more than `bytes`
            }
        }
        __syncwarp();
        at += row;
    }
}

// One round of pointer doubling.  All rounds a chain can need (32: hops are 31-bit) are queued at
// once, without a host round trip in between: round r raises flag[r % 3] when some hop has not
// reached its literal yet, and a round whose predecessor raised nothing returns at once -- every
// block reads the same flag, written by a kernel that has finished.  The third flag is the one
// the next round will raise; this round clears it.
__global__ void __launch_bounds__(256)
double_hops(uint32_t* __restrict__ hop, uint64_t bytes, int* __restrict__ flag, int round) {
    if (round > 0 && flag[(round + 2) % 3] == 0) {          // the previous round found every chain landed
        if (blockIdx.x == 0 && threadIdx.x == 0) { flag[(round + 1) % 3] = 0; flag[round % 3] = 0; }
        return;
    }
    if (blockIdx.x == 0 && threadIdx.x == 0) { flag[(round + 1) % 3] = 0; }
    const uint64_t stride = (uint64_t)gridDim.x * blockDim.x;
    bool any = false;
    for (uint64_t j = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; j < bytes; j += stride) {
        const uint32_t h = hop[j];
        if (h == 0 || (h & kLanded) != 0) { continue; }       // a literal, or already on its literal
        const uint32_t g = hop[j - h];
        if (g == 0) {
            hop[j] = h | kLanded;
        } else if ((g & kLanded) != 0) {
            hop[j] = (h + (g & ~kLanded)) | kLanded;
        } else {
            hop[j] = h + g;
            any = true;                                       // still on its way
        }
    }
    if (__syncthreads_or(any) && threadIdx.x == 0) { flag[round % 3] = 1; }
}

__global__ void __launch_bounds__(256)
fetch_bytes(const uint32_t* __restrict__ hop, uint8_t* __restrict__ out, uint64_t bytes) {
    const uint64_t stride = (uint64_t)gridDim.x * blockDim.x;
    for (uint64_t j = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; j < bytes; j += stride) {
        const uint32_t h = hop[j] & ~kLanded;
        if (h != 0) { out[j] = out[j - h]; }
    }
}

}  // namespace expand
