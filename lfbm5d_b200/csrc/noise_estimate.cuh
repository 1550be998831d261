// Noise-level estimate of a light field (lfbm5d_estimate_sigma): Donoho's median absolute deviation of the finest-scale diagonal
// Haar detail, on the input as given (RGB or grey, before any colour transform).
//
// For every non-masked SAI st, channel c and 2 x 2 block at (2i, 2j), i < H/2, j < W/2 (an odd last row / column is dropped):
//   d = ((x00 - x01) - (x10 - x11)) * 0.5f      (float, no contraction; white noise of std sigma gives d of std sigma)
// key = |d|. M(S) = the key of 0-based rank (n - 1) / 2 of the n keys of a set S (lower median, an element of S), and
// sigma = M / 0.6744897501960817f, one correctly rounded float division. Segments: 0 = pooled over all keys, 1 + c = channel c,
// 1 + C + st = SAI st (all its channels).
//
// The medians are exact radix selects over the key bits: non-negative floats order like their uint32 patterns. Three passes take the
// digits [31:21], [20:10] and [9:0]; each pass recomputes the keys from the light field (nothing is materialised) and counts, per
// segment, the keys whose higher bits equal the prefix the segment has selected so far. A CTA covers a tile of block rows of one
// (SAI, channel) plane, so it feeds exactly three segments; it histograms in shared memory and adds its non-zero bins to 64-bit
// global counters. Integer counts: the result does not depend on the order the CTAs run in. Between passes k_ne_select (one CTA per
// segment) finds the bin that holds the remaining rank and extends the prefix; after the third pass the prefix is the key.
#pragma once
#include "common.cuh"

#define NE_BINS    2048      // 11-bit digits (the last pass uses 10 of them)
#define NE_THREADS 256
#define NE_UNROLL  4         // keys per thread per iteration: 16 independent loads in flight
#define NE_TILE_KEYS 32768   // keys per CTA at most (whole block rows); keeps the per-CTA clear / flush of 3 x 2048 bins below 5 %
#define NE_SIGMA_DIV 0.6744897501960817f   // median(|N(0, 1)|)

struct NeSeg {
    unsigned long long rank;   // rank of the median among the keys that still match the prefix
    unsigned prefix;           // key bits selected so far (the key itself after the last pass)
    unsigned empty;            // no key in this segment (masked SAI): sigma 0
};

// digit position of pass p: shift and width; a key belongs to a segment in pass p > 0 when key >> (shift + width) == prefix
__host__ __device__ __forceinline__ int ne_shift(int pass) { return pass == 0 ? 21 : pass == 1 ? 10 : 0; }
__host__ __device__ __forceinline__ int ne_width(int pass) { return pass == 2 ? 10 : 11; }

__device__ __forceinline__ unsigned ne_key(float x00, float x01, float x10, float x11)
{
    const float d = __fmul_rn(__fsub_rn(__fsub_rn(x00, x01), __fsub_rn(x10, x11)), 0.5f);
    return __float_as_uint(d) & 0x7FFFFFFFu;
}

// grid (tiles of `rows` block rows, C, asize). lf: [asize][C][H][W]; seg: 1 + C + asize segment states; hist: [1 + C + asize][NE_BINS].
__global__ void __launch_bounds__(NE_THREADS) k_ne_hist(const float *__restrict__ lf, const unsigned *__restrict__ mask, int W, int H, int rows,
                                                          int pass, const NeSeg *__restrict__ seg, unsigned long long *__restrict__ hist)
{
    const int st = blockIdx.z, c = blockIdx.y, C = gridDim.y;
    if (!mask[st]) return;
    __shared__ __align__(16) unsigned h[3][NE_BINS];
    for (int i = threadIdx.x; i < 3 * NE_BINS / 4; i += NE_THREADS) reinterpret_cast<uint4 *>(&h[0][0])[i] = make_uint4(0, 0, 0, 0);
    const int sg[3] = { 0, 1 + c, 1 + C + st };
    const int shift = ne_shift(pass), top = shift + ne_width(pass);
    unsigned pre[3] = { 0, 0, 0 };
    if (pass > 0)
#pragma unroll
        for (int s = 0; s < 3; s++) pre[s] = seg[sg[s]].prefix;
    __syncthreads();

    const int W2 = W >> 1, H2 = H >> 1;
    const int i0 = blockIdx.x * rows, i1 = min(H2, i0 + rows);
    const unsigned nkeys = (unsigned) (i1 - i0) * (unsigned) W2;
    const float *plane = lf + ((size_t) st * C + c) * H * W;
    const unsigned lane = threadIdx.x & 31;
    // every lane runs the same number of iterations (the warp-wide match below needs all 32)
    const unsigned step = NE_THREADS * NE_UNROLL;
    for (unsigned base = 0; base < nkeys; base += step) {
        float x[NE_UNROLL][4];
        bool ok[NE_UNROLL];
#pragma unroll
        for (int u = 0; u < NE_UNROLL; u++) {
            const unsigned k = base + u * NE_THREADS + threadIdx.x;
            ok[u] = k < nkeys;
            const unsigned i = k / W2, j = k - i * W2;
            const float *r0 = plane + (size_t) (i0 + i) * 2 * W + 2 * j;
            if (ok[u]) {
                x[u][0] = __ldg(r0); x[u][1] = __ldg(r0 + 1); x[u][2] = __ldg(r0 + W); x[u][3] = __ldg(r0 + W + 1);
            }
        }
#pragma unroll
        for (int u = 0; u < NE_UNROLL; u++) {
            unsigned m = 0, digit = 0;
            if (ok[u]) {
                const unsigned key = ne_key(x[u][0], x[u][1], x[u][2], x[u][3]);
                digit = (key >> shift) & (NE_BINS - 1);
                if (pass == 0) m = 1;     // all three segments take every key: one histogram, flushed three times
                else {
                    const unsigned hi = key >> top;
#pragma unroll
                    for (int s = 0; s < 3; s++) m |= (hi == pre[s]) << s;
                }
            }
            // warp aggregation: lanes with the same (digit, segments) add once. Noise puts most keys of pass 0 into a few bins; in
            // passes 1 and 2 most keys match no prefix, and a warp without a match skips the step.
            if (!__ballot_sync(0xFFFFFFFFu, m != 0)) continue;
            const unsigned v = m ? digit | (m << 11) : 0xFFFFFFFFu;
            const unsigned peers = __match_any_sync(0xFFFFFFFFu, v);
            if (m && lane == (unsigned) (__ffs(peers) - 1)) {
                const unsigned n = __popc(peers);
#pragma unroll
                for (int s = 0; s < 3; s++)
                    if (m & (1u << s)) atomicAdd(&h[s][digit], n);
            }
        }
    }
    __syncthreads();
#pragma unroll
    for (int s = 0; s < 3; s++) {
        const unsigned *src = h[pass == 0 ? 0 : s];
        unsigned long long *dst = hist + (size_t) sg[s] * NE_BINS;
        for (int i = threadIdx.x; i < NE_BINS; i += NE_THREADS) {
            const unsigned n = src[i];
            if (n) atomicAdd(&dst[i], (unsigned long long) n);
        }
    }
}

// One CTA per segment: the bin of this pass that holds the segment's remaining rank. Pass 0 also sets the rank, (n - 1) / 2 of the
// n keys counted. Clears the bins it read for the next pass.
__global__ void __launch_bounds__(NE_THREADS) k_ne_select(unsigned long long *__restrict__ hist, NeSeg *__restrict__ seg, int pass)
{
    constexpr int PER = NE_BINS / NE_THREADS;
    __shared__ unsigned long long wsum[NE_THREADS / 32];
    __shared__ unsigned long long total;
    unsigned long long *hs = hist + (size_t) blockIdx.x * NE_BINS;
    NeSeg *S = seg + blockIdx.x;
    const int t = threadIdx.x, lane = t & 31, w = t >> 5;
    unsigned long long b[PER], sum = 0;
#pragma unroll
    for (int q = 0; q < PER; q++) { b[q] = hs[t * PER + q]; hs[t * PER + q] = 0; sum += b[q]; }
    // inclusive scan of the per-thread sums over the CTA
    unsigned long long inc = sum;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const unsigned long long v = __shfl_up_sync(0xFFFFFFFFu, inc, o);
        if (lane >= o) inc += v;
    }
    if (lane == 31) wsum[w] = inc;
    __syncthreads();
    if (t == 0) {
        unsigned long long a = 0;
        for (int q = 0; q < NE_THREADS / 32; q++) { const unsigned long long v = wsum[q]; wsum[q] = a; a += v; }
        total = a;
    }
    __syncthreads();
    const unsigned long long excl = wsum[w] + inc - sum;
    if (pass == 0) {
        if (total == 0) { if (t == 0) { S->empty = 1; S->prefix = 0; S->rank = 0; } return; }
    } else if (S->empty) return;
    const unsigned long long rank = pass == 0 ? (total - 1) / 2 : S->rank;
    __syncthreads();      // every thread has read S->rank before the owner of the bin rewrites it
    if (rank >= excl && rank < excl + sum) {
        unsigned long long r = rank - excl;
        int q = PER - 1;
        bool found = false;
#pragma unroll
        for (int u = 0; u < PER; u++)
            if (!found) {
                if (r < b[u]) { q = u; found = true; }
                else r -= b[u];
            }
        const unsigned digit = (unsigned) (t * PER + q);
        S->prefix = pass == 0 ? digit : (S->prefix << ne_width(pass)) | digit;
        S->rank = r;
        S->empty = 0;
    }
}
