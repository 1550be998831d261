// Group kernel of 5x5 angular windows (an = 2, A = 25 SAIs): the arithmetic of k_groups (groups.cuh) — gather, 2-D
// id / dct / bior, 5x5 angular DCT or SA-DCT, haar / hw / dct along the similar patches, hard threshold or Wiener
// shrinkage, useSD, the inverses, staging for k_aggregate — in a layout that fits 25 SAIs into one CTA.
//
// One CTA per reference patch, one colour channel at a time, as k_groups. The channel's group is N * 25 * k^2 floats
// (twice that in step 2); validate() keeps N * k^2 * (step 2 ? 2 : 1) <= 2048, i.e. at most 204,800 B of dynamic shared
// memory. The row padding of k_groups (k + 1 floats per row) would not fit: patches are stored densely, k^2 floats each,
// with the rows XOR-swizzled so that the 2-D row and column passes and the per-position passes (angular, 5th dimension,
// gather, staging) stay free of bank conflicts (g25_at). Only one CTA fits on an SM, so it runs 512 threads.
#pragma once
#include "groups.cuh"

#define G25_NT 512
#define G25_SW 5
#define G25_A  (G25_SW * G25_SW)

// Position (p, q) of patch pa in the dense layout. L = 32 / K patch rows share one line of the 32 banks. Row p of patch pa is
// stored as row p ^ (pa mod L), which puts the L consecutive patches of a row pass (and the L rows of a column pass) into
// different lines; inside its row, column q moves to q ^ (p / L | (pa mod L) << log2(K / L)), which spreads the rows of one
// line over all K banks of a row.
template <int K> __device__ __forceinline__ int g25_at(int pa, int p, int q)
{
    constexpr int L = 32 / K, SH = K == 16 ? 3 : 1;
    const int h = pa & (L - 1);
    return pa * (K * K) + (p ^ h) * K + (q ^ ((p / L) | (h << SH)));
}

// 2-D DCT of npatch patches in place: lf_dct2d's arithmetic (rows, then columns with the normalisers)
template <int K> __device__ __forceinline__ void g25_dct2d(float *B, int npatch, bool fwd)
{
    const float *T = fwd ? c_tab.dct2f : c_tab.dct2i;
    for (int item = threadIdx.x; item < npatch * K; item += blockDim.x) {      // rows
        const int pa = item / K, p = item % K;
        float v[K], o[K];
#pragma unroll
        for (int j = 0; j < K; ++j) { const float x = B[g25_at<K>(pa, p, j)]; v[j] = fwd ? x : x * c_tab.cni2[p * K + j]; }
#pragma unroll
        for (int kk = 0; kk < K; ++kk) {
            float acc = 0.f;
#pragma unroll
            for (int j = 0; j < K; ++j) acc = fmaf(v[j], T[kk * K + j], acc);
            o[kk] = acc;
        }
#pragma unroll
        for (int j = 0; j < K; ++j) B[g25_at<K>(pa, p, j)] = o[j];
    }
    __syncthreads();
    for (int item = threadIdx.x; item < npatch * K; item += blockDim.x) {      // columns
        const int pa = item / K, q = item % K;
        float v[K], o[K];
#pragma unroll
        for (int j = 0; j < K; ++j) v[j] = B[g25_at<K>(pa, j, q)];
#pragma unroll
        for (int kk = 0; kk < K; ++kk) {
            float acc = 0.f;
#pragma unroll
            for (int j = 0; j < K; ++j) acc = fmaf(v[j], T[kk * K + j], acc);
            o[kk] = acc;
        }
#pragma unroll
        for (int j = 0; j < K; ++j) B[g25_at<K>(pa, j, q)] = fwd ? o[j] * c_tab.cn2[j * K + q] : c_tab.coef2inv * o[j];
    }
    __syncthreads();
}

// one level of the Bior1.5 decomposition / reconstruction on the top-left N1 x N1 corner (lf_bior_level)
template <int K, int N1> __device__ __forceinline__ void g25_bior_level(float *B, int npatch, bool fwd)
{
#pragma unroll 1
    for (int pass = 0; pass < 2; ++pass) {
        const bool rows = fwd == (pass == 0);       // forward: rows then columns; inverse: columns then rows
        for (int item = threadIdx.x; item < npatch * N1; item += blockDim.x) {
            const int pa = item / N1, l = item % N1;
            float x[N1];
#pragma unroll
            for (int j = 0; j < N1; ++j) x[j] = B[rows ? g25_at<K>(pa, l, j) : g25_at<K>(pa, j, l)];
            if (fwd) lf_bior_line_fwd<N1>(x, 1); else lf_bior_line_inv<N1>(x, 1);
#pragma unroll
            for (int j = 0; j < N1; ++j) B[rows ? g25_at<K>(pa, l, j) : g25_at<K>(pa, j, l)] = x[j];
        }
        __syncthreads();
    }
}
template <int K> __device__ __forceinline__ void g25_t2d(float *B, int npatch, unsigned tau_2D, bool fwd)
{
    if (tau_2D == 5) g25_dct2d<K>(B, npatch, fwd);
    else if (tau_2D == 7) {
        if (fwd) {
            if (K >= 16) g25_bior_level<K, 16>(B, npatch, true);
            g25_bior_level<K, 8>(B, npatch, true);
            g25_bior_level<K, 4>(B, npatch, true);
            g25_bior_level<K, 2>(B, npatch, true);
        } else {
            g25_bior_level<K, 2>(B, npatch, false);
            g25_bior_level<K, 4>(B, npatch, false);
            g25_bior_level<K, 8>(B, npatch, false);
            if (K >= 16) g25_bior_level<K, 16>(B, npatch, false);
        }
    }
}

// 5th dimension of the (st, p, q) vector across the NS similar patches: loaded to registers, lf_filter5d, stored back
template <int STEP, int K, int NS>
__device__ __forceinline__ float g25_filter5d(float *X, float *E, int st, int p, int q, unsigned tau_5D, bool shrink, int c, int lg)
{
    float x[NS], e[NS];
#pragma unroll
    for (int n = 0; n < NS; ++n) {
        const int o = g25_at<K>(n * G25_A + st, p, q);
        x[n] = X[o];
        if (STEP == 2) e[n] = E[o];
    }
    const float w = lf_filter5d<STEP, NS>(x, e, 0, 1, tau_5D, shrink, c, lg);
    float *dst = STEP == 1 ? X : E;
    const float *src = STEP == 1 ? x : e;
#pragma unroll
    for (int n = 0; n < NS; ++n) dst[g25_at<K>(n * G25_A + st, p, q)] = src[n];
    return w;
}
// the rare 5-D DCT: through the out-of-line lf_filter5d_dct on local copies
template <int STEP, int K>
__device__ __forceinline__ float g25_filter5d_dct(float *X, float *E, int st, int p, int q, int ns, bool shrink, int c, int lg)
{
    float x[LF_MAXN], e[LF_MAXN];
    for (int n = 0; n < ns; ++n) {
        const int o = g25_at<K>(n * G25_A + st, p, q);
        x[n] = X[o];
        if (STEP == 2) e[n] = E[o];
    }
    const float w = lf_filter5d_dct(STEP, x, e, 0, 1, ns, shrink, c, lg);
    float *dst = STEP == 1 ? X : E;
    const float *src = STEP == 1 ? x : e;
    for (int n = 0; n < ns; ++n) dst[g25_at<K>(n * G25_A + st, p, q)] = src[n];
    return w;
}

template <int STEP, int K>
__device__ __forceinline__ void g25_body(const GroupArgs25 &g, int r, int nSx, const GroupShapeT<G25_SW> &sh, const unsigned *sofs,
                                         const unsigned char *szero, float *smem, float *red)
{
    constexpr int A = G25_A, k2 = K * K, LK = K == 16 ? 4 : 3;
    constexpr int PPI = G25_NT / k2;                // patches per sweep of the block: 2 for k = 16, 8 for k = 8
    const int tid = threadIdx.x;
    const int lg = 31 - __clz(nSx);
    const unsigned plane = (unsigned) g.w * (unsigned) g.h;
    const int sub = tid >> (2 * LK), pq = tid & (k2 - 1);
    const int p = pq >> LK, q = pq & (K - 1);
    const int npatch = nSx * A;
    const bool use_sadct = sh.use_sadct != 0 && g.tau_4D == 6;
    float *X = smem;
    float *E = smem + (size_t) g.N * A * k2;        // step 2 only
    float *zdst = g.zbuf + (size_t) r * g.N * A * g.C * k2 + pq;
    float sd_w = 0.f;

    for (int c = 0; c < g.C; ++c) {
        // ---- gather (core:286-299): raw patches ----
        {
            const unsigned tofs = (unsigned) c * plane + (unsigned) (p * g.w + q);
            for (int pa = sub; pa < npatch; pa += PPI) {
                const int o = g25_at<K>(pa, p, q);
                if (!szero[pa]) {
                    const unsigned src = sofs[pa] + tofs;
                    lf_cp_async4(&X[o], g.nsym + src);
                    if (STEP == 2) lf_cp_async4(&E[o], g.bsym + src);
                } else {
                    X[o] = 0.f;
                    if (STEP == 2) E[o] = 0.f;
                }
            }
            lf_cp_async_wait_all();
        }
        __syncthreads();
        // ---- 2-D spatial transform ----
        g25_t2d<K>(X, npatch, g.tau_2D, true);
        if (STEP == 2) g25_t2d<K>(E, npatch, g.tau_2D, true);
        // ---- angular transform (core:354-360) ----
        if (g.tau_4D != 4) {
            for (int n = sub; n < nSx; n += PPI) {
#pragma unroll 1
                for (int rep = 0; rep < STEP; ++rep) {
                    float *B = rep == 0 ? X : E;
                    float v[A];
#pragma unroll
                    for (int st = 0; st < A; ++st) v[st] = B[g25_at<K>(n * A + st, p, q)];
                    if (use_sadct) {
                        float u[A];
#pragma unroll
                        for (int st = 0; st < A; ++st) u[st] = v[st];
                        lf_sadct_fwd(u, sh, G25_SW);
#pragma unroll
                        for (int st = 0; st < A; ++st) v[st] = u[st];
                    } else lf_dct4_fwd<G25_SW>(v);
#pragma unroll
                    for (int st = 0; st < A; ++st) B[g25_at<K>(n * A + st, p, q)] = v[st];
                }
            }
            __syncthreads();
        }
        // ---- 5th dimension + shrinkage (core:371-410 / :1170-1210) ----
        float wpart = 0.f;
        for (int st = sub; st < A; st += PPI) {
            const bool shrink = !use_sadct || sh.mask_dct[st];
            if (g.tau_5D == 5) { wpart += g25_filter5d_dct<STEP, K>(X, E, st, p, q, nSx, shrink, c, lg); continue; }
            switch (nSx) {
                case 1:  wpart += g25_filter5d<STEP, K, 1>(X, E, st, p, q, g.tau_5D, shrink, c, lg); break;
                case 2:  wpart += g25_filter5d<STEP, K, 2>(X, E, st, p, q, g.tau_5D, shrink, c, lg); break;
                case 4:  wpart += g25_filter5d<STEP, K, 4>(X, E, st, p, q, g.tau_5D, shrink, c, lg); break;
                case 8:  wpart += g25_filter5d<STEP, K, 8>(X, E, st, p, q, g.tau_5D, shrink, c, lg); break;
                // validate(): N k^2 (step 2: 2 N k^2) <= 2048, so step 2 has at most 16 patches
                case 16: wpart += g25_filter5d<STEP, K, 16>(X, E, st, p, q, g.tau_5D, shrink, c, lg); break;
                default:
                    if (STEP == 1) wpart += g25_filter5d<STEP, K, 32>(X, E, st, p, q, g.tau_5D, shrink, c, lg);
                    break;
            }
        }
        const float wsum = lf_block_sum_f(wpart, red);     // also a barrier for the phase above
        const float sg = c_tab.sigma[c];
        float wgt = wsum > 0.0f ? (sg > 0.0f ? 1.0f / (c_tab.sigma2[c] * wsum) : 1.0f / wsum) : 1.0f;   // core:419-420
        float *Z = STEP == 1 ? X : E;
        if (g.use_sd) {      // sd_weighting_5d (core:3140-3173), as k_groups
            if (g.use_sd == 1 || c == 0) {
                float m1 = 0.f, m2 = 0.f;
                for (int pa = sub; pa < npatch; pa += PPI) { const float xv = Z[g25_at<K>(pa, p, q)]; m1 += xv; m2 += xv * xv; }
                const float mean = lf_block_sum_f(m1, red);
                const float sq = lf_block_sum_f(m2, red);
                const float Nn = (float) (g.use_sd == 1 ? nSx * A : nSx * k2);
                const float res = (sq - mean * mean / Nn) / (Nn - 1.0f);
                sd_w = res > 0.0f ? 1.0f / sqrtf(res) : 0.0f;
            }
            wgt = sd_w;
        }
        // ---- inverse angular transform (core:432-451) ----
        if (g.tau_4D != 4) {
            for (int n = sub; n < nSx; n += PPI) {
                float v[A];
#pragma unroll
                for (int st = 0; st < A; ++st) v[st] = Z[g25_at<K>(n * A + st, p, q)];
                if (use_sadct) {
                    float u[A];
#pragma unroll
                    for (int st = 0; st < A; ++st) u[st] = v[st];
                    lf_sadct_inv(u, sh, G25_SW);
#pragma unroll
                    for (int st = 0; st < A; ++st) v[st] = u[st];
                } else lf_dct4_inv<G25_SW>(v);
#pragma unroll
                for (int st = 0; st < A; ++st) Z[g25_at<K>(n * A + st, p, q)] = v[st];
            }
            __syncthreads();
        }
        // ---- inverse 2-D transform (core:489-493) ----
        g25_t2d<K>(Z, npatch, g.tau_2D, false);
        // ---- stage the filtered patches and the weight for k_aggregate ----
        if (tid == 0) g.wbuf[(size_t) r * g.C + c] = wgt;
        for (int pa = sub; pa < npatch; pa += PPI) zdst[(pa * g.C + c) * k2] = Z[g25_at<K>(pa, p, q)];
        __syncthreads();
    }
}

template <int STEP>
__global__ void __launch_bounds__(G25_NT, 1) k_groups25(GroupArgs25 g)
{
    extern __shared__ float smem[];
    __shared__ GroupShapeT<G25_SW> sh;
    __shared__ float red[G25_NT / 32];
    __shared__ unsigned sofs[LF_MAXN * G25_A];          // per gathered patch: st*C*plane + position
    __shared__ unsigned char szero[LF_MAXN * G25_A];    // patch reads as zeros (empty SAI, or column w-k: core:1697)
    const int r = blockIdx.x + g.r0;
    const int nSx = (int) g.bm_count[r];
    if (!lf_group_setup<false, G25_SW, GroupArgs25>(g, r, nSx, sh, sofs, szero)) return;
    if (g.k == 8) g25_body<STEP, 8>(g, r, nSx, sh, sofs, szero, smem, red);
    else g25_body<STEP, 16>(g, r, nSx, sh, sofs, szero, smem, red);
}
