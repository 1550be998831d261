// Group kernel of 5x5 angular windows (an = 2, A = 25 SAIs): the arithmetic of k_groups (groups.cuh) — gather, 2-D
// id / dct / bior, 5x5 angular DCT or SA-DCT, haar / hw / dct along the similar patches, hard threshold or Wiener
// shrinkage, useSD, the inverses, staging for k_aggregate — in a layout that fits 25 SAIs into one CTA.
//
// One CTA per reference patch, one colour channel at a time, as k_groups. The channel's group is N * 25 * k^2 floats
// (twice that in step 2); validate() keeps N * k^2 * (step 2 ? 2 : 1) <= 2048, i.e. at most 204,800 B of dynamic shared
// memory. The row padding of k_groups (k + 1 floats per row) would not fit: patches are stored densely, k^2 floats each,
// with the rows XOR-swizzled so that the 2-D row and column passes and the per-position passes (angular, 5th dimension,
// gather, staging) stay free of bank conflicts (LfSwizzled in groups.cuh). Only one CTA fits on an SM, so it runs 512 threads.
#pragma once
#include "groups.cuh"

#define G25_NT 512
#define G25_SW 5
#define G25_A  (G25_SW * G25_SW)

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
    const LfSwizzled<K> lay;
    float *X = smem;
    float *E = smem + (size_t) g.N * A * k2;        // step 2 only
    float *zdst = g.zbuf + (size_t) r * g.N * A * g.C * k2 + pq;
    float sd_w = 0.f;

    for (int c = 0; c < g.C; ++c) {
        // ---- gather (core:286-299): raw patches ----
        {
            const unsigned tofs = (unsigned) c * plane + (unsigned) (p * g.w + q);
            for (int pa = sub; pa < npatch; pa += PPI) {
                const int o = lay.at(pa, p, q);
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
        lf_t2d<K>(X, npatch, lay, g.tau_2D, true);
        if (STEP == 2) lf_t2d<K>(E, npatch, lay, g.tau_2D, true);
        // ---- angular transform (core:354-360) ----
        if (g.tau_4D != 4) {
            for (int n = sub; n < nSx; n += PPI) {
#pragma unroll 1
                for (int rep = 0; rep < STEP; ++rep) {
                    float *B = rep == 0 ? X : E;
                    float v[A];
#pragma unroll
                    for (int st = 0; st < A; ++st) v[st] = B[lay.at(n * A + st, p, q)];
                    if (use_sadct) {
                        float u[A];
#pragma unroll
                        for (int st = 0; st < A; ++st) u[st] = v[st];
                        lf_sadct_fwd(u, sh, G25_SW);
#pragma unroll
                        for (int st = 0; st < A; ++st) v[st] = u[st];
                    } else lf_dct4_fwd<G25_SW>(v);
#pragma unroll
                    for (int st = 0; st < A; ++st) B[lay.at(n * A + st, p, q)] = v[st];
                }
            }
            __syncthreads();
        }
        // ---- 5th dimension + shrinkage (core:371-410 / :1170-1210) ----
        float wpart = 0.f;
        for (int st = sub; st < A; st += PPI) {
            const bool shrink = !use_sadct || sh.mask_dct[st];
            if (g.tau_5D == 5) { wpart += lf_filter5d_dct_group<STEP, A, 1>(&X, &E, lay, st, p, q, nSx, shrink, c, lg); continue; }
            switch (nSx) {
                case 1:  wpart += lf_filter5d_group<STEP, 1, A, 1>(&X, &E, lay, st, p, q, g.tau_5D, shrink, c, lg); break;
                case 2:  wpart += lf_filter5d_group<STEP, 2, A, 1>(&X, &E, lay, st, p, q, g.tau_5D, shrink, c, lg); break;
                case 4:  wpart += lf_filter5d_group<STEP, 4, A, 1>(&X, &E, lay, st, p, q, g.tau_5D, shrink, c, lg); break;
                case 8:  wpart += lf_filter5d_group<STEP, 8, A, 1>(&X, &E, lay, st, p, q, g.tau_5D, shrink, c, lg); break;
                // validate(): N k^2 (step 2: 2 N k^2) <= 2048, so step 2 has at most 16 patches
                case 16: wpart += lf_filter5d_group<STEP, 16, A, 1>(&X, &E, lay, st, p, q, g.tau_5D, shrink, c, lg); break;
                default:
                    if (STEP == 1) wpart += lf_filter5d_group<STEP, 32, A, 1>(&X, &E, lay, st, p, q, g.tau_5D, shrink, c, lg);
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
                for (int pa = sub; pa < npatch; pa += PPI) { const float xv = Z[lay.at(pa, p, q)]; m1 += xv; m2 += xv * xv; }
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
                for (int st = 0; st < A; ++st) v[st] = Z[lay.at(n * A + st, p, q)];
                if (use_sadct) {
                    float u[A];
#pragma unroll
                    for (int st = 0; st < A; ++st) u[st] = v[st];
                    lf_sadct_inv(u, sh, G25_SW);
#pragma unroll
                    for (int st = 0; st < A; ++st) v[st] = u[st];
                } else lf_dct4_inv<G25_SW>(v);
#pragma unroll
                for (int st = 0; st < A; ++st) Z[lay.at(n * A + st, p, q)] = v[st];
            }
            __syncthreads();
        }
        // ---- inverse 2-D transform (core:489-493) ----
        lf_t2d<K>(Z, npatch, lay, g.tau_2D, false);
        // ---- stage the filtered patches and the weight for k_aggregate ----
        if (tid == 0) g.wbuf[(size_t) r * g.C + c] = wgt;
        for (int pa = sub; pa < npatch; pa += PPI) zdst[(pa * g.C + c) * k2] = Z[lay.at(pa, p, q)];
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
