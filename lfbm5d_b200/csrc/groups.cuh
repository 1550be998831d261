// 5-D group processing: gather -> 2-D spatial transform -> angular (SA-)DCT -> 1-D transform along the similar
// patches -> hard threshold / Wiener shrinkage -> inverses (group kernels, one CTA per reference patch: the generic
// k_groups with one colour channel at a time in shared memory, the register-resident k_groups_id16, and the packed
// k_groups_w8 in groups_wiener8.cuh), then the ordered weighted aggregation of the staged patches (k_aggregate).
// Restates core:277-528 (step 1) and :1054-1329 (step 2).
#pragma once
#include "common.cuh"
#include <cooperative_groups.h>
namespace cg = cooperative_groups;

template <int SW> struct GroupShapeT;

struct GroupArgsBase {
    int C, asw, A, k, log2k, N, w, h, pst, nc;
    int r0;                           // first reference patch of the launch (blockIdx.x + r0; row bands of the multi-GPU path)
    int RS, PS;                       // shared-memory row stride / patch stride (floats)
    unsigned tau_2D, tau_4D, tau_5D;
    const int *rows, *cols;
    const unsigned *bm_count, *bm_idx;            // [R], [R*(N+1)]
    const unsigned *first;                        // [A][plane] disparity argmin
    const unsigned char *shape;                   // [A][plane]
    const float *nsym, *bsym;                     // [A][C][plane]
    float *numsym, *densym;
    // staging for the ordered aggregation kernel (k_aggregate): filtered patches, weights, positions, flags
    float *zbuf;                                  // [R][N][A][C][k2]
    float *wbuf;                                  // [R][C]
    const unsigned short *gmask;                  // [R] bit st = SAI st takes part in the group's angular shape (k_group_masks), A <= 9
    const struct GroupShapeT<LF_LUTASW> *shape_lut;   // [2^A] SA-DCT index tables per shape (host-built, core:300-330), A <= 9
    const unsigned char *act;                     // partial-window branch: [R] 1 = reference patch still to be processed; nullptr = all
    int use_sd;                                   // 1: weight = 1 / sample std of the filtered group (core:3140-3173); 2: BM3D's variant (bm3d.cpp:1345)
    int partial;                                  // pst != cst: local 2-D variants (no zero column, core:1735)
    unsigned *ent;                                // [A][R*N] (y << 16 | x) of every patch that is aggregated, else LF_NOENT
    int R;
};
struct GroupArgs : GroupArgsBase {                // k_groups, k_groups_id16, k_groups_w8: windows up to 3x3
    LfWindow9 win;
};
struct GroupArgs25 : GroupArgsBase {              // k_groups25: 5x5 windows
    LfWindow win;
    const unsigned *gmask32;                      // [R] 25-bit angular shape masks (k_group_masks32); the SA-DCT tables are built per group
};

#define LF_NOENT 0xffffffffu

// SA-DCT index tables of one angular shape of a window of side up to SW
template <int SW> struct GroupShapeT {
    unsigned mask[SW * SW], idx[SW * SW], idx_col[SW * SW], mask_dct[SW * SW];
    unsigned row_size[SW], col_size[SW];
    int use_sadct;
};
typedef GroupShapeT<LF_LUTASW> GroupShape;        // the host table's entries (windows up to 3x3)

// The tables of the shape `bits` (bit st: SAI st takes part) of an asw x asw window, as sadct_4d_process builds them
// (core:1969-2010); ensure_shape_lut runs the same construction on the host for every shape of a window up to 3x3.
template <int SW>
__host__ __device__ inline void lf_shape_build(GroupShapeT<SW> &sh, unsigned bits, unsigned asw)
{
    const unsigned A = asw * asw;
    unsigned size = 0;
    for (unsigned st = 0; st < SW * SW; st++) { sh.mask[st] = st < A ? (bits >> st) & 1u : 0u; sh.idx[st] = sh.idx_col[st] = sh.mask_dct[st] = 0; size += sh.mask[st]; }
    sh.use_sadct = size != A;
    unsigned mask_col[SW * SW] = { 0 };
    for (unsigned s = 0; s < asw; s++) {
        unsigned rr = 0;
        for (unsigned t = 0; t < asw; t++) if (sh.mask[s * asw + t]) sh.idx[s * asw + rr++] = t;
        sh.row_size[s] = rr;
        for (unsigned t = 0; t < rr; t++) mask_col[s * asw + t] = 1;
    }
    for (unsigned t = 0; t < asw; t++) {
        unsigned rr = 0;
        for (unsigned s = 0; s < asw; s++) if (mask_col[s * asw + t]) sh.idx_col[(rr++) * asw + t] = s;
        sh.col_size[t] = rr;
        for (unsigned s = 0; s < rr; s++) sh.mask_dct[s * asw + t] = 1;
    }
    for (unsigned s = asw; s < SW; s++) sh.row_size[s] = sh.col_size[s] = 0;
}

// ---- 1-D transforms along the similar patches (lib_transforms.cpp:290-321, :403-471), fully unrolled ----
template <int NS> __device__ __forceinline__ void lf_haar_fwd(float *v)
{
    float tmp[NS > 1 ? NS : 1];
#pragma unroll
    for (int N = NS; N >= 2; N >>= 1) {
        const int n = N / 2;
#pragma unroll
        for (int i = 0; i < n; ++i) {
            const float a = v[2 * i], b = v[2 * i + 1];
            tmp[i] = (a + b) * LF_SQRT2_INV_F;
            tmp[n + i] = (a - b) * LF_SQRT2_INV_F;
        }
#pragma unroll
        for (int i = 0; i < N; ++i) v[i] = tmp[i];
    }
}
template <int NS> __device__ __forceinline__ void lf_haar_inv(float *v)
{
    float tmp[NS > 1 ? NS : 1];
#pragma unroll
    for (int n = 1; n < NS; n *= 2) {
#pragma unroll
        for (int i = 0; i < n; ++i) {
            const float a = v[i], b = v[n + i];
            tmp[2 * i] = (a + b) * LF_SQRT2_INV_F;
            tmp[2 * i + 1] = (a - b) * LF_SQRT2_INV_F;
        }
#pragma unroll
        for (int i = 0; i < 2 * n; ++i) v[i] = tmp[i];
    }
}
template <int NS> __device__ __forceinline__ void lf_hadamard(float *v)
{
    float tmp[NS > 1 ? NS : 1];
#pragma unroll
    for (int len = NS; len >= 2; len >>= 1) {
        const int n = len / 2;
#pragma unroll
        for (int base = 0; base < NS; base += len) {
#pragma unroll
            for (int i = 0; i < n; ++i) {
                const float a = v[base + 2 * i], b = v[base + 2 * i + 1];
                tmp[base + i] = a + b;
                tmp[base + n + i] = a - b;
            }
        }
#pragma unroll
        for (int i = 0; i < NS; ++i) v[i] = tmp[i];
    }
}

__device__ __forceinline__ float lf_block_sum_f(float v, float *sh)
{
    for (int o = 16; o > 0; o >>= 1) v += __shfl_down_sync(0xffffffffu, v, o);
    __syncthreads();
    if ((threadIdx.x & 31) == 0) sh[threadIdx.x >> 5] = v;
    __syncthreads();
    float r = 0.f;
    const int nw = (blockDim.x + 31) >> 5;
    for (int i = 0; i < nw; ++i) r += sh[i];
    return r;
}

// 1-D DCT of length ns = 2^lg along the similar patches with the normalisers of preProcess_5d (core:2544-2556, :2578-2593).
// A rarely used option: kept out of line with rolled loops (compile time and register pressure of the common paths).
__device__ __noinline__ void lf_dct5(float *v, int ns, int lg, bool fwd)
{
    const float *T = (fwd ? c_tab.dct5f : c_tab.dct5i) + ((1 << (2 * lg)) - 1) / 3;
    float a[LF_MAXN], o[LF_MAXN];
#pragma unroll 1
    for (int n = 0; n < ns; ++n) a[n] = fwd ? v[n] : v[n] * (n == 0 ? LF_SQRT2_F : 1.0f);
#pragma unroll 1
    for (int kk = 0; kk < ns; ++kk) {
        float acc = 0.f;
#pragma unroll 1
        for (int j = 0; j < ns; ++j) acc = fmaf(a[j], T[kk * ns + j], acc);
        o[kk] = acc;
    }
#pragma unroll 1
    for (int n = 0; n < ns; ++n) v[n] = fwd ? o[n] * (n == 0 ? c_tab.cn5_0[lg] : c_tab.cn5_c[lg]) : o[n] * c_tab.coef5inv[lg];
}

// 5th-dimension filtering with the DCT (ht_filtering_dct_5d core:2524-2700, wiener_filtering_dct_5d :2943-3130) of one
// (st, pq) vector; out of line like lf_dct5, its arrays live in local memory.
__device__ __noinline__ float lf_filter5d_dct(int step, float *X, float *E, int base, int nstride, int ns, bool shrink, int c, int lg)
{
    float vo[LF_MAXN], ve[LF_MAXN];
#pragma unroll 1
    for (int n = 0; n < ns; ++n) { vo[n] = X[base + n * nstride]; if (step == 2) ve[n] = E[base + n * nstride]; }
    lf_dct5(vo, ns, lg, true);
    if (step == 2) lf_dct5(ve, ns, lg, true);
    float wsum = 0.f;
    if (shrink) {
        const float T = c_tab.thr_dct[c], s2 = c_tab.sigma2[c];
#pragma unroll 1
        for (int n = 0; n < ns; ++n) {
            if (step == 1) { if (fabsf(vo[n]) > T) wsum += 1.0f; else vo[n] = 0.0f; }
            else {
                float value = ve[n] * ve[n];
                value = value / (value + s2);
                ve[n] = vo[n] * value;
                wsum += value;
            }
        }
    }
    float *out = step == 1 ? vo : ve;
    lf_dct5(out, ns, lg, false);
    float *dst = step == 1 ? X : E;
#pragma unroll 1
    for (int n = 0; n < ns; ++n) dst[base + n * nstride] = out[n];
    return wsum;
}

// ---- 5th-dimension filtering of one (st, pq) vector; returns this thread's contribution to weight_table[c] ----
template <int STEP, int NS>
__device__ __forceinline__ float lf_filter5d(float *X, float *E, int base, int nstride, unsigned tau_5D, bool shrink, int c, int lg)
{
    float vo[NS], ve[NS];
#pragma unroll
    for (int n = 0; n < NS; ++n) vo[n] = X[base + n * nstride];
    if (STEP == 2) {
#pragma unroll
        for (int n = 0; n < NS; ++n) ve[n] = E[base + n * nstride];
    }
    const bool haar = tau_5D == 9;
    if (NS > 1) {
        if (haar) { lf_haar_fwd<NS>(vo); if (STEP == 2) lf_haar_fwd<NS>(ve); }
        else { lf_hadamard<NS>(vo); if (STEP == 2) lf_hadamard<NS>(ve); }
    }
    float wsum = 0.f;
    if (shrink) {
        if (STEP == 1) {
            const float T = haar ? c_tab.thr[c][0] : c_tab.thr[c][lg];
#pragma unroll
            for (int n = 0; n < NS; ++n) {
                if (fabsf(vo[n]) > T) wsum += 1.0f; else vo[n] = 0.0f;
            }
        } else {
            const float s2 = c_tab.sigma2[c];
            const float hc = c_tab.hadcoef[lg];
#pragma unroll
            for (int n = 0; n < NS; ++n) {
                float value;
                if (haar) {
                    value = ve[n] * ve[n];
                    value = value / (value + s2);
                    ve[n] = vo[n] * value;
                } else {
                    value = ve[n] * ve[n] * hc;
                    value = value / (value + s2);
                    ve[n] = vo[n] * value * hc;
                }
                wsum += value;
            }
        }
    }
    float *out = STEP == 1 ? vo : ve;
    if (NS > 1) {
        if (haar) lf_haar_inv<NS>(out);
        else {
            lf_hadamard<NS>(out);
            if (STEP == 1) {
                const float hc = c_tab.hadcoef[lg];
#pragma unroll
                for (int n = 0; n < NS; ++n) out[n] *= hc;
            }
        }
    }
    float *dst = STEP == 1 ? X : E;
#pragma unroll
    for (int n = 0; n < NS; ++n) dst[base + n * nstride] = out[n];
    return wsum;
}

// ---- angular tables of windows up to TW x TW (LfTables: windows up to 3x3 and 5x5 windows have their own) ----
template <int TW> __device__ __forceinline__ const float *lf_tab_dcta(int n, bool fwd)      // 1-D DCT of length n
{
    if constexpr (TW > LF_LUTASW) return fwd ? c_tab.dctaf5[n - 1] : c_tab.dctai5[n - 1];
    else return fwd ? c_tab.dctaf[n - 1] : c_tab.dctai[n - 1];
}
template <int TW> __device__ __forceinline__ const float *lf_tab_cn4(bool fwd)
{
    if constexpr (TW > LF_LUTASW) return fwd ? c_tab.cn4_5 : c_tab.cni4_5;
    else return fwd ? c_tab.cn4 : c_tab.cni4;
}
template <int TW> __device__ __forceinline__ const float *lf_tab_cnsa(int n, bool fwd)
{
    if constexpr (TW > LF_LUTASW) return fwd ? c_tab.cnsa5[n - 2] : c_tab.cnisa5[n - 2];
    else return fwd ? c_tab.cnsa[n - 2] : c_tab.cnisa[n - 2];
}
template <int TW> __device__ __forceinline__ float lf_tab_coefsa_inv(int n)
{
    if constexpr (TW > LF_LUTASW) return c_tab.coefsa_inv5[n];
    else return c_tab.coefsa_inv[n];
}

// ---- angular transforms of one (n, pq) vector v[A] (st fastest) ----
template <int ASW> __device__ __forceinline__ void lf_dct4_fwd(float *v)
{
    constexpr int TW = ASW > LF_LUTASW ? LF_MAXASW : LF_LUTASW;
    const float *T = lf_tab_dcta<TW>(ASW, true);
    const float *cn4 = lf_tab_cn4<TW>(true);
    float y[ASW * ASW];
#pragma unroll
    for (int s = 0; s < ASW; ++s)
#pragma unroll
        for (int kk = 0; kk < ASW; ++kk) {
            float acc = 0.f;
#pragma unroll
            for (int t = 0; t < ASW; ++t) acc = fmaf(v[s * ASW + t], T[kk * ASW + t], acc);
            y[s * ASW + kk] = acc;
        }
#pragma unroll
    for (int t = 0; t < ASW; ++t)
#pragma unroll
        for (int kk = 0; kk < ASW; ++kk) {
            float acc = 0.f;
#pragma unroll
            for (int s = 0; s < ASW; ++s) acc = fmaf(y[s * ASW + t], T[kk * ASW + s], acc);
            v[kk * ASW + t] = acc * cn4[kk * ASW + t];
        }
}
template <int ASW> __device__ __forceinline__ void lf_dct4_inv(float *v)
{
    constexpr int TW = ASW > LF_LUTASW ? LF_MAXASW : LF_LUTASW;
    const float *T = lf_tab_dcta<TW>(ASW, false);
    const float *cni4 = lf_tab_cn4<TW>(false);
    float a[ASW * ASW], y[ASW * ASW];
#pragma unroll
    for (int st = 0; st < ASW * ASW; ++st) a[st] = v[st] * cni4[st];
#pragma unroll
    for (int s = 0; s < ASW; ++s)
#pragma unroll
        for (int kk = 0; kk < ASW; ++kk) {
            float acc = 0.f;
#pragma unroll
            for (int t = 0; t < ASW; ++t) acc = fmaf(a[s * ASW + t], T[kk * ASW + t], acc);
            y[s * ASW + kk] = acc;
        }
#pragma unroll
    for (int t = 0; t < ASW; ++t)
#pragma unroll
        for (int kk = 0; kk < ASW; ++kk) {
            float acc = 0.f;
#pragma unroll
            for (int s = 0; s < ASW; ++s) acc = fmaf(y[s * ASW + t], T[kk * ASW + s], acc);
            v[kk * ASW + t] = acc * c_tab.coef4inv;
        }
}
// generic 1-D r2r of length n (1..SW) on a small array
template <int SW> __device__ __forceinline__ void lf_r2r_small(const float *in, float *out, int n, bool fwd)
{
    const float *T = lf_tab_dcta<SW>(n, fwd);
    for (int kk = 0; kk < n; ++kk) {
        float acc = 0.f;
        for (int j = 0; j < n; ++j) acc = fmaf(in[j], T[kk * n + j], acc);
        out[kk] = acc;
    }
}
// shape-adaptive variants (core:1969-2116, :2131-2264); rare path, generic code
template <int SW> __device__ __noinline__ void lf_sadct_fwd(float *v, const GroupShapeT<SW> &sh, int asw)
{
    float a[SW], b[SW];
    for (int s = 0; s < asw; ++s) {
        const int n = sh.row_size[s];
        if (n == 1) v[s * asw] = v[s * asw + sh.idx[s * asw]];
        else if (n > 1) {
            for (int t = 0; t < n; ++t) a[t] = v[s * asw + sh.idx[s * asw + t]];
            lf_r2r_small<SW>(a, b, n, true);
            for (int t = 0; t < n; ++t) v[s * asw + t] = b[t] * lf_tab_cnsa<SW>(n, true)[t];
        }
    }
    for (int t = 0; t < asw; ++t) {
        const int n = sh.col_size[t];
        if (n == 1) v[t] = v[sh.idx_col[t] * asw + t];
        else if (n > 1) {
            for (int s = 0; s < n; ++s) a[s] = v[sh.idx_col[s * asw + t] * asw + t];
            lf_r2r_small<SW>(a, b, n, true);
            for (int s = 0; s < n; ++s) v[s * asw + t] = b[s] * lf_tab_cnsa<SW>(n, true)[s];
        }
    }
    const float coef = 0.5f * LF_SQRT2_INV_F;
    for (int st = 0; st < asw * asw; ++st) v[st] *= (float) sh.mask_dct[st] * coef;
}
template <int SW> __device__ __noinline__ void lf_sadct_inv(float *v, const GroupShapeT<SW> &sh, int asw)
{
    float a[SW], b[SW];
    const float c2 = 2.0f * LF_SQRT2_F;
    for (int t = 0; t < asw; ++t) {
        const int n = sh.col_size[t];
        if (n == 1) v[sh.idx_col[t] * asw + t] = v[t] * c2;
        else if (n > 1) {
            for (int s = 0; s < n; ++s) a[s] = v[s * asw + t] * lf_tab_cnsa<SW>(n, false)[s] * c2;
            lf_r2r_small<SW>(a, b, n, false);
            const float coef = lf_tab_coefsa_inv<SW>(n);
            for (int s = 0; s < n; ++s) v[sh.idx_col[s * asw + t] * asw + t] = b[s] * coef;
        }
    }
    for (int s = 0; s < asw; ++s) {
        const int n = sh.row_size[s];
        if (n == 1) v[s * asw + sh.idx[s * asw]] = v[s * asw];
        else if (n > 1) {
            for (int t = 0; t < n; ++t) a[t] = v[s * asw + t] * lf_tab_cnsa<SW>(n, false)[t];
            lf_r2r_small<SW>(a, b, n, false);
            const float coef = lf_tab_coefsa_inv<SW>(n);
            for (int t = 0; t < n; ++t) v[s * asw + sh.idx[s * asw + t]] = b[t] * coef;
        }
    }
    for (int st = 0; st < asw * asw; ++st) v[st] = v[st] * (float) sh.mask[st];
}

// ---- shared-memory layouts of a channel's group: at(pa, p, q) is the offset of position (p, q) of local patch pa ----
// rows padded to RS floats, patches PS floats apart (3x3 windows: RS = k + 1 removes the bank conflicts of the 2-D passes)
struct LfPadded {
    int RS, PS;
    __device__ __forceinline__ int at(int pa, int p, int q) const { return pa * PS + p * RS + q; }
};
// 5x5 windows: patches stored densely, k^2 floats each (the padding would not fit 25 SAIs into one CTA). L = 32 / K patch rows
// share one line of the 32 banks. Row p of patch pa is stored as row p ^ (pa mod L), which puts the L consecutive patches of a
// row pass (and the L rows of a column pass) into different lines; inside its row, column q moves to
// q ^ (p / L | (pa mod L) << log2(K / L)), which spreads the rows of one line over all K banks of a row.
template <int K> struct LfSwizzled {
    __device__ __forceinline__ int at(int pa, int p, int q) const
    {
        constexpr int L = 32 / K, SH = K == 16 ? 3 : 1;
        const int h = pa & (L - 1);
        return pa * (K * K) + (p ^ h) * K + (q ^ ((p / L) | (h << SH)));
    }
};

// ---- 2-D spatial transforms, in place on npatch patches of the layout lay ----
template <int K, class L> __device__ __forceinline__ void lf_dct2d(float *B, int npatch, const L &lay, bool fwd)
{
    const float *T = fwd ? c_tab.dct2f : c_tab.dct2i;
    for (int item = threadIdx.x; item < npatch * K; item += blockDim.x) {      // rows (contiguous dimension first)
        const int pa = item / K, p = item % K;
        float v[K], o[K];
#pragma unroll
        for (int j = 0; j < K; ++j) { const float x = B[lay.at(pa, p, j)]; v[j] = fwd ? x : x * c_tab.cni2[p * K + j]; }
#pragma unroll
        for (int kk = 0; kk < K; ++kk) {
            float acc = 0.f;
#pragma unroll
            for (int j = 0; j < K; ++j) acc = fmaf(v[j], T[kk * K + j], acc);
            o[kk] = acc;
        }
#pragma unroll
        for (int j = 0; j < K; ++j) B[lay.at(pa, p, j)] = o[j];
    }
    __syncthreads();
    for (int item = threadIdx.x; item < npatch * K; item += blockDim.x) {      // columns
        const int pa = item / K, q = item % K;
        float v[K], o[K];
#pragma unroll
        for (int j = 0; j < K; ++j) v[j] = B[lay.at(pa, j, q)];
#pragma unroll
        for (int kk = 0; kk < K; ++kk) {
            float acc = 0.f;
#pragma unroll
            for (int j = 0; j < K; ++j) acc = fmaf(v[j], T[kk * K + j], acc);
            o[kk] = acc;
        }
#pragma unroll
        for (int j = 0; j < K; ++j) B[lay.at(pa, j, q)] = fwd ? o[j] * c_tab.cn2[j * K + q] : c_tab.coef2inv * o[j];
    }
    __syncthreads();
}

// Bior1.5 full decomposition / reconstruction (lib_transforms.cpp:46-204) of the line B[at(0)], ..., B[at(N1 - 1)];
// all indices compile-time so that the line lives in registers
template <int N1, class I> __device__ __forceinline__ void lf_bior_line_fwd(float *B, const I &at)
{
    float v[N1], o[N1];
    constexpr int N2 = N1 / 2;
#pragma unroll
    for (int j = 0; j < N1; ++j) v[j] = B[at(j)];
#pragma unroll
    for (int j = 0; j < N2; ++j) {
        float vl = 0.0f, vh = 0.0f;
#pragma unroll
        for (int t = 0; t < 10; ++t) {
            const float xv = v[(t + 2 * j + 4 * N1 - 4) % N1];      // periodic extension by 4 samples (per_ext_ind)
            vl += xv * c_tab.lpd[t];
            if (t == 4 || t == 5) vh += xv * c_tab.hpd[t];           // the other high-pass taps are exactly zero
        }
        o[j] = vl; o[j + N2] = vh;
    }
#pragma unroll
    for (int j = 0; j < N1; ++j) B[at(j)] = o[j];
}
template <int N1, class I> __device__ __forceinline__ void lf_bior_line_inv(float *B, const I &at)
{
    float v[N1], o[N1];
    constexpr int N2 = N1 / 2;
#pragma unroll
    for (int j = 0; j < N1; ++j) v[j] = B[at(j)];
#pragma unroll
    for (int i = 0; i < N2; ++i) {
        float vl = 0.0f, vh = 0.0f;
#pragma unroll
        for (int t = 0; t < 10; ++t) {
            const float xv = v[(t * N2 + i) % N1];                    // extension by 4*N2 = 2*N1 samples: index mod N1
            if (t == 4 || t == 5) vl += c_tab.lpr[t] * xv;            // the other low-pass reconstruction taps are zero
            vh += c_tab.hpr[t] * xv;
        }
        o[2 * i] = vh; o[2 * i + 1] = vl;
    }
#pragma unroll
    for (int j = 0; j < N1; ++j) B[at(j)] = o[j];
}
// one pass of a level on the top-left N1 x N1 corner of every patch, one thread per (patch, line): rows or columns
template <int N1, bool FWD, class L> __device__ __forceinline__ void lf_bior_pass(float *B, int npatch, const L &lay, bool rows)
{
    for (int item = threadIdx.x; item < npatch * N1; item += blockDim.x) {
        const int pa = item / N1, l = item % N1;
        const auto at = [&](int j) { return rows ? lay.at(pa, l, j) : lay.at(pa, j, l); };
        if (FWD) lf_bior_line_fwd<N1>(B, at); else lf_bior_line_inv<N1>(B, at);
    }
    __syncthreads();
}
template <int N1, class L> __device__ __forceinline__ void lf_bior_level(float *B, int npatch, const L &lay, bool fwd)
{
    if (fwd) { lf_bior_pass<N1, true>(B, npatch, lay, true); lf_bior_pass<N1, true>(B, npatch, lay, false); }
    else { lf_bior_pass<N1, false>(B, npatch, lay, false); lf_bior_pass<N1, false>(B, npatch, lay, true); }     // columns first
}
template <int K, class L> __device__ __forceinline__ void lf_bior2d(float *B, int npatch, const L &lay, bool fwd)
{
    if (fwd) {
        if (K >= 16) lf_bior_level<16>(B, npatch, lay, true);
        lf_bior_level<8>(B, npatch, lay, true);
        lf_bior_level<4>(B, npatch, lay, true);
        lf_bior_level<2>(B, npatch, lay, true);
    } else {
        lf_bior_level<2>(B, npatch, lay, false);
        lf_bior_level<4>(B, npatch, lay, false);
        lf_bior_level<8>(B, npatch, lay, false);
        if (K >= 16) lf_bior_level<16>(B, npatch, lay, false);
    }
}
// tau_2D: dct or bior (id: nothing to do); k = 12 takes id or dct (validate(): Bior1.5 needs a power of two)
template <int K, class L> __device__ __forceinline__ void lf_t2d(float *B, int npatch, const L &lay, unsigned tau_2D, bool fwd)
{
    if (tau_2D == 5) lf_dct2d<K>(B, npatch, lay, fwd);
    else if constexpr ((K & (K - 1)) == 0) {
        if (tau_2D == 7) lf_bior2d<K>(B, npatch, lay, fwd);
    }
}

// Per-group set-up shared by the group kernels (core:277-299, :486-503): SA-DCT shape of the group, source offset of every
// gathered patch (ZB: patches that read as zeros point at the zero block behind the window buffers, else szero marks them),
// and the aggregation entries: (y << 16 | x) of every patch that k_aggregate has to add, LF_NOENT otherwise.
// Returns false (after marking the group's entries empty) for reference patches the partial-window branch skips.
// SW: window side the shared arrays are sized for; windows up to 3x3 copy their shape from the host table, 5x5 ones build it.
// ENT = false: leave the aggregation entries to another CTA of the group (k_groups_cl: rank 0 writes them).
template <bool ZB, int SW = LF_LUTASW, class GA = GroupArgs, bool ENT = true>
__device__ __forceinline__ bool lf_group_setup(const GA &g, int r, int nSx, GroupShapeT<SW> &sh, unsigned *sofs, unsigned char *szero)
{
    __shared__ unsigned s_yx[LF_MAXN * SW * SW];
    const int A = g.A, w = g.w, k = g.k;
    const int tid = threadIdx.x, nt = blockDim.x;
    const unsigned plane = (unsigned) g.w * (unsigned) g.h;
    if (g.act && !g.act[r]) {        // den-aware ind_initialize (utilities_LF.cpp:1031-1099): every pixel of the patch already has a weight
        if constexpr (ENT)
            for (int t = tid; t < g.N * A; t += nt) {
                const int n = t / A, st = t - n * A;
                g.ent[(size_t) st * g.R * g.N + (size_t) r * g.N + n] = LF_NOENT;
            }
        return false;
    }
    if constexpr (SW == LF_LUTASW) {
        if (tid >= nt - 32) {        // the last warp copies the group's SA-DCT tables, beside the offset loop of the first warps
            const unsigned *src = reinterpret_cast<const unsigned *>(g.shape_lut + g.gmask[r]);
            unsigned *dst = reinterpret_cast<unsigned *>(&sh);
            for (int i = tid - (nt - 32); i < (int) (sizeof(GroupShape) / 4); i += 32) dst[i] = src[i];
        }
    } else if (tid == nt - 32) lf_shape_build<SW>(sh, g.gmask32[r], (unsigned) g.asw);     // 2^25 shapes: no table, built per group
    for (int t = tid; t < nSx * A; t += nt) {
        const int n = t / A, st = t - n * A;
        const unsigned ind = g.bm_idx[(size_t) r * (g.N + 1) + n];
        const unsigned pv = (st == g.pst) ? ind : (g.win.mask[st] ? g.first[(size_t) st * plane + ind] : 0u);
        const unsigned py = pv / (unsigned) w, px = pv - py * (unsigned) w;
        const bool zero = !g.win.mask[st] || (!g.partial && (int) px >= w - k);       // empty SAI, or column w-k (core:1697)
        if (ZB) sofs[t] = zero ? (unsigned) A * (unsigned) g.C * plane : (unsigned) st * (unsigned) g.C * plane + pv;
        else { sofs[t] = (unsigned) st * (unsigned) g.C * plane + pv; szero[t] = zero ? 1 : 0; }
        s_yx[t] = (py << 16) | px;
    }
    __syncthreads();
    if constexpr (ENT)
        for (int t = tid; t < g.N * A; t += nt) {
            const int n = t / A, st = t - n * A;
            // core:486, :503: which SAIs receive this group's patches
            const bool on = n < nSx && !g.win.proc[st] && !(g.tau_4D == 6 && st != g.pst && !sh.mask[st]);
            g.ent[(size_t) st * g.R * g.N + (size_t) r * g.N + n] = on ? s_yx[t] : LF_NOENT;
        }
    return true;
}

// partial-window branch: reference patches of the grid that still contain a pixel without weight in SAI pst (channel 0)
__global__ void k_active_refs(const float *__restrict__ den0, const int *__restrict__ rows, const int *__restrict__ cols, int nc, int R, int w,
                              int k, unsigned char *__restrict__ act, unsigned *__restrict__ count)
{
    const int r = blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= R) return;
    const int ry = rows[r / nc], rx = cols[r % nc];
    const float *pp = den0 + (size_t) ry * w + rx;
    bool open = false;
    for (int p = 0; p < k && !open; ++p)
        for (int q = 0; q < k; ++q)
            if (pp[p * w + q] == 0.0f) { open = true; break; }
    act[r] = open ? 1 : 0;
    if (open) {      // count[1], count[2]: last row / column of an active reference patch (block matching stops behind them)
        atomicAdd(count, 1u);
        atomicMax(count + 1, (unsigned) ry);
        atomicMax(count + 2, (unsigned) rx);
    }
}

// bit st of gmask[r]: SAI st belongs to the angular shape of reference patch r (core:300-312)
template <typename M>
__device__ __forceinline__ void lf_group_mask(const int *__restrict__ rows, const int *__restrict__ cols, int nc, int r0, int r1, int w, unsigned plane,
                                              int A, int pst, const LfWindow &win, const unsigned char *__restrict__ shape, M *__restrict__ gmask)
{
    const int r = r0 + blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= r1) return;
    const int k_r = rows[r / nc] * w + cols[r % nc];
    unsigned m = 0;
    for (int st = 0; st < A; ++st) {
        const unsigned b = (st == pst) ? 1u : (win.mask[st] ? (unsigned) shape[(size_t) st * plane + k_r] : 0u);
        m |= (b ? 1u : 0u) << st;
    }
    gmask[r] = (M) m;
}
__global__ void k_group_masks(const int *__restrict__ rows, const int *__restrict__ cols, int nc, int r0, int r1, int w, unsigned plane, int A, int pst,
                              LfWindow win, const unsigned char *__restrict__ shape, unsigned short *__restrict__ gmask)
{
    lf_group_mask(rows, cols, nc, r0, r1, w, plane, A, pst, win, shape, gmask);
}
// 5x5 windows: 25 bits
__global__ void k_group_masks32(const int *__restrict__ rows, const int *__restrict__ cols, int nc, int r0, int r1, int w, unsigned plane, int A, int pst,
                                LfWindow win, const unsigned char *__restrict__ shape, unsigned *__restrict__ gmask)
{
    lf_group_mask(rows, cols, nc, r0, r1, w, plane, A, pst, win, shape, gmask);
}

// k = 12 (k_groups12): 288 threads, two patches of 144 positions per sweep. validate() keeps the group of one channel
// (N * A * k * (k + 1) floats, twice that in step 2) within LF_G12_SMEM bytes of dynamic shared memory.
#define LF_G12_NT 288
#define LF_G12_SMEM (220 * 1024)

// 2-D transform of the generic body: K = 0 dispatches on g.k (8 or 16)
template <int K> __device__ __forceinline__ void lf_t2d_k(float *B, int npatch, const GroupArgs &g, bool fwd)
{
    const LfPadded lay{ g.RS, g.PS };
    if constexpr (K != 0) lf_t2d<K>(B, npatch, lay, g.tau_2D, fwd);
    else if (g.k == 8) lf_t2d<8>(B, npatch, lay, g.tau_2D, fwd);
    else lf_t2d<16>(B, npatch, lay, g.tau_2D, fwd);
}

// Body of the generic group kernels. K = 0: k = 8 or 16 from the arguments, 256 threads (k_groups); K = 12: LF_G12_NT threads
// (k_groups12). The kernels declare the shared arrays (smem: the dynamic one): an extern declaration in this function would
// move the module's first extern shared array, and with it the dynamic shared-memory base of other kernels (k_groups25).
template <int STEP, int ASW, int K>
__device__ __forceinline__ void lf_groups_body(const GroupArgs &g, float *smem, GroupShape &sh, float *red, unsigned *sofs, unsigned char *szero)
{
    constexpr int A = ASW * ASW;
    const int tid = threadIdx.x;
    const int r = blockIdx.x + g.r0;
    const int k = K ? K : g.k, k2 = k * k, w = g.w;
    const unsigned plane = (unsigned) g.w * (unsigned) g.h;
    const int nSx = (int) g.bm_count[r];
    const int lg = 31 - __clz(nSx);
    const int PS = g.PS, RS = g.RS;
    float *X = smem;
    float *E = smem + (size_t) g.N * A * PS;      // step 2 only (N >= nSx except the duplicated single match: N >= 2)
    // thread <-> (sub, pq): a thread keeps its pixel/coefficient position and strides over patches
    const int PPI = K ? LF_G12_NT / (K * K) : 256 >> (2 * g.log2k);     // patches handled per sweep of the block (1 for k = 16, 2 for k = 12, 4 for k = 8)
    const int sub = K ? tid / (K * K) : tid >> (2 * g.log2k), pq = K ? tid - sub * (K * K) : tid & (k2 - 1);
    const int p = K ? pq / K : pq >> g.log2k, q = K ? pq - p * K : pq & (k - 1);
    const int poff = p * RS + q;
    const int npatch = nSx * A;
    if (!lf_group_setup<false>(g, r, nSx, sh, sofs, szero)) return;
    const bool use_sadct = sh.use_sadct != 0 && g.tau_4D == 6;
    float *zdst = g.zbuf + (size_t) r * g.N * A * g.C * k2 + pq;
    float sd_w = 0.f;

    for (int c = 0; c < g.C; ++c) {
        // ---- gather (core:286-299): raw patches ----
        {
            const unsigned tofs = (unsigned) c * plane + (unsigned) (p * w + q);
            // asynchronous global->shared copies: all of a thread's loads are in flight at once
            for (int pa = sub; pa < npatch; pa += PPI) {
                float *dx = &X[pa * PS + poff];
                if (!szero[pa]) {
                    const unsigned src = sofs[pa] + tofs;
                    lf_cp_async4(dx, g.nsym + src);
                    if (STEP == 2) lf_cp_async4(&E[pa * PS + poff], g.bsym + src);
                } else {
                    *dx = 0.f;
                    if (STEP == 2) E[pa * PS + poff] = 0.f;
                }
            }
            lf_cp_async_wait_all();
        }
        __syncthreads();
        // ---- 2-D spatial transform; patches that read as zeros stay zero under any of the transforms ----
        lf_t2d_k<K>(X, npatch, g, true);
        if (STEP == 2) lf_t2d_k<K>(E, npatch, g, true);
        // ---- angular transform (core:354-360) ----
        if (g.tau_4D != 4) {
            for (int n = sub; n < nSx; n += PPI) {
                const int off = n * A * PS + poff;
                for (int rep = 0; rep < STEP; ++rep) {
                    float *B = rep == 0 ? X : E;
                    float v[A];
#pragma unroll
                    for (int st = 0; st < A; ++st) v[st] = B[off + st * PS];
                    if (use_sadct) {        // rare: keep the dynamically indexed copy away from the register-resident one
                        float u[A];
#pragma unroll
                        for (int st = 0; st < A; ++st) u[st] = v[st];
                        lf_sadct_fwd(u, sh, ASW);
#pragma unroll
                        for (int st = 0; st < A; ++st) v[st] = u[st];
                    } else lf_dct4_fwd<ASW>(v);
#pragma unroll
                    for (int st = 0; st < A; ++st) B[off + st * PS] = v[st];
                }
            }
            __syncthreads();
        }
        // ---- 5th dimension + shrinkage (core:371-410 / :1170-1210) ----
        float wpart = 0.f;
        for (int st = sub; st < A; st += PPI) {
            const int base = st * PS + poff;
            const bool shrink = !use_sadct || sh.mask_dct[st];
            const int ns = A * PS;
            if (g.tau_5D == 5) { wpart += lf_filter5d_dct(STEP, X, E, base, ns, nSx, shrink, c, lg); continue; }
            switch (nSx) {
                case 1:  wpart += lf_filter5d<STEP, 1>(X, E, base, ns, g.tau_5D, shrink, c, lg); break;
                case 2:  wpart += lf_filter5d<STEP, 2>(X, E, base, ns, g.tau_5D, shrink, c, lg); break;
                case 4:  wpart += lf_filter5d<STEP, 4>(X, E, base, ns, g.tau_5D, shrink, c, lg); break;
                case 8:  wpart += lf_filter5d<STEP, 8>(X, E, base, ns, g.tau_5D, shrink, c, lg); break;
                case 16: wpart += lf_filter5d<STEP, 16>(X, E, base, ns, g.tau_5D, shrink, c, lg); break;
                default: wpart += lf_filter5d<STEP, 32>(X, E, base, ns, g.tau_5D, shrink, c, lg); break;
            }
        }
        const float wsum = lf_block_sum_f(wpart, red);     // also a barrier for the phase above
        const float sg = c_tab.sigma[c];
        float wgt = wsum > 0.0f ? (sg > 0.0f ? 1.0f / (c_tab.sigma2[c] * wsum) : 1.0f / wsum) : 1.0f;   // core:419-420
        float *Z = STEP == 1 ? X : E;
        if (g.use_sd) {      // sd_weighting_5d (core:3140-3173; N without the k^2 factor as written there); BM3D reads channel 0 for every c
            if (g.use_sd == 1 || c == 0) {
                float m1 = 0.f, m2 = 0.f;
                for (int pa = sub; pa < npatch; pa += PPI) { const float xv = Z[pa * PS + poff]; m1 += xv; m2 += xv * xv; }
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
                const int off = n * A * PS + poff;
                float v[A];
#pragma unroll
                for (int st = 0; st < A; ++st) v[st] = Z[off + st * PS];
                if (use_sadct) {
                    float u[A];
#pragma unroll
                    for (int st = 0; st < A; ++st) u[st] = v[st];
                    lf_sadct_inv(u, sh, ASW);
#pragma unroll
                    for (int st = 0; st < A; ++st) v[st] = u[st];
                } else lf_dct4_inv<ASW>(v);
#pragma unroll
                for (int st = 0; st < A; ++st) Z[off + st * PS] = v[st];
            }
            __syncthreads();
        }
        // ---- inverse 2-D transform (core:489-493) ----
        lf_t2d_k<K>(Z, npatch, g, false);
        // ---- stage the filtered patches and the weight; k_aggregate adds them in the reference's order ----
        if (tid == 0) g.wbuf[(size_t) r * g.C + c] = wgt;
        for (int pa = sub; pa < npatch; pa += PPI) zdst[(pa * g.C + c) * k2] = Z[pa * PS + poff];
        __syncthreads();
    }
}

template <int STEP, int ASW>
__global__ void __launch_bounds__(256) k_groups(GroupArgs g)
{
    extern __shared__ float smem[];
    __shared__ GroupShape sh;
    __shared__ float red[8];
    __shared__ unsigned sofs[LF_MAXN * LF_LUTA];          // per gathered patch: st*C*plane + position
    __shared__ unsigned char szero[LF_MAXN * LF_LUTA];    // patch reads as zeros (empty SAI, or column w-k: core:1697)
    lf_groups_body<STEP, ASW, 0>(g, smem, sh, red, sofs, szero);
}

template <int STEP, int ASW>
__global__ void __launch_bounds__(LF_G12_NT) k_groups12(GroupArgs g)
{
    extern __shared__ float smem[];
    __shared__ GroupShape sh;
    __shared__ float red[LF_G12_NT / 32];
    __shared__ unsigned sofs[LF_MAXN * LF_LUTA];
    __shared__ unsigned char szero[LF_MAXN * LF_LUTA];
    lf_groups_body<STEP, ASW, 12>(g, smem, sh, red, sofs, szero);
}

// ------------------------------------------------------------------------------------------------------------
// k = 16 groups of 3x3 windows whose channel does not fit into the shared memory of one CTA (N = 32 in step 1, N >= 16 in
// step 2 with 2-D dct / bior): the group of one reference patch runs on a cluster of CL CTAs of 256 threads (thread <-> pixel
// position, as k_groups at k = 16). Patch n of the group lives on CTA n % CL in local slot n / CL, with all of its SAIs, so
// the gather, the 2-D transforms, the angular transforms and the staging stay local. The 5th dimension runs across the
// cluster: the (st, pq) vectors are dealt out by st (CTA `rank` takes st = rank, rank + CL, ...), each thread loads its nSx
// values from the CTAs that own them through distributed shared memory, filters them with lf_filter5d / lf_filter5d_dct and
// stores them back. Group-wide sums (Wiener weight, useSD) are reduced per CTA and then added in rank order, so that the
// result does not depend on scheduling. Same per-element arithmetic as k_groups: step 1 is bit-identical to it.
// ------------------------------------------------------------------------------------------------------------
// 5th dimension of the (st, p, q) vector of the layout lay whose value n is local patch (n / CL) * A + st of CTA n % CL (Xr, Er:
// every CTA's X and E; k_groups_cl, and k_groups25 with CL = 1): loaded to registers, lf_filter5d, stored back
template <int STEP, int NS, int A, int CL, class L>
__device__ __forceinline__ float lf_filter5d_group(float *const *Xr, float *const *Er, const L &lay, int st, int p, int q, unsigned tau_5D,
                                                   bool shrink, int c, int lg)
{
    float x[NS], e[NS];
#pragma unroll
    for (int n = 0; n < NS; ++n) {
        const int o = lay.at((n / CL) * A + st, p, q);
        x[n] = Xr[n % CL][o];
        if (STEP == 2) e[n] = Er[n % CL][o];
    }
    const float w = lf_filter5d<STEP, NS>(x, e, 0, 1, tau_5D, shrink, c, lg);
    float *const *dst = STEP == 1 ? Xr : Er;
#pragma unroll
    for (int n = 0; n < NS; ++n) dst[n % CL][lay.at((n / CL) * A + st, p, q)] = STEP == 1 ? x[n] : e[n];
    return w;
}
// the rare 5-D DCT: through the out-of-line lf_filter5d_dct on local copies
template <int STEP, int A, int CL, class L>
__device__ __forceinline__ float lf_filter5d_dct_group(float *const *Xr, float *const *Er, const L &lay, int st, int p, int q, int ns,
                                                       bool shrink, int c, int lg)
{
    float x[LF_MAXN], e[LF_MAXN];
#pragma unroll 1
    for (int n = 0; n < ns; ++n) {
        const int o = lay.at((n / CL) * A + st, p, q);
        x[n] = Xr[n % CL][o];
        if (STEP == 2) e[n] = Er[n % CL][o];
    }
    const float w = lf_filter5d_dct(STEP, x, e, 0, 1, ns, shrink, c, lg);
    float *const *dst = STEP == 1 ? Xr : Er;
#pragma unroll 1
    for (int n = 0; n < ns; ++n) dst[n % CL][lay.at((n / CL) * A + st, p, q)] = STEP == 1 ? x[n] : e[n];
    return w;
}
// sum of the CTAs' partial sums part[i], in rank order (the same value in every thread of the cluster)
template <int CL>
__device__ __forceinline__ float lf_cluster_sum(cg::cluster_group &cluster, float *part, int i)
{
    float s = *cluster.map_shared_rank(part + i, 0);
#pragma unroll
    for (int j = 1; j < CL; ++j) s += *cluster.map_shared_rank(part + i, j);
    return s;
}

template <int STEP, int CL>
__global__ void __cluster_dims__(CL, 1, 1) __launch_bounds__(256) k_groups_cl(GroupArgs g)
{
    extern __shared__ float smem[];                       // this CTA's patches: N / CL slots of A patches (twice that in step 2)
    __shared__ GroupShape sh;
    __shared__ float red[8];
    __shared__ float part[3];                             // this CTA's partial sums: weight, useSD's sum and sum of squares
    __shared__ unsigned sofs[LF_MAXN * LF_LUTA];
    __shared__ unsigned char szero[LF_MAXN * LF_LUTA];
    constexpr int A = 9, k2 = 256;
    cg::cluster_group cluster = cg::this_cluster();
    const int rank = (int) cluster.block_rank();
    const int tid = threadIdx.x;
    const int r = blockIdx.x / CL + g.r0;
    const int w = g.w;
    const unsigned plane = (unsigned) g.w * (unsigned) g.h;
    const int nSx = (int) g.bm_count[r];
    const int lg = 31 - __clz(nSx);
    const int PS = g.PS, RS = g.RS;
    const int SS = A * PS;                                // slot stride (floats)
    float *X = smem;
    float *E = smem + (size_t) (g.N / CL) * SS;          // step 2 only
    const int pq = tid, p = pq >> 4, q = pq & 15;
    const int poff = p * RS + q;
    const int nloc = (nSx - rank + CL - 1) / CL;          // patches n = rank, rank + CL, ... of the group (0 when nSx <= rank)
    const int npl = nloc * A;
    // every CTA of the cluster reads the same act[r] and bm_count[r]: a skipped group is skipped by all of them, before any
    // cluster barrier
    if (!(rank == 0 ? lf_group_setup<false>(g, r, nSx, sh, sofs, szero)
                    : lf_group_setup<false, LF_LUTASW, GroupArgs, false>(g, r, nSx, sh, sofs, szero))) return;
    const bool use_sadct = sh.use_sadct != 0 && g.tau_4D == 6;
    float *zdst = g.zbuf + (size_t) r * g.N * A * g.C * k2 + pq;
    const LfPadded lay{ RS, PS };
    float *Xr[CL], *Er[CL];
#pragma unroll
    for (int j = 0; j < CL; ++j) { Xr[j] = cluster.map_shared_rank(X, j); Er[j] = STEP == 2 ? cluster.map_shared_rank(E, j) : nullptr; }
    float sd_w = 0.f;

    for (int c = 0; c < g.C; ++c) {
        // ---- gather (core:286-299) of this CTA's patches: local patch pl = slot * A + st is group patch (slot * CL + rank, st) ----
        {
            const unsigned tofs = (unsigned) c * plane + (unsigned) (p * w + q);
            for (int pl = 0; pl < npl; ++pl) {
                const int slot = pl / A, st = pl - slot * A;
                const int pa = (slot * CL + rank) * A + st;
                float *dx = &X[pl * PS + poff];
                if (!szero[pa]) {
                    const unsigned src = sofs[pa] + tofs;
                    lf_cp_async4(dx, g.nsym + src);
                    if (STEP == 2) lf_cp_async4(&E[pl * PS + poff], g.bsym + src);
                } else {
                    *dx = 0.f;
                    if (STEP == 2) E[pl * PS + poff] = 0.f;
                }
            }
            lf_cp_async_wait_all();
        }
        __syncthreads();
        // ---- 2-D spatial transform and angular transform (core:354-360) of the local patches ----
        // g.k is always 16 here; the run-time dispatch of k_groups is kept because ptxas allocates this kernel better with it
        // (lf_t2d<16> directly: 16 -> 24 B spills in <1,4>, 0 -> 52 B in <2,2>)
        lf_t2d_k<0>(X, npl, g, true);
        if (STEP == 2) lf_t2d_k<0>(E, npl, g, true);
        if (g.tau_4D != 4) {
            for (int slot = 0; slot < nloc; ++slot) {
                const int off = slot * SS + poff;
                for (int rep = 0; rep < STEP; ++rep) {
                    float *B = rep == 0 ? X : E;
                    float v[A];
#pragma unroll
                    for (int st = 0; st < A; ++st) v[st] = B[off + st * PS];
                    if (use_sadct) {
                        float u[A];
#pragma unroll
                        for (int st = 0; st < A; ++st) u[st] = v[st];
                        lf_sadct_fwd(u, sh, 3);
#pragma unroll
                        for (int st = 0; st < A; ++st) v[st] = u[st];
                    } else lf_dct4_fwd<3>(v);
#pragma unroll
                    for (int st = 0; st < A; ++st) B[off + st * PS] = v[st];
                }
            }
        }
        cluster.sync();        // the peers read this CTA's coefficients
        // ---- 5th dimension + shrinkage (core:371-410 / :1170-1210) across the cluster ----
        float wpart = 0.f;
        for (int st = rank; st < A; st += CL) {
            const bool shrink = !use_sadct || sh.mask_dct[st];
            if (g.tau_5D == 5) { wpart += lf_filter5d_dct_group<STEP, A, CL>(Xr, Er, lay, st, p, q, nSx, shrink, c, lg); continue; }
            switch (nSx) {
                case 1:  wpart += lf_filter5d_group<STEP, 1, A, CL>(Xr, Er, lay, st, p, q, g.tau_5D, shrink, c, lg); break;
                case 2:  wpart += lf_filter5d_group<STEP, 2, A, CL>(Xr, Er, lay, st, p, q, g.tau_5D, shrink, c, lg); break;
                case 4:  wpart += lf_filter5d_group<STEP, 4, A, CL>(Xr, Er, lay, st, p, q, g.tau_5D, shrink, c, lg); break;
                case 8:  wpart += lf_filter5d_group<STEP, 8, A, CL>(Xr, Er, lay, st, p, q, g.tau_5D, shrink, c, lg); break;
                case 16: wpart += lf_filter5d_group<STEP, 16, A, CL>(Xr, Er, lay, st, p, q, g.tau_5D, shrink, c, lg); break;
                default: wpart += lf_filter5d_group<STEP, 32, A, CL>(Xr, Er, lay, st, p, q, g.tau_5D, shrink, c, lg); break;
            }
        }
        const float wloc = lf_block_sum_f(wpart, red);
        if (tid == 0) part[0] = wloc;
        cluster.sync();        // the peers wrote this CTA's coefficients back; every partial weight is visible
        // step 1: the weight is a count of coefficients, exact in any order; step 2: rank order
        const float wsum = lf_cluster_sum<CL>(cluster, part, 0);
        const float sg = c_tab.sigma[c];
        float wgt = wsum > 0.0f ? (sg > 0.0f ? 1.0f / (c_tab.sigma2[c] * wsum) : 1.0f / wsum) : 1.0f;   // core:419-420
        float *Z = STEP == 1 ? X : E;
        if (g.use_sd) {      // sd_weighting_5d (core:3140-3173), as k_groups
            if (g.use_sd == 1 || c == 0) {
                float m1 = 0.f, m2 = 0.f;
                for (int pl = 0; pl < npl; ++pl) { const float xv = Z[pl * PS + poff]; m1 += xv; m2 += xv * xv; }
                const float s1 = lf_block_sum_f(m1, red);
                const float s2 = lf_block_sum_f(m2, red);
                if (tid == 0) { part[1] = s1; part[2] = s2; }
                cluster.sync();
                const float mean = lf_cluster_sum<CL>(cluster, part, 1);
                const float sq = lf_cluster_sum<CL>(cluster, part, 2);
                const float Nn = (float) (g.use_sd == 1 ? nSx * A : nSx * k2);
                const float res = (sq - mean * mean / Nn) / (Nn - 1.0f);
                sd_w = res > 0.0f ? 1.0f / sqrtf(res) : 0.0f;
            }
            wgt = sd_w;
        }
        // ---- inverse angular transform (core:432-451) and inverse 2-D transform (core:489-493) of the local patches ----
        if (g.tau_4D != 4) {
            for (int slot = 0; slot < nloc; ++slot) {
                const int off = slot * SS + poff;
                float v[A];
#pragma unroll
                for (int st = 0; st < A; ++st) v[st] = Z[off + st * PS];
                if (use_sadct) {
                    float u[A];
#pragma unroll
                    for (int st = 0; st < A; ++st) u[st] = v[st];
                    lf_sadct_inv(u, sh, 3);
#pragma unroll
                    for (int st = 0; st < A; ++st) v[st] = u[st];
                } else lf_dct4_inv<3>(v);
#pragma unroll
                for (int st = 0; st < A; ++st) Z[off + st * PS] = v[st];
            }
            __syncthreads();
        }
        lf_t2d_k<0>(Z, npl, g, false);
        // ---- stage the filtered patches (zbuf layout of k_groups) and, on rank 0, the weight ----
        if (rank == 0 && tid == 0) g.wbuf[(size_t) r * g.C + c] = wgt;
        for (int pl = 0; pl < npl; ++pl) {
            const int slot = pl / A, st = pl - slot * A;
            zdst[(((slot * CL + rank) * A + st) * g.C + c) * k2] = Z[pl * PS + poff];
        }
        __syncthreads();
    }
    cluster.sync();            // no CTA exits while a peer may still read its partial sums
}

// ---- packed FP32x2 versions of the 3x3 angular DCT: two independent signals per register pair ----
typedef unsigned long long lf_f2;

__device__ __forceinline__ lf_f2 lf_dup(float c) { return lf_pk(c, c); }

__device__ __forceinline__ void w8_dct4_fwd(lf_f2 (&v)[9], lf_f2 nz2)
{
    const float *T = c_tab.dctaf[2];
    lf_f2 y[9];
#pragma unroll
    for (int s = 0; s < 3; ++s)
#pragma unroll
        for (int kk = 0; kk < 3; ++kk) {
            lf_f2 acc = 0ull;
#pragma unroll
            for (int t = 0; t < 3; ++t) acc = lf_fma2(v[s * 3 + t], lf_dup(T[kk * 3 + t]), acc);
            y[s * 3 + kk] = acc;
        }
#pragma unroll
    for (int t = 0; t < 3; ++t)
#pragma unroll
        for (int kk = 0; kk < 3; ++kk) {
            lf_f2 acc = 0ull;
#pragma unroll
            for (int s = 0; s < 3; ++s) acc = lf_fma2(y[s * 3 + t], lf_dup(T[kk * 3 + s]), acc);
            v[kk * 3 + t] = lf_mul2(acc, lf_dup(c_tab.cn4[kk * 3 + t]), nz2);
        }
}
__device__ __forceinline__ void w8_dct4_inv(lf_f2 (&v)[9], lf_f2 nz2)
{
    const float *T = c_tab.dctai[2];
    lf_f2 a[9], y[9];
#pragma unroll
    for (int st = 0; st < 9; ++st) a[st] = lf_mul2(v[st], lf_dup(c_tab.cni4[st]), nz2);
#pragma unroll
    for (int s = 0; s < 3; ++s)
#pragma unroll
        for (int kk = 0; kk < 3; ++kk) {
            lf_f2 acc = 0ull;
#pragma unroll
            for (int t = 0; t < 3; ++t) acc = lf_fma2(a[s * 3 + t], lf_dup(T[kk * 3 + t]), acc);
            y[s * 3 + kk] = acc;
        }
#pragma unroll
    for (int t = 0; t < 3; ++t)
#pragma unroll
        for (int kk = 0; kk < 3; ++kk) {
            lf_f2 acc = 0ull;
#pragma unroll
            for (int s = 0; s < 3; ++s) acc = lf_fma2(y[s * 3 + t], lf_dup(T[kk * 3 + s]), acc);
            v[kk * 3 + t] = lf_mul2(acc, lf_dup(c_tab.coef4inv), nz2);
        }
}

// ------------------------------------------------------------------------------------------------------------
// Register-resident variant for tau_2D = id, k = 16, step 1 (configs 1, 3, 5 of BASELINE.json): thread <-> pixel position
// of the patch, the N x 9 samples of that position across the group live in registers through the angular DCT, the Haar
// transform along the similar patches, the hard threshold and both inverses. No shared-memory staging, all gathers of a
// thread in flight at once, one block reduction per channel for the weight. Same arithmetic as k_groups (bit-identical).
// ------------------------------------------------------------------------------------------------------------
// 3x3 angular transform of the NS vectors x[n][.]: two consecutive n per packed FP32x2 operation (SA-DCT groups: scalar path)
template <int NS>
__device__ __forceinline__ void lf_id_angular(float (&x)[NS][9], const GroupShape &sh, bool use_sadct, bool fwd, lf_f2 nz2)
{
    if (use_sadct) {
#pragma unroll
        for (int n = 0; n < NS; ++n) {
            float u[9];
#pragma unroll
            for (int st = 0; st < 9; ++st) u[st] = x[n][st];
            if (fwd) lf_sadct_fwd(u, sh, 3); else lf_sadct_inv(u, sh, 3);
#pragma unroll
            for (int st = 0; st < 9; ++st) x[n][st] = u[st];
        }
        return;
    }
    if (NS == 1) { if (fwd) lf_dct4_fwd<3>(x[0]); else lf_dct4_inv<3>(x[0]); return; }
#pragma unroll
    for (int h = 0; h < NS / 2; ++h) {
        lf_f2 v[9];
#pragma unroll
        for (int st = 0; st < 9; ++st) v[st] = lf_pk(x[2 * h][st], x[2 * h + 1][st]);
        if (fwd) w8_dct4_fwd(v, nz2); else w8_dct4_inv(v, nz2);
#pragma unroll
        for (int st = 0; st < 9; ++st) lf_upk(v[st], x[2 * h][st], x[2 * h + 1][st]);
    }
}

template <int NS, int CC>
__device__ __forceinline__ float lf_group_id_channel(const GroupArgs &g, const unsigned *sofs, const GroupShape &sh, bool use_sadct,
                                                     unsigned tofs, int c, int lg, float *zdst, lf_f2 nz2)
{
    constexpr int A = 9, k2 = 256;
    const int C = CC ? CC : g.C;
    float x[NS][A];
    {   // masked / out-of-row patches point at the zero block behind the window buffers: no predicates in the gather
        const uint4 *s4 = reinterpret_cast<const uint4 *>(sofs);
#pragma unroll
        for (int q4 = 0; q4 < (NS * A + 3) / 4; ++q4) {
            const uint4 o = s4[q4];
            const unsigned ov[4] = {o.x, o.y, o.z, o.w};
#pragma unroll
            for (int e = 0; e < 4; ++e) {
                const int pa = q4 * 4 + e;
                if (pa < NS * A) x[pa / A][pa % A] = __ldg(g.nsym + (ov[e] + tofs));
            }
        }
    }
    if (g.tau_4D != 4) lf_id_angular<NS>(x, sh, use_sadct, true, nz2);
    float wpart = 0.f;
    const bool haar = g.tau_5D == 9;
    const float T = haar ? c_tab.thr[c][0] : c_tab.thr[c][lg];
#pragma unroll
    for (int st = 0; st < A; ++st) {
        float v[NS];
#pragma unroll
        for (int n = 0; n < NS; ++n) v[n] = x[n][st];
        if (NS > 1) { if (haar) lf_haar_fwd<NS>(v); else lf_hadamard<NS>(v); }
        if (!use_sadct || sh.mask_dct[st]) {
#pragma unroll
            for (int n = 0; n < NS; ++n) { if (fabsf(v[n]) > T) wpart += 1.0f; else v[n] = 0.0f; }
        }
        if (NS > 1) {
            if (haar) lf_haar_inv<NS>(v);
            else {
                lf_hadamard<NS>(v);
                const float hc = c_tab.hadcoef[lg];
#pragma unroll
                for (int n = 0; n < NS; ++n) v[n] *= hc;
            }
        }
#pragma unroll
        for (int n = 0; n < NS; ++n) x[n][st] = v[n];
    }
    if (g.tau_4D != 4) lf_id_angular<NS>(x, sh, use_sadct, false, nz2);
    float *zc = zdst + c * k2;
#pragma unroll
    for (int n = 0; n < NS; ++n)
#pragma unroll
        for (int st = 0; st < A; ++st) zc[(n * A + st) * C * k2] = x[n][st];
    return wpart;
}

template <int CC>
__global__ void __launch_bounds__(256) k_groups_id16(GroupArgs g, unsigned long long nz2)
{
    __shared__ GroupShape sh;
    __shared__ float red[8];
    __shared__ __align__(16) unsigned sofs[8 * 9];
    constexpr int A = 9, k = 16, k2 = 256;
    const int tid = threadIdx.x;
    const int r = blockIdx.x + g.r0;
    const int w = g.w;
    const unsigned plane = (unsigned) g.w * (unsigned) g.h;
    const int nSx = (int) g.bm_count[r];
    const int lg = 31 - __clz(nSx);
    const int pq = tid, p = pq >> 4, q = pq & 15;
    if (!lf_group_setup<true>(g, r, nSx, sh, sofs, nullptr)) return;
    const bool use_sadct = sh.use_sadct != 0 && g.tau_4D == 6;
    float *zdst = g.zbuf + (size_t) r * g.N * A * g.C * k2 + pq;
    for (int c = 0; c < g.C; ++c) {
        const unsigned tofs = (unsigned) c * plane + (unsigned) (p * w + q);
        float wpart;
        switch (nSx) {
            case 1:  wpart = lf_group_id_channel<1, CC>(g, sofs, sh, use_sadct, tofs, c, lg, zdst, nz2); break;
            case 2:  wpart = lf_group_id_channel<2, CC>(g, sofs, sh, use_sadct, tofs, c, lg, zdst, nz2); break;
            case 4:  wpart = lf_group_id_channel<4, CC>(g, sofs, sh, use_sadct, tofs, c, lg, zdst, nz2); break;
            default: wpart = lf_group_id_channel<8, CC>(g, sofs, sh, use_sadct, tofs, c, lg, zdst, nz2); break;
        }
        const float wsum = lf_block_sum_f(wpart, red);
        const float sg = c_tab.sigma[c];
        if (tid == 0) g.wbuf[(size_t) r * g.C + c] = wsum > 0.0f ? (sg > 0.0f ? 1.0f / (c_tab.sigma2[c] * wsum) : 1.0f / wsum) : 1.0f;
    }
}

// ------------------------------------------------------------------------------------------------------------
// Weighted aggregation (core:496-526 / :1297-1327), deterministic and in the reference's order. One CTA per
// 16x16 pixel tile of one SAI: every thread owns one pixel (all channels) and adds, in (reference patch, n) order —
// the order the reference's serial loops produce for any given pixel — the contributions of every staged patch
// that covers it: num += (kaiser*w)*z, den += kaiser*w. No atomics: results do not depend on scheduling, and
// the accumulators are bit-identical to the reference's.
// ------------------------------------------------------------------------------------------------------------
struct AggArgs {
    int C, A, k, N, log2N, w, h, nc;
    int R;
    const unsigned *ent;           // [A][R*N] (y << 16 | x) of the patches to add, LF_NOENT for the others (lf_group_setup)
    const float *zbuf, *wbuf;
    float *numsym, *densym;
    const int *arange, *brange;    // per tile row / tile column: first and last candidate reference row / column index
    int y_lo, y_hi;                // pixel rows of this launch; reference rows a_min..a_max only (row bands of the multi-GPU path)
    int a_min, a_max, ty0;         // ty0: first tile row of the grid
    LfWindow win;
};
#define AGG_CAP_K8 1024     // list capacity for k = 8 (more, smaller patches per tile: one flush per tile) ...
#define AGG_CAP_K16 768     // ... and otherwise (measured: 768 is faster for k = 16, 1024 for k = 8)

// K, CC: compile-time patch size / channel count (0 = take them from the arguments); BAND: the launch covers the pixel rows
// [y_lo, y_hi) and the reference rows a_min .. a_max only (team path) — kept out of the whole-plane variant, which sits exactly
// at its register budget
template <int K, int CC, bool BAND>
__global__ void __launch_bounds__(256, 4) k_aggregate(AggArgs g)
{
    constexpr int AGG_CAP = K == 8 ? AGG_CAP_K8 : AGG_CAP_K16;
    __shared__ uint2 lpos[AGG_CAP];                  // (y << 16 | x) of the patch, index of its first channel in zbuf (units of k^2)
    __shared__ float4 lw[AGG_CAP];                   // per-channel weights of its group
    __shared__ unsigned short wlist[8][AGG_CAP];     // per warp: the listed patches that touch the warp's 8x4 pixels, in list order
    __shared__ float skaiser[LF_MAXK * LF_MAXK];
    __shared__ int wcount[2][8];
    const int st = blockIdx.z;
    if (!g.win.mask[st] || g.win.proc[st]) return;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int k = K ? K : g.k, k2 = k * k, A = g.A, C = CC ? CC : g.C, N = g.N;
    const int tyb = BAND ? blockIdx.y + g.ty0 : blockIdx.y;
    const int y0 = tyb * 16, x0 = blockIdx.x * 16;
    // a warp owns an 8 (x) by 4 (y) block of the tile: the squarer the footprint, the fewer patches touch it and the more
    // of its lanes each of them covers
    const int wy0 = y0 + (warp >> 1) * 4, wx0 = x0 + (warp & 1) * 8;
    const int y = wy0 + (lane >> 3), x = wx0 + (lane & 7);
    const bool inimg = BAND ? (y < g.y_hi && y >= g.y_lo && x < g.w) : (y < g.h && x < g.w);
    const size_t plane = (size_t) g.w * g.h;
    for (int t = tid; t < k2; t += 256) skaiser[t] = c_tab.kaiser[t];
    const int a_lo = BAND ? max(g.arange[2 * tyb], g.a_min) : g.arange[2 * tyb], a_hi = BAND ? min(g.arange[2 * tyb + 1], g.a_max) : g.arange[2 * tyb + 1];
    const int b_lo = g.brange[2 * blockIdx.x], b_hi = g.brange[2 * blockIdx.x + 1];
    const int nbn = (b_hi - b_lo + 1) * N;                 // candidates per reference row: (column, n)
    float num[3] = { 0.f, 0.f, 0.f }, den[3] = { 0.f, 0.f, 0.f };
    const size_t pix = ((size_t) st * C) * plane + (size_t) y * g.w + x;
    if (inimg)
        for (int c = 0; c < C; ++c) { num[c] = g.numsym[pix + c * plane]; den[c] = g.densym[pix + c * plane]; }
    // pixels outside the image never match: their coordinates are moved out of every patch's reach
    const int ty = inimg ? y : -0x4000, tx = inimg ? x : -0x4000;
    const float *__restrict__ zb = g.zbuf;

    // add the listed patches in list order; the loads of eight consecutive entries are issued before any of them is added
    // (memory-level parallelism: about half of the lanes are covered by a given patch)
    auto flush = [&](const int total) {
        __syncthreads();                 // the list is complete
        int cnt = 0;
        for (int i0 = 0; i0 < total; i0 += 32) {
            const int i = i0 + lane;
            bool ov = false;
            if (i < total) {
                const unsigned yx = lpos[i].x;
                const int py = (int) (yx >> 16), px = (int) (yx & 0xffffu);
                ov = py < wy0 + 4 && py + k > wy0 && px < wx0 + 8 && px + k > wx0;
            }
            const unsigned m = __ballot_sync(0xffffffffu, ov);
            if (ov) wlist[warp][cnt + __popc(m & ((1u << lane) - 1u))] = (unsigned short) i;
            cnt += __popc(m);
        }
        // pad to a multiple of the batch with an entry that covers nothing (index AGG_CAP - 1 is reserved for it)
        constexpr int U = 8;
        const int cpad = (cnt + U - 1) / U * U;
        if (lane < cpad - cnt) wlist[warp][cnt + lane] = (unsigned short) (AGG_CAP - 1);
        __syncwarp();
        const unsigned short *wl = wlist[warp];
        for (int i0 = 0; i0 < cpad; i0 += U) {
            float z[U][3], kv[U];
            int idx[U];
            bool on[U];
#pragma unroll
            for (int u = 0; u < U; ++u) {
                const int i = idx[u] = wl[i0 + u];
                const uint2 e = lpos[i];
                const int dy = ty - (int) (e.x >> 16), dx = tx - (int) (e.x & 0xffffu);
                on[u] = (unsigned) dy < (unsigned) k && (unsigned) dx < (unsigned) k;
                const int pq = dy * k + dx;
                if (on[u]) {
                    if (K != 16) kv[u] = skaiser[pq];      // the Kaiser window is all ones for k = 16 (bm3d.cpp:1144-1146): 1 * w == w
                    const float *zp = zb + ((size_t) e.y * (unsigned) k2 + (unsigned) pq);
#pragma unroll
                    for (int c = 0; c < 3; ++c) z[u][c] = c < C ? __ldg(zp + c * k2) : 0.f;
                }
            }
#pragma unroll
            for (int u = 0; u < U; ++u) {
                const float4 wv = lw[idx[u]];
                if (on[u]) {
                    const float wc[3] = {wv.x, wv.y, wv.z};
#pragma unroll
                    for (int c = 0; c < 3; ++c)
                        if (c < C) {
                            const float kw = K == 16 ? wc[c] : kv[u] * wc[c];
                            num[c] += kw * z[u][c];
                            den[c] += kw;
                        }
                }
            }
        }
        __syncthreads();                 // the list can be overwritten
    };

    if (tid == 0) lpos[AGG_CAP - 1] = make_uint2(0x7fff7fffu, 0u);     // the padding entry: far away from every pixel
    if (a_hi >= a_lo && nbn > 0) {
        const unsigned *ent = g.ent + (size_t) st * g.R * N;
        int total = 0, buf = 0;            // entries listed so far (identical in every thread)
        // candidates (a, b, n) in the reference's order, flattened: f = (a - a_lo) * nbn + (b - b_lo) * N + n; the (b, n) of a
        // reference row are contiguous in ent. 256 candidates per round, whatever the row length.
        const int nf = (a_hi - a_lo + 1) * nbn;
        for (int base = 0; base < nf; base += 256) {
            if (total + 256 > AGG_CAP - 1) { flush(total); total = 0; }
            const int f = base + tid;
            bool hit = false;
            unsigned yx = 0;
            int rn = 0;
            if (f < nf) {
                const int da = f / nbn, bn = f - da * nbn;
                rn = ((a_lo + da) * g.nc + b_lo) * N + bn;       // r * N + n
                yx = __ldg(ent + rn);
                const int py = (int) (yx >> 16), px = (int) (yx & 0xffffu);       // LF_NOENT: far outside
                hit = py < y0 + 16 && py + k > y0 && px < x0 + 16 && px + k > x0;       // keep those whose patch covers the tile
            }
            const unsigned m = __ballot_sync(0xffffffffu, hit);
            if (lane == 0) wcount[buf][warp] = __popc(m);
            __syncthreads();
            int off = total;
#pragma unroll
            for (int wv = 0; wv < 8; ++wv) { const int cw = wcount[buf][wv]; if (wv < warp) off += cw; total += cw; }
            if (hit) {
                const int o = off + __popc(m & ((1u << lane) - 1u));
                const int r = rn >> g.log2N;
                lpos[o] = make_uint2(yx, (unsigned) (((size_t) rn * A + st) * C));
                float4 ew = make_float4(0.f, 0.f, 0.f, 0.f);
                ew.x = g.wbuf[(size_t) r * C];
                if (C > 1) { ew.y = g.wbuf[(size_t) r * C + 1]; ew.z = g.wbuf[(size_t) r * C + 2]; }
                lw[o] = ew;
            }
            buf ^= 1;
        }
        flush(total);
    }
    if (inimg)
        for (int c = 0; c < C; ++c) { g.numsym[pix + c * plane] = num[c]; g.densym[pix + c * plane] = den[c]; }
}
