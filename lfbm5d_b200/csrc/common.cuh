// Common definitions of the LFBM5D CUDA path (sm_100a). Compiled with -fmad=false: every a*b+c in this
// translation unit is a separate multiply and add, like the reference's x86-64 build; fused multiply-adds
// appear only where written explicitly (fmaf in the DCT passes, matching oracle DCT mode 0).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#define LF_MAXK      16      // largest patch side handled by the transform kernels
#define LF_MAXASW    5       // angular window side (2*an+1), an <= 2
#define LF_MAXA      (LF_MAXASW * LF_MAXASW)
// windows up to 3x3 (an <= 1): SA-DCT shapes from a host table of 2^A entries, 16-bit group masks, and the group kernels
// k_groups / k_groups_id16 / k_groups_w8 with their shared arrays sized for 9 SAIs; 5x5 windows take k_groups25
#define LF_LUTASW    3
#define LF_LUTA      (LF_LUTASW * LF_LUTASW)
#define LF_MAXN      32      // largest number of similar patches
#define LF_MAXDISP   16      // largest disparity half window nDisp: (2*nDisp+1)^2 <= 1089 disparity offsets
#define LF_SQRT2_INV_F ((float) 0.7071067811865475)
#define LF_SQRT2_F     ((float) 1.414213562373095)

// Per-step constants. Filled on the host with the reference's expressions (bm3d.cpp:1101-1169 preProcess,
// core:3191-3252 preProcess_4d / preProcess_4d_sadct, utilities.cpp:633-684 estimate_sigma) and the FFTW
// REDFT10/REDFT01 cosine tables (oracle DCT mode 0), then copied to constant memory.
struct LfTables {
    float dct2f[LF_MAXK * LF_MAXK];      // [kk*k + j] = (float)(2 cos(pi (j+1/2) kk / k))
    float dct2i[LF_MAXK * LF_MAXK];      // [kk*k + j] = j ? (float)(2 cos(pi j (kk+1/2) / k)) : 1
    float cn2[LF_MAXK * LF_MAXK], cni2[LF_MAXK * LF_MAXK], kaiser[LF_MAXK * LF_MAXK];
    float coef2inv;                      // 1 / (2k)
    float dctaf[LF_LUTASW][LF_LUTASW * LF_LUTASW];   // [n-1][kk*n + j], 1-D tables for lengths 1..asw (windows up to 3x3)
    float dctai[LF_LUTASW][LF_LUTASW * LF_LUTASW];
    float cn4[LF_LUTA], cni4[LF_LUTA];
    float coef4inv;                      // 1 / (sqrt(aw) sqrt(ah) 2)
    float cnsa[LF_LUTASW][LF_LUTASW], cnisa[LF_LUTASW][LF_LUTASW];   // [n-2][t]
    float coefsa_inv[LF_LUTASW + 1];     // [n] = 0.5 (float)SQRT2_INV / sqrt(n)
    float lpd[10], hpd[10], lpr[10], hpr[10];
    float sigma[3], sigma2[3];
    float thr[3][8];                     // hard threshold per channel and log2(nSx)
    float hadcoef[8];                    // 1 / nSx
    // 5-D DCT along the similar patches (core:2524-2700, :2943-3130): REDFT10 / REDFT01 tables of length 2^lg packed one after
    // the other (offset (4^lg - 1) / 3), preProcess_5d normalisers (core:3262-3276) and the hard threshold lambda sigma 2 sqrt2
    float dct5f[1365], dct5i[1365];
    float cn5_0[6], cn5_c[6], coef5inv[6];
    float thr_dct[3];
    // the angular tables above for 5x5 windows (lengths 1..5, k_groups25). Kept apart: the 3x3 group kernels read theirs at
    // the offsets and strides they were tuned with (a 5x5 layout of the same arrays costs k_groups_id16 16 registers).
    float dctaf5[LF_MAXASW][LF_MAXASW * LF_MAXASW], dctai5[LF_MAXASW][LF_MAXASW * LF_MAXASW];
    float cn4_5[LF_MAXA], cni4_5[LF_MAXA];
    float cnsa5[LF_MAXASW][LF_MAXASW], cnisa5[LF_MAXASW][LF_MAXASW];
    float coefsa_inv5[LF_MAXASW + 1];
};

__constant__ LfTables c_tab;

// Multi-GPU team path: where the sampled self sums of every offset plane live (rank q holds the planes pl0[q] .. pl0[q+1]-1 in ITS
// s_at / s_mir, reached through peer pointers: NVLink loads), for the reference patches whose selection needs the complete candidate
// sequence (exact distance ties).
#define LF_MAXRANKS 16
struct PeerTable {
    const float *s_at[LF_MAXRANKS];
    const float *s_mir[LF_MAXRANKS];
    int pl0[LF_MAXRANKS + 1];
    int G;                        // 0: no table, everything is local
};
__device__ __forceinline__ float lf_peer_sum(const PeerTable &pt, bool mir, const float *local, int ddk, size_t R, int r)
{
    if (pt.G == 0) return local[(size_t) ddk * R + r];
    int q = 0;
    while (q + 1 < pt.G && ddk >= pt.pl0[q + 1]) ++q;
    return (mir ? pt.s_mir[q] : pt.s_at[q])[(size_t) ddk * R + r];
}

struct LfWindow {
    int      st[LF_MAXA];        // global SAI index of each window slot
    unsigned mask[LF_MAXA];
    unsigned proc[LF_MAXA];
    int      A;
};
// The window as the group kernels of windows up to 3x3 receive it: their parameter block keeps its 3x3 size (a larger one
// costs k_groups_id16 16 registers)
struct LfWindow9 {
    int      st[LF_LUTA];
    unsigned mask[LF_LUTA];
    unsigned proc[LF_LUTA];
    int      A;
};

__device__ __forceinline__ void lf_cp_async4(float *smem_dst, const float *gsrc)
{
    const unsigned sa = (unsigned) __cvta_generic_to_shared(smem_dst);
    asm volatile("cp.async.ca.shared.global [%0], [%1], 4;\n" ::"r"(sa), "l"(gsrc));
}
__device__ __forceinline__ void lf_cp_async_wait_all()
{
    asm volatile("cp.async.commit_group;\n cp.async.wait_group 0;\n" ::: "memory");
}


// ---- packed FP32x2 arithmetic (two independent IEEE operations per instruction; sm_100 FADD2 / FFMA2) ----
__device__ __forceinline__ unsigned long long lf_pk(float lo, float hi)
{
    unsigned long long r;
    asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(lo), "f"(hi));
    return r;
}
__device__ __forceinline__ void lf_upk(unsigned long long v, float &lo, float &hi)
{
    asm("mov.b64 {%0, %1}, %2;" : "=f"(lo), "=f"(hi) : "l"(v));
}
__device__ __forceinline__ unsigned long long lf_add2(unsigned long long a, unsigned long long b)
{
    unsigned long long r;
    asm("add.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b));
    return r;
}
__device__ __forceinline__ unsigned long long lf_sub2(unsigned long long a, unsigned long long b)
{
    unsigned long long r;
    asm("sub.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b));
    return r;
}
// Exact packed product. ptxas contracts mul.rn.f32x2 + add.rn.f32x2 into FFMA2 (observed, CUDA 12.9) even with
// -fmad=false — also when the product is written as fma(a, b, -0) with a literal -0 — which would change the rounding of
// the recurrence. With the -0 addend supplied at run time (SatGeom::negzero2) ptxas cannot fold it: fma(a, b, -0) is the
// exact product (round(a*b + -0) = round(a*b), +0 for a zero product) and stays separate from the following add.
__device__ __forceinline__ unsigned long long lf_mul2(unsigned long long a, unsigned long long b, unsigned long long negzero)
{
    unsigned long long r;
    asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(r) : "l"(a), "l"(b), "l"(negzero));
    return r;
}
__device__ __forceinline__ unsigned long long lf_fma2(unsigned long long a, unsigned long long b, unsigned long long c)
{
    unsigned long long r;
    asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(r) : "l"(a), "l"(b), "l"(c));
    return r;
}

// 64-bit (value, tag) words handed from CTA to CTA through L2: a naturally aligned 64-bit access is single-copy atomic, so a
// consumer that finds the tag it expects also has the value that was written with it — no flag, no fence
__device__ __forceinline__ void lf_st_relaxed64(unsigned long long *p, unsigned long long v)
{
    asm volatile("st.relaxed.gpu.global.b64 [%0], %1;\n" ::"l"(p), "l"(v) : "memory");
}
__device__ __forceinline__ unsigned long long lf_ld_relaxed64(const unsigned long long *p)
{
    unsigned long long v;
    asm volatile("ld.relaxed.gpu.global.b64 %0, [%1];\n" : "=l"(v) : "l"(p) : "memory");
    return v;
}

// release/acquire flag accesses at GPU scope (producer/consumer hand-off between CTAs)
__device__ __forceinline__ void lf_st_release(int *p, int v)
{
    asm volatile("st.release.gpu.global.s32 [%0], %1;\n" ::"l"(p), "r"(v) : "memory");
}
// polling load: strong at GPU scope (served by L2) but without the L1 invalidation an acquire load carries (CCTL.IVALL on sm_100);
// spin on this one, then read the flag once more with lf_ld_acquire before touching the data it guards
__device__ __forceinline__ int lf_ld_relaxed(const int *p)
{
    int v;
    asm volatile("ld.relaxed.gpu.global.s32 %0, [%1];\n" : "=r"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ int lf_ld_acquire(const int *p)
{
    int v;
    asm volatile("ld.acquire.gpu.global.s32 %0, [%1];\n" : "=r"(v) : "l"(p) : "memory");
    return v;
}
