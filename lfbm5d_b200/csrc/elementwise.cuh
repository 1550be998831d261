// Colour transform, mirror padding / cropping, running estimate, final estimate and the small reductions of the step drivers.
// Every kernel works on a range of rows: one GPU and LFBM3D pass all rows, a rank of a team (team.cuh) the rows of its band, so
// that both run the same per-pixel arithmetic.
#pragma once
#include "common.cuh"

// utilities.cpp:482-599, evaluated left to right in float (no contraction). One thread per pixel of one SAI.
__device__ __forceinline__ void lf_color_px(unsigned cs, bool fwd, float x, float y, float z, float &o0, float &o1, float &o2)
{
    if (cs == 0) {            // YUV
        if (fwd) {
            o0 = 0.299f * x + 0.587f * y + 0.114f * z;
            o1 = -0.14713f * x - 0.28886f * y + 0.436f * z;
            o2 = 0.615f * x - 0.51498f * y - 0.10001f * z;
        } else {
            o0 = x + 1.13983f * z;
            o1 = x - 0.39465f * y - 0.5806f * z;
            o2 = x + 2.03211f * y;
        }
    } else if (cs == 1) {     // YCbCr
        if (fwd) {
            o0 = 0.299f * x + 0.587f * y + 0.114f * z;
            o1 = -0.169f * x - 0.331f * y + 0.500f * z;
            o2 = 0.500f * x - 0.419f * y - 0.081f * z;
        } else {
            o0 = 1.000f * x + 0.000f * y + 1.402f * z;
            o1 = 1.000f * x - 0.344f * y - 0.714f * z;
            o2 = 1.000f * x + 1.772f * y + 0.000f * z;
        }
    } else {                  // OPP
        if (fwd) {
            o0 = 0.333f * x + 0.333f * y + 0.333f * z;
            o1 = 0.500f * x + 0.000f * y - 0.500f * z;
            o2 = 0.250f * x - 0.500f * y + 0.250f * z;
        } else {
            o0 = 1.0f * x + 1.0f * y + 0.666f * z;
            o1 = 1.0f * x + 0.0f * y - 1.333f * z;
            o2 = 1.0f * x - 1.0f * y + 0.666f * z;
        }
    }
}

// Colour transform of the rows [i_lo, i_lo + ni) of every non-masked SAI of a [nsai][3][H][W] light field, written to out (which
// may be lf itself). mode 0: inverse, 1: forward, 2: forward then inverse: what the reference leaves in LF_noisy / LF_basic after a
// step (bm5d.cpp:133, 711-714; not the identity for OPP / YUV / YCbCr).
__global__ void k_color(const float *lf, float *out, const unsigned *mask, unsigned nsai, int W, int H, unsigned cs, int mode, int i_lo, int ni)
{
    const size_t HW = (size_t) W * H, band = (size_t) ni * W, total = (size_t) nsai * band;
    for (size_t t = (size_t) blockIdx.x * blockDim.x + threadIdx.x; t < total; t += (size_t) gridDim.x * blockDim.x) {
        const unsigned st = (unsigned) (t / band);
        if (!mask[st]) continue;
        const size_t o = (size_t) st * 3 * HW + (size_t) i_lo * W + (t - (size_t) st * band);
        const float *b = lf + o;
        float o0, o1, o2;
        if (mode == 2) {
            float f0, f1, f2;
            lf_color_px(cs, true, b[0], b[HW], b[2 * HW], f0, f1, f2);
            lf_color_px(cs, false, f0, f1, f2, o0, o1, o2);
        } else lf_color_px(cs, mode != 0, b[0], b[HW], b[2 * HW], o0, o1, o2);
        float *r = out + o;
        r[0] = o0; r[HW] = o1; r[2 * HW] = o2;
    }
}

__device__ __forceinline__ int lf_mirror(int v, int n)   // utilities.cpp:215-263 (edge pixel repeated)
{
    return v < 0 ? -v - 1 : (v >= n ? 2 * n - 1 - v : v);
}

// Build the padded working set of one angular window (bm5d.cpp:254-265) on the padded rows [y_lo, y_lo + nrows), and below
// row est_hi the channel-0 running estimate block matching reads (utilities_LF.cpp:913-954 via core:169 / :937). sub = noisy
// (step 1) or basic (step 2). Outputs: nsym/bsym/numsym/densym [A][C][hb][wb], est0 [A][hb][wb]. bsym/basic may be null.
// One GPU builds all rows (est_hi = hb); a team rank builds the rows its groups touch and leaves the estimate of the rows it
// shares with the next rank to their owner.
__global__ void k_pad(const float *__restrict__ noisy, const float *__restrict__ basic, const float *__restrict__ num,
                      const float *__restrict__ den, float *__restrict__ nsym, float *__restrict__ bsym,
                      float *__restrict__ numsym, float *__restrict__ densym, float *__restrict__ est0,
                      LfWindow win, int W, int H, int C, int n, int y_lo, int nrows, int est_hi)
{
    const int wb = W + 2 * n, hb = H + 2 * n;
    const size_t plane_b = (size_t) wb * hb, plane = (size_t) W * H, band = (size_t) nrows * wb;
    const size_t total = (size_t) win.A * band;
    for (size_t t = (size_t) blockIdx.x * blockDim.x + threadIdx.x; t < total; t += (size_t) gridDim.x * blockDim.x) {
        const int a = (int) (t / band);
        if (!win.mask[a]) continue;
        const size_t rb = t - (size_t) a * band;
        const int i = y_lo + (int) (rb / wb), j = (int) (rb % wb);
        const size_t r = (size_t) i * wb + j;
        const int si = lf_mirror(i - n, H), sj = lf_mirror(j - n, W);
        const size_t src = (size_t) win.st[a] * C * plane + (size_t) si * W + sj;
        const size_t dst = (size_t) a * C * plane_b + r;
        for (int c = 0; c < C; c++) {
            const float nv = noisy[src + c * plane], uv = num[src + c * plane], dv = den[src + c * plane];
            nsym[dst + c * plane_b] = nv;
            numsym[dst + c * plane_b] = uv;
            densym[dst + c * plane_b] = dv;
            float bv = 0.f;
            if (basic) { bv = basic[src + c * plane]; bsym[dst + c * plane_b] = bv; }
            if (c == 0 && i < est_hi) est0[(size_t) a * plane_b + r] = dv ? uv / dv : (basic ? bv : nv);
        }
    }
}

// Same estimate from the window's padded buffers (after a core call, or as the debug pass uploaded them), padded rows
// [y_lo, y_lo + nrows)
__global__ void k_est0(const float *__restrict__ sub, const float *__restrict__ numsym, const float *__restrict__ densym,
                       float *__restrict__ est0, LfWindow win, int wb, int hb, int C, int y_lo, int nrows)
{
    const size_t plane_b = (size_t) wb * hb, band = (size_t) nrows * wb, total = (size_t) win.A * band;
    for (size_t t = (size_t) blockIdx.x * blockDim.x + threadIdx.x; t < total; t += (size_t) gridDim.x * blockDim.x) {
        const int a = (int) (t / band);
        if (!win.mask[a]) continue;
        const size_t r = (size_t) y_lo * wb + (t - (size_t) a * band), o = (size_t) a * C * plane_b + r;
        const float dv = densym[o];
        est0[(size_t) a * plane_b + r] = dv ? numsym[o] / dv : sub[o];
    }
}

__device__ __forceinline__ unsigned long long lf_block_sum_u64(unsigned long long v)
{
    __shared__ unsigned long long sh[32];
    for (int o = 16; o > 0; o >>= 1) v += __shfl_down_sync(0xffffffffu, v, o);
    if ((threadIdx.x & 31) == 0) sh[threadIdx.x >> 5] = v;
    __syncthreads();
    if (threadIdx.x < 32) {
        v = threadIdx.x < (blockDim.x + 31) / 32 ? sh[threadIdx.x] : 0ull;
        for (int o = 16; o > 0; o >>= 1) v += __shfl_down_sync(0xffffffffu, v, o);
    }
    return v;
}

// Crop the interior rows [i_lo, i_lo + ni) of the window's padded accumulators back into the light field (bm5d.cpp:388-396).
// With `count` it also counts the entries with den > 0 in the top-left (H-k+1) x (W-k+1) of every SAI (LF_denoised_percent,
// utilities_LF.cpp:967-995): the single-GPU step driver runs it after every core call, so the coverage test costs no extra pass
// over the accumulators.
__global__ void k_unpad(float *__restrict__ num, float *__restrict__ den, const float *__restrict__ numsym,
                        const float *__restrict__ densym, LfWindow win, int W, int H, int C, int n, int i_lo, int ni, int k,
                        unsigned long long *count)
{
    unsigned long long cnt = 0;
    const int wb = W + 2 * n, hb = H + 2 * n;
    const size_t plane_b = (size_t) wb * hb, plane = (size_t) W * H, band = (size_t) ni * W;
    const size_t total = (size_t) win.A * C * band;
    for (size_t t = (size_t) blockIdx.x * blockDim.x + threadIdx.x; t < total; t += (size_t) gridDim.x * blockDim.x) {
        const int ac = (int) (t / band), a = ac / C, c = ac - a * C;
        if (!win.mask[a]) continue;
        const size_t rb = t - (size_t) ac * band;
        const int i = i_lo + (int) (rb / W), j = (int) (rb % W);
        const size_t src = ((size_t) a * C + c) * plane_b + (size_t) (i + n) * wb + (j + n);
        const size_t dst = ((size_t) win.st[a] * C + c) * plane + (size_t) i * W + j;
        const float dv = densym[src];
        num[dst] = numsym[src];
        den[dst] = dv;
        if (count && i < H - k + 1 && j < W - k + 1 && dv > 0.0f) cnt++;
    }
    if (count) {
        cnt = lf_block_sum_u64(cnt);
        if (threadIdx.x == 0 && cnt) atomicAdd(count, cnt);
    }
}

// Number of entries equal to 0.0 on the rows [y_lo, y_lo + nrows) of nplanes planes of rowlen floats (bm5d.cpp:195 / :318-333)
__global__ void k_count_zero(const float *__restrict__ den, int nplanes, size_t plane_stride, int rowlen, int y_lo, int nrows,
                             unsigned long long *out)
{
    unsigned long long cnt = 0;
    const size_t band = (size_t) nrows * rowlen;
    for (int pl = 0; pl < nplanes; pl++) {      // the rows of one plane are contiguous: no index division in the loop
        const float *d = den + (size_t) pl * plane_stride + (size_t) y_lo * rowlen;
        for (size_t t = (size_t) blockIdx.x * blockDim.x + threadIdx.x; t < band; t += (size_t) gridDim.x * blockDim.x)
            if (d[t] == 0.0f) cnt++;
    }
    cnt = lf_block_sum_u64(cnt);
    if (threadIdx.x == 0 && cnt) atomicAdd(out, cnt);
}

// Final estimate (bm5d.cpp:405 / :706) fused with the inverse colour transforms of the outputs (bm5d.cpp:711-714, 1414-1419) on
// the rows [i_lo, i_lo + ni) of every non-masked SAI: out = den ? num/den : sub, then out and, with inputs_back, noisy (and basic)
// go back to RGB. inputs_back = 0: noisy / basic stay in the working colour space (the host entry points returned their
// round-tripped copies early). For C == 1 or the RGB colour space `docolor` is 0.
__global__ void k_final(const float *__restrict__ num, const float *__restrict__ den, float *noisy, float *basic, float *out,
                        const unsigned *mask, unsigned nsai, int W, int H, int C, int step, unsigned cs, int docolor, int inputs_back,
                        int i_lo, int ni)
{
    const size_t HW = (size_t) W * H, band = (size_t) ni * W, total = (size_t) nsai * band;
    for (size_t t = (size_t) blockIdx.x * blockDim.x + threadIdx.x; t < total; t += (size_t) gridDim.x * blockDim.x) {
        const unsigned st = (unsigned) (t / band);
        if (!mask[st]) continue;
        const size_t base = (size_t) st * C * HW + (size_t) i_lo * W + (t - (size_t) st * band);
        float e[3], nz[3], bs[3];
        for (int c = 0; c < C; c++) {
            const float nv = noisy[base + c * HW], dv = den[base + c * HW];
            nz[c] = nv;
            bs[c] = step == 2 ? basic[base + c * HW] : 0.f;
            e[c] = dv ? num[base + c * HW] / dv : (step == 2 ? bs[c] : nv);
        }
        if (docolor) {
            float a, b, c2;
            lf_color_px(cs, false, e[0], e[1], e[2], a, b, c2); e[0] = a; e[1] = b; e[2] = c2;
            if (inputs_back) {
                lf_color_px(cs, false, nz[0], nz[1], nz[2], a, b, c2); nz[0] = a; nz[1] = b; nz[2] = c2;
                if (step == 2) { lf_color_px(cs, false, bs[0], bs[1], bs[2], a, b, c2); bs[0] = a; bs[1] = b; bs[2] = c2; }
            }
        }
        for (int c = 0; c < C; c++) {
            out[base + c * HW] = e[c];
            if (docolor && inputs_back) {
                noisy[base + c * HW] = nz[c];
                if (step == 2) basic[base + c * HW] = bs[c];
            }
        }
    }
}
