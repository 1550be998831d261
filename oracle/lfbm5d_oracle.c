/* TEST INFRASTRUCTURE ONLY — see lfbm5d_oracle.h for scope, pinning status and who may call this.
 *
 * CPU restatement of the LFBM5D hot path (reference: V-Sense/LFBM5D, files cited per function as
 * file:line into /root/reference/src). Written from the algorithm's description, not copied: the
 * data flow is restructured (no per-row 2-D tables, no full summed-area planes kept, matches found
 * by argmin unless a tie forces the libstdc++ sort to be emulated) but every floating-point
 * operation that reaches an output is performed with the reference's operands, precision and order,
 * so results are bit-identical to the reference built with oracle/Makefile (-O2, no FMA contraction).
 */
#include "lfbm5d_oracle.h"
#include <math.h>
#include <stdlib.h>
#include <string.h>
#include <stdio.h>
#ifdef _OPENMP
#include <omp.h>
#endif

#define SQRT2_D     1.414213562373095
#define SQRT2_INV_D 0.7071067811865475

static int g_dct_mode = 0;
static int g_use_sd = 0;    /* useSD of the next orc_pass / orc_run_* calls (test infrastructure; see orc_set_use_sd) */
static int g_sum_mode = 0;  /* 1: group weight sums in double (test infrastructure; see orc_set_sum_mode) */
static int g_bm3d = 0;      /* set while orc_run_bm3d_LF drives orc_pass: BM3D thresholds (bm3d.cpp:340, :532, :940) */
static int g_threads = 0;
void orc_set_dct_mode(int mode) { g_dct_mode = mode; }
void orc_set_sum_mode(int mode) { g_sum_mode = mode; }
void orc_set_threads(int n) { g_threads = n; }
static int nthreads(void)
{
#ifdef _OPENMP
    return g_threads > 0 ? g_threads : omp_get_max_threads();
#else
    return 1;
#endif
}

/* ------------------------------------------------------------------------------------------ */
/* small utilities                                                                             */
/* ------------------------------------------------------------------------------------------ */

/* utilities.cpp:697-712 */
unsigned orc_ind_initialize(unsigned *out, unsigned max_size, unsigned N, unsigned step)
{
    unsigned cnt = 0, ind = N;
    while (ind < max_size - N) { out[cnt++] = ind; ind += step; }
    if (cnt == 0 || out[cnt - 1] < max_size - N - 1) out[cnt++] = max_size - N - 1;
    return cnt;
}

/* utilities.cpp:608-616 */
static unsigned closest_power_of_2(unsigned n)
{
    unsigned r = 1;
    while (r * 2 <= n) r *= 2;
    return r;
}

/* utilities.cpp:482-599; expressions evaluated left to right in float */
int orc_color_space_transform(float *img, unsigned cs, unsigned width, unsigned height, unsigned chnls, int fwd)
{
    if (chnls == 1 || cs == ORC_RGB) return 0;
    if (cs != ORC_YUV && cs != ORC_YCBCR && cs != ORC_OPP) return 1;
    const size_t n = (size_t) width * height;
    float *r = img, *g = img + n, *b = img + 2 * n;
    for (size_t k = 0; k < n; k++) {
        const float x = r[k], y = g[k], z = b[k];
        float o0, o1, o2;
        if (cs == ORC_YUV) {
            if (fwd) {
                o0 = 0.299f * x + 0.587f * y + 0.114f * z;
                o1 = -0.14713f * x - 0.28886f * y + 0.436f * z;
                o2 = 0.615f * x - 0.51498f * y - 0.10001f * z;
            } else {
                o0 = x + 1.13983f * z;
                o1 = x - 0.39465f * y - 0.5806f * z;
                o2 = x + 2.03211f * y;
            }
        } else if (cs == ORC_YCBCR) {
            if (fwd) {
                o0 = 0.299f * x + 0.587f * y + 0.114f * z;
                o1 = -0.169f * x - 0.331f * y + 0.500f * z;
                o2 = 0.500f * x - 0.419f * y - 0.081f * z;
            } else {
                o0 = 1.000f * x + 0.000f * y + 1.402f * z;
                o1 = 1.000f * x - 0.344f * y - 0.714f * z;
                o2 = 1.000f * x + 1.772f * y + 0.000f * z;
            }
        } else {
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
        r[k] = o0; g[k] = o1; b[k] = o2;
    }
    return 0;
}

/* utilities.cpp:633-684 */
int orc_estimate_sigma(float sigma, float *t, unsigned chnls, unsigned cs)
{
    if (chnls == 1) { t[0] = sigma; return 0; }
    if (cs == ORC_YUV) {
        t[0] = sqrtf(0.299f * 0.299f + 0.587f * 0.587f + 0.114f * 0.114f) * sigma;
        t[1] = sqrtf(0.14713f * 0.14713f + 0.28886f * 0.28886f + 0.436f * 0.436f) * sigma;
        t[2] = sqrtf(0.615f * 0.615f + 0.51498f * 0.51498f + 0.10001f * 0.10001f) * sigma;
    } else if (cs == ORC_YCBCR) {
        t[0] = sqrtf(0.299f * 0.299f + 0.587f * 0.587f + 0.114f * 0.114f) * sigma;
        t[1] = sqrtf(0.169f * 0.169f + 0.331f * 0.331f + 0.500f * 0.500f) * sigma;
        t[2] = sqrtf(0.500f * 0.500f + 0.419f * 0.419f + 0.081f * 0.081f) * sigma;
    } else if (cs == ORC_OPP) {
        t[0] = sqrtf(0.333f * 0.333f + 0.333f * 0.333f + 0.333f * 0.333f) * sigma;
        t[1] = sqrtf(0.5f * 0.5f + 0.0f * 0.0f + 0.5f * 0.5f) * sigma;
        t[2] = sqrtf(0.25f * 0.25f + 0.5f * 0.5f + 0.25f * 0.25f) * sigma;
    } else if (cs == ORC_RGB) {
        t[0] = t[1] = t[2] = sigma;
    } else return 1;
    return 0;
}

/* utilities.cpp:215-263: mirror padding with the edge pixel repeated */
void orc_symetrize(const float *img, float *out, unsigned width, unsigned height, unsigned chnls, unsigned N)
{
    const unsigned w = width + 2 * N, h = height + 2 * N;
    for (unsigned c = 0; c < chnls; c++) {
        const float *src = img + (size_t) c * width * height;
        float *dst = out + (size_t) c * w * h;
        for (unsigned i = 0; i < h; i++) {
            int si = (int) i - (int) N;
            if (si < 0) si = -si - 1; else if (si >= (int) height) si = 2 * (int) height - 1 - si;
            for (unsigned j = 0; j < w; j++) {
                int sj = (int) j - (int) N;
                if (sj < 0) sj = -sj - 1; else if (sj >= (int) width) sj = 2 * (int) width - 1 - sj;
                dst[(size_t) i * w + j] = src[(size_t) si * width + sj];
            }
        }
    }
}

/* utilities.cpp:275-298 */
void orc_unsymetrize(float *img, const float *sym, unsigned width, unsigned height, unsigned chnls, unsigned N)
{
    const unsigned w = width + 2 * N, h = height + 2 * N;
    for (unsigned c = 0; c < chnls; c++)
        for (unsigned i = 0; i < height; i++)
            memcpy(img + (size_t) c * width * height + (size_t) i * width,
                   sym + (size_t) c * w * h + (size_t) (i + N) * w + N, width * sizeof(float));
}

/* utilities_LF.cpp:881-901 */
void orc_angular_search_window(int *c_asw, int *min_asw, int *max_asw, unsigned aidx, unsigned asize, unsigned asize_sw)
{
    int mn = (int) aidx - (int) asize_sw, mx = (int) aidx + (int) asize_sw;
    int shift = mn < 0 ? -mn : 0;
    mn += shift; mx += shift;
    int c = (int) asize_sw - shift;
    shift = mx >= (int) asize ? ((int) asize - mx - 1) : 0;
    mn += shift; mx += shift; c -= shift;
    *c_asw = c; *min_asw = mn; *max_asw = mx;
}

/* utilities_LF.cpp:967-995: counts every channel but normalises by pixels */
float orc_LF_denoised_percent(const float *den_sym, const unsigned *mask, unsigned A, unsigned width, unsigned height,
                              unsigned chnls, unsigned N, unsigned kHW)
{
    const unsigned w_b = width + 2 * N, h_b = height + 2 * N;
    float cnt = 0.0f;
    unsigned nmask = 0;
    for (unsigned st = 0; st < A; st++) {
        if (!mask[st]) continue;
        nmask++;
        const float *d = den_sym + (size_t) st * chnls * w_b * h_b;
        for (unsigned i = 0; i < height - kHW + 1; i++)
            for (unsigned j = 0; j < width - kHW + 1; j++)
                for (unsigned c = 0; c < chnls; c++)
                    if (d[(size_t) c * w_b * h_b + (size_t) (i + N) * w_b + N + j] > 0.0) cnt++;
    }
    return cnt * 100.0f / (float) nmask / (float) (height - kHW + 1) / (float) (width - kHW + 1);
}

/* ------------------------------------------------------------------------------------------ */
/* libstdc++ (GCC 13, bits/stl_algo.h + bits/stl_heap.h) sort algorithms on (d, idx) pairs,     */
/* comparator = d_a < d_b. Needed because the reference's tie behaviour is that of these        */
/* algorithms (core:3435 partial_sort, core:3600 sort; comparator bm3d.cpp:1377).               */
/* ------------------------------------------------------------------------------------------ */
typedef struct { float d; unsigned i; } pr_t;
#define LESS(a, b) ((a).d < (b).d)

static void push_heap_(pr_t *first, long hole, long top, pr_t value)
{
    long parent = (hole - 1) / 2;
    while (hole > top && LESS(first[parent], value)) {
        first[hole] = first[parent];
        hole = parent;
        parent = (hole - 1) / 2;
    }
    first[hole] = value;
}
static void adjust_heap_(pr_t *first, long hole, long len, pr_t value)
{
    const long top = hole;
    long child = hole;
    while (child < (len - 1) / 2) {
        child = 2 * (child + 1);
        if (LESS(first[child], first[child - 1])) child--;
        first[hole] = first[child];
        hole = child;
    }
    if ((len & 1) == 0 && child == (len - 2) / 2) {
        child = 2 * (child + 1);
        first[hole] = first[child - 1];
        hole = child - 1;
    }
    push_heap_(first, hole, top, value);
}
static void make_heap_(pr_t *first, long len)
{
    if (len < 2) return;
    long parent = (len - 2) / 2;
    for (;;) {
        pr_t v = first[parent];
        adjust_heap_(first, parent, len, v);
        if (parent == 0) return;
        parent--;
    }
}
static void pop_heap_(pr_t *first, pr_t *last, pr_t *result)
{
    pr_t v = *result;
    *result = *first;
    adjust_heap_(first, 0, last - first, v);
}
static void partial_sort_(pr_t *first, pr_t *middle, pr_t *last)
{
    make_heap_(first, middle - first);
    for (pr_t *i = middle; i < last; ++i)
        if (LESS(*i, *first)) pop_heap_(first, middle, i);
    while (middle - first > 1) { --middle; pop_heap_(first, middle, middle); }
}
static void swap_(pr_t *a, pr_t *b) { pr_t t = *a; *a = *b; *b = t; }
static void move_median_to_first_(pr_t *result, pr_t *a, pr_t *b, pr_t *c)
{
    if (LESS(*a, *b)) {
        if (LESS(*b, *c)) swap_(result, b);
        else if (LESS(*a, *c)) swap_(result, c);
        else swap_(result, a);
    } else if (LESS(*a, *c)) swap_(result, a);
    else if (LESS(*b, *c)) swap_(result, c);
    else swap_(result, b);
}
static pr_t *unguarded_partition_(pr_t *first, pr_t *last, pr_t *pivot)
{
    for (;;) {
        while (LESS(*first, *pivot)) ++first;
        --last;
        while (LESS(*pivot, *last)) --last;
        if (!(first < last)) return first;
        swap_(first, last);
        ++first;
    }
}
static void introsort_loop_(pr_t *first, pr_t *last, long depth)
{
    while (last - first > 16) {
        if (depth == 0) { partial_sort_(first, last, last); return; }
        --depth;
        pr_t *mid = first + (last - first) / 2;
        move_median_to_first_(first, first + 1, mid, last - 1);
        pr_t *cut = unguarded_partition_(first + 1, last, first);
        introsort_loop_(cut, last, depth);
        last = cut;
    }
}
static void unguarded_linear_insert_(pr_t *last)
{
    pr_t v = *last;
    pr_t *next = last - 1;
    while (LESS(v, *next)) { *last = *next; last = next; --next; }
    *last = v;
}
static void insertion_sort_(pr_t *first, pr_t *last)
{
    if (first == last) return;
    for (pr_t *i = first + 1; i != last; ++i) {
        if (LESS(*i, *first)) {
            pr_t v = *i;
            memmove(first + 1, first, (size_t) (i - first) * sizeof(pr_t));
            *first = v;
        } else unguarded_linear_insert_(i);
    }
}
static void std_sort_(pr_t *first, pr_t *last)
{
    if (first == last) return;
    long n = last - first, lg = 0;
    while ((n >> (lg + 1)) > 0) lg++;
    introsort_loop_(first, last, lg * 2);
    if (last - first > 16) {
        insertion_sort_(first, first + 16);
        for (pr_t *i = first + 16; i != last; ++i) unguarded_linear_insert_(i);
    } else insertion_sort_(first, last);
}

void orc_std_partial_sort(float *d, unsigned *idx, unsigned n, unsigned middle)
{
    pr_t *v = (pr_t *) malloc(sizeof(pr_t) * (n ? n : 1));
    for (unsigned i = 0; i < n; i++) { v[i].d = d[i]; v[i].i = idx[i]; }
    partial_sort_(v, v + middle, v + n);
    for (unsigned i = 0; i < n; i++) { d[i] = v[i].d; idx[i] = v[i].i; }
    free(v);
}
void orc_std_sort(float *d, unsigned *idx, unsigned n)
{
    pr_t *v = (pr_t *) malloc(sizeof(pr_t) * (n ? n : 1));
    for (unsigned i = 0; i < n; i++) { v[i].d = d[i]; v[i].i = idx[i]; }
    std_sort_(v, v + n);
    for (unsigned i = 0; i < n; i++) { d[i] = v[i].d; idx[i] = v[i].i; }
    free(v);
}

/* ------------------------------------------------------------------------------------------ */
/* block matching                                                                              */
/* ------------------------------------------------------------------------------------------ */

/* One summed-area plane, exactly the recurrence and evaluation order of core:3335-3389 (self) and
 * core:3520-3573 (stereo): diff[] must already hold the squared differences inside
 * [lo, h-lo) x [lo, w-lo) and zeros elsewhere; sums are produced for rows/cols [lo, h-hi_cut) /
 * [lo, w-hi_cut) into sum[] (other entries untouched). */
static void sat_plane(const float *diff, float *sum, unsigned w, unsigned h, unsigned k, unsigned lo, unsigned row_end, unsigned col_end)
{
    const unsigned dn = lo * w + lo;
    float value = 0.0f;
    for (unsigned p = 0; p < k; p++)
        for (unsigned q = 0; q < k; q++) value += diff[dn + p * w + q];
    sum[dn] = value;
    for (unsigned j = lo + 1; j < col_end; j++) {
        const unsigned ind = lo * w + j - 1;
        float s = sum[ind];
        for (unsigned p = 0; p < k; p++) s += diff[ind + p * w + k] - diff[ind + p * w];
        sum[ind + 1] = s;
    }
    for (unsigned i = lo + 1; i < row_end; i++) {
        const unsigned ind = (i - 1) * w + lo;
        float s = sum[ind];
        for (unsigned q = 0; q < k; q++) s += diff[ind + k * w + q] - diff[ind + q];
        sum[ind + w] = s;
        unsigned kk = i * w + lo + 1;
        unsigned pq = (i + k - 1) * w + k - 1 + lo + 1;
        for (unsigned j = lo + 1; j < col_end; j++, kk++, pq++)
            sum[kk] = sum[kk - 1] + sum[kk - w] - sum[kk - 1 - w]
                    + diff[pq] - diff[pq - k] - diff[pq - k * w] + diff[pq - k - k * w];
    }
}

/* core:3301-3461 */
void orc_bm_self(const float *img, unsigned width, unsigned height, unsigned kHW, unsigned NHW, unsigned nHW,
                 unsigned nHW_sim, unsigned pHW, float tauMatch, unsigned *out_count, unsigned *out_idx, unsigned maxN)
{
    const unsigned Ns = 2 * nHW_sim + 1;
    const float threshold = tauMatch * kHW * kHW;
    const size_t plane = (size_t) width * height;
    unsigned *rows = (unsigned *) malloc(sizeof(unsigned) * (height + 2));
    unsigned *cols = (unsigned *) malloc(sizeof(unsigned) * (width + 2));
    const unsigned nr = orc_ind_initialize(rows, height - kHW + 1, nHW, pHW);
    const unsigned nc = orc_ind_initialize(cols, width - kHW + 1, nHW, pHW);
    const size_t R = (size_t) nr * nc;
    memset(out_count, 0, plane * sizeof(unsigned));

    if (NHW <= 1) {
        for (unsigned a = 0; a < nr; a++)
            for (unsigned b = 0; b < nc; b++) {
                const unsigned k_r = rows[a] * width + cols[b];
                out_count[k_r] = 1;
                out_idx[(size_t) k_r * maxN] = k_r;
            }
        free(rows); free(cols);
        return;
    }

    /* Per plane (di in [0,nSim], dj index in [0,Ns)) only two samples per reference patch are ever read
     * (core:3410-3419): the table at k_r, and the table at k_r - di*w + (nSim - djx) (the "value" of the
     * mirrored candidate). Planes are independent, so they are computed in parallel and sampled. */
    const unsigned nplanes = (nHW_sim + 1) * Ns;
    float *s_at = (float *) malloc(sizeof(float) * nplanes * R);    /* table[ddk][k_r] */
    float *s_mir = (float *) malloc(sizeof(float) * nplanes * R);   /* table[ddk][k_r - di*w + nSim - djx] */
#pragma omp parallel num_threads(nthreads())
    {
        float *diff = (float *) calloc(plane, sizeof(float));
        float *sum = (float *) malloc(plane * sizeof(float));
#pragma omp for schedule(dynamic)
        for (unsigned ddk = 0; ddk < nplanes; ddk++) {
            const unsigned di = ddk / Ns, djx = ddk % Ns;
            const int dk = (int) (di * width + djx) - (int) nHW_sim;
            for (size_t t = 0; t < plane; t++) sum[t] = 2 * threshold;
            for (unsigned i = nHW; i < height - nHW; i++) {
                unsigned k = i * width + nHW;
                for (unsigned j = nHW; j < width - nHW; j++, k++)
                    diff[k] = (img[k + dk] - img[k]) * (img[k + dk] - img[k]);
            }
            sat_plane(diff, sum, width, height, kHW, nHW, height - nHW, width - nHW);
            for (unsigned a = 0; a < nr; a++)
                for (unsigned b = 0; b < nc; b++) {
                    const unsigned k_r = rows[a] * width + cols[b];
                    const size_t r = (size_t) a * nc + b;
                    s_at[(size_t) ddk * R + r] = sum[k_r];
                    s_mir[(size_t) ddk * R + r] = sum[(int) k_r - (int) (di * width) + (int) nHW_sim - (int) djx];
                }
        }
        free(diff); free(sum);
    }

#pragma omp parallel num_threads(nthreads())
    {
        pr_t *td = (pr_t *) malloc(sizeof(pr_t) * (Ns * Ns + 1));
#pragma omp for schedule(dynamic, 16)
        for (size_t r = 0; r < R; r++) {
            const unsigned k_r = rows[r / nc] * width + cols[r % nc];
            unsigned cnt = 0;
            for (int dj = -(int) nHW_sim; dj <= (int) nHW_sim; dj++) {
                for (int di = 0; di <= (int) nHW_sim; di++) {
                    const float v = s_at[(size_t) (dj + (int) nHW_sim + di * (int) Ns) * R + r];
                    if (v < threshold) { td[cnt].d = v; td[cnt].i = k_r + di * width + dj; cnt++; }
                }
                for (int di = -(int) nHW_sim; di < 0; di++) {
                    const size_t ddk = (size_t) (-dj + (int) nHW_sim + (-di) * (int) Ns);
                    if (s_at[ddk * R + r] < threshold) { td[cnt].d = s_mir[ddk * R + r]; td[cnt].i = k_r + di * (int) width + dj; cnt++; }
                }
            }
            const unsigned nSx_r = NHW > cnt ? closest_power_of_2(cnt) : NHW;
            if (nSx_r == 1 && cnt == 0) { td[0].d = 0.0f; td[0].i = k_r; cnt = 1; }
            partial_sort_(td, td + nSx_r, td + cnt);
            unsigned o = 0;
            for (unsigned n = 0; n < nSx_r; n++) out_idx[(size_t) k_r * maxN + o++] = td[n].i;
            if (nSx_r == 1) out_idx[(size_t) k_r * maxN + o++] = td[0].i;
            out_count[k_r] = o;
        }
        free(td);
    }
    free(s_at); free(s_mir); free(rows); free(cols);
}

/* core:3479-3611 with pHW = 1. Only element [0] of the sorted list and the shape flag are consumed
 * downstream (core:294, 310, 503, 510), so the full std::sort is emulated only where the minimum is tied. */
void orc_bm_stereo(const float *img1, const float *img2, unsigned width, unsigned height, unsigned kHW, unsigned nHW,
                   unsigned nHW_disp, float tauMatch, unsigned *out_first, unsigned *out_shape, unsigned *out_ties)
{
    (void) nHW;
    const unsigned Ns = 2 * nHW_disp + 1, np = Ns * Ns;
    const float threshold = tauMatch * kHW * kHW;
    const size_t plane = (size_t) width * height;
    const unsigned row_end = height - nHW_disp - kHW + 1, col_end = width - nHW_disp - kHW + 1;
    float **sums = (float **) malloc(sizeof(float *) * np);
    for (unsigned t = 0; t < np; t++) sums[t] = (float *) calloc(plane, sizeof(float));
#pragma omp parallel num_threads(nthreads())
    {
        float *diff = (float *) calloc(plane, sizeof(float));
#pragma omp for schedule(dynamic)
        for (unsigned ddk = 0; ddk < np; ddk++) {
            const unsigned di = ddk / Ns, dj = ddk % Ns;
            const int dk = (int) (di * width + dj) - (int) (nHW_disp * (1 + width));
            for (unsigned i = nHW_disp; i < height - nHW_disp; i++) {
                unsigned k = i * width + nHW_disp;
                for (unsigned j = nHW_disp; j < width - nHW_disp; j++, k++)
                    diff[k] = (img2[k + dk] - img1[k]) * (img2[k + dk] - img1[k]);
            }
            sat_plane(diff, sums[ddk], width, height, kHW, nHW_disp, row_end, col_end);
        }
        free(diff);
    }
    for (size_t t = 0; t < plane; t++) { out_first[t] = 0xFFFFFFFFu; out_shape[t] = 0; if (out_ties) out_ties[t] = 0; }
    /* grid = ind_initialize(dim - k + 1, nDisp, 1) = [nDisp, dim - k + 1 - nDisp) */
#pragma omp parallel num_threads(nthreads())
    {
        pr_t *td = (pr_t *) malloc(sizeof(pr_t) * np);
#pragma omp for schedule(dynamic, 4)
        for (unsigned i = nHW_disp; i < row_end; i++)
            for (unsigned j = nHW_disp; j < col_end; j++) {
                const unsigned k_r = i * width + j;
                unsigned c = 0, nmin = 0, amin = 0;
                float best = 0.0f;
                for (int dj = -(int) nHW_disp; dj <= (int) nHW_disp; dj++)
                    for (int di = -(int) nHW_disp; di <= (int) nHW_disp; di++) {
                        td[c].d = sums[(dj + (int) nHW_disp) + (di + (int) nHW_disp) * (int) Ns][k_r];
                        td[c].i = k_r + di * (int) width + dj;
                        if (c == 0 || td[c].d < best) { best = td[c].d; nmin = 1; amin = c; }
                        else if (td[c].d == best) nmin++;
                        c++;
                    }
                unsigned first = td[amin].i;
                if (nmin > 1) { std_sort_(td, td + np); first = td[0].i; }
                out_first[k_r] = first;
                out_shape[k_r] = best < threshold ? 1u : 0u;
                if (out_ties) out_ties[k_r] = nmin > 1;
            }
        free(td);
    }
    for (unsigned t = 0; t < np; t++) free(sums[t]);
    free(sums);
}

/* ------------------------------------------------------------------------------------------ */
/* 1-D / 2-D transforms                                                                        */
/* ------------------------------------------------------------------------------------------ */

/* FFTW r2r kinds, unnormalised (FFTW manual "1d Real-even DFTs"); arithmetic per orc_set_dct_mode */
#define MAXDCT 64
typedef struct { int n; float f2[MAXDCT * MAXDCT], f3[MAXDCT * MAXDCT]; double d2[MAXDCT * MAXDCT], d3[MAXDCT * MAXDCT]; } dct_tab_t;
static dct_tab_t *volatile g_tabs[MAXDCT + 1];
static const dct_tab_t *dct_tab(int n)
{
    dct_tab_t *t = g_tabs[n];
    if (t) return t;
#pragma omp critical(orc_dct_tab)
    {
        t = g_tabs[n];
        if (!t) {
            t = (dct_tab_t *) malloc(sizeof(dct_tab_t));
            t->n = n;
            for (int k = 0; k < n; k++)
                for (int j = 0; j < n; j++) {
                    const double a = 2.0 * cos(M_PI * ((double) j + 0.5) * (double) k / (double) n);
                    const double b = (j == 0) ? 1.0 : 2.0 * cos(M_PI * (double) j * ((double) k + 0.5) / (double) n);
                    t->d2[k * n + j] = a; t->f2[k * n + j] = (float) a;
                    t->d3[k * n + j] = b; t->f3[k * n + j] = (float) b;
                }
            g_tabs[n] = t;
        }
    }
    return t;
}
/* 1-D transform of n values read with stride s; kind 2 = REDFT10, 3 = REDFT01 (f32 mode) */
static void dct1_f32(const float *x, int sx, float *y, int sy, int n, int kind)
{
    const dct_tab_t *t = dct_tab(n);
    const float *tab = kind == 2 ? t->f2 : t->f3;
    float tmp[MAXDCT];
    for (int k = 0; k < n; k++) {
        float acc = 0.0f;
        for (int j = 0; j < n; j++) acc = fmaf(x[j * sx], tab[k * n + j], acc);
        tmp[k] = acc;
    }
    for (int k = 0; k < n; k++) y[k * sy] = tmp[k];
}
static void dct1_f64(const double *x, int sx, double *y, int sy, int n, int kind)
{
    const dct_tab_t *t = dct_tab(n);
    const double *tab = kind == 2 ? t->d2 : t->d3;
    double tmp[MAXDCT];
    for (int k = 0; k < n; k++) {
        double acc = 0.0;
        for (int j = 0; j < n; j++) acc += x[j * sx] * tab[k * n + j];
        tmp[k] = acc;
    }
    for (int k = 0; k < n; k++) y[k * sy] = tmp[k];
}
/* rank-1 transform, contiguous, in -> out */
static void r2r_1d(const float *in, float *out, int n, int kind)
{
    if (g_dct_mode == 0) { dct1_f32(in, 1, out, 1, n, kind); return; }
    double a[MAXDCT], b[MAXDCT];
    for (int i = 0; i < n; i++) a[i] = in[i];
    dct1_f64(a, 1, b, 1, n, kind);
    for (int i = 0; i < n; i++) out[i] = (float) b[i];
}
/* rank-2 transform of an n0 x n1 row-major array: contiguous dimension first, then the strided one */
static void r2r_2d(const float *in, float *out, int n0, int n1, int kind)
{
    if (g_dct_mode == 0) {
        float tmp[1024];
        for (int r = 0; r < n0; r++) dct1_f32(in + r * n1, 1, tmp + r * n1, 1, n1, kind);
        for (int c = 0; c < n1; c++) dct1_f32(tmp + c, n1, out + c, n1, n0, kind);
    } else {
        double a[1024], b[1024];
        for (int i = 0; i < n0 * n1; i++) a[i] = in[i];
        for (int r = 0; r < n0; r++) dct1_f64(a + r * n1, 1, b + r * n1, 1, n1, kind);
        for (int c = 0; c < n1; c++) dct1_f64(b + c, n1, a + c, n1, n0, kind);
        for (int i = 0; i < n0 * n1; i++) out[i] = (float) a[i];
    }
}

/* bm3d.cpp:1101-1169 */
void orc_preProcess(float *kaiser, float *coef_norm, float *coef_norm_inv, unsigned kHW)
{
    static const float k8[16] = { 0.1924f, 0.2989f, 0.3846f, 0.4325f, 0.2989f, 0.4642f, 0.5974f, 0.6717f,
                                  0.3846f, 0.5974f, 0.7688f, 0.8644f, 0.4325f, 0.6717f, 0.8644f, 0.9718f };
    static const float k12[36] = { 0.1924f, 0.2615f, 0.3251f, 0.3782f, 0.4163f, 0.4362f, 0.2615f, 0.3554f, 0.4419f, 0.5139f, 0.5657f, 0.5927f,
                                   0.3251f, 0.4419f, 0.5494f, 0.6390f, 0.7033f, 0.7369f, 0.3782f, 0.5139f, 0.6390f, 0.7433f, 0.8181f, 0.8572f,
                                   0.4163f, 0.5657f, 0.7033f, 0.8181f, 0.9005f, 0.9435f, 0.4362f, 0.5927f, 0.7369f, 0.8572f, 0.9435f, 0.9885f };
    if (kHW == 8 || kHW == 12) {
        const float *q = kHW == 8 ? k8 : k12;
        const unsigned hh = kHW / 2;
        for (unsigned i = 0; i < kHW; i++)
            for (unsigned j = 0; j < kHW; j++) {
                const unsigned a = i < hh ? i : kHW - 1 - i, b = j < hh ? j : kHW - 1 - j;
                kaiser[i * kHW + j] = q[a * hh + b];
            }
    } else
        for (unsigned i = 0; i < kHW * kHW; i++) kaiser[i] = 1.0f;
    const float coef = 0.5f / ((float) kHW);
    for (unsigned i = 0; i < kHW; i++)
        for (unsigned j = 0; j < kHW; j++) {
            if (i == 0 && j == 0) { coef_norm[i * kHW + j] = 0.5f * coef; coef_norm_inv[i * kHW + j] = 2.0f; }
            else if (i * j == 0) { coef_norm[i * kHW + j] = (float) (SQRT2_INV_D * coef); coef_norm_inv[i * kHW + j] = (float) SQRT2_D; }
            else { coef_norm[i * kHW + j] = 1.0f * coef; coef_norm_inv[i * kHW + j] = 1.0f; }
        }
}
/* core:3191-3216 */
void orc_preProcess_4d(float *coef_norm, float *coef_norm_inv, unsigned awidth, unsigned aheight)
{
    const float coef = 0.5f / (sqrtf((float) awidth) * sqrtf((float) aheight));
    for (unsigned i = 0; i < aheight; i++)
        for (unsigned j = 0; j < awidth; j++) {
            if (i == 0 && j == 0) { coef_norm[i * awidth + j] = (float) (0.5f * coef); coef_norm_inv[i * awidth + j] = 2.0f; }
            else if (i * j == 0) { coef_norm[i * awidth + j] = (float) (SQRT2_INV_D * coef); coef_norm_inv[i * awidth + j] = (float) SQRT2_D; }
            else { coef_norm[i * awidth + j] = (float) (1.0f * coef); coef_norm_inv[i * awidth + j] = 1.0f; }
        }
}
/* core:3229-3252, packed [size-2][max] */
void orc_preProcess_4d_sadct(float *coef_norm, float *coef_norm_inv, unsigned max_dct_size)
{
    for (unsigned k = 0; k + 1 < max_dct_size; k++) {
        const unsigned n = k + 2;
        const float coef = (float) ((float) SQRT2_D / sqrt((double) n));
        coef_norm[k * max_dct_size] = (float) (SQRT2_INV_D * coef);
        coef_norm_inv[k * max_dct_size] = (float) SQRT2_D;
        for (unsigned i = 1; i < n; i++) { coef_norm[k * max_dct_size + i] = coef; coef_norm_inv[k * max_dct_size + i] = 1.0f; }
    }
}

/* lib_transforms.cpp:403-433 */
void orc_haar_forward(float *v, unsigned N)
{
    float tmp[MAXDCT];
    const float c = (float) SQRT2_INV_D;
    while (N >= 2) {
        const unsigned n = N / 2;
        for (unsigned k = 0; k < n; k++) {
            const float a = v[2 * k], b = v[2 * k + 1];
            tmp[k] = (a + b) * c;
            tmp[n + k] = (a - b) * c;
        }
        for (unsigned k = 0; k < N; k++) v[k] = tmp[k];
        N = n;
    }
}
/* lib_transforms.cpp:447-471 */
void orc_haar_inverse(float *v, unsigned N)
{
    float tmp[MAXDCT];
    const float c = (float) SQRT2_INV_D;
    for (unsigned n = 1; n < N; n *= 2) {
        for (unsigned k = 0; k < n; k++) {
            const float a = v[k], b = v[n + k];
            tmp[2 * k] = (a + b) * c;
            tmp[2 * k + 1] = (a - b) * c;
        }
        for (unsigned k = 0; k < 2 * n; k++) v[k] = tmp[k];
    }
}
/* lib_transforms.cpp:290-321 */
void orc_hadamard(float *v, unsigned N)
{
    if (N <= 1) return;
    if (N == 2) { const float a = v[0], b = v[1]; v[0] = a + b; v[1] = a - b; return; }
    float tmp[MAXDCT];
    const unsigned n = N / 2;
    for (unsigned k = 0; k < n; k++) {
        const float a = v[2 * k], b = v[2 * k + 1];
        v[k] = a + b;
        tmp[k] = a - b;
    }
    for (unsigned k = 0; k < n; k++) v[n + k] = tmp[k];
    orc_hadamard(v, n);
    orc_hadamard(v + n, n);
}

/* lib_transforms.cpp:215-277 */
static void bior15(float *lpd, float *hpd, float *lpr, float *hpr)
{
    const float coef_norm = 1.f / (sqrtf(2.f) * 128.f);
    const float sqrt2_inv = 1.f / sqrtf(2.f);
    static const float a[10] = { 3.f, -3.f, -22.f, 22.f, 128.f, 128.f, 22.f, -22.f, -3.f, 3.f };
    static const float d[10] = { 3.f, 3.f, -22.f, -22.f, 128.f, -128.f, 22.f, 22.f, -3.f, -3.f };
    for (int i = 0; i < 10; i++) {
        lpd[i] = a[i] * coef_norm;
        hpr[i] = d[i] * coef_norm;
        hpd[i] = i == 4 ? -sqrt2_inv : (i == 5 ? sqrt2_inv : 0.f);
        lpr[i] = (i == 4 || i == 5) ? sqrt2_inv : 0.f;
    }
}
/* periodic extension index, lib_transforms.cpp:352-373 */
static void per_ext_ind(unsigned *ind, unsigned N, unsigned L)
{
    for (unsigned k = 0; k < N; k++) ind[k + L] = k;
    int i1 = (int) N - (int) L;
    while (i1 < 0) i1 += (int) N;
    unsigned i2 = 0;
    for (unsigned k = 0; k < L; k++) {
        ind[k] = (unsigned) i1;
        ind[k + L + N] = i2;
        i1 = ((unsigned) i1 < N - 1) ? i1 + 1 : 0;
        i2 = (i2 < N - 1) ? i2 + 1 : 0;
    }
}
static unsigned ilog2_ceil(unsigned N) { unsigned k = 1, n = 0; while (k < N) { k *= 2; n++; } return n; }

/* lib_transforms.cpp:46-120 */
void orc_bior_2d_forward(const float *patch, float *out, unsigned N)
{
    float lpd[10], hpd[10], lpr[10], hpr[10];
    bior15(lpd, hpd, lpr, hpr);
    for (unsigned i = 0; i < N * N; i++) out[i] = patch[i];
    const unsigned iters = ilog2_ceil(N);
    unsigned N1 = N, N2 = N / 2;
    float tmp[MAXDCT + 8];
    unsigned ind[MAXDCT + 8];
    for (unsigned it = 0; it < iters; it++) {
        const unsigned len = N1 + 8;
        per_ext_ind(ind, N1, 4);
        for (unsigned i = 0; i < N1; i++) {
            for (unsigned j = 0; j < len; j++) tmp[j] = out[i * N + ind[j]];
            for (unsigned j = 0; j < N2; j++) {
                float vl = 0.0f, vh = 0.0f;
                for (unsigned t = 0; t < 10; t++) { vl += tmp[t + j * 2] * lpd[t]; vh += tmp[t + j * 2] * hpd[t]; }
                out[i * N + j] = vl;
                out[i * N + j + N2] = vh;
            }
        }
        for (unsigned j = 0; j < N1; j++) {
            for (unsigned i = 0; i < len; i++) tmp[i] = out[j + ind[i] * N];
            for (unsigned i = 0; i < N2; i++) {
                float vl = 0.0f, vh = 0.0f;
                for (unsigned t = 0; t < 10; t++) { vl += tmp[t + i * 2] * lpd[t]; vh += tmp[t + i * 2] * hpd[t]; }
                out[j + i * N] = vl;
                out[j + (i + N2) * N] = vh;
            }
        }
        N1 /= 2; N2 /= 2;
    }
}
/* lib_transforms.cpp:135-204 */
void orc_bior_2d_inverse(float *sig, unsigned N)
{
    float lpd[10], hpd[10], lpr[10], hpr[10];
    bior15(lpd, hpd, lpr, hpr);
    const unsigned iters = ilog2_ceil(N);
    unsigned N1 = 2, N2 = 1;
    float tmp[5 * MAXDCT];
    unsigned ind[5 * MAXDCT];
    for (unsigned it = 0; it < iters; it++) {
        const unsigned len = N1 + 4 * N1;
        per_ext_ind(ind, N1, 4 * N2);
        for (unsigned j = 0; j < N1; j++) {
            for (unsigned i = 0; i < len; i++) tmp[i] = sig[j + ind[i] * N];
            for (unsigned i = 0; i < N2; i++) {
                float vl = 0.0f, vh = 0.0f;
                for (unsigned t = 0; t < 10; t++) { vl += lpr[t] * tmp[t * N2 + i]; vh += hpr[t] * tmp[t * N2 + i]; }
                sig[i * 2 * N + j] = vh;
                sig[(i * 2 + 1) * N + j] = vl;
            }
        }
        for (unsigned i = 0; i < N1; i++) {
            for (unsigned j = 0; j < len; j++) tmp[j] = sig[i * N + ind[j]];
            for (unsigned j = 0; j < N2; j++) {
                float vl = 0.0f, vh = 0.0f;
                for (unsigned t = 0; t < 10; t++) { vl += lpr[t] * tmp[t * N2 + j]; vh += hpr[t] * tmp[t * N2 + j]; }
                sig[i * N + j * 2] = vh;
                sig[i * N + j * 2 + 1] = vl;
            }
        }
        N1 *= 2; N2 *= 2;
    }
}

/* bm3d.cpp:745-757: REDFT10 x REDFT10 then coef_norm */
void orc_dct_2d_forward(const float *patch, float *out, unsigned k)
{
    float kais[1024], cn[1024], cni[1024];
    orc_preProcess(kais, cn, cni, k);
    float tmp[1024];
    r2r_2d(patch, tmp, (int) k, (int) k, 2);
    for (unsigned i = 0; i < k * k; i++) out[i] = tmp[i] * cn[i];
}
/* bm3d.cpp:1039-1071 */
void orc_dct_2d_inverse(float *patch, unsigned k)
{
    float kais[1024], cn[1024], cni[1024], a[1024], b[1024];
    orc_preProcess(kais, cn, cni, k);
    for (unsigned i = 0; i < k * k; i++) a[i] = patch[i] * cni[i];
    r2r_2d(a, b, (int) k, (int) k, 3);
    const float coef = 1.0f / (float) (k * 2);
    for (unsigned i = 0; i < k * k; i++) patch[i] = coef * b[i];
}

/* ------------------------------------------------------------------------------------------ */
/* one window pass                                                                             */
/* ------------------------------------------------------------------------------------------ */
#define MAXA 81     /* (2*an+1)^2 up to an = 4 */
#define MAXASW 9

typedef struct {
    unsigned asw, A, chnls, k, k2, N;
    unsigned tau_2D, tau_4D, tau_5D;
    float cn2[1024], cni2[1024], kaiser[1024];
    float cn4[MAXA], cni4[MAXA];
    float cnsa[MAXASW * MAXASW], cnisa[MAXASW * MAXASW];
    float sigma_table[3];
    float lambda;
    int partial;          /* `pst != cst` branch: 2-D transforms of the local variants (core:1715, :1756, :1822) */
} pass_ctx;

/* 2-D spatial transform of the k x k patch of `plane` at flat position pos (core:1679 / bm3d.cpp:705 / :831);
 * a patch whose column is w_b - k is never written into the reference's table and reads as zeros (core:1697). */
static void t2d_forward(const pass_ctx *cx, const float *plane, unsigned w_b, unsigned pos, float *out)
{
    const unsigned k = cx->k, k2 = cx->k2;
    /* the row-band variants fill columns j < w_b - k only (core:1697): column w_b - k stays zero; the local variants of the
       partial-window branch write every column they read (core:1735) */
    if (!cx->partial && pos % w_b >= w_b - k) { for (unsigned i = 0; i < k2; i++) out[i] = 0.0f; return; }
    float patch[1024];
    for (unsigned p = 0; p < k; p++)
        for (unsigned q = 0; q < k; q++) patch[p * k + q] = plane[pos + p * w_b + q];
    if (cx->tau_2D == ORC_ID) memcpy(out, patch, k2 * sizeof(float));
    else if (cx->tau_2D == ORC_DCT) {
        float tmp[1024];
        r2r_2d(patch, tmp, (int) k, (int) k, 2);
        for (unsigned i = 0; i < k2; i++) out[i] = tmp[i] * cx->cn2[i];
    } else orc_bior_2d_forward(patch, out, k);
}
static void t2d_inverse(const pass_ctx *cx, float *patch)
{
    const unsigned k = cx->k, k2 = cx->k2;
    if (cx->tau_2D == ORC_DCT) {
        float a[1024], b[1024];
        for (unsigned i = 0; i < k2; i++) a[i] = patch[i] * cx->cni2[i];
        r2r_2d(a, b, (int) k, (int) k, 3);
        const float coef = 1.0f / (float) (k * 2);
        for (unsigned i = 0; i < k2; i++) patch[i] = coef * b[i];
    } else if (cx->tau_2D == ORC_BIOR) orc_bior_2d_inverse(patch, k);
}

/* shape bookkeeping of one group (core:302-323 and the mask updates inside sadct_4d_process :2036-2105) */
typedef struct {
    unsigned mask[MAXA], idx[MAXA], mask_col[MAXA], idx_col[MAXA], mask_dct[MAXA];
    unsigned row_size[MAXASW], col_size[MAXASW];
    int use_sadct;
} shape_t;

static void shape_build(shape_t *sh, unsigned asw)
{
    const unsigned A = asw * asw;
    memset(sh->idx, 0, sizeof(sh->idx)); memset(sh->mask_col, 0, sizeof(sh->mask_col));
    memset(sh->idx_col, 0, sizeof(sh->idx_col)); memset(sh->mask_dct, 0, sizeof(sh->mask_dct));
    unsigned size = 0;
    for (unsigned st = 0; st < A; st++) size += sh->mask[st];
    sh->use_sadct = size != A;
    for (unsigned s = 0; s < asw; s++) {
        unsigned r = 0;
        for (unsigned t = 0; t < asw; t++) if (sh->mask[s * asw + t]) sh->idx[s * asw + r++] = t;
        sh->row_size[s] = r;
        for (unsigned t = 0; t < r; t++) sh->mask_col[s * asw + t] = 1;
    }
    for (unsigned t = 0; t < asw; t++) {
        unsigned r = 0;
        for (unsigned s = 0; s < asw; s++) if (sh->mask_col[s * asw + t]) sh->idx_col[(r++) * asw + t] = s;
        sh->col_size[t] = r;
        for (unsigned s = 0; s < r; s++) sh->mask_dct[s * asw + t] = 1;
    }
}

/* angular transform of one (n, c, pq) vector v[A] (st fastest): full DCT core:1862-1901, SA-DCT core:1969-2116 */
static void t4d_forward(const pass_ctx *cx, const shape_t *sh, float *v)
{
    const unsigned asw = cx->asw, A = cx->A;
    if (cx->tau_4D == ORC_ID) return;
    if (!sh->use_sadct) {
        float o[MAXA];
        r2r_2d(v, o, (int) asw, (int) asw, 2);
        for (unsigned st = 0; st < A; st++) v[st] = o[st] * cx->cn4[st];
        return;
    }
    float a[MAXASW], b[MAXASW];
    for (unsigned s = 0; s < asw; s++) {
        const unsigned n = sh->row_size[s];
        if (n == 1) v[s * asw] = v[s * asw + sh->idx[s * asw]];
        else if (n > 1) {
            for (unsigned t = 0; t < n; t++) a[t] = v[s * asw + sh->idx[s * asw + t]];
            r2r_1d(a, b, (int) n, 2);
            for (unsigned t = 0; t < n; t++) v[s * asw + t] = b[t] * cx->cnsa[(n - 2) * asw + t];
        }
    }
    for (unsigned t = 0; t < asw; t++) {
        const unsigned n = sh->col_size[t];
        if (n == 1) v[t] = v[sh->idx_col[t] * asw + t];
        else if (n > 1) {
            for (unsigned s = 0; s < n; s++) a[s] = v[sh->idx_col[s * asw + t] * asw + t];
            r2r_1d(a, b, (int) n, 2);
            for (unsigned s = 0; s < n; s++) v[s * asw + t] = b[s] * cx->cnsa[(n - 2) * asw + s];
        }
    }
    const float coef = (float) (0.5 * (float) SQRT2_INV_D);
    for (unsigned st = 0; st < A; st++) v[st] *= (float) sh->mask_dct[st] * coef;
}
/* inverse: core:1913-1954 (full) / core:2131-2264 (SA-DCT); output still indexed by st */
static void t4d_inverse(const pass_ctx *cx, const shape_t *sh, float *v)
{
    const unsigned asw = cx->asw, A = cx->A;
    if (cx->tau_4D == ORC_ID) return;
    if (!sh->use_sadct) {
        float a[MAXA], o[MAXA];
        for (unsigned st = 0; st < A; st++) a[st] = v[st] * cx->cni4[st];
        r2r_2d(a, o, (int) asw, (int) asw, 3);
        const float coef = 1.0f / (sqrtf((float) asw) * sqrtf((float) asw) * 2.0f);
        for (unsigned st = 0; st < A; st++) v[st] = o[st] * coef;
        return;
    }
    float a[MAXASW], b[MAXASW];
    const float c2 = (float) (2.0 * (float) SQRT2_D);
    for (unsigned t = 0; t < asw; t++) {
        const unsigned n = sh->col_size[t];
        if (n == 1) v[sh->idx_col[t] * asw + t] = v[t] * c2;
        else if (n > 1) {
            for (unsigned s = 0; s < n; s++) a[s] = v[s * asw + t] * cx->cnisa[(n - 2) * asw + s] * c2;
            r2r_1d(a, b, (int) n, 3);
            const float coef = 0.5f * (float) (SQRT2_INV_D) / sqrtf((float) n);
            for (unsigned s = 0; s < n; s++) v[sh->idx_col[s * asw + t] * asw + t] = b[s] * coef;
        }
    }
    for (unsigned s = 0; s < asw; s++) {
        const unsigned n = sh->row_size[s];
        if (n == 1) v[s * asw + sh->idx[s * asw]] = v[s * asw];
        else if (n > 1) {
            for (unsigned t = 0; t < n; t++) a[t] = v[s * asw + t] * cx->cnisa[(n - 2) * asw + t];
            r2r_1d(a, b, (int) n, 3);
            const float coef = 0.5f * (float) (SQRT2_INV_D) / sqrtf((float) n);
            for (unsigned t = 0; t < n; t++) v[s * asw + sh->idx[s * asw + t]] = b[t] * coef;
        }
    }
    for (unsigned st = 0; st < A; st++) v[st] = v[st] * (float) sh->mask[st];
}

/* result of one reference patch */
typedef struct {
    unsigned nSx;
    unsigned pos[64 * MAXA];    /* [n][st] flat positions in the padded plane (undefined for masked-out SAIs) */
    float w[3];
    unsigned shape[MAXA];       /* shape_table_LF[st][k_r] (1 for pst) */
    float *Z;                   /* [st][c][n][pq] filtered pixel-domain patches */
} group_out;

/* core:277-480 (step 1) / :1054-1281 (step 2) for one reference patch */
static void process_group(const pass_ctx *cx, int step, const float *noisy, const float *basic, unsigned w_b, unsigned h_b,
                          const unsigned *mask_asw, unsigned pst, unsigned k_r,
                          const unsigned *bm_count, const unsigned *bm_idx, unsigned maxN,
                          const unsigned *st_first, const unsigned *st_shape, group_out *go, float *scratch)
{
    const unsigned A = cx->A, C = cx->chnls, k2 = cx->k2;
    const size_t plane = (size_t) w_b * h_b;
    const unsigned nSx = bm_count[k_r];
    go->nSx = nSx;
    /* group buffers G[n][c][pq][st] */
    float *G = scratch, *E = scratch + (size_t) nSx * C * k2 * A;
    memset(G, 0, sizeof(float) * 2 * nSx * C * k2 * A);
    float patch[1024];
    for (unsigned n = 0; n < nSx; n++) {
        const unsigned ind_pst = bm_idx[(size_t) k_r * maxN + n];
        for (unsigned st = 0; st < A; st++) {
            if (!mask_asw[st]) continue;
            const unsigned pos = (st == pst) ? ind_pst : st_first[(size_t) st * plane + ind_pst];
            go->pos[n * A + st] = pos;
            for (unsigned c = 0; c < C; c++) {
                t2d_forward(cx, noisy + ((size_t) st * C + c) * plane, w_b, pos, patch);
                for (unsigned pq = 0; pq < k2; pq++) G[((size_t) (n * C + c) * k2 + pq) * A + st] = patch[pq];
                if (step == 2) {
                    t2d_forward(cx, basic + ((size_t) st * C + c) * plane, w_b, pos, patch);
                    for (unsigned pq = 0; pq < k2; pq++) E[((size_t) (n * C + c) * k2 + pq) * A + st] = patch[pq];
                }
            }
        }
    }
    shape_t sh;
    memset(&sh, 0, sizeof(sh));
    for (unsigned st = 0; st < A; st++) {
        const unsigned s = (st == pst) ? 1u : (mask_asw[st] ? st_shape[(size_t) st * plane + k_r] : 0u);
        go->shape[st] = s;
        sh.mask[st] = s;
    }
    if (cx->tau_4D == ORC_SADCT) shape_build(&sh, cx->asw); else sh.use_sadct = 0;

    for (unsigned n = 0; n < nSx; n++)
        for (unsigned c = 0; c < C; c++)
            for (unsigned pq = 0; pq < k2; pq++) {
                t4d_forward(cx, &sh, G + ((size_t) (n * C + c) * k2 + pq) * A);
                if (step == 2) t4d_forward(cx, &sh, E + ((size_t) (n * C + c) * k2 + pq) * A);
            }

    /* 5th dimension: per pq, vectors along n for each (c, st); core:2281-2505 / :2706-2925 */
    float wt[3] = { 0.0f, 0.0f, 0.0f };
    double wtd[3] = { 0.0, 0.0, 0.0 };           /* step-2 weight sums of sum mode 1 */
    float vo[64], ve[64];
    const float hcoef = 1.0f / (float) nSx;
    float cn5[64], cni5[64];                     /* preProcess_5d, core:3262-3276 */
    {
        const float coef = (float) (SQRT2_D) / sqrt(nSx);
        cn5[0] = (float) (SQRT2_INV_D * coef); cni5[0] = (float) (SQRT2_D);
        for (unsigned i = 1; i < nSx; i++) { cn5[i] = coef; cni5[i] = 1.0; }
    }
    for (unsigned pq = 0; pq < k2; pq++) {
        /* forward along n */
        for (unsigned c = 0; c < C; c++)
            for (unsigned st = 0; st < A; st++) {
                if (cx->tau_5D == ORC_DCT) {      /* core:2544-2556 / :2974-2989: REDFT10 of length nSx, then coef_norm_5d */
                    for (int rep = 0; rep < step; rep++) {
                        float *B = rep == 0 ? G : E;
                        for (unsigned n = 0; n < nSx; n++) vo[n] = B[((size_t) (n * C + c) * k2 + pq) * A + st];
                        r2r_1d(vo, ve, (int) nSx, 2);
                        for (unsigned n = 0; n < nSx; n++) B[((size_t) (n * C + c) * k2 + pq) * A + st] = ve[n] * cn5[n];
                    }
                } else if (nSx > 1) {
                    for (unsigned n = 0; n < nSx; n++) vo[n] = G[((size_t) (n * C + c) * k2 + pq) * A + st];
                    if (cx->tau_5D == ORC_HAAR) orc_haar_forward(vo, nSx); else orc_hadamard(vo, nSx);
                    for (unsigned n = 0; n < nSx; n++) G[((size_t) (n * C + c) * k2 + pq) * A + st] = vo[n];
                    if (step == 2) {
                        for (unsigned n = 0; n < nSx; n++) ve[n] = E[((size_t) (n * C + c) * k2 + pq) * A + st];
                        if (cx->tau_5D == ORC_HAAR) orc_haar_forward(ve, nSx); else orc_hadamard(ve, nSx);
                        for (unsigned n = 0; n < nSx; n++) E[((size_t) (n * C + c) * k2 + pq) * A + st] = ve[n];
                    }
                }
            }
        /* shrinkage, in the reference's accumulation order: c, then st, then n */
        for (unsigned c = 0; c < C; c++) {
            const float sg = cx->sigma_table[c];
            float T;
            if (g_bm3d) T = cx->lambda * sg * sqrtf((float) nSx);                 /* bm3d.cpp:940 */
            else if (cx->tau_5D == ORC_HAAR) T = cx->lambda * sg * (float) (SQRT2_D);
            else if (cx->tau_5D == ORC_DCT) T = cx->lambda * sg * 2.0f * (float) (SQRT2_D);       /* core:2566 */
            else T = cx->lambda * sg * sqrtf((float) nSx) * (float) (SQRT2_D);
            for (unsigned st = 0; st < A; st++) {
                if (sh.use_sadct && !sh.mask_dct[st]) continue;
                for (unsigned n = 0; n < nSx; n++) {
                    float *g = &G[((size_t) (n * C + c) * k2 + pq) * A + st];
                    if (step == 1) {
                        if (fabsf(*g) > T) wt[c]++; else *g = 0.0f;
                    } else {
                        float *e = &E[((size_t) (n * C + c) * k2 + pq) * A + st];
                        float value;
                        if (cx->tau_5D == ORC_HAAR || cx->tau_5D == ORC_DCT) {
                            value = (*e) * (*e);
                            value /= (value + sg * sg);
                            *e = (*g) * value;
                        } else {
                            value = (*e) * (*e) * hcoef;
                            value /= (value + sg * sg);
                            *e = (*g) * value * hcoef;
                        }
                        if (g_sum_mode) wtd[c] += value; else wt[c] += value;
                    }
                }
            }
        }
        /* inverse along n (of G in step 1, of E in step 2) */
        float *X = step == 1 ? G : E;
        for (unsigned c = 0; c < C; c++)
            for (unsigned st = 0; st < A; st++) {
                if (cx->tau_5D == ORC_DCT) {      /* core:2578-2593: coef_norm_inv_5d, REDFT01, 0.5 / sqrt(2 nSx) */
                    for (unsigned n = 0; n < nSx; n++) vo[n] = X[((size_t) (n * C + c) * k2 + pq) * A + st] * cni5[n];
                    r2r_1d(vo, ve, (int) nSx, 3);
                    const float coef5 = 0.5f * (float) (SQRT2_INV_D) / sqrtf((float) nSx);
                    for (unsigned n = 0; n < nSx; n++) X[((size_t) (n * C + c) * k2 + pq) * A + st] = ve[n] * coef5;
                } else if (nSx > 1) {
                    for (unsigned n = 0; n < nSx; n++) vo[n] = X[((size_t) (n * C + c) * k2 + pq) * A + st];
                    if (cx->tau_5D == ORC_HAAR) orc_haar_inverse(vo, nSx);
                    else {
                        orc_hadamard(vo, nSx);
                        if (step == 1) for (unsigned n = 0; n < nSx; n++) vo[n] *= hcoef;
                    }
                    for (unsigned n = 0; n < nSx; n++) X[((size_t) (n * C + c) * k2 + pq) * A + st] = vo[n];
                }
            }
    }
    if (g_sum_mode && step == 2)                 /* rounded to float once; the weight below is the same float expression */
        for (unsigned c = 0; c < C; c++) wt[c] = (float) wtd[c];
    for (unsigned c = 0; c < C; c++) {
        const float sg = cx->sigma_table[c];
        go->w[c] = wt[c] > 0.0f ? (sg > 0.0 ? 1.0f / (float) (sg * sg * wt[c]) : 1.0f / (float) (wt[c])) : 1.0f;
    }
    if (g_use_sd) {      /* sd_weighting_5d, core:3140-3173 (N without the k^2 factor, as written there); bm3d.cpp:1345-1372 reads channel 0 for every c */
        const float *X = step == 1 ? G : E;
        const unsigned Nn = g_bm3d ? nSx * k2 : nSx * A;
        for (unsigned c = 0; c < C; c++) {
            const unsigned cc = g_bm3d ? 0 : c;
            float mean = 0.0f, std = 0.0f;
            double meand = 0.0, stdd = 0.0;      /* sum mode 1 */
            for (unsigned pq = 0; pq < k2; pq++)
                for (unsigned st = 0; st < A; st++)
                    for (unsigned n = 0; n < nSx; n++) {
                        const float x = X[((size_t) (n * C + cc) * k2 + pq) * A + st];
                        if (g_sum_mode) { meand += x; stdd += x * x; }
                        else { mean += x; std += x * x; }
                    }
            if (g_sum_mode) { mean = (float) meand; std = (float) stdd; }
            const float res = (std - mean * mean / (float) Nn) / (float) (Nn - 1);
            go->w[c] = res > 0.0f ? 1.0f / sqrtf(res) : 0.0f;
        }
    }
    /* inverse angular + inverse spatial transforms; output Z[st][c][n][pq] */
    float *X = step == 1 ? G : E;
    for (unsigned n = 0; n < nSx; n++)
        for (unsigned c = 0; c < C; c++) {
            for (unsigned pq = 0; pq < k2; pq++) t4d_inverse(cx, &sh, X + ((size_t) (n * C + c) * k2 + pq) * A);
            for (unsigned st = 0; st < A; st++) {
                for (unsigned pq = 0; pq < k2; pq++) patch[pq] = X[((size_t) (n * C + c) * k2 + pq) * A + st];
                t2d_inverse(cx, patch);
                memcpy(go->Z + (((size_t) st * C + c) * nSx + n) * k2, patch, k2 * sizeof(float));
            }
        }
}

void orc_set_use_sd(int on) { g_use_sd = on; }

int orc_pass(int step, float sigma, float lambda, const float *noisy_sym, const float *basic_sym, float *num_sym, float *den_sym,
             const unsigned *mask_asw, const unsigned *procSAI_asw, unsigned pst, unsigned asw, unsigned w_b, unsigned h_b,
             unsigned chnls, unsigned nSim, unsigned nDisp, unsigned k, unsigned N, unsigned p, unsigned color_space,
             unsigned tau_2D, unsigned tau_4D, unsigned tau_5D,
             unsigned *dbg_count, unsigned *dbg_idx, unsigned *dbg_first, unsigned *dbg_shape)
{
    return orc_pass_ex(step, sigma, lambda, noisy_sym, basic_sym, num_sym, den_sym, mask_asw, procSAI_asw, pst, pst, asw, w_b, h_b, chnls,
                       nSim, nDisp, k, N, p, color_space, tau_2D, tau_4D, tau_5D, dbg_count, dbg_idx, dbg_first, dbg_shape);
}

/* utilities_LF.cpp:1000-1016 */
static int patch_denoised(const float *den0, unsigned p_idx, unsigned w_b, unsigned k)
{
    for (unsigned p = 0; p < k; p++)
        for (unsigned q = 0; q < k; q++)
            if (den0[p_idx + p * w_b + q] == 0.0) return 0;
    return 1;
}

/* One core call. cst = window slot of the SAI the window was centred on; pst == cst is the full-grid branch (core:223-530 /
   :986-1331), pst != cst the partial-window branch (core:531-821 / :1332-1658): only the grid patches of SAI pst that still
   contain a pixel with den == 0 are processed (den-aware ind_initialize, utilities_LF.cpp:1031-1099), block matching is the
   same computation restricted to them (core:3631-3788, :3806-3945) and the 2-D transforms are the local variants. */
int orc_pass_ex(int step, float sigma, float lambda, const float *noisy_sym, const float *basic_sym, float *num_sym, float *den_sym,
                const unsigned *mask_asw, const unsigned *procSAI_asw, unsigned cst, unsigned pst, unsigned asw, unsigned w_b, unsigned h_b,
                unsigned chnls, unsigned nSim, unsigned nDisp, unsigned k, unsigned N, unsigned p, unsigned color_space,
                unsigned tau_2D, unsigned tau_4D, unsigned tau_5D,
                unsigned *dbg_count, unsigned *dbg_idx, unsigned *dbg_first, unsigned *dbg_shape)
{
    const unsigned A = asw * asw, n = nSim + nDisp, k2 = k * k;
    const size_t plane = (size_t) w_b * h_b;
    if (asw > MAXASW || chnls > 3 || k2 > 1024 || N > 64) return 1;
    if (tau_2D != ORC_ID && tau_2D != ORC_DCT && tau_2D != ORC_BIOR) return 1;
    if (tau_4D != ORC_ID && tau_4D != ORC_DCT && tau_4D != ORC_SADCT) return 1;
    if (tau_5D != ORC_HAAR && tau_5D != ORC_HADAMARD && tau_5D != ORC_DCT) return 1;

    pass_ctx *cx = (pass_ctx *) calloc(1, sizeof(pass_ctx));
    cx->asw = asw; cx->A = A; cx->chnls = chnls; cx->k = k; cx->k2 = k2; cx->N = N;
    cx->tau_2D = tau_2D; cx->tau_4D = tau_4D; cx->tau_5D = tau_5D;
    if (orc_estimate_sigma(sigma, cx->sigma_table, chnls, color_space)) { free(cx); return 1; }
    orc_preProcess(cx->kaiser, cx->cn2, cx->cni2, k);
    orc_preProcess_4d(cx->cn4, cx->cni4, asw, asw);
    if (asw > 1) orc_preProcess_4d_sadct(cx->cnsa, cx->cnisa, asw);
    cx->lambda = lambda;
    if (step == 1 && tau_2D == ORC_ID && tau_4D == ORC_DCT) cx->lambda = lambda / (float) (SQRT2_D);   /* core:206-207 */
    float tauMatch = (chnls == 1 ? 3.f : 1.f) * (cx->sigma_table[0] < 35.0f ? (step == 1 ? 3000 : 2000) : 5000);  /* core:146 / :915 */
    if (g_bm3d) tauMatch = step == 1 ? (chnls == 1 ? 3.f : 1.f) * (cx->sigma_table[0] < 35.0f ? 2500 : 5000)      /* bm3d.cpp:340 */
                                     : (cx->sigma_table[0] < 35.0f ? 400 : 3500);                                /* bm3d.cpp:532 */

    unsigned *rows = (unsigned *) malloc(sizeof(unsigned) * (h_b + 2)), *cols = (unsigned *) malloc(sizeof(unsigned) * (w_b + 2));
    const unsigned nr = orc_ind_initialize(rows, h_b - k + 1, n, p), nc = orc_ind_initialize(cols, w_b - k + 1, n, p);
    cx->partial = pst != cst;
    unsigned char *act = (unsigned char *) malloc((size_t) nr * nc);
    {
        size_t nact = 0;
        const float *den0 = den_sym + (size_t) pst * chnls * plane;
        for (unsigned a = 0; a < nr; a++)
            for (unsigned b = 0; b < nc; b++) {
                act[(size_t) a * nc + b] = cx->partial ? !patch_denoised(den0, rows[a] * w_b + cols[b], w_b, k) : 1;
                nact += act[(size_t) a * nc + b];
            }
        if (nact == 0) { free(act); free(rows); free(cols); free(cx); return 0; }   /* core:160-165 */
    }

    /* running estimate, channel 0 only (the only one block matching reads): core:169 / :937 */
    const float *sub = step == 1 ? noisy_sym : basic_sym;
    float *est0 = (float *) malloc(sizeof(float) * A * plane);
    for (unsigned st = 0; st < A; st++) {
        if (!mask_asw[st]) continue;
        const size_t o = (size_t) st * chnls * plane;
        for (size_t t = 0; t < plane; t++)
            est0[(size_t) st * plane + t] = den_sym[o + t] ? num_sym[o + t] / den_sym[o + t] : sub[o + t];
    }
    const unsigned maxN = N + 1;
    unsigned *bm_count = dbg_count ? dbg_count : (unsigned *) malloc(sizeof(unsigned) * plane);
    unsigned *bm_idx = dbg_idx ? dbg_idx : (unsigned *) malloc(sizeof(unsigned) * plane * maxN);
    unsigned *st_first = dbg_first ? dbg_first : (unsigned *) malloc(sizeof(unsigned) * A * plane);
    unsigned *st_shape = dbg_shape ? dbg_shape : (unsigned *) malloc(sizeof(unsigned) * A * plane);
    orc_bm_self(est0 + (size_t) pst * plane, w_b, h_b, k, N, n, nSim, p, tauMatch, bm_count, bm_idx, maxN);
    for (unsigned st = 0; st < A; st++) {
        if (st == pst || !mask_asw[st]) {
            for (size_t t = 0; t < plane; t++) { st_first[(size_t) st * plane + t] = 0xFFFFFFFFu; st_shape[(size_t) st * plane + t] = 0; }
            continue;
        }
        orc_bm_stereo(est0 + (size_t) pst * plane, est0 + (size_t) st * plane, w_b, h_b, k, n, nDisp, tauMatch,
                      st_first + (size_t) st * plane, st_shape + (size_t) st * plane, NULL);
    }
    free(est0);

    /* per reference row: groups in parallel, aggregation serial in the reference's order (core:484-528) */
    const size_t zsz = (size_t) A * chnls * (N + 1) * k2;
    group_out *gos = (group_out *) calloc(nc, sizeof(group_out));
    for (unsigned b = 0; b < nc; b++) gos[b].Z = (float *) malloc(sizeof(float) * zsz);
    const int nt = nthreads();
    float **scr = (float **) malloc(sizeof(float *) * nt);
    for (int t = 0; t < nt; t++) scr[t] = (float *) malloc(sizeof(float) * 2 * (N + 1) * chnls * k2 * A);
    for (unsigned a = 0; a < nr; a++) {
        const unsigned i_r = rows[a];
#pragma omp parallel for schedule(dynamic) num_threads(nt)
        for (unsigned b = 0; b < nc; b++) {
#ifdef _OPENMP
            const int tid = omp_get_thread_num();
#else
            const int tid = 0;
#endif
            if (!act[(size_t) a * nc + b]) continue;
            process_group(cx, step, noisy_sym, basic_sym, w_b, h_b, mask_asw, pst, i_r * w_b + cols[b],
                          bm_count, bm_idx, maxN, st_first, st_shape, &gos[b], scr[tid]);
        }
        for (unsigned st = 0; st < A; st++) {
            if (procSAI_asw[st]) continue;
            for (unsigned b = 0; b < nc; b++) {
                const group_out *go = &gos[b];
                if (!act[(size_t) a * nc + b]) continue;
                if (!(tau_4D != ORC_SADCT || st == pst || go->shape[st])) continue;
                for (unsigned c = 0; c < chnls; c++) {
                    float *num = num_sym + ((size_t) st * chnls + c) * plane;
                    float *den = den_sym + ((size_t) st * chnls + c) * plane;
                    for (unsigned nn = 0; nn < go->nSx; nn++) {
                        const unsigned pos = go->pos[nn * A + st];
                        const float *z = go->Z + (((size_t) st * chnls + c) * go->nSx + nn) * k2;
                        for (unsigned pp = 0; pp < k; pp++)
                            for (unsigned q = 0; q < k; q++) {
                                const unsigned ind = pos + pp * w_b + q;
                                num[ind] += cx->kaiser[pp * k + q] * go->w[c] * z[pp * k + q];
                                den[ind] += cx->kaiser[pp * k + q] * go->w[c];
                            }
                    }
                }
            }
        }
    }
    for (unsigned b = 0; b < nc; b++) free(gos[b].Z);
    for (int t = 0; t < nt; t++) free(scr[t]);
    free(scr); free(gos); free(rows); free(cols); free(cx); free(act);
    if (!dbg_count) free(bm_count);
    if (!dbg_idx) free(bm_idx);
    if (!dbg_first) free(st_first);
    if (!dbg_shape) free(st_shape);
    return 0;
}

/* ------------------------------------------------------------------------------------------ */
/* step drivers, nb_threads == 1 semantics (bm5d.cpp:165-407 and :861-1106)                     */
/* ------------------------------------------------------------------------------------------ */
static int run_step(int step, float sigma, float lambda, float *noisy, const unsigned *mask, float *basic, float *denoised,
                    unsigned ang_major, unsigned awidth, unsigned aheight, unsigned an, unsigned width, unsigned height,
                    unsigned chnls, unsigned N, unsigned nSim, unsigned nDisp, unsigned k, unsigned p, unsigned tau_2D,
                    unsigned tau_4D, unsigned tau_5D, unsigned color_space, unsigned *sched, unsigned max_sched,
                    unsigned *n_sched, unsigned max_passes)
{
    const unsigned asize = awidth * aheight, asw = 2 * an + 1, Aw = asw * asw;
    const unsigned cs = aheight / 2, ct = awidth / 2;
    const unsigned cst = ang_major == ORC_ROWMAJOR ? cs * awidth + ct : cs + ct * aheight;
    if (asw > aheight || asw > awidth) return 1;
    const unsigned n = nSim + nDisp, w_b = width + 2 * n, h_b = height + 2 * n;
    const size_t each = (size_t) width * height * chnls, each_b = (size_t) w_b * h_b * chnls;
    float *out = step == 1 ? basic : denoised;
    if (n_sched) *n_sched = 0;

    for (unsigned st = 0; st < asize; st++) {
        if (!mask[st]) continue;
        if (orc_color_space_transform(noisy + st * each, color_space, width, height, chnls, 1)) return 1;
        if (step == 2 && orc_color_space_transform(basic + st * each, color_space, width, height, chnls, 1)) return 1;
    }
    float *num = (float *) calloc(asize * each, sizeof(float)), *den = (float *) calloc(asize * each, sizeof(float));
    unsigned *proc = (unsigned *) malloc(sizeof(unsigned) * asize);
    unsigned remaining = 0;
    for (unsigned st = 0; st < asize; st++) { proc[st] = !mask[st]; remaining += proc[st] == 0; }
    const unsigned max_proc = remaining;
    float *nsym = (float *) malloc(sizeof(float) * Aw * each_b), *bsym = step == 2 ? (float *) malloc(sizeof(float) * Aw * each_b) : NULL;
    float *numsym = (float *) malloc(sizeof(float) * Aw * each_b), *densym = (float *) malloc(sizeof(float) * Aw * each_b);
    unsigned *st_idx = (unsigned *) malloc(sizeof(unsigned) * Aw), *mask_asw = (unsigned *) malloc(sizeof(unsigned) * Aw),
             *proc_asw = (unsigned *) malloc(sizeof(unsigned) * Aw);
    int rc = 0;
    unsigned passes = 0;

    while (remaining && rc == 0) {
        unsigned ps, pt, pst = 0;
        if (remaining == max_proc && mask[cst]) { ps = cs; pt = ct; }
        else {
            long best = -1;
            for (unsigned st = 0; st < asize; st++) {
                if (proc[st]) continue;
                long z = 0;
                const float *d = den + st * each;
                for (size_t t = 0; t < each; t++) z += d[t] == 0.0;
                if (z >= best) { pst = st; best = z; }
            }
            if (ang_major == ORC_ROWMAJOR) { ps = pst / awidth; pt = pst - ps * awidth; }
            else { pt = pst / aheight; ps = pst - pt * aheight; }
        }
        int cs_asw, min_s, max_s, ct_asw, min_t, max_t;
        orc_angular_search_window(&cs_asw, &min_s, &max_s, ps, aheight, an);
        orc_angular_search_window(&ct_asw, &min_t, &max_t, pt, awidth, an);
        const unsigned cst_asw = ang_major == ORC_ROWMAJOR ? (unsigned) cs_asw * asw + ct_asw : (unsigned) cs_asw + (unsigned) ct_asw * asw;
        for (unsigned s_a = 0; s_a < asw; s_a++)
            for (unsigned t_a = 0; t_a < asw; t_a++) {
                const unsigned s = s_a + min_s, t = t_a + min_t;
                if (ang_major == ORC_ROWMAJOR) st_idx[s_a * asw + t_a] = s * awidth + t;
                else st_idx[s_a + t_a * asw] = s + t * aheight;
            }
        unsigned n_unproc = 0;
        unsigned tau4 = tau_4D;
        for (unsigned a = 0; a < Aw; a++) {
            const unsigned st = st_idx[a];
            mask_asw[a] = mask[st];
            proc_asw[a] = !mask[st];
            n_unproc += mask[st] != 0;
            if (mask[st]) {
                orc_symetrize(noisy + st * each, nsym + a * each_b, width, height, chnls, n);
                if (step == 2) orc_symetrize(basic + st * each, bsym + a * each_b, width, height, chnls, n);
                orc_symetrize(num + st * each, numsym + a * each_b, width, height, chnls, n);
                orc_symetrize(den + st * each, densym + a * each_b, width, height, chnls, n);
            }
        }
        if (n_unproc != Aw && tau4 == ORC_DCT) tau4 = ORC_SADCT;   /* bm5d.cpp:276-280 */
        const unsigned max_unproc = n_unproc;
        unsigned calls = 0;
        while (n_unproc && rc == 0) {
            unsigned pst_asw = 0;
            if (n_unproc == max_unproc && mask_asw[cst_asw]) pst_asw = cst_asw;
            else {   /* the unprocessed SAI of the window with the most zero weights in its padded den, ties to the highest slot */
                int best = -1;
                for (unsigned a = 0; a < Aw; a++) {
                    if (proc_asw[a]) continue;
                    int z = 0;
                    const float *d = densym + a * each_b;
                    for (size_t t = 0; t < each_b; t++) z += d[t] == 0.0;
                    if (z >= best) { pst_asw = a; best = z; }
                }
            }
            rc = orc_pass_ex(step, sigma, lambda, nsym, bsym, numsym, densym, mask_asw, proc_asw, cst_asw, pst_asw, asw, w_b, h_b, chnls,
                             nSim, nDisp, k, N, p, color_space, tau_2D, tau4, tau_5D, NULL, NULL, NULL, NULL);
            if (rc) break;
            calls++;
            proc_asw[pst_asw] += 1;
            proc[st_idx[pst_asw]] += 1;
            const float pct = orc_LF_denoised_percent(densym, mask_asw, Aw, width, height, chnls, n, k);
            if (pct >= 100.0f)
                for (unsigned a = 0; a < Aw; a++)
                    if (proc_asw[a] == 0) { proc_asw[a] += 1; proc[st_idx[a]] += 1; }
            n_unproc = 0;
            for (unsigned a = 0; a < Aw; a++) n_unproc += proc_asw[a] == 0;
        }
        if (sched && n_sched && *n_sched < max_sched) {
            unsigned *e = sched + 4 * (*n_sched);
            e[0] = st_idx[cst_asw]; e[1] = (unsigned) min_s; e[2] = (unsigned) min_t; e[3] = calls;
            (*n_sched)++;
        }
        for (unsigned a = 0; a < Aw; a++) {
            const unsigned st = st_idx[a];
            if (!mask[st]) continue;
            orc_unsymetrize(num + st * each, numsym + a * each_b, width, height, chnls, n);
            orc_unsymetrize(den + st * each, densym + a * each_b, width, height, chnls, n);
        }
        remaining = 0;
        for (unsigned st = 0; st < asize; st++) remaining += proc[st] == 0;
        passes++;
        if (max_passes && passes >= max_passes) break;
    }
    if (rc == 0) {
        const float *sub = step == 1 ? noisy : basic;
        for (unsigned st = 0; st < asize; st++) {
            if (!mask[st]) continue;
            for (size_t t = 0; t < each; t++) {
                const size_t o = st * each + t;
                out[o] = den[o] ? num[o] / den[o] : sub[o];
            }
        }
        for (unsigned st = 0; st < asize; st++) {
            if (!mask[st]) continue;
            orc_color_space_transform(out + st * each, color_space, width, height, chnls, 0);
            if (step == 2) orc_color_space_transform(basic + st * each, color_space, width, height, chnls, 0);
            orc_color_space_transform(noisy + st * each, color_space, width, height, chnls, 0);
        }
    }
    free(num); free(den); free(proc); free(nsym); free(bsym); free(numsym); free(densym); free(st_idx); free(mask_asw); free(proc_asw);
    return rc;
}

int orc_run_step1(float sigma, float lambda, float *noisy, const unsigned *mask, float *basic, unsigned ang_major,
                  unsigned awidth, unsigned aheight, unsigned an, unsigned width, unsigned height, unsigned chnls,
                  unsigned N, unsigned nSim, unsigned nDisp, unsigned k, unsigned p, unsigned tau_2D, unsigned tau_4D,
                  unsigned tau_5D, unsigned color_space, unsigned *sched, unsigned max_sched, unsigned *n_sched, unsigned max_passes)
{
    return run_step(1, sigma, lambda, noisy, mask, basic, NULL, ang_major, awidth, aheight, an, width, height, chnls, N, nSim,
                    nDisp, k, p, tau_2D, tau_4D, tau_5D, color_space, sched, max_sched, n_sched, max_passes);
}
int orc_run_step2(float sigma, float *noisy, const unsigned *mask, float *basic, float *denoised, unsigned ang_major,
                  unsigned awidth, unsigned aheight, unsigned an, unsigned width, unsigned height, unsigned chnls,
                  unsigned N, unsigned nSim, unsigned nDisp, unsigned k, unsigned p, unsigned tau_2D, unsigned tau_4D,
                  unsigned tau_5D, unsigned color_space, unsigned *sched, unsigned max_sched, unsigned *n_sched, unsigned max_passes)
{
    return run_step(2, sigma, 0.0f, noisy, mask, basic, denoised, ang_major, awidth, aheight, an, width, height, chnls, N, nSim,
                    nDisp, k, p, tau_2D, tau_4D, tau_5D, color_space, sched, max_sched, n_sched, max_passes);
}

/* ------------------------------------------------------------------------------------------ */
/* noise + PSNR                                                                                */
/* ------------------------------------------------------------------------------------------ */
/* MT19937 (Matsumoto & Nishimura 2002, the generator of mt19937ar.c:60-160), init_genrand + genrand_res53 */
static unsigned long g_mt[624];
static int g_mti = 625;
void orc_mt_seed(unsigned long s)
{
    g_mt[0] = s & 0xffffffffUL;
    for (g_mti = 1; g_mti < 624; g_mti++) {
        g_mt[g_mti] = (1812433253UL * (g_mt[g_mti - 1] ^ (g_mt[g_mti - 1] >> 30)) + (unsigned long) g_mti);
        g_mt[g_mti] &= 0xffffffffUL;
    }
}
static unsigned long mt_int32(void)
{
    static const unsigned long mag01[2] = { 0x0UL, 0x9908b0dfUL };
    unsigned long y;
    if (g_mti >= 624) {
        int kk;
        if (g_mti == 625) orc_mt_seed(5489UL);
        for (kk = 0; kk < 624 - 397; kk++) {
            y = (g_mt[kk] & 0x80000000UL) | (g_mt[kk + 1] & 0x7fffffffUL);
            g_mt[kk] = g_mt[kk + 397] ^ (y >> 1) ^ mag01[y & 0x1UL];
        }
        for (; kk < 623; kk++) {
            y = (g_mt[kk] & 0x80000000UL) | (g_mt[kk + 1] & 0x7fffffffUL);
            g_mt[kk] = g_mt[kk + (397 - 624)] ^ (y >> 1) ^ mag01[y & 0x1UL];
        }
        y = (g_mt[623] & 0x80000000UL) | (g_mt[0] & 0x7fffffffUL);
        g_mt[623] = g_mt[396] ^ (y >> 1) ^ mag01[y & 0x1UL];
        g_mti = 0;
    }
    y = g_mt[g_mti++];
    y ^= (y >> 11);
    y ^= (y << 7) & 0x9d2c5680UL;
    y ^= (y << 15) & 0xefc60000UL;
    y ^= (y >> 18);
    return y & 0xffffffffUL;
}
double orc_mt_res53(void)
{
    const unsigned long a = mt_int32() >> 5, b = mt_int32() >> 6;
    return (1.0 * a * 67108864.0 + b) * (1.0 / 9007199254740992.0);
}
/* utilities.cpp:177-184 with a caller-chosen seed instead of time+pid (utilities.cpp:165-175) */
void orc_add_noise(const float *img, float *out, size_t n, float sigma, unsigned long seed)
{
    orc_mt_seed(seed);
    for (size_t k = 0; k < n; k++) {
        const double a = orc_mt_res53();
        const double b = orc_mt_res53();
        const double z = (double) (sigma) * sqrt(-2.0 * log(a)) * cos(2.0 * M_PI * b);
        out[k] = img[k] + (float) z;
    }
}
/* utilities.cpp:412-435 */
void orc_psnr(const float *a, const float *b, size_t n, float *psnr, float *rmse)
{
    float tmp = 0.0f;
    for (size_t k = 0; k < n; k++) tmp += (a[k] - b[k]) * (a[k] - b[k]);
    *rmse = sqrtf(tmp / (float) n);
    *psnr = 20.0f * log10f(255.0f / (*rmse));
}

/* ------------------------------------------------------------------------------------------ */
/* per-SAI BM3D (bm3d_LF.cpp:69-122 -> bm3d.cpp:86-287, nb_threads == 1): the A = 1, no-disparity,   */
/* Hadamard specialisation of a window pass with BM3D's own thresholds                              */
/* ------------------------------------------------------------------------------------------ */
/* bm3d.cpp:1187-1330 is the self block matching with search radius = border */
void orc_bm3d_bm(const float *img, unsigned width, unsigned height, unsigned kHW, unsigned NHW, unsigned nHW,
                 unsigned pHW, float tauMatch, unsigned *out_count, unsigned *out_idx, unsigned maxN)
{
    orc_bm_self(img, width, height, kHW, NHW, nHW, nHW, pHW, tauMatch, out_count, out_idx, maxN);
}

int orc_run_bm3d_LF(float sigma, float *noisy, const unsigned *mask, float *basic, float *denoised, unsigned asize,
                    unsigned width, unsigned height, unsigned chnls, unsigned nHard, unsigned nWien, unsigned kHard,
                    unsigned kWien, unsigned NHard, unsigned NWien, unsigned pHard, unsigned pWien,
                    unsigned tau_2D_hard, unsigned tau_2D_wien, float lambdaHard3D, unsigned color_space)
{
    if (nHard != nWien || NHard < 2 || NWien < 2) return 1;      /* bm3d.cpp:175 passes the nHard-padded buffers with nWien */
    if ((tau_2D_hard != ORC_DCT && tau_2D_hard != ORC_BIOR) || (tau_2D_wien != ORC_DCT && tau_2D_wien != ORC_BIOR)) return 1;
    const size_t each = (size_t) width * height * chnls;
    const unsigned w_b = width + 2 * nHard, h_b = height + 2 * nHard;
    const size_t each_b = (size_t) w_b * h_b * chnls;
    float *nsym = (float *) malloc(sizeof(float) * each_b), *bsym = (float *) malloc(sizeof(float) * each_b);
    float *num = (float *) malloc(sizeof(float) * each_b), *den = (float *) malloc(sizeof(float) * each_b);
    const unsigned one = 1, zero = 0;
    int rc = 0;
    g_bm3d = 1;
    for (unsigned st = 0; st < asize && rc == 0; st++) {
        if (!mask[st]) continue;
        float *nz = noisy + st * each, *bs = basic + st * each, *dn = denoised + st * each;
        if (orc_color_space_transform(nz, color_space, width, height, chnls, 1)) { rc = 1; break; }      /* bm3d.cpp:117 */
        orc_symetrize(nz, nsym, width, height, chnls, nHard);
        memset(num, 0, sizeof(float) * each_b); memset(den, 0, sizeof(float) * each_b);
        rc = orc_pass(1, sigma, lambdaHard3D, nsym, NULL, num, den, &one, &zero, 0, 1, w_b, h_b, chnls, nHard, 0, kHard, NHard, pHard,
                      color_space, tau_2D_hard, ORC_ID, ORC_HADAMARD, NULL, NULL, NULL, NULL);
        if (rc) break;
        for (size_t t = 0; t < each_b; t++) num[t] = num[t] / den[t];                                    /* bm3d.cpp:476-477 */
        orc_unsymetrize(bs, num, width, height, chnls, nHard);
        orc_symetrize(bs, bsym, width, height, chnls, nHard);                                            /* bm3d.cpp:152-160 */
        memset(num, 0, sizeof(float) * each_b); memset(den, 0, sizeof(float) * each_b);
        rc = orc_pass(2, sigma, 0.0f, nsym, bsym, num, den, &one, &zero, 0, 1, w_b, h_b, chnls, nWien, 0, kWien, NWien, pWien,
                      color_space, tau_2D_wien, ORC_ID, ORC_HADAMARD, NULL, NULL, NULL, NULL);
        if (rc) break;
        for (size_t t = 0; t < each_b; t++) num[t] = num[t] / den[t];                                    /* bm3d.cpp:682-683 */
        orc_unsymetrize(dn, num, width, height, chnls, nWien);
        orc_color_space_transform(dn, color_space, width, height, chnls, 0);                             /* bm3d.cpp:269-274 */
        orc_color_space_transform(nz, color_space, width, height, chnls, 0);
        orc_color_space_transform(bs, color_space, width, height, chnls, 0);
    }
    g_bm3d = 0;
    free(nsym); free(bsym); free(num); free(den);
    return rc;
}
