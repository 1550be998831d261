// Block matching: exact float32 summed-area recurrences (a warp sweeps two offset planes as a skewed
// wavefront), top-N selection for self similarity and argmin for disparity matching, with the libstdc++
// sort algorithms emulated where exact float ties make the reference's result algorithm-dependent.
//
// Reference behaviour restated: precompute_BM (bm5d_core_processing.cpp:3301-3461) and precompute_BM_stereo
// (:3479-3611): per offset, a table of squared differences, then patch sums by the recurrence
//   s[k] = s[k-1] + s[k-w] - s[k-1-w] + d[pq] - d[pq-kHW] - d[pq-kHW*w] + d[pq-kHW-kHW*w]
// evaluated left to right in float, with dedicated formulas for the first patch, first row and first column.
// The rounding of that recurrence decides ~1 % of the match lists, so it is reproduced operation for operation.
#pragma once
#include "common.cuh"
#include <cuda.h>

// ---- geometry shared by all planes of one launch ----
struct SatGeom {
    int w, h, k;
    int lo;                 // first row/column of the summed region
    int row_end, col_end;   // one past its last row/column
    int ylim, xlim;         // squared differences are zero for rows >= ylim or columns >= xlim (self: dim - nHW)
    int nstrips;            // 32-column strips
    int pstrips;            // strips per plane in the hand-off buffers (bnd / progress): the same for every launch that
                            // shares them, so that disjoint plane ids give disjoint ranges (>= nstrips)
    int SR;                 // skewed rows per strip in the stereo output: (row_end - lo) + 31
    int nc;                 // number of reference-patch columns (self)
    const int *rowmap;      // [h] row -> reference row index or -1 (self)
    const int *colmap;      // [w]
    int gp, nreg, rlast, nr;     // reference rows (self): lo + a*gp for a < nreg, plus rlast (index nr-1)
    unsigned long long negzero2; // packed (-0.f, -0.f) supplied at run time (see lf_mul2)
    unsigned epoch;         // launch counter: tags the boundary words of this launch (stale words of earlier launches never match)
    const float *frow;      // [plane][w] first row of every plane's sums, [plane][h] first column (k_sat_edges)
    const float *fcol;
};
// One offset plane: d(y,x) = (img2[y+oy][x+ox] - img1[y][x])^2, oy shared by the group.
struct SatPlane {
    int    ox;
    float *out_skew;        // stereo: sums in skewed layout [strip][sidx][lane], sidx = (i - lo) + lane
    float *out_at;          // self: sums sampled at the reference patches, [nr*nc]
    float *out_mir;         // self: sums sampled at (ref - (mir_di, -mir_dc)) (pre-filled with 2*threshold)
    int    mir_di, mir_dc;
};
// Up to 2*SAT_NW planes that share the two source images and the row offset: one CTA per (group, strip).
#define SAT_NW 7          // warps per CTA; each warp sweeps two planes
#define SAT_SUB 8         // steps per hand-off between neighbouring strips
struct SatGroup {
    const float *img1, *img2;
    int oy, oxmin, nplanes, first_plane;
    int z1, z2;             // plane indices of img1 / img2 in the tensor map of the estimate planes (TMA path)
};

// ---- TMA (cp.async.bulk.tensor) + mbarrier, as used for the source-row rings of k_sat2 ----
__device__ __forceinline__ void lf_mbar_init(unsigned long long *bar, unsigned count)
{
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;\n" ::"r"((unsigned) __cvta_generic_to_shared(bar)), "r"(count) : "memory");
    asm volatile("fence.mbarrier_init.release.cluster;\n" ::: "memory");
}
__device__ __forceinline__ void lf_mbar_expect_tx(unsigned long long *bar, unsigned bytes)
{
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;\n" ::"r"((unsigned) __cvta_generic_to_shared(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void lf_mbar_wait(unsigned long long *bar, unsigned parity)
{
    const unsigned a = (unsigned) __cvta_generic_to_shared(bar);
    unsigned done;
    do {
        asm volatile("{\n .reg .pred p;\n mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n selp.u32 %0, 1, 0, p;\n}\n"
                     : "=r"(done) : "r"(a), "r"(parity) : "memory");
    } while (!done);
}
// one box of the 3-D tensor (x, y, plane) into shared memory; elements outside the tensor arrive as zeros
__device__ __forceinline__ void lf_tma_load_3d(float *smem_dst, const CUtensorMap *map, unsigned long long *bar, int x, int y, int z)
{
    asm volatile("cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];\n"
                 ::"r"((unsigned) __cvta_generic_to_shared(smem_dst)), "l"(map), "r"((unsigned) __cvta_generic_to_shared(bar)), "r"(x), "r"(y), "r"(z)
                 : "memory");
}

template <int IMM> __device__ __forceinline__ float lf_lds(unsigned addr)
{
    float v;
    asm volatile("ld.shared.f32 %0, [%1+%2];\n" : "=f"(v) : "r"(addr), "n"(IMM));
    return v;
}

// Summed-area planes. Work unit = (group of <= 2 * SAT_NW planes sharing their source rows, 32-column strip). A warp sweeps
// TWO planes (column offsets ox and ox + 1 of the group): lane l owns column c0 + l and runs one row behind lane l - 1 (skewed
// wavefront, one 64-bit shuffle per step); the img1 operand is shared, the img2 operands are adjacent ring entries, and all
// floating-point work of a step runs as packed FP32x2 instructions (bit-identical per half).
// The strips of a plane are pipelined across CTAs: strip c consumes the last column of strip c - 1 through global memory with
// tagged 64-bit words (see the hand-off comment in the kernel), and CTAs take their work from a ticket counter in strip-major order so that a producer
// has always started before its consumer (no deadlock). Source rows of both images are staged once per CTA with cp.async
// into two 128(+K)-row shared-memory rings (row stride 64 floats: the skewed reads are bank-conflict free) and reused by all
// planes of the group; squared differences are formed on the fly.
// TMA: the source rows arrive as 8-row x 64-column boxes of the estimate planes (cp.async.bulk.tensor, one elected thread, an
// mbarrier per CTA; out-of-image elements are zero-filled by the hardware) instead of 4-byte cp.async copies issued by every thread;
// needs a 16-byte multiple as the row pitch of the planes (the host picks the variant).
template <bool SELF, int K, bool TMA>
__global__ void __launch_bounds__(SAT_NW * 32, 3) k_sat2(SatGeom g, const SatGroup *__restrict__ groups, const SatPlane *__restrict__ planes,
                                                          int ngroups, unsigned long long *bnd, int *ticket_counter,
                                                          const __grid_constant__ CUtensorMap tmap)
{
    extern __shared__ __align__(128) float s_dyn[];
    __shared__ __align__(8) unsigned long long s_mbar;
    // source-row rings of img1 / img2: 128 rows + K mirror rows (slot s < K is also stored at s + 128, so that the
    // row K below any slot is always at slot + K without wrapping)
    float *R1 = s_dyn, *R2 = s_dyn + (128 + K) * 64;
    __shared__ int s_ticket;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const unsigned FULL = 0xffffffffu;
    if (tid == 0) s_ticket = atomicAdd(ticket_counter, 1);
    __syncthreads();
    const int strip = s_ticket / ngroups, gi = s_ticket - strip * ngroups;
    const SatGroup G = groups[gi];
    const bool hasplane = 2 * warp < G.nplanes;
    const bool hasB = 2 * warp + 1 < G.nplanes;
    const int pid = G.first_plane + (hasplane ? 2 * warp : 0);        // plane A; plane B = pid + 1 (A again when absent)
    const SatPlane PA = planes[pid], PB = planes[hasB ? pid + 1 : pid];
    const int w = g.w, h = g.h, lo = g.lo;
    constexpr int k = K;
    const int W = g.col_end - lo, Hh = g.row_end - lo;
    const int c0 = lo + (strip << 5);
    const int j = c0 + lane;
    const bool valid = hasplane && j < g.col_end;
    const int lastlane = min(31, W - 1 - (strip << 5));
    const bool has_next = strip + 1 < g.nstrips;
    const int xb1 = c0 - 1, xb2 = c0 - 1 + G.oxmin;
    // TMA boxes start at a 16-byte multiple of the row (an unaligned innermost coordinate faults, tools/probe/tma_probe.cu): the
    // box starts up to three columns early and the lanes read at that shift; img2 needs 32 + 13 + K <= 61 columns, so 64 still do
    const int xs1 = TMA ? (xb1 & 3) : 0, xs2 = TMA ? (xb2 & 3) : 0;
    const int oxo = PA.ox - G.oxmin;                   // column shift of plane A inside the img2 ring (plane B: +1)
    const int ymax = min(g.row_end - 1 + k - 1, h - 1);
    const size_t pstride = (size_t) g.pstrips * h;
    // hand-off words of the last column of a strip: [plane][strip][row] = (sum, epoch << 16 | row)
    const unsigned long long *bnd_prev = bnd + (size_t) pid * pstride + (size_t) (strip > 0 ? strip - 1 : 0) * h;
    unsigned long long *bnd_next = bnd + (size_t) pid * pstride + (size_t) strip * h;
    const size_t bB = hasB ? pstride : 0;              // offset from plane A's boundary column to plane B's
    const unsigned tag_hi = g.epoch << 16;

    // ring slot of source row y of img1 (and of row y + oy of img2): counted from row lo + k, so that the 32-row loads of the
    // chunks start at multiples of 32 (no box straddles the end of the ring)
    const int rbase = lo + k;
    unsigned mbar_parity = 0;
    auto load_rows = [&](int y0, int y1) {
        if (TMA) {
            if (y0 > ymax) return;
            if (tid == 0) {
                const int nbox = (y1 - y0 + 1) >> 3;
                int nmir = 0;
                for (int b = 0; b < nbox; ++b) nmir += (((y0 + 8 * b - rbase) & 127) < K) ? 1 : 0;
                lf_mbar_expect_tx(&s_mbar, (unsigned) (2 * (nbox + nmir)) * 8u * 64u * 4u);
                for (int b = 0; b < nbox; ++b) {
                    const int y = y0 + 8 * b, sl = (y - rbase) & 127;
                    lf_tma_load_3d(R1 + sl * 64, &tmap, &s_mbar, xb1 - xs1, y, G.z1);
                    lf_tma_load_3d(R2 + sl * 64, &tmap, &s_mbar, xb2 - xs2, y + G.oy, G.z2);
                    if (sl < K) {
                        lf_tma_load_3d(R1 + (sl + 128) * 64, &tmap, &s_mbar, xb1 - xs1, y, G.z1);
                        lf_tma_load_3d(R2 + (sl + 128) * 64, &tmap, &s_mbar, xb2 - xs2, y + G.oy, G.z2);
                    }
                }
            }
            return;
        }
        if (y1 > ymax) y1 = ymax;
        const int n = (y1 - y0 + 1) * 128;
        for (int t = tid; t < n; t += blockDim.x) {
            const int y = y0 + (t >> 7), c = t & 63, which = (t >> 6) & 1;
            if (which == 0) {
                const int x = xb1 + c, sl = (y - rbase) & 127;
                float *dst = &R1[sl * 64 + c];
                if (x < w) {
                    lf_cp_async4(dst, G.img1 + (size_t) y * w + x);
                    if (sl < K) lf_cp_async4(dst + 128 * 64, G.img1 + (size_t) y * w + x);
                } else { *dst = 0.f; if (sl < K) dst[128 * 64] = 0.f; }
            } else {
                const int yy = y + G.oy, x = xb2 + c, sl = (y - rbase) & 127;
                float *dst = &R2[sl * 64 + c];
                if (yy >= 0 && yy < h && x >= 0 && x < w) {
                    lf_cp_async4(dst, G.img2 + (size_t) yy * w + x);
                    if (sl < K) lf_cp_async4(dst + 128 * 64, G.img2 + (size_t) yy * w + x);
                } else { *dst = 0.f; if (sl < K) dst[128 * 64] = 0.f; }
            }
        }
    };
    // per-lane constants of the sampled outputs (self) / the skewed output pointers (stereo)
    int colb = -1, colbA2 = -1, colbB2 = -1;
    float *outA = nullptr, *outB = nullptr;
    if (SELF) {
        if (j < w) colb = g.colmap[j];
        const int jA = j - PA.mir_dc, jB = j - PB.mir_dc;
        if (PA.mir_di > 0 && jA >= 0 && jA < w) colbA2 = g.colmap[jA];
        if (PB.mir_di > 0 && jB >= 0 && jB < w && hasB) colbB2 = g.colmap[jB];
    } else {
        outA = PA.out_skew + ((size_t) strip * g.SR) * 32 + lane;      // + sidx*32, sidx = (i - lo) + lane
        outB = PB.out_skew + ((size_t) strip * g.SR) * 32 + lane;
    }
    // reference-row index of row i (or -1), by arithmetic (self planes)
    auto row_index = [&](int i) -> int {
        const int d = i - lo;
        if (i == g.rlast) return g.nr - 1;
        if (d >= 0 && d % g.gp == 0 && d / g.gp < g.nreg) return d / g.gp;
        return -1;
    };
    auto emit_self = [&](int a, int a2, float vA, float vB) {     // a / a2: reference-row index of rows i and i + mir_di
        if (a >= 0 && colb >= 0) { PA.out_at[a * g.nc + colb] = vA; if (hasB) PB.out_at[a * g.nc + colb] = vB; }
        if (a2 >= 0) {
            if (colbA2 >= 0) PA.out_mir[a2 * g.nc + colbA2] = vA;
            if (colbB2 >= 0) PB.out_mir[a2 * g.nc + colbB2] = vB;
        }
    };
    auto emit = [&](int i, float vA, float vB) {     // cold paths (first row / first column)
        if (SELF) emit_self(row_index(i), PA.mir_di > 0 ? row_index(i + PA.mir_di) : -1, vA, vB);
        else {
            const size_t o = (size_t) ((i - lo) + lane) * 32;
            outA[o] = vA;
            if (hasB) outB[o] = vB;
        }
    };
    // rows the loads of a chunk wait for: cp.async groups of the thread, or the transaction count of the CTA's mbarrier
    auto rows_wait = [&](int y0) {
        if (TMA) { if (y0 <= ymax) { lf_mbar_wait(&s_mbar, mbar_parity); mbar_parity ^= 1u; } }
        else lf_cp_async_wait_all();
    };
    // ---- prologue: source rows of chunk 0; the first row of the sums comes from k_sat_edges ----
    if (TMA) { if (tid == 0) lf_mbar_init(&s_mbar, 1); __syncthreads(); }
    load_rows(lo, lo + 32 + k - 1);
    rows_wait(lo);
    __syncthreads();

    float curv[2] = { 0.f, 0.f }, prevv[2] = { 0.f, 0.f };
    if (hasplane) {
        const float *frA = g.frow + (size_t) pid * w, *frB = g.frow + (size_t) (hasB ? pid + 1 : pid) * w;
        if (j < g.col_end) { curv[0] = __ldg(frA + j); curv[1] = __ldg(frB + j); }
        if (j - 1 >= lo && j - 1 < g.col_end) { prevv[0] = __ldg(frA + j - 1); prevv[1] = __ldg(frB + j - 1); }      // s(lo, j-1); lane 0 of strip 0: unused
        if (valid) emit(lo, curv[0], curv[1]);
    }

    // ---- wavefront over the remaining rows in chunks of 32 steps (core:3365-3387 / :3550-3572) ----
    // Per lane, ro1 / ro2 = byte offset of the ring row holding source row i-1 (img1) / i-1+oy (img2); source row
    // i+K-1 is K ring rows further (mirror rows: no wrap). Both advance by one ring row (256 B) per step.
    const int nsteps = (Hh - 1) + 31;
    const int nchunks = (nsteps + 31) >> 5;
    const unsigned sb1 = (unsigned) __cvta_generic_to_shared(R1) + 4u * (unsigned) (lane + xs1);
    const unsigned sb2 = (unsigned) __cvta_generic_to_shared(R2) + 4u * (unsigned) (lane + oxo + xs2);
    unsigned ro1 = (unsigned) (((lo + 1 - lane - 1 - rbase) & 127) * 256);
    unsigned ro2 = ro1;      // both rings are indexed by the img1 row
    const bool colz = SELF && (j + k - 1 >= g.xlim);
    // lane 0 of strip 0 owns the first column of the plane: its sums come from k_sat_edges (through the same per-chunk staging the
    // other strips use for the last column of their predecessor) and replace what the general recurrence would give
    const bool lane0 = lane == 0;
    const bool ovr = strip == 0 && lane0;
    // lane is active at steps s in [lane + 1, lane + Hh - 1]
    const unsigned s_first = valid ? (unsigned) (lane + 1) : 0x40000000u;
    const unsigned s_span = (unsigned) (Hh - 1);
    const bool bstore = has_next && lane == 31;
    unsigned long long *bpA = bnd_next + (lo - lane) + 1, *bpB = bpA + bB;       // running: bnd_next[i] of the current step
    unsigned btag = tag_hi | (unsigned) ((lo - lane + 1) & 0xffff);               // running: its tag
    float *opA = outA + 32, *opB = outB + 32;                       // running: skewed output slot of the current step
    // reference-row counters (self): phase and index of rows i and i + mir_di, advanced with the step
    int ph1 = 0, ai1 = 0, ph2 = 0, ai2 = 0;
    if (SELF) {
        const int v1 = 1 - lane + 64 * g.gp, v2 = v1 + PA.mir_di;
        ph1 = v1 % g.gp; ai1 = v1 / g.gp - 64;
        ph2 = v2 % g.gp; ai2 = v2 / g.gp - 64;
    }
    const unsigned long long nz2 = g.negzero2;
    unsigned long long cur2 = lf_pk(curv[0], curv[1]), prevL2 = lf_pk(prevv[0], prevv[1]);
    auto step_general = [&](int s, unsigned long long Lin2) {
        if ((unsigned) s - s_first < s_span) {
            const unsigned a1 = sb1 + ro1, a2 = sb2 + ro2;
            const float aNK = lf_lds<K * 256 + K * 4>(a1), aN0 = lf_lds<K * 256>(a1), aOK = lf_lds<K * 4>(a1), aO0 = lf_lds<0>(a1);
            unsigned long long t1 = lf_sub2(lf_pk(lf_lds<K * 256 + K * 4>(a2), lf_lds<K * 256 + K * 4 + 4>(a2)), lf_pk(aNK, aNK));
            unsigned long long t2 = lf_sub2(lf_pk(lf_lds<K * 256>(a2), lf_lds<K * 256 + 4>(a2)), lf_pk(aN0, aN0));
            unsigned long long t3 = lf_sub2(lf_pk(lf_lds<K * 4>(a2), lf_lds<K * 4 + 4>(a2)), lf_pk(aOK, aOK));
            unsigned long long t4 = lf_sub2(lf_pk(lf_lds<0>(a2), lf_lds<4>(a2)), lf_pk(aO0, aO0));
            t1 = lf_mul2(t1, t1, nz2); t2 = lf_mul2(t2, t2, nz2); t3 = lf_mul2(t3, t3, nz2); t4 = lf_mul2(t4, t4, nz2);
            if (SELF) {
                const bool rowz = lo + s - lane + k - 1 >= g.ylim;
                if (rowz || colz) t1 = 0ull;
                if (rowz) t2 = 0ull;
                if (colz) t3 = 0ull;
            }
            unsigned long long nv = lf_add2(Lin2, cur2);
            nv = lf_sub2(nv, prevL2);
            nv = lf_add2(nv, t1);
            nv = lf_sub2(nv, t2);
            nv = lf_sub2(nv, t3);
            nv = lf_add2(nv, t4);
            if (ovr) nv = Lin2;
            prevL2 = Lin2;
            cur2 = nv;
            float vA, vB;
            lf_upk(nv, vA, vB);
            if (SELF) {
                const int i = lo + s - lane;
                const int a = (i == g.rlast) ? g.nr - 1 : ((ph1 == 0 && ai1 < g.nreg) ? ai1 : -1);
                const int a2 = (i + PA.mir_di == g.rlast) ? g.nr - 1 : ((ph2 == 0 && ai2 < g.nreg) ? ai2 : -1);
                if ((a >= 0) | (a2 >= 0)) emit_self(a, PA.mir_di > 0 ? a2 : -1, vA, vB);
            } else {
                *opA = vA;
                if (hasB) *opB = vB;
            }
            if (bstore) {
                lf_st_relaxed64(bpA, ((unsigned long long) btag << 32) | __float_as_uint(vA));
                if (hasB) lf_st_relaxed64(bpB, ((unsigned long long) btag << 32) | __float_as_uint(vB));
            }
        }
        ro1 = (ro1 + 256u) & 32767u;
        ro2 = (ro2 + 256u) & 32767u;
        ++bpA; ++bpB;
        btag = tag_hi | ((btag + 1u) & 0xffffu);
        if (SELF) {
            if (++ph1 == g.gp) { ph1 = 0; ++ai1; }
            if (++ph2 == g.gp) { ph2 = 0; ++ai2; }
        } else { opA += 32; opB += 32; }
    };
    // Hand-off between the strips of a plane: lane 31 of the producer writes the sums of its last column as 64-bit (value, tag)
    // words, tag = (launch epoch, row); the consumer stages the SAT_SUB pairs of its next sub-chunk of steps in shared memory (lane 0
    // reads one pair per step), fetching them one sub-chunk ahead and re-reading only the words whose tag is not there yet. A
    // 64-bit access is single-copy atomic: the matching tag guarantees the value, without flags or fences. A strip runs about
    // 31 (skew of the wavefront) + 2 * SAT_SUB steps behind its predecessor. Strip 0 takes the plane's first column (k_sat_edges)
    // through the same staging.
    constexpr int SUB = SAT_SUB;
    __shared__ unsigned long long s_bnd[SAT_NW][2][SUB];
    const unsigned sbn = (unsigned) __cvta_generic_to_shared(&s_bnd[warp][0][0]);
    const float *fcA = g.fcol + (size_t) pid * h, *fcB = fcA + (hasB ? (size_t) h : 0);
    // boundary pair of this lane's row of sub-chunk v; *ok = both tags matched (spin: retry until they do)
    auto sub_fetch = [&](int v, bool spin, bool *ok) -> unsigned long long {
        const int r = lo + SUB * v + 1 + lane;
        *ok = true;
        if (lane >= SUB || r >= g.row_end) return 0ull;
        if (strip == 0) return lf_pk(__ldg(fcA + r), __ldg(fcB + r));
        const unsigned want = tag_hi | (unsigned) (r & 0xffff);
        for (;;) {
            const unsigned long long wa = lf_ld_relaxed64(bnd_prev + r), wb = lf_ld_relaxed64(bnd_prev + r + bB);
            if ((unsigned) (wa >> 32) == want && (unsigned) (wb >> 32) == want)
                return lf_pk(__uint_as_float((unsigned) wa), __uint_as_float((unsigned) wb));
            if (!spin) { *ok = false; return 0ull; }
            __nanosleep(20);
        }
    };
    unsigned long long nb2 = 0ull;
    bool nb_have = false;
    const int nsub = (nsteps + SUB - 1) / SUB;
    for (int q = 0; q < nchunks; ++q) {
        // stage the source rows of the next chunk while this one runs
        load_rows(lo + 32 * (q + 1) + k, lo + 32 * (q + 1) + 32 + k - 1);
        if (hasplane) {
            const int send = min(32 * q + 32, nsteps);
            for (int v = (32 / SUB) * q; v < (32 / SUB) * (q + 1) && SUB * v < send; ++v) {
                const int s0 = SUB * v + 1, s1 = min(SUB * v + SUB, send);
                bool ok;
                if (!nb_have) nb2 = sub_fetch(v, true, &ok);
                if (lane < SUB) s_bnd[warp][v & 1][lane] = nb2;
                __syncwarp();
                nb_have = false;
                if (v + 1 < nsub) {      // one sub-chunk ahead, if the producer is already there
                    nb2 = sub_fetch(v + 1, false, &ok);
                    nb_have = __all_sync(FULL, ok);
                }
                unsigned bo = sbn + (unsigned) (v & 1) * (SUB * 8);
#pragma unroll 2
                for (int s = s0; s <= s1; ++s, bo += 8) {
                    unsigned long long Lin2 = __shfl_up_sync(FULL, cur2, 1);
                    if (lane0) asm volatile("ld.shared.b64 %0, [%1];" : "=l"(Lin2) : "r"(bo));
                    step_general(s, Lin2);
                }
                __syncwarp();
            }
        }
        rows_wait(lo + 32 * (q + 1) + k);
        __syncthreads();
    }
}

// First row and first column of every plane's sums (core:3345-3372 / :3530-3557): the reference's dedicated formulas — the first
// patch as a row-major running sum of its k*k squared differences, then per column j (row i) the running value plus the k
// differences d[.][j-1+k] - d[.][j-1] (d[i-1+k][.] - d[i-1][.]) added strictly in order. These chains of W*k (H*k) dependent float
// additions per plane cannot be shortened, but the planes are independent and the squared differences do not depend on the
// running sums: one CTA per (group of planes sharing their source rows, direction); seven warps produce the squared differences
// of the next 32 positions into shared memory (lanes <-> planes: neighbouring pixels) while lane p of warp 0 runs the chain of
// plane p over the current 32. k_sat2 then starts every strip from these values instead of waiting for the strip to its left.
#define SATE_NT 256
#define SATE_B 32
// dynamic shared memory of k_sat_edges: two difference buffers + the img1 / img2 source tiles
inline size_t sate_smem(int k) { return ((size_t) 2 * (SATE_B + k) * k * 16 + (size_t) (SATE_B + k) * k + (size_t) (SATE_B + k + 16) * (k + 16)) * 4; }
template <bool SELF, int K>
__global__ void __launch_bounds__(SATE_NT) k_sat_edges(SatGeom g, const SatGroup *__restrict__ groups, const SatPlane *__restrict__ planes,
                                                       float *__restrict__ frow, float *__restrict__ fcol)
{
    extern __shared__ float s_d[];                 // two buffers of [SATE_B + K][K][16] squared differences, then the source tiles
    constexpr int NA = SATE_B + K, BUF = NA * K * 16;
    constexpr int T2A = NA + 16, T2C = K + 16;     // img2 tile: room for the 14 column offsets of a group along x
    float *T1 = s_d + 2 * BUF, *T2 = T1 + NA * K;  // img1 tile [a][c]; img2 tile [a2][c2]
    const SatGroup G = groups[blockIdx.x];
    const int dir = blockIdx.y;                    // 0: first row (scan along x), 1: first column (scan along y)
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int w = g.w, h = g.h, lo = g.lo;
    const int end = dir == 0 ? g.col_end : g.row_end;
    const int nblk = (end - lo - 1 + SATE_B - 1) / SATE_B;      // positions lo + 1 .. end - 1; at least one block (first patch)
    const int pl = tid & 15;
    const int e = pl < G.nplanes ? planes[G.first_plane + pl].ox - G.oxmin : 0;      // column shift of the lane's plane inside the img2 tile
    const float *__restrict__ i1 = G.img1, *__restrict__ i2 = G.img2;
    // squared differences of block b: along positions a0 .. a0 + NA - 1 (a0 = lo + b * SATE_B), across lo .. lo + K - 1.
    // The source pixels are staged first (coalesced, all loads of a thread in flight; pixels outside the image read as 0 like the
    // zero fill of k_sat2's row rings), then every (position, plane) difference comes from shared memory.
    auto produce = [&](int b, int first_thread, int nthreads, int barrier_id) {
        float *D = s_d + (b & 1) * BUF;
        const int a0 = lo + b * SATE_B, t0 = tid - first_thread;
        const int n2a = dir == 0 ? T2A : NA, n2c = dir == 0 ? K : T2C;
        for (int t = t0; t < NA * K; t += nthreads) {
            const int a = dir == 0 ? t % NA : t / K, c = dir == 0 ? t / NA : t % K;
            const int y = dir == 0 ? lo + c : a0 + a, x = dir == 0 ? a0 + a : lo + c;
            T1[a * K + c] = (y < h && x < w) ? __ldg(i1 + (size_t) y * w + x) : 0.f;
        }
        for (int t = t0; t < n2a * n2c; t += nthreads) {
            const int a = dir == 0 ? t % n2a : t / n2c, c = dir == 0 ? t / n2a : t % n2c;
            const int y = (dir == 0 ? lo + c : a0 + a) + G.oy, x = (dir == 0 ? a0 + a : lo + c) + G.oxmin;
            T2[a * T2C + c] = (y >= 0 && y < h && x >= 0 && x < w) ? __ldg(i2 + (size_t) y * w + x) : 0.f;
        }
        asm volatile("bar.sync %0, %1;" ::"r"(barrier_id), "r"(nthreads) : "memory");
        for (int t = t0; t < NA * K * 16; t += nthreads) {
            const int ac = t >> 4, a = ac / K, c = ac - a * K;
            if (pl >= G.nplanes) continue;
            const float df = (dir == 0 ? T2[(a + e) * T2C + c] : T2[a * T2C + c + e]) - T1[a * K + c];
            float v = df * df;
            if (SELF) {
                const int y = dir == 0 ? lo + c : a0 + a, x = dir == 0 ? a0 + a : lo + c;
                if (y >= g.ylim || x >= g.xlim) v = 0.f;
            }
            D[t] = v;
        }
    };
    produce(0, 0, SATE_NT, 1);
    __syncthreads();
    float s = 0.0f;
    float *out = nullptr;
    if (warp == 0 && lane < G.nplanes) {
        const float *D = s_d;
        // first patch: row-major over its k x k squared differences (p outer, t inner)
        for (int p = 0; p < K; ++p)
#pragma unroll
            for (int t = 0; t < K; ++t) s += dir == 0 ? D[(t * K + p) * 16 + lane] : D[(p * K + t) * 16 + lane];
        out = dir == 0 ? frow + (size_t) (G.first_plane + lane) * w : fcol + (size_t) (G.first_plane + lane) * h;
        out[lo] = s;
    }
    for (int b = 0; b < nblk; ++b) {
        if (warp == 0) {
            if (lane < G.nplanes) {
                const float *D = s_d + (b & 1) * BUF + lane;
                const int p0 = lo + 1 + b * SATE_B;
                const int np = min(SATE_B, end - p0);
                for (int q = 0; q < np; ++q) {
                    float e[K];
#pragma unroll
                    for (int c = 0; c < K; ++c) e[c] = D[((q + K) * K + c) * 16] - D[(q * K + c) * 16];
#pragma unroll
                    for (int c = 0; c < K; ++c) s += e[c];
                    out[p0 + q] = s;
                }
            }
        } else if (b + 1 < nblk) produce(b + 1, 32, SATE_NT - 32, 2);
        __syncthreads();
    }
}

__global__ void k_fill(float *p, float v, size_t n)
{
    for (size_t t = (size_t) blockIdx.x * blockDim.x + threadIdx.x; t < n; t += (size_t) gridDim.x * blockDim.x) p[t] = v;
}

// ------------------------------------------------------------------------------------------------------------
// libstdc++ (GCC 13 bits/stl_algo.h, bits/stl_heap.h) partial_sort / sort on (distance, index) pairs compared on the
// distance only (bm3d.cpp:1377-1380), restated for one thread. Only executed where exact ties make the reference's
// output depend on the algorithm.
// ------------------------------------------------------------------------------------------------------------
struct LfPair { float d; unsigned i; };
#define LF_LESS(a, b) ((a).d < (b).d)

__device__ inline void lfs_push_heap(LfPair *first, int hole, int top, LfPair value)
{
    int parent = (hole - 1) / 2;
    while (hole > top && LF_LESS(first[parent], value)) {
        first[hole] = first[parent];
        hole = parent;
        parent = (hole - 1) / 2;
    }
    first[hole] = value;
}
__device__ inline void lfs_adjust_heap(LfPair *first, int hole, int len, LfPair value)
{
    const int top = hole;
    int child = hole;
    while (child < (len - 1) / 2) {
        child = 2 * (child + 1);
        if (LF_LESS(first[child], first[child - 1])) child--;
        first[hole] = first[child];
        hole = child;
    }
    if ((len & 1) == 0 && child == (len - 2) / 2) {
        child = 2 * (child + 1);
        first[hole] = first[child - 1];
        hole = child - 1;
    }
    lfs_push_heap(first, hole, top, value);
}
__device__ inline void lfs_make_heap(LfPair *first, int len)
{
    if (len < 2) return;
    int parent = (len - 2) / 2;
    for (;;) {
        const LfPair v = first[parent];
        lfs_adjust_heap(first, parent, len, v);
        if (parent == 0) return;
        parent--;
    }
}
// pop_heap(first, first+len, result): *result receives the top, its old value is sifted in
__device__ inline void lfs_pop_heap(LfPair *first, int len, LfPair *result)
{
    const LfPair v = *result;
    *result = *first;
    lfs_adjust_heap(first, 0, len, v);
}
__device__ inline void lfs_partial_sort(LfPair *first, int middle, int last)
{
    lfs_make_heap(first, middle);
    for (int i = middle; i < last; ++i)
        if (LF_LESS(first[i], first[0])) lfs_pop_heap(first, middle, &first[i]);
    while (middle > 1) { --middle; lfs_pop_heap(first, middle, &first[middle]); }
}
__device__ inline void lfs_swap(LfPair *a, LfPair *b) { const LfPair t = *a; *a = *b; *b = t; }
__device__ inline void lfs_unguarded_linear_insert(LfPair *v, int last)
{
    const LfPair val = v[last];
    int next = last - 1;
    while (LF_LESS(val, v[next])) { v[last] = v[next]; last = next; --next; }
    v[last] = val;
}
__device__ inline void lfs_insertion_sort(LfPair *v, int first, int last)
{
    if (first == last) return;
    for (int i = first + 1; i != last; ++i) {
        if (LF_LESS(v[i], v[first])) {
            const LfPair val = v[i];
            for (int t = i; t > first; --t) v[t] = v[t - 1];
            v[first] = val;
        } else lfs_unguarded_linear_insert(v, i);
    }
}
__device__ inline void lfs_sort(LfPair *v, int n)
{
    if (n == 0) return;
    int lg = 0;
    while ((n >> (lg + 1)) > 0) lg++;
    // introsort loop with an explicit stack for the recursion on the right part
    int stf[64], stl[64], std_[64], sp = 0;
    stf[0] = 0; stl[0] = n; std_[0] = lg * 2; sp = 1;
    while (sp > 0) {
        --sp;
        int first = stf[sp], last = stl[sp], depth = std_[sp];
        // emulate: while (last - first > 16) {...; introsort_loop(cut, last, depth); last = cut;}
        // The recursive call on [cut, last) runs BEFORE the loop continues on [first, cut): keep that order by
        // pushing the left continuation and then processing the right part first.
        while (last - first > 16) {
            if (depth == 0) { lfs_partial_sort(v + first, last - first, last - first); break; }
            --depth;
            const int mid = first + (last - first) / 2;
            {   // move_median_to_first(first, first+1, mid, last-1)
                LfPair *r = &v[first], *a = &v[first + 1], *b = &v[mid], *c = &v[last - 1];
                if (LF_LESS(*a, *b)) {
                    if (LF_LESS(*b, *c)) lfs_swap(r, b);
                    else if (LF_LESS(*a, *c)) lfs_swap(r, c);
                    else lfs_swap(r, a);
                } else if (LF_LESS(*a, *c)) lfs_swap(r, a);
                else if (LF_LESS(*b, *c)) lfs_swap(r, c);
                else lfs_swap(r, b);
            }
            int f = first + 1, l = last;
            for (;;) {   // unguarded_partition(first+1, last, pivot = first)
                while (LF_LESS(v[f], v[first])) ++f;
                --l;
                while (LF_LESS(v[first], v[l])) --l;
                if (!(f < l)) break;
                lfs_swap(&v[f], &v[l]);
                ++f;
            }
            const int cut = f;
            // right part [cut, last) first (recursion), left part [first, cut) afterwards (loop continuation).
            // The two ranges are disjoint and nothing else touches them, so deferring the left part is equivalent.
            stf[sp] = first; stl[sp] = cut; std_[sp] = depth; ++sp;
            first = cut;
        }
    }
    if (n > 16) {
        lfs_insertion_sort(v, 0, 16);
        for (int i = 16; i != n; ++i) lfs_unguarded_linear_insert(v, i);
    } else lfs_insertion_sort(v, 0, n);
}

// ------------------------------------------------------------------------------------------------------------
// Self-similarity selection (core:3397-3445): one warp per reference patch.
// ------------------------------------------------------------------------------------------------------------
__device__ __forceinline__ unsigned lf_fkey(float v)     // monotonic float -> unsigned
{
    const unsigned b = __float_as_uint(v);
    return (b & 0x80000000u) ? ~b : (b | 0x80000000u);
}
__device__ __forceinline__ float lf_fkey_inv(unsigned key)
{
    return __uint_as_float((key & 0x80000000u) ? (key & 0x7fffffffu) : ~key);
}

#define LF_SEL_SMALL 128

struct SelGeom {
    int w, nSim, Ns, N, R, nc;
    float threshold;
    const int *rows, *cols;       // reference rows / columns
};

// One warp selects the matches of reference patch r exactly like the reference (also under exact float ties).
__device__ __forceinline__ void lf_bm_select_one(const SelGeom &g, const int r, unsigned long long *keys, const float *__restrict__ s_at,
                                                 const float *__restrict__ s_mir, unsigned *__restrict__ out_count, unsigned *__restrict__ out_idx,
                                                 const PeerTable &pt)
{
    const unsigned FULL = 0xffffffffu;
    const int lane = threadIdx.x;
    const int k_r = g.rows[r / g.nc] * g.w + g.cols[r % g.nc];
    const int Ns = g.Ns, nSim = g.nSim, total = Ns * Ns;

    // candidates in the reference's push order: for dj { di = 0..nSim ; di = -nSim..-1 }
    int cnt = 0;
    unsigned long long lmin = ~0ull;       // smallest key seen by this lane
    for (int base = 0; base < total; base += 32) {
        const int o = base + lane;
        bool keep = false;
        float val = 0.f;
        if (o < total) {
            const int djx = o / Ns, rem = o - djx * Ns;
            float test;
            if (rem <= nSim) {
                const int ddk = djx + rem * Ns;
                test = val = lf_peer_sum(pt, false, s_at, ddk, (size_t) g.R, r);
            } else {
                const int a = nSim - (rem - nSim - 1);            // a = -di, di = -nSim + (rem - nSim - 1)
                const int ddk = (Ns - 1 - djx) + a * Ns;
                test = lf_peer_sum(pt, false, s_at, ddk, (size_t) g.R, r);
                val = lf_peer_sum(pt, true, s_mir, ddk, (size_t) g.R, r);
            }
            keep = test < g.threshold;
        }
        const unsigned m = __ballot_sync(FULL, keep);
        if (keep) {
            const int slot = cnt + __popc(m & ((1u << lane) - 1u));
            const unsigned long long kk = ((unsigned long long) lf_fkey(val + 0.0f) << 32) | (unsigned) o;
            keys[slot] = kk;
            lmin = kk < lmin ? kk : lmin;
        }
        cnt += __popc(m);
    }
    __syncwarp();
    unsigned nSx;
    if ((unsigned) g.N > (unsigned) cnt) { nSx = 1; while (nSx * 2 <= (unsigned) cnt) nSx *= 2; } else nSx = g.N;
    unsigned *dst = out_idx + (size_t) r * (g.N + 1);
    if (cnt == 0) {      // nSx == 1: the reference pushes (0, k_r) and duplicates it
        if (lane == 0) { dst[0] = k_r; dst[1] = k_r; out_count[r] = 2; }
        return;
    }
    // the M = min(cnt, nSx+1) smallest keys, ascending; lane t keeps the t-th (t < 32), `extra` the 33rd
    const int M = min(cnt, (int) nSx + 1);
    // pruning: the M-th smallest of the 32 per-lane minima bounds the M-th smallest key from above; the selection rounds
    // then run on the few keys below that bound (the full list stays in place for the tie path)
    __shared__ unsigned long long small[LF_SEL_SMALL];
    const unsigned long long *sel = keys;
    int nsel = cnt;
    if (cnt > LF_SEL_SMALL && M <= 32) {
        unsigned long long bound = 0, pv = 0;
        for (int t = 0; t < M; ++t) {
            unsigned long long best = (t == 0 || lmin > pv) ? lmin : ~0ull;
            for (int o = 16; o > 0; o >>= 1) {
                const unsigned long long other = __shfl_xor_sync(FULL, best, o);
                best = other < best ? other : best;
            }
            pv = bound = best;
        }
        if (bound != ~0ull) {           // at least M lanes hold a candidate
            int c2 = 0;
            for (int base = 0; base < cnt; base += 32) {
                const int q = base + lane;
                const unsigned long long kq = q < cnt ? keys[q] : ~0ull;
                const bool keep = kq <= bound;
                const unsigned m = __ballot_sync(FULL, keep);
                const int slot = c2 + __popc(m & ((1u << lane) - 1u));
                if (keep && slot < LF_SEL_SMALL) small[slot] = kq;
                c2 += __popc(m);
            }
            __syncwarp();
            if (c2 <= LF_SEL_SMALL) { sel = small; nsel = c2; }
        }
    }
    unsigned long long prev = 0, mine = ~0ull, extra = ~0ull;
    for (int t = 0; t < M; ++t) {
        unsigned long long best = ~0ull;
        for (int q = lane; q < nsel; q += 32) {
            const unsigned long long kq = sel[q];
            if ((t == 0 || kq > prev) && kq < best) best = kq;
        }
        for (int o = 16; o > 0; o >>= 1) {
            const unsigned long long other = __shfl_xor_sync(FULL, best, o);
            best = other < best ? other : best;
        }
        prev = best;
        if (t < 32) { if (lane == t) mine = best; } else extra = best;
    }
    // exact float ties among the M smallest make the result depend on the heap algorithm
    unsigned long long nxt = __shfl_down_sync(FULL, mine, 1);
    if (lane == 31) nxt = extra;
    const bool tie_here = (lane + 1 < M) && ((unsigned) (mine >> 32) == (unsigned) (nxt >> 32));
    const bool tie = __any_sync(FULL, tie_here);
    auto idx_of = [&](unsigned o) -> unsigned {
        const int djx = (int) o / Ns, rem = (int) o - djx * Ns;
        const int di = rem <= nSim ? rem : -nSim + (rem - nSim - 1);
        return (unsigned) (k_r + di * g.w + (djx - nSim));
    };
    if (!tie) {
        if (lane < (int) nSx) dst[lane] = idx_of((unsigned) (mine & 0xffffffffu));
        if (lane == 0) {
            if (nSx == 1) { dst[1] = dst[0] = idx_of((unsigned) (mine & 0xffffffffu)); out_count[r] = 2; }
            else out_count[r] = nSx;
        }
        return;
    }
    // slow path: one thread runs the reference's partial_sort on the pairs in push order
    LfPair *pairs = reinterpret_cast<LfPair *>(keys);
    for (int q = lane; q < cnt; q += 32) {
        const unsigned long long kq = keys[q];
        LfPair pr;
        pr.d = lf_fkey_inv((unsigned) (kq >> 32));
        pr.i = idx_of((unsigned) (kq & 0xffffffffu));
        pairs[q] = pr;          // same 8-byte slot, each lane converts its own entries
    }
    __syncwarp();
    if (lane == 0) {
        lfs_partial_sort(pairs, (int) nSx, cnt);
        for (unsigned t = 0; t < nSx; ++t) dst[t] = pairs[t].i;
        if (nSx == 1) { dst[1] = pairs[0].i; out_count[r] = 2; } else out_count[r] = nSx;
    }
}

// General path: one warp per reference patch, either all of them (list == nullptr) or the ones k_bm_select_fast deferred.
__global__ void __launch_bounds__(32) k_bm_select(SelGeom g, const float *__restrict__ s_at, const float *__restrict__ s_mir,
                                                  unsigned *__restrict__ out_count, unsigned *__restrict__ out_idx,
                                                  const unsigned *__restrict__ list, const unsigned *__restrict__ list_count, const PeerTable pt)
{
    extern __shared__ unsigned long long keys[];      // up to Ns*Ns entries, later reused as LfPair[]
    const int n = list ? (int) *list_count : g.R;
    for (int i = blockIdx.x; i < n; i += gridDim.x) {
        lf_bm_select_one(g, list ? (int) list[i] : i, keys, s_at, s_mir, out_count, out_idx, pt);
        __syncwarp();
    }
}

// Fast path: one thread per reference patch (coalesced reads of the sampled sums, lane <-> r), the NM = N + 1 smallest
// (distance, push order) keys kept sorted in registers. Without an exact float tie among the selected distances the
// reference's partial_sort returns exactly these, in this order; reference patches with a tie are deferred to k_bm_select.
template <int NM>
__global__ void __launch_bounds__(128) k_bm_select_fast(SelGeom g, const float *__restrict__ s_at, const float *__restrict__ s_mir,
                                                        unsigned *__restrict__ out_count, unsigned *__restrict__ out_idx,
                                                        unsigned *__restrict__ list, unsigned *__restrict__ list_count)
{
    const int r = blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= g.R) return;
    const int k_r = g.rows[r / g.nc] * g.w + g.cols[r % g.nc];
    const int Ns = g.Ns, nSim = g.nSim;
    const size_t R = (size_t) g.R;
    unsigned long long top[NM];
#pragma unroll
    for (int t = 0; t < NM; ++t) top[t] = ~0ull;
    int cnt = 0;
    auto offer = [&](float test, float val, unsigned o) {
        if (test < g.threshold) {
            ++cnt;
            const unsigned long long key = ((unsigned long long) lf_fkey(val + 0.0f) << 32) | o;
            if (key < top[NM - 1]) {
                top[NM - 1] = key;
#pragma unroll
                for (int t = NM - 1; t > 0; --t) {
                    const unsigned long long a = top[t - 1], b = top[t];
                    const bool sw = b < a;
                    top[t - 1] = sw ? b : a;
                    top[t] = sw ? a : b;
                }
            }
        }
    };
    // candidates in the reference's push order: for dj { di = 0..nSim ; di = -nSim..-1 }
    unsigned o = 0;
    for (int djx = 0; djx < Ns; ++djx) {
        const float *pa = s_at + (size_t) djx * R + r;
        int rem = 0;
        for (; rem + 4 <= nSim + 1; rem += 4, o += 4) {
            float v[4];
#pragma unroll
            for (int u = 0; u < 4; ++u) v[u] = __ldg(pa + (size_t) (rem + u) * Ns * R);
#pragma unroll
            for (int u = 0; u < 4; ++u) offer(v[u], v[u], o + u);
        }
        for (; rem <= nSim; ++rem, ++o) { const float v = __ldg(pa + (size_t) rem * Ns * R); offer(v, v, o); }
        // di = -nSim + j, j = 0..nSim-1: sums of the mirrored pair, stored at plane (Ns-1-djx) + (nSim - j) * Ns
        const size_t mb = (size_t) (Ns - 1 - djx) * R + r;
        int j = 0;
        for (; j + 4 <= nSim; j += 4, o += 4) {
            float t4[4], v4[4];
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                const size_t off = mb + (size_t) (nSim - (j + u)) * Ns * R;
                t4[u] = __ldg(s_at + off);
                v4[u] = __ldg(s_mir + off);
            }
#pragma unroll
            for (int u = 0; u < 4; ++u) offer(t4[u], v4[u], o + u);
        }
        for (; j < nSim; ++j, ++o) {
            const size_t off = mb + (size_t) (nSim - j) * Ns * R;
            offer(__ldg(s_at + off), __ldg(s_mir + off), o);
        }
    }
    unsigned nSx;
    if ((unsigned) g.N > (unsigned) cnt) { nSx = 1; while (nSx * 2 <= (unsigned) cnt) nSx *= 2; } else nSx = g.N;
    unsigned *dst = out_idx + (size_t) r * (g.N + 1);
    if (cnt == 0) { dst[0] = k_r; dst[1] = k_r; out_count[r] = 2; return; }
    const int M = min(cnt, (int) nSx + 1);
    bool tie = false;
#pragma unroll
    for (int t = 0; t + 1 < NM; ++t)
        if (t + 1 < M && (unsigned) (top[t] >> 32) == (unsigned) (top[t + 1] >> 32)) tie = true;
    if (tie) { list[atomicAdd(list_count, 1u)] = (unsigned) r; return; }
    auto idx_of = [&](unsigned oo) -> unsigned {
        const int djx = (int) oo / Ns, rem = (int) oo - djx * Ns;
        const int di = rem <= nSim ? rem : -nSim + (rem - nSim - 1);
        return (unsigned) (k_r + di * g.w + (djx - nSim));
    };
#pragma unroll
    for (int t = 0; t < NM - 1; ++t)
        if (t < (int) nSx) dst[t] = idx_of((unsigned) (top[t] & 0xffffffffu));
    if (nSx == 1) { dst[1] = idx_of((unsigned) (top[0] & 0xffffffffu)); out_count[r] = 2; } else out_count[r] = nSx;
}

// N = 1 has no self search: every reference patch r in [r0, r1) is its own only match (core:3448-3460)
__global__ void k_bm_identity(const int *rows, const int *cols, int nc, int w, int r0, int r1, int N, unsigned *out_count, unsigned *out_idx)
{
    const int r = r0 + blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= r1) return;
    out_count[r] = 1;
    out_idx[(size_t) r * (N + 1)] = (unsigned) (rows[r / nc] * w + cols[r % nc]);
}

// ------------------------------------------------------------------------------------------------------------
// Disparity matching (core:3576-3608): one thread per position, walking the skewed layout k_sat2 writes so that
// the (2*nDisp+1)^2 plane reads are coalesced. Only element [0] of the sorted list and the shape flag are consumed
// downstream (core:294, 310, 503, 510); the full std::sort is emulated only where the minimum is tied.
// ------------------------------------------------------------------------------------------------------------
__global__ void k_stereo_argmin(const float *__restrict__ sums, size_t plane_stride, int w, int nDisp, int lo, int row_end, int col_end,
                                int nstrips, int SR, float threshold, unsigned *__restrict__ out_first, unsigned char *__restrict__ out_shape,
                                unsigned slot, uint2 *__restrict__ tie_list, unsigned *__restrict__ tie_count)
{
    const int Ns = 2 * nDisp + 1;
    const size_t total = (size_t) nstrips * SR * 32;
    for (size_t t = (size_t) blockIdx.x * blockDim.x + threadIdx.x; t < total; t += (size_t) gridDim.x * blockDim.x) {
        const int lane = (int) (t & 31);
        const size_t rs = t >> 5;
        const int strip = (int) (rs / SR), sidx = (int) (rs - (size_t) strip * SR);
        const int i = lo + sidx - lane, j = lo + (strip << 5) + lane;
        if (i < lo || i >= row_end || j >= col_end) continue;
        const int k_r = i * w + j;
        float best = 0.f;
        int nmin = 0, amin = 0, c = 0;
        for (int djx = 0; djx < Ns; ++djx)
            for (int dix = 0; dix < Ns; ++dix, ++c) {
                const float v = sums[(size_t) (djx + dix * Ns) * plane_stride + t];
                if (c == 0 || v < best) { best = v; nmin = 1; amin = c; }
                else if (v == best) nmin++;
            }
        out_first[k_r] = (unsigned) (k_r + (amin % Ns - nDisp) * w + (amin / Ns - nDisp));
        out_shape[k_r] = best < threshold ? 1 : 0;
        // a tied minimum: element [0] of the reference's std::sort depends on the sort's moves; k_stereo_ties redoes these
        if (nmin > 1) tie_list[atomicAdd(tie_count, 1u)] = make_uint2(slot, (unsigned) t);
    }
}

// Positions whose minimum distance is tied (mirror-symmetric borders, flat regions): one thread per listed position runs the
// re-implemented libstdc++ std::sort on the (distance, index) pairs in the reference's push order (core:3590-3606). Each thread
// keeps its (2*nDisp+1)^2 pairs in dynamic shared memory; the host sizes the CTA to fit them.
struct TieGeom {
    size_t plane_stride;
    int w, nDisp, lo, nstrips, SR;
    unsigned plane;                     // w * h
    int nbuf;                           // stereo slots the sums buffer holds: slot s sits at s % nbuf
    int sai[LF_MAXA];                   // window slot of every stereo slot
};
__global__ void k_stereo_ties(TieGeom g, const float *__restrict__ sums, const uint2 *__restrict__ tie_list, const unsigned *__restrict__ tie_count,
                              unsigned *__restrict__ first)
{
    const int Ns = 2 * g.nDisp + 1, np = Ns * Ns;
    const unsigned n = *tie_count;
    for (unsigned e = blockIdx.x * blockDim.x + threadIdx.x; e < n; e += gridDim.x * blockDim.x) {
        const uint2 en = tie_list[e];
        const size_t t = en.y;
        const int lane = (int) (t & 31);
        const size_t rs = t >> 5;
        const int strip = (int) (rs / g.SR), sidx = (int) (rs - (size_t) strip * g.SR);
        const int i = g.lo + sidx - lane, j = g.lo + (strip << 5) + lane;
        const int k_r = i * g.w + j;
        const float *sp = sums + (size_t) (en.x % (unsigned) g.nbuf) * np * g.plane_stride + t;
        // the pairs live in shared memory: the emulated sort is a chain of dependent accesses (one thread per position, few
        // positions), its time is memory latency
        extern __shared__ LfPair s_td[];
        LfPair *td = s_td + (size_t) threadIdx.x * np;
        int c = 0;
        for (int djx = 0; djx < Ns; ++djx)
            for (int dix = 0; dix < Ns; ++dix, ++c) {
                td[c].d = sp[(size_t) (djx + dix * Ns) * g.plane_stride];
                td[c].i = (unsigned) (k_r + (dix - g.nDisp) * g.w + (djx - g.nDisp));
            }
        lfs_sort(td, np);
        first[(size_t) g.sai[en.x] * g.plane + k_r] = td[0].i;
    }
}
