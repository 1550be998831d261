// Kernels of the multi-GPU team path (team.cuh): one light field on G GPUs, every window pass split inside the window —
// offset planes of the block matching over the ranks, reference rows (and the pixel rows they aggregate into) in bands.
// Only what one GPU has no use for: the coverage count of a band (the team sums it over the ranks before it crops the
// accumulators back), the packing of row bands for their gather, the two-stage selection of the self matches — every rank keeps
// the N + 1 best candidates of its own offset planes (k_bm_partial), the owner of a reference row merges the partial lists
// (k_bm_merge); the (distance, push order) keys are totally ordered, so the merge gives exactly the list of k_bm_select_fast —
// and the exchanges over peer memory. The per-pixel kernels both drivers run on row ranges are in elementwise.cuh.
#pragma once
#include "common.cuh"
#include "elementwise.cuh"
#include "block_matching.cuh"

// LF_denoised_percent (utilities_LF.cpp:967-995) on the interior rows [i_lo, i_lo + ni) of the padded weights: entries with
// den > 0 in the top-left (H-k+1) x (W-k+1) of every SAI of the window
__global__ void k_count_cov_rows(const float *__restrict__ densym, LfWindow win, int W, int H, int C, int n, int k, int i_lo, int ni,
                                 unsigned long long *count)
{
    unsigned long long cnt = 0;
    const int wb = W + 2 * n, hb = H + 2 * n;
    const size_t plane_b = (size_t) wb * hb, band = (size_t) ni * W;
    const size_t total = (size_t) win.A * C * band;
    for (size_t t = (size_t) blockIdx.x * blockDim.x + threadIdx.x; t < total; t += (size_t) gridDim.x * blockDim.x) {
        const int ac = (int) (t / band), a = ac / C;
        if (!win.mask[a]) continue;
        const size_t rb = t - (size_t) ac * band;
        const int i = i_lo + (int) (rb / W), j = (int) (rb % W);
        if (i < H - k + 1 && j < W - k + 1 && densym[(size_t) ac * plane_b + (size_t) (i + n) * wb + (j + n)] > 0.0f) cnt++;
    }
    cnt = lf_block_sum_u64(cnt);
    if (threadIdx.x == 0 && cnt) atomicAdd(count, cnt);
}

// rows [i_lo, i_lo + ni) of every plane of a [nplanes][H][W] array <-> a contiguous [nplanes][ni][W] block (gather of the bands)
__global__ void k_pack_rows(const float *__restrict__ lf, float *__restrict__ blk, size_t nplanes, int W, int H, int i_lo, int ni, int unpack)
{
    const size_t HW = (size_t) W * H, band = (size_t) ni * W, total = nplanes * band;
    for (size_t t = (size_t) blockIdx.x * blockDim.x + threadIdx.x; t < total; t += (size_t) gridDim.x * blockDim.x) {
        const size_t pl = t / band, o = pl * HW + (size_t) i_lo * W + (t - pl * band);
        if (unpack) const_cast<float *>(lf)[o] = blk[t]; else blk[t] = lf[o];
    }
}

// ---- two-stage selection of the self matches ----
// Stage 1: one thread per reference patch over the offset planes ddk in [pl0, pl1) of this rank (ddk = di * Ns + djx): every
// plane gives the candidate (dj = djx - nSim, di) and, for di > 0, the mirrored candidate (-dj, -di) whose test is the same sum
// and whose value is the sum sampled at the mirrored patch (core:3407-3420). Output: number of candidates below the threshold
// and the NM smallest (distance, push order) keys, ascending (~0 = none).
template <int NM>
__global__ void __launch_bounds__(128) k_bm_partial(SelGeom g, const float *__restrict__ s_at, const float *__restrict__ s_mir, int pl0, int pl1,
                                                    unsigned *__restrict__ out_cnt, unsigned long long *__restrict__ out_keys)
{
    const int r = blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= g.R) return;
    const int Ns = g.Ns, nSim = g.nSim;
    const size_t R = (size_t) g.R;
    unsigned long long top[NM];
#pragma unroll
    for (int t = 0; t < NM; ++t) top[t] = ~0ull;
    unsigned cnt = 0;
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
    for (int ddk = pl0; ddk < pl1; ++ddk) {
        const int di = ddk / Ns, djx = ddk - di * Ns;
        const float v = __ldg(s_at + (size_t) ddk * R + r);
        offer(v, v, (unsigned) (djx * Ns + di));
        if (di > 0) offer(v, __ldg(s_mir + (size_t) ddk * R + r), (unsigned) ((Ns - 1 - djx) * Ns + (2 * nSim + 1 - di)));
    }
    out_cnt[r] = cnt;
#pragma unroll
    for (int t = 0; t < NM; ++t) out_keys[(size_t) r * NM + t] = top[t];
}

// Stage 2: the owner of reference patch r merges the partial lists of the G ranks ([G][R] counts, [G][R][NM] keys) and finishes
// like k_bm_select_fast: nSx = min(N, 2^floor(log2 count)), indices in list order, duplicate when only one match; reference
// patches with an exact float tie among the selected distances are listed: k_bm_select then runs the re-implemented libstdc++
// partial_sort on their complete candidate sequence, reading the sums of the other ranks' planes through peer pointers.
template <int NM>
__global__ void __launch_bounds__(128) k_bm_merge(SelGeom g, int G, int r0, int r1, const unsigned *__restrict__ cnt_all,
                                                  const unsigned long long *__restrict__ keys_all, unsigned *__restrict__ out_count,
                                                  unsigned *__restrict__ out_idx, unsigned *__restrict__ tie_list, unsigned *__restrict__ tie_count)
{
    const int r = r0 + blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= r1) return;
    const int k_r = g.rows[r / g.nc] * g.w + g.cols[r % g.nc];
    const int Ns = g.Ns, nSim = g.nSim;
    unsigned long long top[NM];
#pragma unroll
    for (int t = 0; t < NM; ++t) top[t] = ~0ull;
    int cnt = 0;
    for (int q = 0; q < G; ++q) {
        cnt += (int) cnt_all[(size_t) q * g.R + r];
        const unsigned long long *src = keys_all + ((size_t) q * g.R + r) * NM;
        for (int u = 0; u < NM; ++u) {
            const unsigned long long key = src[u];
            if (key >= top[NM - 1]) break;          // ascending: nothing smaller follows
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
    unsigned nSx;
    if ((unsigned) g.N > (unsigned) cnt) { nSx = 1; while (nSx * 2 <= (unsigned) cnt) nSx *= 2; } else nSx = g.N;
    unsigned *dst = out_idx + (size_t) r * (g.N + 1);
    if (cnt == 0) { dst[0] = k_r; dst[1] = k_r; out_count[r] = 2; return; }
    const int M = min(cnt, (int) nSx + 1);
    bool tie = false;
#pragma unroll
    for (int t = 0; t + 1 < NM; ++t)
        if (t + 1 < M && (unsigned) (top[t] >> 32) == (unsigned) (top[t + 1] >> 32)) tie = true;
    if (tie) {      // the values written below are then provisional: k_bm_select redoes the listed patches from the complete sums
        const unsigned slot = atomicAdd(tie_count, 1u);
        if (tie_list) tie_list[slot] = (unsigned) r;
    }
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

// ---- exchanges over peer memory (NVLink stores into the other ranks' buffers, mapped with cudaIpc) ----
// One kernel per exchange copies this rank's outgoing segments straight into their place in the receivers' buffers; the last CTA
// to finish then writes the exchange number into every peer's flag slot (after a system-scope fence: a peer that sees the number
// also sees the data). k_peer_wait is the other half: it returns once every peer's number has arrived.
struct PeerSegD { const char *src; char *dst; unsigned long long bytes; unsigned long long first_chunk; };
#define PEER_CHUNK 16384u

__global__ void __launch_bounds__(256) k_peer_copy(const PeerSegD *__restrict__ segs, int nseg, unsigned nchunks, unsigned *done_counter,
                                                   unsigned *const *peer_flags, int me, int G, unsigned epoch)
{
    __shared__ int s_seg;
    for (unsigned ch = blockIdx.x; ch < nchunks; ch += gridDim.x) {
        if (threadIdx.x == 0) {      // which segment this chunk belongs to (few segments: linear scan)
            int q = 0;
            while (q + 1 < nseg && segs[q + 1].first_chunk <= ch) ++q;
            s_seg = q;
        }
        __syncthreads();
        const PeerSegD sg = segs[s_seg];
        const unsigned long long off = (unsigned long long) (ch - sg.first_chunk) * PEER_CHUNK;
        const unsigned n = (unsigned) min((unsigned long long) PEER_CHUNK, sg.bytes - off);
        const char *s = sg.src + off;
        char *d = sg.dst + off;
        if ((((size_t) s | (size_t) d) & 15) == 0) {
            const unsigned nv = n >> 4;
            for (unsigned i = threadIdx.x; i < nv; i += blockDim.x) reinterpret_cast<uint4 *>(d)[i] = reinterpret_cast<const uint4 *>(s)[i];
            for (unsigned i = (nv << 4) + threadIdx.x; i < n; i += blockDim.x) d[i] = s[i];
        } else if ((((size_t) s | (size_t) d) & 3) == 0) {
            const unsigned nv = n >> 2;
            for (unsigned i = threadIdx.x; i < nv; i += blockDim.x) reinterpret_cast<unsigned *>(d)[i] = reinterpret_cast<const unsigned *>(s)[i];
            for (unsigned i = (nv << 2) + threadIdx.x; i < n; i += blockDim.x) d[i] = s[i];
        } else
            for (unsigned i = threadIdx.x; i < n; i += blockDim.x) d[i] = s[i];
        __syncthreads();
    }
    // last CTA out: publish
    __threadfence_system();
    __syncthreads();
    __shared__ unsigned s_last;
    if (threadIdx.x == 0) s_last = atomicAdd(done_counter, 1u) == gridDim.x - 1 ? 1u : 0u;
    __syncthreads();
    if (s_last) {
        if (threadIdx.x == 0) *done_counter = 0u;
        __threadfence_system();
        if ((int) threadIdx.x < G && (int) threadIdx.x != me)
            asm volatile("st.release.sys.global.u32 [%0], %1;\n" ::"l"(peer_flags[threadIdx.x] + me), "r"(epoch) : "memory");
    }
}

__global__ void k_peer_wait(const unsigned *flags, int me, int G, unsigned epoch, unsigned *timed_out)
{
    const int q = threadIdx.x;
    if (q < G && q != me) {
        unsigned v;
        const long long t0 = clock64();
        for (;;) {
            asm volatile("ld.acquire.sys.global.u32 %0, [%1];\n" : "=r"(v) : "l"(flags + q) : "memory");
            if ((int) (v - epoch) >= 0) break;
            if (clock64() - t0 > 20000000000ll) { *timed_out = 1u; break; }      // ~10 s: a lost peer must not hang the device (the step then fails)
            __nanosleep(100);
        }
    }
}
