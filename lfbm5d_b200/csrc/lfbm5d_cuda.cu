// Host side of the C ABI (include/lfbm5d_cuda.h): device buffers, per-step constant tables, the window schedule of
// the reference's step drivers (bm5d.cpp:165-407 / :861-1106, nb_threads == 1 semantics) and the per-pass kernel
// sequence (bm5d_core_processing.cpp:90-530 / :859-1331, `pst == cst` branch).
#include "lfbm5d_cuda.h"
#include "common.cuh"
#include "elementwise.cuh"
#include "block_matching.cuh"
#include "groups.cuh"
#include "groups_wiener8.cuh"
#include "groups25.cuh"

#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <vector>
#include <algorithm>
#include <array>
#include <map>
#include <mutex>
#include <memory>

namespace {

thread_local std::string g_err;
int fail(const std::string &m) { g_err = m; return 1; }

#define CK(x)                                                                                              \
    do {                                                                                                   \
        cudaError_t e_ = (x);                                                                              \
        if (e_ != cudaSuccess)                                                                             \
            return fail(std::string(#x) + ": " + cudaGetErrorString(e_) + " (" + __FILE__ + ":" + std::to_string(__LINE__) + ")"); \
    } while (0)

struct DevBuf {
    void *p = nullptr;
    size_t cap = 0;
    bool borrowed = false;      // an alias of another context's allocation (lanes of a team share the accumulators of the light field)
    void borrow(const DevBuf &o) { release(); p = o.p; cap = o.cap; borrowed = true; }
    int ensure(size_t bytes)
    {
        if (bytes <= cap) return 0;
        if (p && !borrowed) cudaFree(p);
        p = nullptr; cap = 0; borrowed = false;
        cudaError_t e = cudaMalloc(&p, bytes);
        if (e != cudaSuccess) return fail(std::string("cudaMalloc(") + std::to_string(bytes) + "): " + cudaGetErrorString(e));
        cap = bytes;
        return 0;
    }
    void release() { if (p && !borrowed) cudaFree(p); p = nullptr; cap = 0; borrowed = false; }
    template <class T> T *as() const { return reinterpret_cast<T *>(p); }
};

const double SQRT2_D = 1.414213562373095, SQRT2_INV_D = 0.7071067811865475;

// utilities.cpp:697-712
std::vector<int> ind_initialize(unsigned max_size, unsigned N, unsigned step)
{
    std::vector<int> v;
    unsigned ind = N;
    while (ind < max_size - N) { v.push_back((int) ind); ind += step; }
    if (v.empty() || (unsigned) v.back() < max_size - N - 1) v.push_back((int) (max_size - N - 1));
    return v;
}

// utilities.cpp:633-684
int estimate_sigma(float sigma, float *t, unsigned chnls, unsigned cs)
{
    if (chnls == 1) { t[0] = sigma; return 0; }
    if (cs == LFBM5D_YUV) {
        t[0] = sqrtf(0.299f * 0.299f + 0.587f * 0.587f + 0.114f * 0.114f) * sigma;
        t[1] = sqrtf(0.14713f * 0.14713f + 0.28886f * 0.28886f + 0.436f * 0.436f) * sigma;
        t[2] = sqrtf(0.615f * 0.615f + 0.51498f * 0.51498f + 0.10001f * 0.10001f) * sigma;
    } else if (cs == LFBM5D_YCBCR) {
        t[0] = sqrtf(0.299f * 0.299f + 0.587f * 0.587f + 0.114f * 0.114f) * sigma;
        t[1] = sqrtf(0.169f * 0.169f + 0.331f * 0.331f + 0.500f * 0.500f) * sigma;
        t[2] = sqrtf(0.500f * 0.500f + 0.419f * 0.419f + 0.081f * 0.081f) * sigma;
    } else if (cs == LFBM5D_OPP) {
        t[0] = sqrtf(0.333f * 0.333f + 0.333f * 0.333f + 0.333f * 0.333f) * sigma;
        t[1] = sqrtf(0.5f * 0.5f + 0.0f * 0.0f + 0.5f * 0.5f) * sigma;
        t[2] = sqrtf(0.25f * 0.25f + 0.5f * 0.5f + 0.25f * 0.25f) * sigma;
    } else if (cs == LFBM5D_RGB) {
        t[0] = t[1] = t[2] = sigma;
    } else return 1;
    return 0;
}

void dct_tables(float *f, float *inv, int n)
{
    for (int kk = 0; kk < n; kk++)
        for (int j = 0; j < n; j++) {
            f[kk * n + j] = (float) (2.0 * cos(M_PI * ((double) j + 0.5) * (double) kk / (double) n));
            inv[kk * n + j] = j == 0 ? 1.0f : (float) (2.0 * cos(M_PI * (double) j * ((double) kk + 0.5) / (double) n));
        }
}

// everything a pass needs to know (padded geometry)
struct PassCfg {
    int step;
    unsigned asw, A, C, W, H, n, nSim, nDisp, k, N, p, wb, hb;
    unsigned tau_2D, tau_4D, tau_5D;
    unsigned useSD = 0;       // 0 none, 1 sd_weighting_5d, 2 BM3D's sd_weighting
    float tauMatch;
    std::vector<int> rows, cols;
};

int make_passcfg(PassCfg &pc, int step, const lfbm5d_params *p, unsigned tau_4D)
{
    pc.step = step;
    pc.asw = 2 * p->an + 1; pc.A = pc.asw * pc.asw; pc.C = p->chnls; pc.W = p->width; pc.H = p->height;
    pc.nSim = p->nSim; pc.nDisp = p->nDisp; pc.n = p->nSim + p->nDisp; pc.k = p->k; pc.N = p->N; pc.p = p->p;
    pc.wb = pc.W + 2 * pc.n; pc.hb = pc.H + 2 * pc.n;
    pc.tau_2D = p->tau_2D; pc.tau_4D = tau_4D; pc.tau_5D = p->tau_5D; pc.useSD = p->useSD ? 1 : 0;
    float st[3];
    if (estimate_sigma(p->sigma, st, p->chnls, p->color_space)) return fail("unknown colour space");
    pc.tauMatch = (p->chnls == 1 ? 3.f : 1.f) * (st[0] < 35.0f ? (step == 1 ? 3000 : 2000) : 5000);   // core:146 / :915
    pc.rows = ind_initialize(pc.hb - pc.k + 1, pc.n, pc.p);
    pc.cols = ind_initialize(pc.wb - pc.k + 1, pc.n, pc.p);
    return 0;
}

// Host description of the offset planes of a pass: depends only on pst, the window mask, the (partial) extents and the buffers.
struct SatPlan {
    std::vector<SatPlane> planes;
    std::vector<SatGroup> groups;
    std::vector<int> stereo_sai;        // window slot of every stereo slot
    int nself_groups = 0, nself_planes = 0, nslots = 0;
    int groups_per_slot = 0, planes_per_slot = 0;      // Nd * ceil(Nd / 14) groups, Nd^2 planes
    int nbuf = 0;                       // stereo slots the sums buffer holds (stereo_buffer_slots): slot s sits at s % nbuf
    int st_lo = 0, st_row_end = 0, st_col_end = 0, st_strips = 0, st_SR = 0;
    size_t st_stride = 0;
    int self_row_end = 0, self_col_end = 0, self_strips = 0, pstrips = 1;
    DevBuf d_planes, d_groups;
    std::vector<size_t> key;
};

// ---- the window schedule of the reference's step drivers (bm5d.cpp:165-407 / :861-1106), shared by the single-GPU driver
// (step_begin ... step_end below) and the multi-GPU team (team.cuh). These rules decide every match list downstream: both
// drivers take them from here. What differs between the drivers is how they count (whole planes / bands + exchange) and
// which kernels pad, unpad and estimate. ----

// Index of SAI (s, t) among aw x ah SAIs in the order p.ang_major: the light field (awidth x aheight) and an angular window
// (asw x asw) use the same order
unsigned sai_index(const lfbm5d_params &p, unsigned s, unsigned t, unsigned aw, unsigned ah)
{
    return p.ang_major == LFBM5D_ROWMAJOR ? s * aw + t : s + t * ah;
}
unsigned sai_index(const lfbm5d_params &p, unsigned s, unsigned t) { return sai_index(p, s, t, p.awidth, p.aheight); }
void sai_coords(const lfbm5d_params &p, unsigned st, unsigned &s, unsigned &t)
{
    if (p.ang_major == LFBM5D_ROWMAJOR) { s = st / p.awidth; t = st - s * p.awidth; }
    else { t = st / p.aheight; s = st - t * p.aheight; }
}

// utilities_LF.cpp:881-901
void angular_search_window(int &c_asw, int &min_asw, int &max_asw, unsigned aidx, unsigned asize, unsigned asize_sw)
{
    min_asw = (int) aidx - (int) asize_sw;
    max_asw = (int) aidx + (int) asize_sw;
    int shift = min_asw < 0 ? -min_asw : 0;
    min_asw += shift; max_asw += shift;
    c_asw = (int) asize_sw - shift;
    shift = max_asw >= (int) asize ? ((int) asize - max_asw - 1) : 0;
    min_asw += shift; max_asw += shift; c_asw -= shift;
}

} // namespace

// state of a step between step_begin and step_end
struct StepState {
    int step = 0;
    lfbm5d_params p{};
    float *d_noisy = nullptr, *d_basic = nullptr;
    std::vector<unsigned> mask, proc;
    std::vector<char> touched;
    unsigned remaining = 0, max_proc = 0, tau_4D = 0, tables_tau4 = 0, passes = 0;
    PassCfg pc;
    bool docolor = false;
    cudaEvent_t e_begin = nullptr;
    float bm0 = 0.f, gr0 = 0.f;
    unsigned asize() const { return p.awidth * p.aheight; }
    size_t each() const { return (size_t) p.width * p.height * p.chnls; }
    unsigned cst() const { return sai_index(p, p.aheight / 2, p.awidth / 2); }      // centre SAI of the light field (bm5d.cpp:182-186)
};

namespace {

// One angular window while its core calls run
struct WindowRun {
    LfWindow win{};
    unsigned cst_asw = 0, pst_asw = 0;         // window slots: the SAI the window is centred on, the SAI of the current core call
    unsigned n_unproc = 0, max_unproc = 0, calls = 0;
    int min_s = 0, min_t = 0;
};

// bm5d.cpp:165-181: nothing processed but the empty SAIs; p has been validated
int step_state_init(StepState &S, int step, const lfbm5d_params *p, const unsigned *mask)
{
    S = StepState();
    S.p = *p; S.step = step;
    const unsigned asize = S.asize();
    S.mask.assign(mask, mask + asize);
    S.proc.assign(asize, 0);
    for (unsigned st = 0; st < asize; st++) { S.proc[st] = !S.mask[st]; S.remaining += S.proc[st] == 0; }
    S.max_proc = S.remaining;
    S.touched.assign(asize, 0);
    S.tau_4D = S.tables_tau4 = p->tau_4D;
    S.docolor = p->chnls == 3 && p->color_space != LFBM5D_RGB;
    return make_passcfg(S.pc, step, p, S.tau_4D);
}

// bm5d.cpp:189-202, :318-333: the unprocessed entry with the most zero weights, ties to the highest index; the reference keeps
// the count in an int
unsigned most_zeros(const unsigned *proc, const unsigned long long *zeros, unsigned n)
{
    long long best = -1;
    unsigned pick = 0;
    for (unsigned i = 0; i < n; i++) {
        if (proc[i]) continue;
        const long long z = (long long) (int) zeros[i];
        if (z >= best) { pick = i; best = z; }
    }
    return pick;
}

// bm5d.cpp:182-202: the centre SAI first, then the unprocessed SAI with the most zero weights in den. count(sais, zeros) counts
// them for the listed SAIs; an SAI no window has touched yet holds nothing but zeros.
template <class Count> int select_window(const StepState &S, unsigned &ps, unsigned &pt, Count count)
{
    const unsigned asize = S.asize();
    unsigned st_g = S.cst();
    if (S.remaining != S.max_proc || !S.mask[st_g]) {
        std::vector<unsigned> need;
        for (unsigned st = 0; st < asize; st++) if (!S.proc[st] && S.touched[st]) need.push_back(st);
        std::vector<unsigned long long> zc(asize, (unsigned long long) S.each()), h;
        if (!need.empty() && count(need, h)) return 1;
        for (size_t i = 0; i < need.size(); i++) zc[need[i]] = h[i];
        st_g = most_zeros(S.proc.data(), zc.data(), asize);
    }
    sai_coords(S.p, st_g, ps, pt);
    return 0;
}

// The window centred (and clamped) on SAI (ps, pt), bm5d.cpp:204-236. A window with an empty SAI turns dct into sadct for the
// rest of the step (bm5d.cpp:276-280); a driver that runs the windows out of their sequential order passes the static plan's
// value for the window instead (force_sadct 0 / 1). Returns whether tau_4D changed: the caller reloads the constant tables.
bool window_open(StepState &S, WindowRun &w, unsigned ps, unsigned pt, int force_sadct = -1)
{
    const lfbm5d_params &p = S.p;
    const unsigned asw = 2 * p.an + 1, A = asw * asw;
    int cs_asw, max_s, ct_asw, max_t;
    angular_search_window(cs_asw, w.min_s, max_s, ps, p.aheight, p.an);
    angular_search_window(ct_asw, w.min_t, max_t, pt, p.awidth, p.an);
    w.cst_asw = sai_index(p, cs_asw, ct_asw, asw, asw);
    w.win = LfWindow{};
    w.win.A = (int) A;
    w.n_unproc = 0;
    for (unsigned s_a = 0; s_a < asw; s_a++)
        for (unsigned t_a = 0; t_a < asw; t_a++) {
            const unsigned st = sai_index(p, s_a + w.min_s, t_a + w.min_t), a = sai_index(p, s_a, t_a, asw, asw);
            w.win.st[a] = (int) st;
            w.win.mask[a] = S.mask[st];
            w.win.proc[a] = !S.mask[st];
            w.n_unproc += S.mask[st] != 0;
        }
    w.max_unproc = w.n_unproc;
    w.calls = 0;
    if (force_sadct >= 0) S.tau_4D = (force_sadct && p.tau_4D == LFBM5D_DCT) ? (unsigned) LFBM5D_SADCT : p.tau_4D;
    else if (w.n_unproc != A && S.tau_4D == LFBM5D_DCT) S.tau_4D = LFBM5D_SADCT;
    if (S.tau_4D == S.tables_tau4) return false;
    S.pc.tau_4D = S.tables_tau4 = S.tau_4D;
    return true;
}

// The SAI of the window's next core call (bm5d.cpp:318-333): the centre slot first, then the unprocessed slot with the most
// zero weights in its padded den (all channels). count(slots, zeros) counts them for the listed window slots.
template <class Count> int window_next(WindowRun &w, Count count)
{
    if (w.n_unproc == w.max_unproc && w.win.mask[w.cst_asw]) { w.pst_asw = w.cst_asw; return 0; }
    const unsigned A = (unsigned) w.win.A;
    std::vector<unsigned> slots;
    for (unsigned a = 0; a < A; a++) if (!w.win.proc[a]) slots.push_back(a);
    std::vector<unsigned long long> zeros(A, 0), h;
    if (count(slots, h)) return 1;
    for (size_t i = 0; i < slots.size(); i++) zeros[slots[i]] = h[i];
    w.pst_asw = most_zeros(w.win.proc, zeros.data(), A);
    return 0;
}

// After a core call that left `covered` entries of the window with a weight. LF_denoised_percent (utilities_LF.cpp:967-995):
// float counter (saturates at 2^24), normalised without C; at 100 % every SAI of the window counts as processed
// (bm5d.cpp:370-382). Returns whether the window has SAIs left.
bool window_after_call(StepState &S, WindowRun &w, unsigned long long covered)
{
    LfWindow &win = w.win;
    const unsigned A = (unsigned) win.A;
    w.calls++;
    win.proc[w.pst_asw] += 1;
    S.proc[win.st[w.pst_asw]] += 1;
    const float fcnt = (float) std::min<unsigned long long>(covered, 16777216ull);
    unsigned nmask = 0;
    for (unsigned a = 0; a < A; a++) nmask += win.mask[a] == 1;
    const float pct = fcnt * 100.0f / (float) nmask / (float) (S.p.height - S.pc.k + 1) / (float) (S.p.width - S.pc.k + 1);
    if (pct >= 100.0f)
        for (unsigned a = 0; a < A; a++)
            if (win.proc[a] == 0) { win.proc[a] += 1; S.proc[win.st[a]] += 1; }
    w.n_unproc = 0;
    for (unsigned a = 0; a < A; a++) w.n_unproc += win.proc[a] == 0;
    return w.n_unproc > 0;
}

// End of the window: its SAIs hold weights now (window selection). Returns the window's schedule entry (centre SAI, first s,
// first t, core calls; lfbm5d_debug_schedule).
std::array<unsigned, 4> window_close(StepState &S, const WindowRun &w)
{
    for (int a = 0; a < w.win.A; a++) if (w.win.mask[a]) S.touched[w.win.st[a]] = 1;
    S.remaining = 0;
    for (unsigned st = 0; st < S.asize(); st++) S.remaining += S.proc[st] == 0;
    S.passes++;
    return { (unsigned) w.win.st[w.cst_asw], (unsigned) w.min_s, (unsigned) w.min_t, w.calls };
}

} // namespace

// Host entry points (lfbm5d_step1 / lfbm5d_step2): the light field travels SAI by SAI. Uploads (and the colour transform of each SAI)
// run on their own stream in the order the static window plan needs the SAIs, every window waits for the events of its SAIs only;
// an SAI is finalised (num / den, inverse colour transform) and sent back as soon as the last window of the plan that contains it
// is done. PCIe traffic so runs under the window passes in both directions.
struct HostIO {
    bool on = false;
    float *const *h_out = nullptr;
    float *d_out = nullptr;
    std::vector<cudaEvent_t> up, fin;      // per SAI: inputs on the device / final estimate computed
    std::vector<int> last_use;             // last plan window containing the SAI
    std::vector<unsigned> plan;            // (ps, pt) per plan window
    std::vector<char> done;
    bool plan_ok = true;
    unsigned window = 0;
};

struct lfbm5d_ctx {
    StepState ss;
    HostIO io;
    cudaStream_t stream4 = nullptr;                       // device -> host copies of finished SAIs
    int device = 0;
    cudaStream_t stream = nullptr, stream2 = nullptr;     // stream2: early device->host copies of the host entry points
    cudaStream_t stream3 = nullptr;                       // disparity matching of a pass, beside the self matching on `stream`
    cudaEvent_t ev_fork = nullptr, ev_join = nullptr, ev_satb = nullptr;
    int num_sms = 148;
    int smem_optin = 0;            // opt-in shared memory per block (bytes)
    DevBuf noisy, basic, out, num, den, mask;
    DevBuf nsym, bsym, numsym, densym, est0;
    DevBuf s_at, s_mir, sums, first, shape, bmcount, bmidx, bnd, progress, rowmap, colmap, rows, cols, counters,
           zbuf, wbuf, spos, arange, brange, gmask, shape_lut, tielist, stielist, act, rt_noisy, rt_basic, frow, fcol;
    unsigned lut_asw = 0;
    lfbm5d_stats stats{};
    bool timing = false;
    unsigned sat_epoch = 0;        // pass counter (16 bits): tags the strip hand-off words of k_sat2
    CUtensorMap tmap_est0;         // TMA view of the running-estimate planes [A][h_b][w_b] (source rows of k_sat2)
    size_t tmap_key[4] = { 0, 0, 0, 0 };
    bool tmap_ok = false;
    bool bm_only = false;          // lfbm5d_debug_block_matching: a pass stops behind the match tables
    cudaEvent_t ev[5]{};
    unsigned max_passes = 0;
    std::vector<unsigned> sched;
    std::vector<std::unique_ptr<SatPlan>> sat_cache;     // plane tables per window shape (sat_plan)
    std::map<std::pair<const void *, size_t>, int> cluster_occ;   // group_cluster: clusters the device holds per (kernel, smem)
    LfTables tab;                 // this context's constants; c_tab (one per device) is reloaded when it holds another context's
};

namespace {

#define LAUNCH(ctx, kern, grid, block, smem, ...)                          \
    do {                                                                    \
        kern<<<(grid), (block), (smem), (ctx)->stream>>>(__VA_ARGS__);      \
        (ctx)->stats.kernel_launches++;                                     \
    } while (0)
#define LAUNCH_ON(ctx, strm, kern, grid, block, smem, ...)                 \
    do {                                                                    \
        kern<<<(grid), (block), (smem), (strm)>>>(__VA_ARGS__);             \
        (ctx)->stats.kernel_launches++;                                     \
    } while (0)

int grid_for(const lfbm5d_ctx *ctx, size_t n, int block = 256)
{
    size_t g = (n + block - 1) / block;
    const size_t cap = (size_t) ctx->num_sms * 16;
    return (int) std::max<size_t>(1, std::min(g, cap));
}

int validate(const lfbm5d_params *p, int step)
{
    if (!p) return fail("null params");
    if (p->chnls != 1 && p->chnls != 3) return fail("chnls must be 1 or 3");
    if (p->awidth == 0 || p->aheight == 0 || p->width == 0 || p->height == 0) return fail("empty light field");
    const unsigned asw = 2 * p->an + 1;
    if (asw > p->aheight || asw > p->awidth)   // bm5d.cpp:120-124
        return fail("Wrong size of angular search window, the angular search window must be smaller than the light field angular size.");
    if (asw > LF_MAXASW) return fail("angular half window an > 2 is not supported by this build (an must be 0, 1 or 2)");
    if (p->k != 8 && p->k != 12 && p->k != 16) return fail("patch size must be 8, 12 or 16 in this build");
    if (p->k == 12) {
        if (p->tau_2D == LFBM5D_BIOR) return fail("tau_2D = bior needs a power-of-two patch size (k = 8 or 16); k = 12 takes id or dct");
        if (asw == 5) return fail("an = 2 is not supported at k = 12 (the 5x5-window group kernel needs 32 / k to be an integer); use k = 8 or 16");
    }
    if (p->N == 0 || p->N > LF_MAXN || (p->N & (p->N - 1))) return fail("N must be a power of two <= 32");
    if (p->nDisp > LF_MAXDISP) return fail("nDisp > 16 is not supported by this build (nDisp must be <= 16)");
    if (p->nSim + p->nDisp + 1 < p->k) return fail("nSim + nDisp must be >= k - 1");
    if (p->p == 0) return fail("processing step must be >= 1");
    if (p->tau_2D != LFBM5D_ID && p->tau_2D != LFBM5D_DCT && p->tau_2D != LFBM5D_BIOR) return fail("tau_2D must be id, dct or bior");
    if (p->tau_4D != LFBM5D_ID && p->tau_4D != LFBM5D_DCT && p->tau_4D != LFBM5D_SADCT) return fail("tau_4D must be id, dct or sadct");
    if (p->tau_5D != LFBM5D_HAAR && p->tau_5D != LFBM5D_HADAMARD && p->tau_5D != LFBM5D_DCT) return fail("tau_5D must be haar, hw or dct");
    if (p->ang_major != LFBM5D_ROWMAJOR && p->ang_major != LFBM5D_COLMAJOR) return fail("ang_major must be row or col");
    if (p->color_space > LFBM5D_RGB) return fail("Wrong type of transform. Must be OPP, YUV, or YCbCr!!");   // utilities.cpp:588-592
    if (p->height < p->k || p->width < p->k) return fail("image smaller than a patch");
    // the mirror padding of nSim + nDisp pixels (utilities.cpp:215-263) reflects once
    if (p->height < p->nSim + p->nDisp || p->width < p->nSim + p->nDisp) return fail("image smaller than the padding nSim + nDisp");
    // 5x5 windows: one channel of the group (twice that in step 2) has to fit into the shared memory of one CTA (k_groups25)
    if (asw == 5 && p->N * p->k * p->k * (step == 2 ? 2 : 1) > 2048)
        return fail("an = 2 needs N * k^2 <= 2048 in step 1 and 2 * N * k^2 <= 2048 in step 2 (k = 16: N <= 8 / N <= 4; k = 8: N <= 32 / N <= 16)");
    // k = 12 (k_groups12): one channel of the group, rows padded to k + 1 floats (twice that in step 2), in the shared memory of one CTA
    if (p->k == 12 && (size_t) p->N * asw * asw * 12 * 13 * 4 * (step == 2 ? 2 : 1) > LF_G12_SMEM)
        return fail("k = 12 needs N * A * k * (k + 1) * 4 B (twice that in step 2) <= " + std::to_string(LF_G12_SMEM) +
                    " B of shared memory per group (an = 1: N <= 32 in step 1, N <= 16 in step 2)");
    return 0;
}

// c_tab is one __constant__ object per device, shared by every context (and host thread) of the process. Each context keeps
// its own tables; before it launches kernels they are compared with what the device holds and reloaded if they differ (after
// a device-wide synchronisation, so that no kernel of another context is reading the old ones).
std::mutex g_tab_mu;
LfTables g_dev_tab[64];
bool g_dev_tab_valid[64];

int ensure_tables(lfbm5d_ctx *ctx)
{
    std::lock_guard<std::mutex> lk(g_tab_mu);
    const int d = ctx->device & 63;
    if (g_dev_tab_valid[d] && memcmp(&g_dev_tab[d], &ctx->tab, sizeof(LfTables)) == 0) return 0;
    CK(cudaDeviceSynchronize());
    CK(cudaMemcpyToSymbol(c_tab, &ctx->tab, sizeof(LfTables), 0, cudaMemcpyHostToDevice));
    g_dev_tab[d] = ctx->tab;
    g_dev_tab_valid[d] = true;
    return 0;
}

int setup_tables(lfbm5d_ctx *ctx, int step, const lfbm5d_params *p, unsigned tau_4D, bool bm3d = false)
{
    LfTables &T = ctx->tab;
    memset(&T, 0, sizeof(T));
    const int k = (int) p->k, asw = (int) (2 * p->an + 1);
    dct_tables(T.dct2f, T.dct2i, k);
    {   // bm3d.cpp:1101-1169
        static const float k8[16] = { 0.1924f, 0.2989f, 0.3846f, 0.4325f, 0.2989f, 0.4642f, 0.5974f, 0.6717f,
                                      0.3846f, 0.5974f, 0.7688f, 0.8644f, 0.4325f, 0.6717f, 0.8644f, 0.9718f };
        static const float k12[36] = { 0.1924f, 0.2615f, 0.3251f, 0.3782f, 0.4163f, 0.4362f, 0.2615f, 0.3554f, 0.4419f, 0.5139f, 0.5657f, 0.5927f,
                                       0.3251f, 0.4419f, 0.5494f, 0.6390f, 0.7033f, 0.7369f, 0.3782f, 0.5139f, 0.6390f, 0.7433f, 0.8181f, 0.8572f,
                                       0.4163f, 0.5657f, 0.7033f, 0.8181f, 0.9005f, 0.9435f, 0.4362f, 0.5927f, 0.7369f, 0.8572f, 0.9435f, 0.9885f };
        if (k == 8) {
            for (int i = 0; i < 8; i++)
                for (int j = 0; j < 8; j++) T.kaiser[i * 8 + j] = k8[(i < 4 ? i : 7 - i) * 4 + (j < 4 ? j : 7 - j)];
        } else if (k == 12) {      // the 6 x 6 quadrant, mirrored about both centre lines
            for (int i = 0; i < 12; i++)
                for (int j = 0; j < 12; j++) T.kaiser[i * 12 + j] = k12[(i < 6 ? i : 11 - i) * 6 + (j < 6 ? j : 11 - j)];
        } else
            for (int i = 0; i < k * k; i++) T.kaiser[i] = 1.0f;
        const float coef = 0.5f / ((float) k);
        for (int i = 0; i < k; i++)
            for (int j = 0; j < k; j++) {
                if (i == 0 && j == 0) { T.cn2[i * k + j] = 0.5f * coef; T.cni2[i * k + j] = 2.0f; }
                else if (i * j == 0) { T.cn2[i * k + j] = (float) (SQRT2_INV_D * coef); T.cni2[i * k + j] = (float) SQRT2_D; }
                else { T.cn2[i * k + j] = 1.0f * coef; T.cni2[i * k + j] = 1.0f; }
            }
        T.coef2inv = 1.0f / (float) (k * 2);
    }
    // angular tables: windows up to 3x3 and 5x5 windows have their own arrays (row length AW)
    const bool a5 = asw > LF_LUTASW;
    const int AW = a5 ? LF_MAXASW : LF_LUTASW;
    float *dctaf = a5 ? &T.dctaf5[0][0] : &T.dctaf[0][0], *dctai = a5 ? &T.dctai5[0][0] : &T.dctai[0][0];
    float *cn4 = a5 ? T.cn4_5 : T.cn4, *cni4 = a5 ? T.cni4_5 : T.cni4;
    float *cnsa = a5 ? &T.cnsa5[0][0] : &T.cnsa[0][0], *cnisa = a5 ? &T.cnisa5[0][0] : &T.cnisa[0][0];
    float *coefsa_inv = a5 ? T.coefsa_inv5 : T.coefsa_inv;
    for (int n = 1; n <= asw; n++) dct_tables(dctaf + (n - 1) * AW * AW, dctai + (n - 1) * AW * AW, n);
    {   // core:3191-3216
        const float coef = 0.5f / (sqrtf((float) asw) * sqrtf((float) asw));
        for (int i = 0; i < asw; i++)
            for (int j = 0; j < asw; j++) {
                if (i == 0 && j == 0) { cn4[i * asw + j] = (float) (0.5f * coef); cni4[i * asw + j] = 2.0f; }
                else if (i * j == 0) { cn4[i * asw + j] = (float) (SQRT2_INV_D * coef); cni4[i * asw + j] = (float) SQRT2_D; }
                else { cn4[i * asw + j] = (float) (1.0f * coef); cni4[i * asw + j] = 1.0f; }
            }
        T.coef4inv = 1.0f / (sqrtf((float) asw) * sqrtf((float) asw) * 2.0f);   // core:1945
    }
    for (int n = 2; n <= asw; n++) {   // core:3229-3252
        const float coef = (float) ((float) SQRT2_D / sqrt((double) n));
        cnsa[(n - 2) * AW] = (float) (SQRT2_INV_D * coef);
        cnisa[(n - 2) * AW] = (float) SQRT2_D;
        for (int i = 1; i < n; i++) { cnsa[(n - 2) * AW + i] = coef; cnisa[(n - 2) * AW + i] = 1.0f; }
    }
    for (int n = 1; n <= asw; n++) coefsa_inv[n] = 0.5f * (float) (SQRT2_INV_D) / sqrtf((float) n);   // core:2190, :2242
    {   // lib_transforms.cpp:215-277
        const float coef_norm = 1.f / (sqrtf(2.f) * 128.f), sqrt2_inv = 1.f / sqrtf(2.f);
        static const float a[10] = { 3.f, -3.f, -22.f, 22.f, 128.f, 128.f, 22.f, -22.f, -3.f, 3.f };
        static const float d[10] = { 3.f, 3.f, -22.f, -22.f, 128.f, -128.f, 22.f, 22.f, -3.f, -3.f };
        for (int i = 0; i < 10; i++) {
            T.lpd[i] = a[i] * coef_norm;
            T.hpr[i] = d[i] * coef_norm;
            T.hpd[i] = i == 4 ? -sqrt2_inv : (i == 5 ? sqrt2_inv : 0.f);
            T.lpr[i] = (i == 4 || i == 5) ? sqrt2_inv : 0.f;
        }
    }
    if (estimate_sigma(p->sigma, T.sigma, p->chnls, p->color_space)) return fail("unknown colour space");
    float lambda = p->lambda;
    if (step == 1 && p->tau_2D == LFBM5D_ID && tau_4D == LFBM5D_DCT) lambda /= (float) (SQRT2_D);   // core:206-207
    for (unsigned c = 0; c < p->chnls; c++) {
        T.sigma2[c] = T.sigma[c] * T.sigma[c];
        for (int lg = 0; lg < 8; lg++)   // core:2306 (hw) and :2431 (haar, lg = 0)
            T.thr[c][lg] = bm3d ? lambda * T.sigma[c] * sqrtf((float) (1u << lg))                       // bm3d.cpp:940
                                : lambda * T.sigma[c] * sqrtf((float) (1u << lg)) * (float) (SQRT2_D);
    }
    for (int lg = 0; lg < 8; lg++) T.hadcoef[lg] = 1.0f / (float) (1u << lg);
    for (int lg = 0; lg < 6; lg++) {     // 5-D DCT: tables of length 2^lg and preProcess_5d (core:3262-3276)
        const int n = 1 << lg, off = ((1 << (2 * lg)) - 1) / 3;
        dct_tables(T.dct5f + off, T.dct5i + off, n);
        const float coef = (float) (SQRT2_D) / sqrt((unsigned) n);
        T.cn5_0[lg] = (float) (SQRT2_INV_D * coef);
        T.cn5_c[lg] = coef;
        T.coef5inv[lg] = 0.5f * (float) (SQRT2_INV_D) / sqrtf((float) n);
    }
    for (unsigned c = 0; c < p->chnls; c++) T.thr_dct[c] = lambda * T.sigma[c] * 2.0f * (float) (SQRT2_D);   // core:2566
    return ensure_tables(ctx);
}

// upload the reference-patch grid (once per step)
int upload_grid(lfbm5d_ctx *ctx, const PassCfg &pc)
{
    std::vector<int> rowmap(pc.hb, -1), colmap(pc.wb, -1);
    for (size_t a = 0; a < pc.rows.size(); a++) rowmap[pc.rows[a]] = (int) a;
    for (size_t b = 0; b < pc.cols.size(); b++) colmap[pc.cols[b]] = (int) b;
    if (ctx->rowmap.ensure(pc.hb * 4) || ctx->colmap.ensure(pc.wb * 4) || ctx->rows.ensure(pc.rows.size() * 4) ||
        ctx->cols.ensure(pc.cols.size() * 4)) return 1;
    CK(cudaMemcpyAsync(ctx->rowmap.p, rowmap.data(), pc.hb * 4, cudaMemcpyHostToDevice, ctx->stream));
    CK(cudaMemcpyAsync(ctx->colmap.p, colmap.data(), pc.wb * 4, cudaMemcpyHostToDevice, ctx->stream));
    CK(cudaMemcpyAsync(ctx->rows.p, pc.rows.data(), pc.rows.size() * 4, cudaMemcpyHostToDevice, ctx->stream));
    CK(cudaMemcpyAsync(ctx->cols.p, pc.cols.data(), pc.cols.size() * 4, cudaMemcpyHostToDevice, ctx->stream));
    // candidate reference rows / columns per 16-pixel tile row / column of the aggregation kernel: a patch gathered
    // for a reference at row i_r starts within [i_r - n, i_r + n] (self +-nSim, then disparity +-nDisp)
    auto ranges = [&](const std::vector<int> &idx, unsigned dim) {
        const int ntile = (int) (dim + 15) / 16;
        std::vector<int> rg(2 * ntile);
        for (int t = 0; t < ntile; t++) {
            const int lo_v = 16 * t - (int) pc.k - (int) pc.n + 1, hi_v = 16 * t + 15 + (int) pc.n;
            int a_lo = (int) idx.size(), a_hi = -1;
            for (int a = 0; a < (int) idx.size(); a++)
                if (idx[a] >= lo_v && idx[a] <= hi_v) { a_lo = std::min(a_lo, a); a_hi = std::max(a_hi, a); }
            rg[2 * t] = a_lo; rg[2 * t + 1] = a_hi;
        }
        return rg;
    };
    const std::vector<int> ar = ranges(pc.rows, pc.hb), br = ranges(pc.cols, pc.wb);
    if (ctx->arange.ensure(ar.size() * 4) || ctx->brange.ensure(br.size() * 4)) return 1;
    CK(cudaMemcpyAsync(ctx->arange.p, ar.data(), ar.size() * 4, cudaMemcpyHostToDevice, ctx->stream));
    CK(cudaMemcpyAsync(ctx->brange.p, br.data(), br.size() * 4, cudaMemcpyHostToDevice, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    return 0;
}

// Stereo slots the disparity sums buffer holds: as many as (A - 1) slots of 13^2 planes (nDisp = 6) take, at least one, at most
// A - 1. Wider disparity windows run the slots of a pass in chunks of this many (launch_stereo).
int stereo_buffer_slots(const PassCfg &pc)
{
    const int Nd = 2 * (int) pc.nDisp + 1, A1 = (int) pc.A - 1;
    return std::min(A1, std::max(1, A1 * 169 / (Nd * Nd)));
}

int ensure_pass_buffers(lfbm5d_ctx *ctx, const PassCfg &pc)
{
    const size_t plane = (size_t) pc.wb * pc.hb, R = pc.rows.size() * pc.cols.size();
    const size_t Ns = 2 * pc.nSim + 1, nself = (pc.nSim + 1) * Ns, Nd = 2 * pc.nDisp + 1;
    if (ctx->nsym.ensure((pc.A + 1) * pc.C * plane * 4) || ctx->numsym.ensure(pc.A * pc.C * plane * 4) ||
        ctx->densym.ensure(pc.A * pc.C * plane * 4) || ctx->est0.ensure(pc.A * plane * 4)) return 1;
    if (pc.step == 2 && ctx->bsym.ensure((pc.A + 1) * pc.C * plane * 4)) return 1;
    if (pc.N > 1 && (ctx->s_at.ensure(nself * R * 4) || ctx->s_mir.ensure(nself * R * 4))) return 1;
    // stereo sums in the skewed layout of k_sat2: [plane][strip][SR][32]
    const size_t st_cols = pc.wb - 2 * pc.nDisp - pc.k + 1, st_rows = pc.hb - 2 * pc.nDisp - pc.k + 1;
    const size_t st_strips = (st_cols + 31) / 32, st_SR = st_rows + 31;
    if (pc.A > 1 && ctx->sums.ensure((size_t) stereo_buffer_slots(pc) * Nd * Nd * st_strips * st_SR * 32 * 4)) return 1;
    if (ctx->first.ensure(pc.A * plane * 4) || ctx->shape.ensure(pc.A * plane)) return 1;
    if (ctx->bmcount.ensure(R * 4) || ctx->bmidx.ensure(R * (pc.N + 1) * 4)) return 1;
    // hand-off words and first row / column are indexed by plane id, unique within a pass even where the chunks of the sums buffer
    // reuse its memory: a word one chunk tagged under this epoch is never at an address the next chunk polls
    const size_t nplanes = nself + (pc.A - 1) * Nd * Nd;
    const size_t max_strips = std::max(st_strips, (size_t) (pc.wb - 2 * pc.n + 31) / 32);
    {   // hand-off words of k_sat2: a fresh buffer holds no valid tag (epochs start at 1)
        const void *before = ctx->bnd.p;
        if (ctx->bnd.ensure(nplanes * max_strips * pc.hb * 8) || ctx->progress.ensure(64)) return 1;
        if (ctx->bnd.p != before) CK(cudaMemsetAsync(ctx->bnd.p, 0, ctx->bnd.cap, ctx->stream));
    }
    if (ctx->frow.ensure(nplanes * pc.wb * 4) || ctx->fcol.ensure(nplanes * pc.hb * 4)) return 1;
    if (ctx->counters.ensure(64 * 8)) return 1;
    if (ctx->zbuf.ensure(R * pc.N * pc.A * pc.C * pc.k * pc.k * 4) || ctx->wbuf.ensure(R * pc.C * 4) ||
        ctx->spos.ensure(R * pc.N * pc.A * 4)) return 1;
    return 0;
}

// SA-DCT index tables for every subset of the angular window (core:300-330: shape_idx, shape_mask_col, shape_idx_col,
// shape_mask_dct as built by sadct_4d_process, core:1969-2010); the group kernels look them up by the group's mask.
int ensure_shape_lut(lfbm5d_ctx *ctx, unsigned asw)
{
    if (ctx->lut_asw == asw) return 0;
    if (asw > LF_LUTASW) return 0;       // 5x5 windows: k_groups25 builds the shape of each group from its 25-bit mask
    const unsigned A = asw * asw, n = 1u << A;
    std::vector<GroupShape> lut(n);
    for (unsigned bits = 0; bits < n; bits++) {
        GroupShape &sh = lut[bits];
        memset(&sh, 0, sizeof(sh));
        lf_shape_build(sh, bits, asw);
    }
    if (ctx->shape_lut.ensure(n * sizeof(GroupShape))) return 1;
    CK(cudaMemcpyAsync(ctx->shape_lut.p, lut.data(), n * sizeof(GroupShape), cudaMemcpyHostToDevice, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    ctx->lut_asw = asw;
    return 0;
}

// ---- one core call, in pieces: the single-GPU run_pass strings them together; the multi-GPU team path (team.cuh) runs them
// band by band with exchanges in between ----

struct PassGeom {      // derived sizes of a pass
    size_t plane;
    int nr, nc, R, Ns, nself, Nd, nd2;
    float threshold;
};
PassGeom pass_geom(const PassCfg &pc)
{
    PassGeom g;
    g.plane = (size_t) pc.wb * pc.hb;
    g.nr = (int) pc.rows.size(); g.nc = (int) pc.cols.size(); g.R = g.nr * g.nc;
    g.Ns = 2 * (int) pc.nSim + 1; g.nself = pc.N > 1 ? ((int) pc.nSim + 1) * g.Ns : 0;
    g.Nd = 2 * (int) pc.nDisp + 1; g.nd2 = g.Nd * g.Nd;
    g.threshold = pc.tauMatch * pc.k * pc.k;       // core:3315
    return g;
}

// geometry the selection kernels of the self matches read
SelGeom sel_geom(const lfbm5d_ctx *ctx, const PassCfg &pc)
{
    const PassGeom pg = pass_geom(pc);
    SelGeom sg{};
    sg.w = pc.wb; sg.nSim = pc.nSim; sg.Ns = pg.Ns; sg.N = pc.N; sg.R = pg.R; sg.nc = pg.nc; sg.threshold = pg.threshold;
    sg.rows = ctx->rows.as<int>(); sg.cols = ctx->cols.as<int>();
    return sg;
}

// Plane tables of a pass, cached per (pst, window mask, extents, buffers): the same few windows shapes recur in every step.
SatPlan *sat_plan(lfbm5d_ctx *ctx, const PassCfg &pc, const LfWindow &win, int pst, bool partial, int act_ymax, int act_xmax)
{
    const PassGeom pg = pass_geom(pc);
    unsigned maskbits = 0;
    for (int st = 0; st < (int) pc.A; st++) maskbits |= (win.mask[st] ? 1u : 0u) << st;
    std::vector<size_t> key = { (size_t) pst, (size_t) maskbits, (size_t) partial, (size_t) (act_ymax + 1), (size_t) (act_xmax + 1),
                                (size_t) pc.wb, (size_t) pc.hb, (size_t) pc.k, (size_t) pc.nSim, (size_t) pc.nDisp, (size_t) pc.N, (size_t) pc.A,
                                (size_t) pg.R, (size_t) ctx->est0.p, (size_t) ctx->s_at.p, (size_t) ctx->s_mir.p, (size_t) ctx->sums.p };
    for (auto &e : ctx->sat_cache) if (e->key == key) return e.get();
    if (ctx->sat_cache.size() >= 48) {      // bounded: drop everything (the in-flight kernels read the tables: wait for them)
        cudaStreamSynchronize(ctx->stream); cudaStreamSynchronize(ctx->stream3);
        for (auto &e : ctx->sat_cache) { e->d_planes.release(); e->d_groups.release(); }
        ctx->sat_cache.clear();
    }
    std::unique_ptr<SatPlan> sp(new SatPlan());
    SatPlan &P = *sp;
    P.key = key;
    const float *est0 = ctx->est0.as<float>();
    const float *ref0 = est0 + (size_t) pst * pg.plane;
    const int Ns = pg.Ns, Nd = pg.Nd, R = pg.R;
    // ---- offset planes: groups of <= 14 planes sharing their source rows (same images, same row offset) ----
    for (int di = 0; di < (pg.nself ? (int) pc.nSim + 1 : 0); di++)
        for (int djx0 = 0; djx0 < Ns; djx0 += 2 * SAT_NW) {
            SatGroup G{};
            G.img1 = ref0; G.img2 = ref0; G.oy = di; G.oxmin = djx0 - (int) pc.nSim;      // core:3331: dk = di*w + djx - nSim
            G.z1 = G.z2 = pst;
            G.first_plane = (int) P.planes.size();
            for (int djx = djx0; djx < std::min(Ns, djx0 + 2 * SAT_NW); djx++) {
                SatPlane Q{};
                const int ddk = di * Ns + djx;
                Q.ox = djx - (int) pc.nSim;
                Q.out_at = ctx->s_at.as<float>() + (size_t) ddk * R;
                Q.out_mir = ctx->s_mir.as<float>() + (size_t) ddk * R;
                Q.mir_di = di; Q.mir_dc = (int) pc.nSim - djx;
                P.planes.push_back(Q);
                G.nplanes++;
            }
            P.groups.push_back(G);
        }
    P.nself_groups = (int) P.groups.size(); P.nself_planes = (int) P.planes.size();
    // The summed-area recurrences run from the top-left corner, so stopping them early changes nothing in what was computed.
    // The partial-window branch needs the self sums up to the last active reference patch (+ nSim columns for the mirrored
    // offsets) and the disparity results up to nSim rows / columns further (positions of the self matches); the reference
    // computes the whole planes there as well (core:3631-3788, :3806-3945) and reads the same values.
    const int st_row_full = pc.hb - pc.nDisp - pc.k + 1, st_col_full = pc.wb - pc.nDisp - pc.k + 1;
    P.st_lo = pc.nDisp;
    P.st_row_end = partial ? std::min(st_row_full, act_ymax + (int) pc.nSim + 1) : st_row_full;
    P.st_col_end = partial ? std::min(st_col_full, act_xmax + (int) pc.nSim + 1) : st_col_full;
    P.st_strips = (P.st_col_end - P.st_lo + 31) / 32; P.st_SR = (P.st_row_end - P.st_lo) + 31;
    P.st_stride = (size_t) ((st_col_full - P.st_lo + 31) / 32) * ((st_row_full - P.st_lo) + 31) * 32;      // allocation: full planes
    // a row offset's Nd column offsets split into ngx balanced groups of <= 14 consecutive ones (one group up to nDisp = 6);
    // plane ids stay [slot][di][dj]
    const int ngx = (Nd + 2 * SAT_NW - 1) / (2 * SAT_NW);
    P.groups_per_slot = Nd * ngx; P.planes_per_slot = pg.nd2;
    P.nbuf = pc.A > 1 ? stereo_buffer_slots(pc) : 1;
    int slot = 0;
    for (int st = 0; st < (int) pc.A; st++) {
        if (st == pst || !win.mask[st]) continue;
        const size_t bslot = (size_t) (slot % P.nbuf);
        for (int di = 0; di < Nd; di++)      // core:3516: dk = (di - nDisp)*w + (dj - nDisp)
            for (int gx = 0, dj0 = 0; gx < ngx; gx++) {
                const int dj1 = dj0 + Nd / ngx + (gx < Nd % ngx ? 1 : 0);
                SatGroup G{};
                G.img1 = ref0; G.img2 = est0 + (size_t) st * pg.plane; G.oy = di - (int) pc.nDisp; G.oxmin = dj0 - (int) pc.nDisp;
                G.z1 = pst; G.z2 = st;
                G.first_plane = (int) P.planes.size();
                for (int dj = dj0; dj < dj1; dj++) {
                    SatPlane Q{};
                    Q.ox = dj - (int) pc.nDisp;
                    Q.out_skew = ctx->sums.as<float>() + (bslot * pg.nd2 + (size_t) di * Nd + dj) * P.st_stride;
                    P.planes.push_back(Q);
                    G.nplanes++;
                }
                P.groups.push_back(G);
                dj0 = dj1;
            }
        P.stereo_sai.push_back(st);
        slot++;
    }
    P.nslots = slot;
    P.self_row_end = partial ? std::min((int) pc.hb - (int) pc.n, act_ymax + 1) : (int) pc.hb - (int) pc.n;
    P.self_col_end = partial ? std::min((int) pc.wb - (int) pc.n, act_xmax + (int) pc.nSim + 1) : (int) pc.wb - (int) pc.n;
    P.self_strips = (P.self_col_end - (int) pc.n + 31) / 32;
    // one plane stride for both launches: they share bnd / progress and are told apart by their plane ids only
    P.pstrips = std::max(std::max(P.self_strips, P.st_strips), 1);
    if (!P.planes.empty()) {
        if (P.d_planes.ensure(P.planes.size() * sizeof(SatPlane)) || P.d_groups.ensure(P.groups.size() * sizeof(SatGroup))) return nullptr;
        // pageable source: the copies are staged before the calls return, the vectors stay alive in the cache anyway
        if (cudaMemcpyAsync(P.d_planes.p, P.planes.data(), P.planes.size() * sizeof(SatPlane), cudaMemcpyHostToDevice, ctx->stream) != cudaSuccess ||
            cudaMemcpyAsync(P.d_groups.p, P.groups.data(), P.groups.size() * sizeof(SatGroup), cudaMemcpyHostToDevice, ctx->stream) != cudaSuccess) {
            fail("upload of the plane tables failed");
            return nullptr;
        }
    }
    ctx->sat_cache.push_back(std::move(sp));
    return ctx->sat_cache.back().get();
}

// Tensor map of the estimate planes for the TMA loads of k_sat2 (cuTensorMapEncodeTiled through the runtime's driver entry point:
// no link-time dependency on libcuda). Needs a row pitch that is a multiple of 16 bytes; otherwise the cp.async variant runs.
int ensure_tmap(lfbm5d_ctx *ctx, const PassCfg &pc)
{
    const size_t key[4] = { (size_t) ctx->est0.p, pc.wb, pc.hb, pc.A };
    if (memcmp(key, ctx->tmap_key, sizeof(key)) == 0) return 0;
    memcpy(ctx->tmap_key, key, sizeof(key));
    ctx->tmap_ok = false;
    memset(&ctx->tmap_est0, 0, sizeof(ctx->tmap_est0));
    if (((size_t) pc.wb * 4) % 16 != 0 || ((size_t) ctx->est0.p % 16) != 0 || getenv("LFBM5D_NO_TMA")) return 0;
    typedef CUresult (*encode_fn)(CUtensorMap *, CUtensorMapDataType, cuuint32_t, void *, const cuuint64_t *, const cuuint64_t *, const cuuint32_t *,
                                  const cuuint32_t *, CUtensorMapInterleave, CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
    static encode_fn enc = nullptr;
    if (!enc) {
        void *fp = nullptr;
        cudaDriverEntryPointQueryResult qr;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fp, cudaEnableDefault, &qr) != cudaSuccess || !fp) { cudaGetLastError(); return 0; }
        enc = (encode_fn) fp;
    }
    const cuuint64_t dims[3] = { pc.wb, pc.hb, pc.A };
    const cuuint64_t strides[2] = { (cuuint64_t) pc.wb * 4, (cuuint64_t) pc.wb * pc.hb * 4 };
    const cuuint32_t box[3] = { 64, 8, 1 }, estr[3] = { 1, 1, 1 };
    if (enc(&ctx->tmap_est0, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 3, ctx->est0.p, dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
            CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) != CUDA_SUCCESS) return 0;
    ctx->tmap_ok = true;
    return 0;
}

// New pass: reset the two ticket counters and move on to the next epoch of the hand-off tags (1 .. 65535; when the counter wraps the
// words are cleared, so that a word written 65535 passes ago under another geometry can never be taken for a fresh one)
int next_sat_epoch(lfbm5d_ctx *ctx)
{
    CK(cudaMemsetAsync(ctx->progress.p, 0, 16, ctx->stream));
    if (++ctx->sat_epoch > 0xffffu) {
        ctx->sat_epoch = 1;
        CK(cudaStreamSynchronize(ctx->stream3));
        CK(cudaMemsetAsync(ctx->bnd.p, 0, ctx->bnd.cap, ctx->stream));
    }
    return 0;
}

// Summed-area planes of the self groups [sg0, sg1) on `strm` (ticket counter 0) ...
int launch_sat_self(lfbm5d_ctx *ctx, const PassCfg &pc, const SatPlan &P, int sg0, int sg1, cudaStream_t strm)
{
    if (sg1 <= sg0) return 0;
    const PassGeom pg = pass_geom(pc);
    int *ticket = ctx->progress.as<int>();
    SatGeom g{};
    g.epoch = ctx->sat_epoch;
    g.w = pc.wb; g.h = pc.hb; g.k = pc.k; g.lo = pc.n; g.row_end = P.self_row_end; g.col_end = P.self_col_end;
    g.ylim = pc.hb - pc.n; g.xlim = pc.wb - pc.n; g.nstrips = P.self_strips; g.pstrips = P.pstrips; g.SR = 0;
    g.nc = pg.nc; g.rowmap = ctx->rowmap.as<int>(); g.colmap = ctx->colmap.as<int>();
    g.gp = pc.p; g.nr = pg.nr; g.rlast = pc.rows.back();
    g.nreg = 0;      // rows produced by the regular stride of ind_initialize (utilities.cpp:697-712)
    for (unsigned ind = pc.n; ind < pc.hb - pc.k + 1 - pc.n; ind += pc.p) g.nreg++;
    g.negzero2 = 0x8000000080000000ull;
    g.frow = ctx->frow.as<float>(); g.fcol = ctx->fcol.as<float>();
    const size_t smem = 2 * (128 + pc.k) * 64 * 4;
    if (ensure_tmap(ctx, pc)) return 1;
    // k = 12: cp.async ring loads (the TMA variant issues 8-row boxes and needs k to be a multiple of 8)
    auto kfn = pc.k == 12 ? k_sat2<true, 12, false>
             : ctx->tmap_ok ? (pc.k == 8 ? k_sat2<true, 8, true> : k_sat2<true, 16, true>) : (pc.k == 8 ? k_sat2<true, 8, false> : k_sat2<true, 16, false>);
    auto kedge = pc.k == 8 ? k_sat_edges<true, 8> : pc.k == 12 ? k_sat_edges<true, 12> : k_sat_edges<true, 16>;
    CK(cudaFuncSetAttribute((const void *) kfn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int) smem));
    const size_t smem_e = sate_smem((int) pc.k);
    CK(cudaFuncSetAttribute((const void *) kedge, cudaFuncAttributeMaxDynamicSharedMemorySize, (int) smem_e));
    kedge<<<dim3(sg1 - sg0, 2), SATE_NT, smem_e, strm>>>(g, P.d_groups.as<SatGroup>() + sg0, P.d_planes.as<SatPlane>(), ctx->frow.as<float>(), ctx->fcol.as<float>());
    ctx->stats.kernel_launches++;
    kfn<<<(sg1 - sg0) * P.self_strips, SAT_NW * 32, smem, strm>>>(g, P.d_groups.as<SatGroup>() + sg0, P.d_planes.as<SatPlane>(), sg1 - sg0,
                                                                  ctx->bnd.as<unsigned long long>(), ticket, ctx->tmap_est0);
    ctx->stats.kernel_launches++;
    return 0;
}
// ... and of the disparity slots [s0, s1) (ticket counter 1)
int launch_sat_stereo(lfbm5d_ctx *ctx, const PassCfg &pc, const SatPlan &P, int s0, int s1, cudaStream_t strm)
{
    if (s1 <= s0) return 0;
    int *ticket = ctx->progress.as<int>();
    SatGeom g{};
    g.epoch = ctx->sat_epoch;
    g.w = pc.wb; g.h = pc.hb; g.k = pc.k; g.lo = P.st_lo; g.row_end = P.st_row_end; g.col_end = P.st_col_end;
    g.ylim = pc.hb; g.xlim = pc.wb; g.nstrips = P.st_strips; g.pstrips = P.pstrips; g.SR = P.st_SR;
    g.gp = 1; g.negzero2 = 0x8000000080000000ull;
    g.frow = ctx->frow.as<float>(); g.fcol = ctx->fcol.as<float>();
    const size_t smem = 2 * (128 + pc.k) * 64 * 4;
    const int ngroups = (s1 - s0) * P.groups_per_slot;
    if (ensure_tmap(ctx, pc)) return 1;
    auto kfn = pc.k == 12 ? k_sat2<false, 12, false>
             : ctx->tmap_ok ? (pc.k == 8 ? k_sat2<false, 8, true> : k_sat2<false, 16, true>) : (pc.k == 8 ? k_sat2<false, 8, false> : k_sat2<false, 16, false>);
    auto kedge = pc.k == 8 ? k_sat_edges<false, 8> : pc.k == 12 ? k_sat_edges<false, 12> : k_sat_edges<false, 16>;
    CK(cudaFuncSetAttribute((const void *) kfn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int) smem));
    const size_t smem_e = sate_smem((int) pc.k);
    CK(cudaFuncSetAttribute((const void *) kedge, cudaFuncAttributeMaxDynamicSharedMemorySize, (int) smem_e));
    kedge<<<dim3(ngroups, 2), SATE_NT, smem_e, strm>>>(g, P.d_groups.as<SatGroup>() + P.nself_groups + s0 * P.groups_per_slot, P.d_planes.as<SatPlane>(),
                                                       ctx->frow.as<float>(), ctx->fcol.as<float>());
    ctx->stats.kernel_launches++;
    kfn<<<ngroups * P.st_strips, SAT_NW * 32, smem, strm>>>(g, P.d_groups.as<SatGroup>() + P.nself_groups + s0 * P.groups_per_slot,
                                                            P.d_planes.as<SatPlane>(), ngroups, ctx->bnd.as<unsigned long long>(), ticket + 1, ctx->tmap_est0);
    ctx->stats.kernel_launches++;
    return 0;
}

// Selection of the self matches of every reference patch from the complete sampled sums (single GPU; team fallback under ties)
int launch_self_select(lfbm5d_ctx *ctx, const PassCfg &pc, cudaStream_t strm)
{
    const PassGeom pg = pass_geom(pc);
    const int R = pg.R;
    const SelGeom sg = sel_geom(ctx, pc);
    void (*kfast)(SelGeom, const float *, const float *, unsigned *, unsigned *, unsigned *, unsigned *) = nullptr;
    switch (pc.N) {
        case 2: kfast = k_bm_select_fast<3>; break;
        case 4: kfast = k_bm_select_fast<5>; break;
        case 8: kfast = k_bm_select_fast<9>; break;
        case 16: kfast = k_bm_select_fast<17>; break;
        case 32: kfast = k_bm_select_fast<33>; break;
        default: break;
    }
    if (kfast) {
        // one thread per reference patch; the few with an exact float tie among the selected distances go to the warp kernel
        if (ctx->tielist.ensure((R + 1) * 4)) return 1;
        unsigned *tl = ctx->tielist.as<unsigned>();
        CK(cudaMemsetAsync(tl + R, 0, 4, strm));
        LAUNCH_ON(ctx, strm, kfast, (R + 127) / 128, 128, 0, sg, ctx->s_at.as<float>(), ctx->s_mir.as<float>(), ctx->bmcount.as<unsigned>(),
                  ctx->bmidx.as<unsigned>(), tl, tl + R);
        LAUNCH_ON(ctx, strm, k_bm_select, std::min<size_t>(R, (size_t) ctx->num_sms * 16), 32, (size_t) pg.Ns * pg.Ns * 8, sg, ctx->s_at.as<float>(),
                  ctx->s_mir.as<float>(), ctx->bmcount.as<unsigned>(), ctx->bmidx.as<unsigned>(), (const unsigned *) tl, (const unsigned *) (tl + R), PeerTable{});
    } else
        LAUNCH_ON(ctx, strm, k_bm_select, R, 32, (size_t) pg.Ns * pg.Ns * 8, sg, ctx->s_at.as<float>(), ctx->s_mir.as<float>(),
                  ctx->bmcount.as<unsigned>(), ctx->bmidx.as<unsigned>(), (const unsigned *) nullptr, (const unsigned *) nullptr, PeerTable{});
    return 0;
}

// Disparity argmin / shape flags of the slots [s0, s1) from their summed-area planes, tied minima redone like std::sort
int launch_stereo_argmin(lfbm5d_ctx *ctx, const PassCfg &pc, const SatPlan &P, int s0, int s1, cudaStream_t strm)
{
    if (s1 <= s0) return 0;
    const PassGeom pg = pass_geom(pc);
    // every position could be tied (a flat light field): room for all of them
    if (ctx->stielist.ensure(((size_t) P.nslots * P.st_stride + 1) * 8)) return 1;
    uint2 *sl = ctx->stielist.as<uint2>();
    unsigned *sc = reinterpret_cast<unsigned *>(sl + (size_t) P.nslots * P.st_stride);
    CK(cudaMemsetAsync(sc, 0, 4, strm));
    TieGeom tg{};
    tg.plane_stride = P.st_stride; tg.w = (int) pc.wb; tg.nDisp = (int) pc.nDisp; tg.lo = P.st_lo; tg.nstrips = P.st_strips; tg.SR = P.st_SR;
    tg.plane = (unsigned) pg.plane; tg.nbuf = P.nbuf;
    for (int s = 0; s < P.nslots; s++) tg.sai[s] = P.stereo_sai[s];
    for (int s = s0; s < s1; s++) {
        const int st = P.stereo_sai[s];
        LAUNCH_ON(ctx, strm, k_stereo_argmin, grid_for(ctx, P.st_stride, 128), 128, 0,
                  ctx->sums.as<float>() + (size_t) (s % P.nbuf) * pg.nd2 * P.st_stride, P.st_stride,
                  (int) pc.wb, (int) pc.nDisp, P.st_lo, P.st_row_end, P.st_col_end, P.st_strips, P.st_SR, pg.threshold,
                  ctx->first.as<unsigned>() + (size_t) st * pg.plane, ctx->shape.as<unsigned char>() + (size_t) st * pg.plane, (unsigned) s, sl, sc);
    }
    // Nd^2 pairs per thread in shared memory: 32 threads per CTA up to nDisp = 6, fewer where a CTA of 32 lists does not fit
    const size_t pair_bytes = (size_t) pg.nd2 * sizeof(LfPair);
    const int nt = (int) std::min<size_t>(32, (size_t) ctx->smem_optin / pair_bytes);
    if (nt < 1) return fail("k_stereo_ties: one sort list of " + std::to_string(pair_bytes) + " bytes exceeds the shared memory of a block");
    const size_t smem_t = (size_t) nt * pair_bytes;
    CK(cudaFuncSetAttribute((const void *) k_stereo_ties, cudaFuncAttributeMaxDynamicSharedMemorySize, (int) smem_t));
    LAUNCH_ON(ctx, strm, k_stereo_ties, ctx->num_sms * 4, nt, smem_t, tg, ctx->sums.as<float>(), (const uint2 *) sl, (const unsigned *) sc,
              ctx->first.as<unsigned>());
    return 0;
}

// Disparity matching of the slots [s0, s1) on strm: planes, argmin and ties, in chunks of P.nbuf slots, the slots the sums buffer
// holds. Each chunk's tie kernel is ordered before the next chunk's planes overwrite the buffer (same stream). between() runs once
// the first chunk's planes are enqueued: the caller's self matching on the other stream then starts behind them. planes_done (if
// set) is recorded on strm behind the last chunk's planes.
template <class F>
int launch_stereo(lfbm5d_ctx *ctx, const PassCfg &pc, const SatPlan &P, int s0, int s1, cudaStream_t strm, cudaEvent_t planes_done, F between)
{
    for (int c0 = s0; c0 < s1 || c0 == s0; c0 += P.nbuf) {
        const int c1 = std::min(s1, c0 + P.nbuf);
        // a launch on a used ticket counter hands out no work: the second and later chunks reset theirs (the pass reset the first)
        if (c0 > s0) CK(cudaMemsetAsync(ctx->progress.as<int>() + 1, 0, 4, strm));
        if (launch_sat_stereo(ctx, pc, P, c0, c1, strm)) return 1;
        if (planes_done && c1 >= s1) CK(cudaEventRecord(planes_done, strm));
        if (c0 == s0 && between()) return 1;
        if (launch_stereo_argmin(ctx, pc, P, c0, c1, strm)) return 1;
    }
    return 0;
}

// Angular shape masks of the reference patches [r0, r1) (bit st: SAI st takes part), with the SA-DCT tables their group kernel
// reads: 16-bit masks into the host-built table for windows up to 3x3, 32-bit masks for 5x5 windows
int launch_group_masks(lfbm5d_ctx *ctx, const PassCfg &pc, const LfWindow &win, int pst, int r0, int r1)
{
    const PassGeom pg = pass_geom(pc);
    if (pc.asw > LF_LUTASW) {
        if (ctx->gmask.ensure((size_t) pg.R * 4)) return 1;
        LAUNCH(ctx, k_group_masks32, (r1 - r0 + 255) / 256, 256, 0, ctx->rows.as<int>(), ctx->cols.as<int>(), pg.nc, r0, r1, (int) pc.wb,
               (unsigned) pg.plane, (int) pc.A, pst, win, ctx->shape.as<unsigned char>(), ctx->gmask.as<unsigned>());
        return 0;
    }
    if (ensure_shape_lut(ctx, pc.asw) || ctx->gmask.ensure((size_t) pg.R * 2)) return 1;
    LAUNCH(ctx, k_group_masks, (r1 - r0 + 255) / 256, 256, 0, ctx->rows.as<int>(), ctx->cols.as<int>(), pg.nc, r0, r1, (int) pc.wb,
           (unsigned) pg.plane, (int) pc.A, pst, win, ctx->shape.as<unsigned char>(), ctx->gmask.as<unsigned short>());
    return 0;
}

// Dynamic shared memory of one channel of a group on one CTA: N patches of A SAIs (twice that in step 2), k rows of RS floats.
// Row padding removes the shared-memory bank conflicts of the 2-D passes (3 CTAs/SM without it measured slower); 5x5 windows
// store their patches densely (LfSwizzled).
static int group_rs(unsigned k, unsigned asw, unsigned tau_2D) { return asw > LF_LUTASW || tau_2D == LFBM5D_ID ? (int) k : (int) k + 1; }
static size_t group_smem(int step, unsigned k, unsigned asw, unsigned N, unsigned tau_2D)
{
    return (size_t) N * asw * asw * k * group_rs(k, asw, tau_2D) * 4 * (step == 2 ? 2 : 1);
}

// k = 16 groups of 3x3 windows whose channel (N * A * k * RS floats, twice that in step 2) needs more than the opt-in shared memory
// of one CTA next to k_groups' static arrays run on a cluster of CL CTAs (k_groups_cl), the smallest power of two for which
// 1 / CL of the group fits next to that kernel's static arrays. cl = 1: k_groups' branch fits (or does not apply). Before the
// first launch of a (kernel, shared memory) pair, the device has to be able to hold at least one such cluster at a time.
struct GroupCluster {
    int cl = 1;
    void (*fn)(GroupArgs) = nullptr;
    size_t smem = 0;                 // dynamic shared memory per CTA
    int max_active = 0;              // cudaOccupancyMaxActiveClusters of this configuration
};
int group_cluster(lfbm5d_ctx *ctx, int step, unsigned k, unsigned asw, unsigned N, unsigned tau_2D, GroupCluster &gc)
{
    gc = GroupCluster{};
    if (k != 16 || asw != 3) return 0;
    const size_t smem = group_smem(step, k, asw, N, tau_2D);
    cudaFuncAttributes fa;
    CK(cudaFuncGetAttributes(&fa, (const void *) (step == 1 ? k_groups<1, 3> : k_groups<2, 3>)));
    if (smem + fa.sharedSizeBytes <= (size_t) ctx->smem_optin) return 0;
    void (*const fns[2][2])(GroupArgs) = { { k_groups_cl<1, 2>, k_groups_cl<1, 4> }, { k_groups_cl<2, 2>, k_groups_cl<2, 4> } };
    for (int i = 0; i < 2 && !gc.fn; i++) {
        void (*fn)(GroupArgs) = fns[step - 1][i];
        CK(cudaFuncGetAttributes(&fa, (const void *) fn));
        if (smem / (2 << i) + fa.sharedSizeBytes <= (size_t) ctx->smem_optin) { gc.cl = 2 << i; gc.fn = fn; gc.smem = smem / gc.cl; }
    }
    if (!gc.fn) return fail("a group of " + std::to_string(smem) + " B of shared memory per channel does not fit a cluster of 4 CTAs");
    const auto key = std::make_pair((const void *) gc.fn, gc.smem);
    const auto it = ctx->cluster_occ.find(key);
    if (it != ctx->cluster_occ.end()) { gc.max_active = it->second; return 0; }
    CK(cudaFuncSetAttribute((const void *) gc.fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int) gc.smem));
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3((unsigned) gc.cl); cfg.blockDim = dim3(256); cfg.dynamicSmemBytes = gc.smem; cfg.stream = ctx->stream;
    cudaLaunchAttribute at;
    at.id = cudaLaunchAttributeClusterDimension;
    at.val.clusterDim.x = (unsigned) gc.cl; at.val.clusterDim.y = 1; at.val.clusterDim.z = 1;
    cfg.attrs = &at; cfg.numAttrs = 1;
    CK(cudaOccupancyMaxActiveClusters(&gc.max_active, (const void *) gc.fn, &cfg));
    if (gc.max_active <= 0)
        return fail("the group kernel needs clusters of " + std::to_string(gc.cl) + " CTAs with " + std::to_string(gc.smem + fa.sharedSizeBytes) +
                    " B of shared memory per CTA, and this device cannot run one");
    ctx->cluster_occ[key] = gc.max_active;
    return 0;
}

// The group kernel a pass runs, chosen from (step, k, asw, N, C, tau_2D, tau_5D, useSD), with its launch shape. Exactly one of
// fn / fn_nz / fn25 is set: fn_nz kernels take the zero-block marker as a second argument. cl > 1: a cluster of cl CTAs per group.
struct GroupKernel {
    const char *name = nullptr;
    void (*fn)(GroupArgs) = nullptr;                                  // k_groups, k_groups12, k_groups_cl
    void (*fn_nz)(GroupArgs, unsigned long long) = nullptr;           // k_groups_id16, k_groups_w8
    void (*fn25)(GroupArgs25) = nullptr;                              // k_groups25
    int threads = 256, cl = 1;
    size_t smem = 0;                                                  // dynamic shared memory per CTA
    const void *func() const { return fn ? (const void *) fn : fn_nz ? (const void *) fn_nz : (const void *) fn25; }
};
int group_kernel(lfbm5d_ctx *ctx, int step, unsigned k, unsigned asw, unsigned N, unsigned C, unsigned tau_2D, unsigned tau_5D,
                 unsigned useSD, GroupKernel &gk)
{
    gk = GroupKernel{};
    gk.smem = group_smem(step, k, asw, N, tau_2D);
    const bool s1 = step == 1, c3 = C == 3;        // validate(): C is 1 or 3
    if (asw == G25_SW) {
        // 5x5 windows: dense swizzled patches (no row padding), one CTA of 512 threads per SM; validate() bounds the group
        gk.fn25 = s1 ? k_groups25<1> : k_groups25<2>;
        gk.name = s1 ? "k_groups25<1>" : "k_groups25<2>";
        gk.threads = G25_NT;
        return 0;
    }
    if (k == 12) {         // 288 threads (2 patches x 144 positions); validate() bounds the group's shared memory
        gk.fn = s1 ? (asw == 3 ? k_groups12<1, 3> : k_groups12<1, 1>) : (asw == 3 ? k_groups12<2, 3> : k_groups12<2, 1>);
        gk.name = s1 ? (asw == 3 ? "k_groups12<1,3>" : "k_groups12<1,1>") : (asw == 3 ? "k_groups12<2,3>" : "k_groups12<2,1>");
        gk.threads = LF_G12_NT;
        return 0;
    }
    GroupCluster gc;
    if (group_cluster(ctx, step, k, asw, N, tau_2D, gc)) return 1;
    if (gc.cl > 1) {       // distributed over a cluster: CTA blockIdx.x % cl of the cluster of reference patch blockIdx.x / cl + r0
        gk.fn = gc.fn; gk.cl = gc.cl; gk.smem = gc.smem;
        gk.name = s1 ? (gc.cl == 2 ? "k_groups_cl<1,2>" : "k_groups_cl<1,4>") : (gc.cl == 2 ? "k_groups_cl<2,2>" : "k_groups_cl<2,4>");
        return 0;
    }
    if (s1 && tau_2D == LFBM5D_ID && k == 16 && asw == 3 && N <= 8 && tau_5D != LFBM5D_DCT && !useSD) {
        // register-resident path (no 2-D transform to stage); patches that contribute zeros read the zero block behind nsym
        gk.fn_nz = c3 ? k_groups_id16<3> : k_groups_id16<1>;
        gk.name = c3 ? "k_groups_id16<3>" : "k_groups_id16<1>";
        gk.smem = 0;
        return 0;
    }
    if (!s1 && tau_2D == LFBM5D_DCT && k == 8 && asw == 3 && N <= 16 && tau_5D == LFBM5D_HAAR && !useSD) {
        // packed X/E path: FP32x2 forward transforms, two rows per lane in the inverses
        gk.fn_nz = c3 ? k_groups_w8<3> : k_groups_w8<1>;
        gk.name = c3 ? "k_groups_w8<3>" : "k_groups_w8<1>";
        gk.threads = W8_NT;
        gk.smem = (size_t) 16 * 9 * W8_PS * 8;
        return 0;
    }
    gk.fn = s1 ? (asw == 3 ? k_groups<1, 3> : k_groups<1, 1>) : (asw == 3 ? k_groups<2, 3> : k_groups<2, 1>);
    gk.name = s1 ? (asw == 3 ? "k_groups<1,3>" : "k_groups<1,1>") : (asw == 3 ? "k_groups<2,3>" : "k_groups<2,1>");
    return 0;
}

// Group kernel for the reference patches [r0, r1) (gather, transforms, shrinkage, inverses, staging for the aggregation)
int launch_groups(lfbm5d_ctx *ctx, const PassCfg &pc, const LfWindow &win, int pst, bool partial, int r0, int r1)
{
    if (r1 <= r0) return 0;
    GroupKernel gk;
    if (group_kernel(ctx, pc.step, pc.k, pc.asw, pc.N, pc.C, pc.tau_2D, pc.tau_5D, pc.useSD, gk)) return 1;
    const PassGeom pg = pass_geom(pc);
    const int R = pg.R;
    GroupArgsBase gb{};
    gb.gmask = ctx->gmask.as<unsigned short>(); gb.shape_lut = ctx->shape_lut.as<GroupShape>();
    gb.act = partial ? ctx->act.as<unsigned char>() : nullptr; gb.partial = partial ? 1 : 0; gb.use_sd = (int) pc.useSD;
    gb.C = pc.C; gb.asw = pc.asw; gb.A = pc.A; gb.k = pc.k; gb.log2k = pc.k == 8 ? 3 : 4; gb.N = pc.N; gb.w = pc.wb; gb.h = pc.hb;
    gb.pst = pst; gb.nc = pg.nc; gb.r0 = r0;
    gb.RS = group_rs(pc.k, pc.asw, pc.tau_2D);
    gb.PS = pc.k * gb.RS;
    gb.tau_2D = pc.tau_2D; gb.tau_4D = pc.tau_4D; gb.tau_5D = pc.tau_5D;
    gb.rows = ctx->rows.as<int>(); gb.cols = ctx->cols.as<int>();
    gb.bm_count = ctx->bmcount.as<unsigned>(); gb.bm_idx = ctx->bmidx.as<unsigned>();
    gb.first = ctx->first.as<unsigned>(); gb.shape = ctx->shape.as<unsigned char>();
    gb.nsym = ctx->nsym.as<float>(); gb.bsym = ctx->bsym.as<float>();
    gb.numsym = ctx->numsym.as<float>(); gb.densym = ctx->densym.as<float>();
    gb.zbuf = ctx->zbuf.as<float>(); gb.wbuf = ctx->wbuf.as<float>(); gb.ent = ctx->spos.as<unsigned>(); gb.R = R;
    const int nblk = r1 - r0;
    if (gk.smem) CK(cudaFuncSetAttribute(gk.func(), cudaFuncAttributeMaxDynamicSharedMemorySize, (int) gk.smem));
    if (gk.fn25) {
        GroupArgs25 g25{};
        static_cast<GroupArgsBase &>(g25) = gb;
        g25.win = win;
        g25.gmask32 = ctx->gmask.as<unsigned>();
        gk.fn25<<<nblk, gk.threads, gk.smem, ctx->stream>>>(g25);
    } else {
        GroupArgs ga{};
        static_cast<GroupArgsBase &>(ga) = gb;
        for (int a = 0; a < LF_LUTA; a++) { ga.win.st[a] = win.st[a]; ga.win.mask[a] = win.mask[a]; ga.win.proc[a] = win.proc[a]; }
        ga.win.A = win.A;
        if (gk.fn_nz) gk.fn_nz<<<nblk, gk.threads, gk.smem, ctx->stream>>>(ga, 0x8000000080000000ull);
        else gk.fn<<<nblk * gk.cl, gk.threads, gk.smem, ctx->stream>>>(ga);
    }
    ctx->stats.kernel_launches++;
    return 0;
}

// Ordered aggregation of the staged patches of the reference rows [a_lo, a_hi) into the pixel rows [y_lo, y_hi)
int launch_aggregate(lfbm5d_ctx *ctx, const PassCfg &pc, const LfWindow &win, int y_lo, int y_hi, int a_lo, int a_hi)
{
    if (y_hi <= y_lo || a_hi <= a_lo) return 0;
    const PassGeom pg = pass_geom(pc);
    AggArgs aa{};
    aa.C = pc.C; aa.A = pc.A; aa.k = pc.k; aa.N = pc.N; aa.log2N = 0;
    while ((1u << aa.log2N) < pc.N) aa.log2N++;
    aa.w = pc.wb; aa.h = pc.hb; aa.nc = pg.nc;
    aa.R = pg.R; aa.ent = ctx->spos.as<unsigned>();
    aa.zbuf = ctx->zbuf.as<float>(); aa.wbuf = ctx->wbuf.as<float>();
    aa.numsym = ctx->numsym.as<float>(); aa.densym = ctx->densym.as<float>();
    aa.arange = ctx->arange.as<int>(); aa.brange = ctx->brange.as<int>();
    aa.win = win;
    aa.y_lo = y_lo; aa.y_hi = y_hi; aa.a_min = a_lo; aa.a_max = a_hi - 1;
    aa.ty0 = y_lo / 16;
    dim3 grid((pc.wb + 15) / 16, (y_hi + 15) / 16 - aa.ty0, pc.A);
    const bool band = !(y_lo == 0 && y_hi == (int) pc.hb && a_lo == 0 && a_hi == pg.nr);
    void (*kagg)(AggArgs) = band ? k_aggregate<8, 1, true> : k_aggregate<8, 1, false>;         // validate(): k is 8, 12 or 16, C is 1 or 3
    if (pc.C == 3 && pc.k == 16) kagg = band ? k_aggregate<16, 3, true> : k_aggregate<16, 3, false>;
    else if (pc.C == 3 && pc.k == 12) kagg = band ? k_aggregate<12, 3, true> : k_aggregate<12, 3, false>;
    else if (pc.C == 1 && pc.k == 12) kagg = band ? k_aggregate<12, 1, true> : k_aggregate<12, 1, false>;
    else if (pc.C == 3 && pc.k == 8) kagg = band ? k_aggregate<8, 3, true> : k_aggregate<8, 3, false>;
    else if (pc.C == 1 && pc.k == 16) kagg = band ? k_aggregate<16, 1, true> : k_aggregate<16, 1, false>;
    LAUNCH(ctx, kagg, grid, 256, 0, aa);
    return 0;
}

// partial-window branch: which reference patches of SAI pst still hold a pixel without weight
int launch_active_refs(lfbm5d_ctx *ctx, const PassCfg &pc, int pst, unsigned **cnt_out)
{
    const size_t Rr = pc.rows.size() * pc.cols.size();
    if (ctx->act.ensure(Rr + 16)) return 1;
    unsigned *cnt = reinterpret_cast<unsigned *>(ctx->act.as<unsigned char>() + ((Rr + 3) & ~(size_t) 3));
    CK(cudaMemsetAsync(cnt, 0, 12, ctx->stream));
    LAUNCH(ctx, k_active_refs, (unsigned) ((Rr + 255) / 256), 256, 0,
           ctx->densym.as<float>() + (size_t) pst * pc.C * pc.wb * pc.hb, ctx->rows.as<int>(), ctx->cols.as<int>(), (int) pc.cols.size(), (int) Rr,
           (int) pc.wb, (int) pc.k, ctx->act.as<unsigned char>(), cnt);
    *cnt_out = cnt;
    return 0;
}

// ---- the elementwise kernels on a range of rows: one GPU passes all of them, a team rank those of its band. An empty range
// launches nothing. ----

// padded working set of the window from noisy / basic and the accumulators, padded rows [y_lo, y_hi); running estimate below est_hi
void launch_pad(lfbm5d_ctx *ctx, const PassCfg &pc, const LfWindow &win, const float *noisy, const float *basic, int y_lo, int y_hi, int est_hi)
{
    if (y_hi <= y_lo) return;
    LAUNCH(ctx, k_pad, grid_for(ctx, (size_t) win.A * (y_hi - y_lo) * pc.wb), 256, 0, noisy, basic, ctx->num.as<float>(), ctx->den.as<float>(),
           ctx->nsym.as<float>(), ctx->bsym.as<float>(), ctx->numsym.as<float>(), ctx->densym.as<float>(), ctx->est0.as<float>(), win,
           (int) pc.W, (int) pc.H, (int) pc.C, (int) pc.n, y_lo, y_hi - y_lo, est_hi);
}

// running estimate of the window on the padded rows [y_lo, y_hi), from its padded buffers
void launch_est0(lfbm5d_ctx *ctx, const PassCfg &pc, const LfWindow &win, int y_lo, int y_hi)
{
    if (y_hi <= y_lo) return;
    LAUNCH(ctx, k_est0, grid_for(ctx, (size_t) win.A * (y_hi - y_lo) * pc.wb), 256, 0, pc.step == 1 ? ctx->nsym.as<float>() : ctx->bsym.as<float>(),
           ctx->numsym.as<float>(), ctx->densym.as<float>(), ctx->est0.as<float>(), win, (int) pc.wb, (int) pc.hb, (int) pc.C, y_lo, y_hi - y_lo);
}

// padded accumulators of the window back into num / den on the interior rows [i_lo, i_hi); count (optional) += covered entries
void launch_unpad(lfbm5d_ctx *ctx, const PassCfg &pc, const LfWindow &win, int i_lo, int i_hi, unsigned long long *count)
{
    if (i_hi <= i_lo) return;
    LAUNCH(ctx, k_unpad, grid_for(ctx, (size_t) win.A * pc.C * (i_hi - i_lo) * pc.W), 256, 0, ctx->num.as<float>(), ctx->den.as<float>(),
           ctx->numsym.as<float>(), ctx->densym.as<float>(), win, (int) pc.W, (int) pc.H, (int) pc.C, (int) pc.n, i_lo, i_hi - i_lo, (int) pc.k, count);
}

// *out += zero weights on the rows [y_lo, y_hi) of the C planes [h][w] from den
void launch_count_zero(lfbm5d_ctx *ctx, const float *den, int C, int w, int h, int y_lo, int y_hi, unsigned long long *out)
{
    if (y_hi <= y_lo) return;
    LAUNCH(ctx, k_count_zero, grid_for(ctx, (size_t) C * (y_hi - y_lo) * w), 256, 0, den, C, (size_t) w * h, w, y_lo, y_hi - y_lo, out);
}

// colour transform (mode: k_color) of the rows [i_lo, i_hi) of nsai SAIs [3][H][W] from lf into out (in place: out = lf)
void launch_color(lfbm5d_ctx *ctx, cudaStream_t strm, const float *lf, float *out, const unsigned *mask, unsigned nsai, unsigned W, unsigned H,
                  unsigned cs, int mode, int i_lo, int i_hi)
{
    if (i_hi <= i_lo) return;
    LAUNCH_ON(ctx, strm, k_color, grid_for(ctx, (size_t) nsai * (i_hi - i_lo) * W), 256, 0, lf, out, mask, nsai, (int) W, (int) H, cs, mode, i_lo, i_hi - i_lo);
}

// final estimate of the step (k_final) on the rows [i_lo, i_hi) of the SAIs [st0, st0 + nsai), from this context's num / den
void launch_final(lfbm5d_ctx *ctx, const StepState &S, float *noisy, float *basic, float *out, unsigned st0, unsigned nsai, int inputs_back,
                  int i_lo, int i_hi)
{
    if (i_hi <= i_lo) return;
    const lfbm5d_params &p = S.p;
    const size_t off = st0 * S.each();
    LAUNCH(ctx, k_final, grid_for(ctx, (size_t) nsai * (i_hi - i_lo) * p.width), 256, 0, ctx->num.as<float>() + off, ctx->den.as<float>() + off,
           noisy + off, basic ? basic + off : nullptr, out + off, ctx->mask.as<unsigned>() + st0, nsai, (int) p.width, (int) p.height, (int) p.chnls,
           S.step, p.color_space, S.docolor ? 1 : 0, inputs_back, i_lo, i_hi - i_lo);
}

// the zero blocks behind nsym / bsym that the packed / register-resident group kernels gather "reads as zeros" patches from
int clear_zero_blocks(lfbm5d_ctx *ctx, const PassCfg &pc)
{
    const size_t plane = (size_t) pc.wb * pc.hb;
    CK(cudaMemsetAsync(ctx->nsym.as<float>() + (size_t) pc.A * pc.C * plane, 0, (size_t) pc.C * plane * 4, ctx->stream));
    if (pc.step == 2) CK(cudaMemsetAsync(ctx->bsym.as<float>() + (size_t) pc.A * pc.C * plane, 0, (size_t) pc.C * plane * 4, ctx->stream));
    return 0;
}

// One core call on the padded device buffers of the window (nsym/bsym/numsym/densym/est0 already filled).
// cst = slot the window was centred on: pst != cst is the partial-window branch (core:531-821 / :1332-1658).
int run_pass(lfbm5d_ctx *ctx, const PassCfg &pc, const LfWindow &win, int pst, int cst = -1)
{
    const bool partial = cst >= 0 && cst != pst;
    if (ensure_tables(ctx)) return 1;
    int act_ymax = -1, act_xmax = -1;       // partial-window branch: last row / column of a reference patch that is still processed
    if (partial) {
        unsigned *cnt = nullptr;
        if (launch_active_refs(ctx, pc, pst, &cnt)) return 1;
        unsigned h3[3] = { 0, 0, 0 };
        CK(cudaMemcpyAsync(h3, cnt, 12, cudaMemcpyDeviceToHost, ctx->stream));
        CK(cudaStreamSynchronize(ctx->stream));
        if (h3[0] == 0) return 0;       // nothing left to denoise in this SAI (core:160-165)
        act_ymax = (int) h3[1]; act_xmax = (int) h3[2];
    }
    const PassGeom pg = pass_geom(pc);
    const int R = pg.R;
    if (ctx->timing) CK(cudaEventRecord(ctx->ev[0], ctx->stream));
    SatPlan *Pp = sat_plan(ctx, pc, win, pst, partial, act_ymax, act_xmax);
    if (!Pp) return 1;
    const SatPlan &P = *Pp;
    if (next_sat_epoch(ctx)) return 1;
    cudaEvent_t sat0 = ctx->ev[2], sat1 = ctx->ev[3];
    if (ctx->timing) CK(cudaEventRecord(sat0, ctx->stream));
    // Self matching (summed-area planes, selection) stays on the main stream; disparity matching (planes, argmin, ties) runs
    // beside it on a second stream: the issue-bound plane kernels overlap with the bandwidth-bound argmin and the latency-bound
    // selection / tie kernels of the other branch. The two launches use disjoint plane indices of bnd / progress.
    cudaStream_t sB = ctx->stream3;
    CK(cudaEventRecord(ctx->ev_fork, ctx->stream));
    CK(cudaStreamWaitEvent(sB, ctx->ev_fork, 0));
    // the disparity planes are launched first: they finish first and their argmin then runs under the self planes
    if (launch_stereo(ctx, pc, P, 0, P.nslots, sB, ctx->timing ? ctx->ev_satb : nullptr, [&]() -> int {
            if (pg.nself > 0) {
                LAUNCH(ctx, k_fill, grid_for(ctx, (size_t) pg.nself * R), 256, 0, ctx->s_mir.as<float>(), 2 * pg.threshold, (size_t) pg.nself * R);   // core:3317
                if (launch_sat_self(ctx, pc, P, 0, P.nself_groups, ctx->stream)) return 1;
            }
            if (ctx->timing) CK(cudaEventRecord(sat1, ctx->stream));
            // ---- selection ----
            if (pg.nself > 0) { if (launch_self_select(ctx, pc, ctx->stream)) return 1; }
            else
                LAUNCH(ctx, k_bm_identity, (R + 255) / 256, 256, 0, ctx->rows.as<int>(), ctx->cols.as<int>(), pg.nc, (int) pc.wb, 0, R, (int) pc.N,
                       ctx->bmcount.as<unsigned>(), ctx->bmidx.as<unsigned>());
            return 0;
        })) return 1;
    CK(cudaEventRecord(ctx->ev_join, sB));
    CK(cudaStreamWaitEvent(ctx->stream, ctx->ev_join, 0));
    if (launch_group_masks(ctx, pc, win, (int) pst, 0, R)) return 1;
    if (ctx->timing) CK(cudaEventRecord(ctx->ev[1], ctx->stream));
    if (ctx->bm_only) { CK(cudaGetLastError()); return 0; }

    // ---- groups, then the ordered aggregation of the staged patches ----
    if (clear_zero_blocks(ctx, pc) || launch_groups(ctx, pc, win, pst, partial, 0, R)) return 1;
    if (ctx->timing) CK(cudaEventRecord(ctx->ev[4], ctx->stream));
    if (launch_aggregate(ctx, pc, win, 0, (int) pc.hb, 0, pg.nr)) return 1;
    CK(cudaGetLastError());
    ctx->stats.window_passes++;
    if (ctx->timing) {
        cudaEvent_t e2;
        CK(cudaEventCreate(&e2));
        CK(cudaEventRecord(e2, ctx->stream));
        CK(cudaEventSynchronize(e2));
        float a = 0, b = 0, c = 0, d = 0;
        cudaEventElapsedTime(&a, ctx->ev[0], ctx->ev[1]);
        cudaEventElapsedTime(&b, ctx->ev[1], ctx->ev[4]);
        cudaEventElapsedTime(&c, sat0, sat1);
        { float cb = 0.f; cudaEventElapsedTime(&cb, sat0, ctx->ev_satb); c = std::max(c, cb); }      // both plane kernels done (several chunks: the last chunk's planes, earlier chunks' argmin included)
        cudaEventElapsedTime(&d, ctx->ev[4], e2);
        ctx->stats.ms_block_matching += a; ctx->stats.ms_groups += b; ctx->stats.ms_sat += c; ctx->stats.ms_aggregate += d;
        cudaEventDestroy(e2);
    }
    return 0;
}

// ---- the reference's step driver for nb_threads == 1 (bm5d.cpp:165-407 / :861-1106) on device-resident light fields, in three parts:
// step_begin (colour transform, zeroed accumulators, tables), step_window (one angular window: pad, core call(s), unpad) and
// step_end (num / den, inverse colour transforms). step_device strings them together with the window selection of the schedule
// section above.
int step_begin(lfbm5d_ctx *ctx, int step, const lfbm5d_params *p, float *d_noisy, float *d_basic, const unsigned *mask)
{
    if (validate(p, step)) return 1;
    CK(cudaSetDevice(ctx->device));
    StepState &S = ctx->ss;
    if (step_state_init(S, step, p, mask)) return 1;
    S.d_noisy = d_noisy; S.d_basic = d_basic;
    const unsigned asize = S.asize();
    const size_t each = S.each();
    ctx->sched.clear();
    if (ctx->timing) { CK(cudaEventCreate(&S.e_begin)); CK(cudaEventRecord(S.e_begin, ctx->stream)); }
    S.bm0 = ctx->stats.ms_block_matching; S.gr0 = ctx->stats.ms_groups;

    if (ctx->mask.ensure(asize * 4) || ctx->num.ensure(asize * each * 4) || ctx->den.ensure(asize * each * 4)) return 1;
    CK(cudaMemcpyAsync(ctx->mask.p, S.mask.data(), asize * 4, cudaMemcpyHostToDevice, ctx->stream));
    if (S.docolor && !ctx->io.on) {      // (host entry points: done SAI by SAI behind the uploads)
        launch_color(ctx, ctx->stream, d_noisy, d_noisy, ctx->mask.as<unsigned>(), asize, p->width, p->height, p->color_space, 1, 0, p->height);
        if (step == 2)
            launch_color(ctx, ctx->stream, d_basic, d_basic, ctx->mask.as<unsigned>(), asize, p->width, p->height, p->color_space, 1, 0, p->height);
    }
    CK(cudaMemsetAsync(ctx->num.p, 0, asize * each * 4, ctx->stream));
    CK(cudaMemsetAsync(ctx->den.p, 0, asize * each * 4, ctx->stream));
    if (setup_tables(ctx, step, p, S.tau_4D)) return 1;
    if (ensure_pass_buffers(ctx, S.pc) || upload_grid(ctx, S.pc)) return 1;
    return 0;
}

// zero weights of the items[i]-th C planes [h][w] from base, one count per item
int count_zeros(lfbm5d_ctx *ctx, const float *base, int C, int w, int h, const std::vector<unsigned> &items, std::vector<unsigned long long> &out)
{
    if (ctx->counters.ensure((items.size() + 8) * 8)) return 1;
    unsigned long long *counters = ctx->counters.as<unsigned long long>();
    CK(cudaMemsetAsync(counters, 0, items.size() * 8, ctx->stream));
    for (size_t i = 0; i < items.size(); i++)
        launch_count_zero(ctx, base + items[i] * (size_t) C * w * h, C, w, h, 0, h, counters + i);
    out.resize(items.size());
    CK(cudaMemcpyAsync(out.data(), counters, items.size() * 8, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    return 0;
}

int step_select(lfbm5d_ctx *ctx, unsigned &ps, unsigned &pt)
{
    const StepState &S = ctx->ss;
    return select_window(S, ps, pt, [&](const std::vector<unsigned> &sais, std::vector<unsigned long long> &zeros) {
        return count_zeros(ctx, ctx->den.as<float>(), (int) S.p.chnls, (int) S.p.width, (int) S.p.height, sais, zeros);
    });
}

// One angular window centred (and clamped) on SAI (ps, pt): bm5d.cpp:204-402
int step_window(lfbm5d_ctx *ctx, unsigned ps, unsigned pt)
{
    StepState &S = ctx->ss;
    const lfbm5d_params *p = &S.p;
    const int step = S.step;
    const PassCfg &pc = S.pc;
    WindowRun w;
    if (window_open(S, w, ps, pt) && setup_tables(ctx, step, p, S.tau_4D)) return 1;
    const LfWindow &win = w.win;
    const unsigned A = (unsigned) win.A;
    if (ctx->io.on)
        for (unsigned a = 0; a < A; a++) if (win.mask[a]) CK(cudaStreamWaitEvent(ctx->stream, ctx->io.up[win.st[a]], 0));
    launch_pad(ctx, pc, win, S.d_noisy, step == 2 ? S.d_basic : nullptr, 0, (int) pc.hb, (int) pc.hb);
    auto count = [&](const std::vector<unsigned> &slots, std::vector<unsigned long long> &zeros) {
        return count_zeros(ctx, ctx->densym.as<float>(), (int) pc.C, (int) pc.wb, (int) pc.hb, slots, zeros);
    };
    while (w.n_unproc) {
        if (window_next(w, count)) return 1;
        if (w.calls > 0) launch_est0(ctx, pc, win, 0, (int) pc.hb);      // the running estimate after the previous core call (core:169 / :937)
        if (run_pass(ctx, pc, win, (int) w.pst_asw, (int) w.cst_asw)) return 1;
        // crop the accumulators back into the light field and count the covered entries in the same pass over them
        unsigned long long *counters = ctx->counters.as<unsigned long long>();
        CK(cudaMemsetAsync(counters, 0, 8, ctx->stream));
        launch_unpad(ctx, pc, win, 0, (int) pc.H, counters);
        unsigned long long cnt = 0;
        CK(cudaMemcpyAsync(&cnt, counters, 8, cudaMemcpyDeviceToHost, ctx->stream));
        CK(cudaStreamSynchronize(ctx->stream));
        window_after_call(S, w, cnt);
    }
    const std::array<unsigned, 4> e = window_close(S, w);
    ctx->sched.insert(ctx->sched.end(), e.begin(), e.end());
    return 0;
}

// final estimate of one SAI (bm5d.cpp:405 / :706 + inverse colour transform) and its way back to the host
int io_finish_sai(lfbm5d_ctx *ctx, unsigned st)
{
    StepState &S = ctx->ss;
    const lfbm5d_params *p = &S.p;
    const size_t each = S.each();
    HostIO &io = ctx->io;
    launch_final(ctx, S, S.d_noisy, S.d_basic, io.d_out, st, 1, 0, 0, (int) p->height);
    CK(cudaEventRecord(io.fin[st], ctx->stream));
    CK(cudaStreamWaitEvent(ctx->stream4, io.fin[st], 0));
    CK(cudaMemcpyAsync(io.h_out[st], io.d_out + st * each, each * 4, cudaMemcpyDeviceToHost, ctx->stream4));
    io.done[st] = 1;
    return 0;
}

// after window number io.window of the step: SAIs no later plan window touches are final
int io_after_window(lfbm5d_ctx *ctx, unsigned ps, unsigned pt, unsigned calls)
{
    HostIO &io = ctx->io;
    const unsigned i = io.window++;
    if (!io.plan_ok) return 0;
    if (2 * i + 1 >= io.plan.size() || io.plan[2 * i] != ps || io.plan[2 * i + 1] != pt || calls != 1) { io.plan_ok = false; return 0; }      // the run left the static plan
    const unsigned asize = ctx->ss.asize();
    for (unsigned st = 0; st < asize; st++)
        if (ctx->ss.mask[st] && !io.done[st] && io.last_use[st] == (int) i && io_finish_sai(ctx, st)) return 1;
    return 0;
}

int step_end(lfbm5d_ctx *ctx, float *d_out)
{
    StepState &S = ctx->ss;
    const unsigned asize = S.asize();
    if (ctx->io.on) {      // whatever the plan did not finish early
        for (unsigned st = 0; st < asize; st++) if (S.mask[st] && !ctx->io.done[st] && io_finish_sai(ctx, st)) return 1;
    } else
        launch_final(ctx, S, S.d_noisy, S.d_basic, d_out, 0, asize, 1, 0, (int) S.p.height);
    CK(cudaGetLastError());
    if (ctx->timing) {
        cudaEvent_t e_end = nullptr;
        CK(cudaEventCreate(&e_end));
        CK(cudaEventRecord(e_end, ctx->stream));
        CK(cudaEventSynchronize(e_end));
        float total = 0;
        cudaEventElapsedTime(&total, S.e_begin, e_end);
        ctx->stats.ms_other += total - (ctx->stats.ms_block_matching - S.bm0) - (ctx->stats.ms_groups - S.gr0);
        cudaEventDestroy(S.e_begin); cudaEventDestroy(e_end);
    }
    CK(cudaStreamSynchronize(ctx->stream));
    return 0;
}

int step_device(lfbm5d_ctx *ctx, int step, const lfbm5d_params *p, float *d_noisy, float *d_basic, float *d_out, const unsigned *mask)
{
    if (step_begin(ctx, step, p, d_noisy, d_basic, mask)) return 1;
    ctx->sched.clear();
    while (ctx->ss.remaining) {
        unsigned ps = 0, pt = 0;
        if (step_select(ctx, ps, pt) || step_window(ctx, ps, pt)) return 1;
        if (ctx->io.on && io_after_window(ctx, ps, pt, ctx->sched.back())) return 1;
        if (ctx->max_passes && ctx->ss.passes >= ctx->max_passes) break;
    }
    return step_end(ctx, d_out);
}

// out[c][i][j] = numsym / densym on the unpadded interior, without a zero guard (bm3d.cpp:476-477, :682-683)
__global__ void k_ratio_crop(const float *__restrict__ numsym, const float *__restrict__ densym, float *__restrict__ out, int W, int H, int C, int n)
{
    const int wb = W + 2 * n, hb = H + 2 * n;
    const size_t plane = (size_t) W * H, plane_b = (size_t) wb * hb, total = plane * C;
    for (size_t t = (size_t) blockIdx.x * blockDim.x + threadIdx.x; t < total; t += (size_t) gridDim.x * blockDim.x) {
        const int c = (int) (t / plane);
        const size_t px = t - (size_t) c * plane;
        const int i = (int) (px / W), j = (int) (px - (size_t) i * W);
        const size_t src = (size_t) c * plane_b + (size_t) (i + n) * wb + (j + n);
        out[t] = numsym[src] / densym[src];
    }
}

int validate_bm3d(const lfbm3d_params *p)
{
    if (!p) return fail("null params");
    if (p->chnls != 1 && p->chnls != 3) return fail("chnls must be 1 or 3");
    if (p->nHard != p->nWien) return fail("nHard must equal nWien (the reference passes the nHard-padded image to its 2nd step, bm3d.cpp:175)");
    for (int s = 0; s < 2; s++) {
        const unsigned k = s ? p->kWien : p->kHard, N = s ? p->NWien : p->NHard, t2 = s ? p->tau_2D_wien : p->tau_2D_hard;
        if (k != 8 && k != 12 && k != 16) return fail("patch size must be 8, 12 or 16 in this build");
        if (k == 12 && t2 == LFBM5D_BIOR) return fail("tau_2D = bior needs a power-of-two patch size (k = 8 or 16); k = 12 takes dct");
        if (N < 2 || N > LF_MAXN || (N & (N - 1))) return fail("N must be a power of two in [2, 32]");
        if (t2 != LFBM5D_DCT && t2 != LFBM5D_BIOR) return fail("tau_2D must be dct or bior for BM3D");
        if ((s ? p->pWien : p->pHard) == 0) return fail("processing step must be >= 1");
    }
    if (p->nHard + 1 < std::max(p->kHard, p->kWien)) return fail("nHard must be >= k - 1");
    if (p->color_space > LFBM5D_RGB) return fail("Wrong type of transform. Must be OPP, YUV, or YCbCr!!");
    if (p->width < 16 || p->height < 16) return fail("image smaller than a patch");
    if (p->width < p->nHard || p->height < p->nHard) return fail("image smaller than the padding nHard");
    return 0;
}

// run_bm3d on every SAI (bm3d_LF.cpp:110-119 -> bm3d.cpp:86-287, nb_threads == 1): each SAI is the A = 1, no-disparity,
// Hadamard case of a window pass with BM3D's thresholds. SAIs are independent, so step 1 runs for all of them before step 2
// (one constant-table switch instead of 2 per SAI); results are identical to the per-SAI order.
int bm3d_device(lfbm5d_ctx *ctx, const lfbm3d_params *p, float *d_noisy, const unsigned *mask, float *d_basic, float *d_out)
{
    if (validate_bm3d(p)) return 1;
    CK(cudaSetDevice(ctx->device));
    const unsigned asize = p->asize, C = p->chnls, W = p->width, H = p->height;
    const size_t HW = (size_t) W * H, each = HW * C;
    const bool docolor = C == 3 && p->color_space != LFBM5D_RGB;
    if (ctx->mask.ensure(asize * 4) || ctx->num.ensure(each * 4) || ctx->den.ensure(each * 4)) return 1;
    CK(cudaMemcpyAsync(ctx->mask.p, mask, asize * 4, cudaMemcpyHostToDevice, ctx->stream));
    if (docolor) launch_color(ctx, ctx->stream, d_noisy, d_noisy, ctx->mask.as<unsigned>(), asize, W, H, p->color_space, 1, 0, H);   // bm3d.cpp:117
    ctx->sched.clear();
    for (int step = 1; step <= 2; step++) {
        lfbm5d_params q{};
        q.sigma = p->sigma; q.lambda = p->lambdaHard3D; q.ang_major = LFBM5D_ROWMAJOR; q.awidth = q.aheight = 1; q.an = 0;
        q.width = W; q.height = H; q.chnls = C;
        q.N = step == 1 ? p->NHard : p->NWien; q.nSim = step == 1 ? p->nHard : p->nWien; q.nDisp = 0;
        q.k = step == 1 ? p->kHard : p->kWien; q.p = step == 1 ? p->pHard : p->pWien;
        q.tau_2D = step == 1 ? p->tau_2D_hard : p->tau_2D_wien; q.tau_4D = LFBM5D_ID; q.tau_5D = LFBM5D_HADAMARD;
        q.color_space = p->color_space; q.nb_threads = 1;
        PassCfg pc;
        if (make_passcfg(pc, step, &q, LFBM5D_ID)) return 1;
        pc.useSD = (step == 1 ? p->useSD_h : p->useSD_w) ? 2 : 0;
        float st3[3];
        if (estimate_sigma(p->sigma, st3, C, p->color_space)) return fail("unknown colour space");
        pc.tauMatch = step == 1 ? (C == 1 ? 3.f : 1.f) * (st3[0] < 35.0f ? 2500 : 5000)      // bm3d.cpp:340
                                : (st3[0] < 35.0f ? 400 : 3500);                             // bm3d.cpp:532
        if (setup_tables(ctx, step, &q, LFBM5D_ID, true) || ensure_pass_buffers(ctx, pc) || upload_grid(ctx, pc)) return 1;
        LfWindow win{};
        win.A = 1; win.st[0] = 0; win.mask[0] = 1; win.proc[0] = 0;
        float *dst = step == 1 ? d_basic : d_out;
        for (unsigned st = 0; st < asize; st++) {
            if (!mask[st]) continue;
            CK(cudaMemsetAsync(ctx->num.p, 0, each * 4, ctx->stream));
            CK(cudaMemsetAsync(ctx->den.p, 0, each * 4, ctx->stream));
            launch_pad(ctx, pc, win, d_noisy + st * each, step == 2 ? d_basic + st * each : nullptr, 0, (int) pc.hb, (int) pc.hb);
            if (run_pass(ctx, pc, win, 0)) return 1;
            LAUNCH(ctx, k_ratio_crop, grid_for(ctx, each), 256, 0, ctx->numsym.as<float>(), ctx->densym.as<float>(), dst + st * each, (int) W,
                   (int) H, (int) C, (int) pc.n);
        }
    }
    if (docolor)      // bm3d.cpp:269-274
        for (float *lf : { d_out, d_noisy, d_basic }) launch_color(ctx, ctx->stream, lf, lf, ctx->mask.as<unsigned>(), asize, W, H, p->color_space, 0, 0, H);
    CK(cudaGetLastError());
    CK(cudaStreamSynchronize(ctx->stream));
    return 0;
}

int upload_lf(lfbm5d_ctx *ctx, DevBuf &buf, float *const *host, const unsigned *mask, unsigned asize, size_t each)
{
    if (buf.ensure(asize * each * 4)) return 1;
    for (unsigned st = 0; st < asize; st++)
        if (mask[st]) CK(cudaMemcpyAsync(buf.as<float>() + st * each, host[st], each * 4, cudaMemcpyHostToDevice, ctx->stream));
    return 0;
}
int download_lf(lfbm5d_ctx *ctx, const DevBuf &buf, float *const *host, const unsigned *mask, unsigned asize, size_t each)
{
    for (unsigned st = 0; st < asize; st++)
        if (mask[st]) CK(cudaMemcpyAsync(host[st], buf.as<float>() + st * each, each * 4, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    return 0;
}

} // namespace

extern "C" {

const char *lfbm5d_last_error(void) { return g_err.c_str(); }

int lfbm5d_create(lfbm5d_ctx **out, int device)
{
    if (!out) return fail("null output pointer");
    int ndev = 0;
    cudaError_t e = cudaGetDeviceCount(&ndev);
    if (e != cudaSuccess || ndev == 0) return fail(std::string("no CUDA device available (") + cudaGetErrorString(e) + "); this library has no CPU fallback");
    if (device < 0 || device >= ndev) return fail("invalid device index");
    CK(cudaSetDevice(device));
    lfbm5d_ctx *ctx = new lfbm5d_ctx();
    ctx->device = device;
    cudaDeviceProp prop;
    CK(cudaGetDeviceProperties(&prop, device));
    ctx->num_sms = prop.multiProcessorCount;
    ctx->smem_optin = (int) prop.sharedMemPerBlockOptin;
    CK(cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking));
    CK(cudaStreamCreateWithFlags(&ctx->stream2, cudaStreamNonBlocking));
    CK(cudaStreamCreateWithFlags(&ctx->stream3, cudaStreamNonBlocking));
    CK(cudaStreamCreateWithFlags(&ctx->stream4, cudaStreamNonBlocking));
    CK(cudaEventCreateWithFlags(&ctx->ev_fork, cudaEventDisableTiming));
    CK(cudaEventCreateWithFlags(&ctx->ev_join, cudaEventDisableTiming));
    CK(cudaEventCreate(&ctx->ev_satb));
    for (auto &ev : ctx->ev) CK(cudaEventCreate(&ev));
    *out = ctx;
    return 0;
}

void lfbm5d_destroy(lfbm5d_ctx *ctx)
{
    if (!ctx) return;
    cudaSetDevice(ctx->device);
    cudaStreamSynchronize(ctx->stream);
    DevBuf *all[] = { &ctx->noisy, &ctx->basic, &ctx->out, &ctx->num, &ctx->den, &ctx->mask, &ctx->nsym, &ctx->bsym, &ctx->numsym,
                      &ctx->densym, &ctx->est0, &ctx->s_at, &ctx->s_mir, &ctx->sums, &ctx->first, &ctx->shape, &ctx->bmcount,
                      &ctx->bmidx, &ctx->bnd, &ctx->progress, &ctx->rowmap, &ctx->colmap, &ctx->rows, &ctx->cols, &ctx->counters,
                      &ctx->zbuf, &ctx->wbuf, &ctx->spos, &ctx->arange, &ctx->brange, &ctx->gmask, &ctx->shape_lut, &ctx->tielist, &ctx->stielist, &ctx->act, &ctx->rt_noisy, &ctx->rt_basic, &ctx->frow, &ctx->fcol };
    for (auto b : all) b->release();
    for (auto &e : ctx->sat_cache) { e->d_planes.release(); e->d_groups.release(); }
    for (auto &ev : ctx->ev) if (ev) cudaEventDestroy(ev);
    cudaStreamDestroy(ctx->stream);
    if (ctx->stream2) cudaStreamDestroy(ctx->stream2);
    if (ctx->stream3) cudaStreamDestroy(ctx->stream3);
    if (ctx->stream4) cudaStreamDestroy(ctx->stream4);
    for (auto e : ctx->io.up) cudaEventDestroy(e);
    for (auto e : ctx->io.fin) cudaEventDestroy(e);
    if (ctx->ev_fork) cudaEventDestroy(ctx->ev_fork);
    if (ctx->ev_join) cudaEventDestroy(ctx->ev_join);
    if (ctx->ev_satb) cudaEventDestroy(ctx->ev_satb);
    delete ctx;
}

void lfbm5d_reset_stats(lfbm5d_ctx *ctx) { if (ctx) ctx->stats = lfbm5d_stats{}; }
void lfbm5d_get_stats(lfbm5d_ctx *ctx, lfbm5d_stats *out) { if (ctx && out) *out = ctx->stats; }
void lfbm5d_enable_timing(lfbm5d_ctx *ctx, int on) { if (ctx) ctx->timing = on != 0; }
void *lfbm5d_stream(lfbm5d_ctx *ctx) { return ctx ? (void *) ctx->stream : nullptr; }
void lfbm5d_set_max_passes(lfbm5d_ctx *ctx, unsigned m) { if (ctx) ctx->max_passes = m; }

int lfbm5d_group_cluster(lfbm5d_ctx *ctx, int step, const lfbm5d_params *p, int *cluster_size, int *max_active_clusters)
{
    if (!ctx || !cluster_size || !max_active_clusters) return fail("null argument");
    if (step != 1 && step != 2) return fail("step must be 1 or 2");
    if (validate(p, step)) return 1;
    CK(cudaSetDevice(ctx->device));
    GroupCluster gc;
    if (group_cluster(ctx, step, p->k, 2 * p->an + 1, p->N, p->tau_2D, gc)) return 1;
    *cluster_size = gc.cl;
    *max_active_clusters = gc.max_active;
    return 0;
}

int lfbm5d_group_kernel(lfbm5d_ctx *ctx, int step, const lfbm5d_params *p, char *name, unsigned cap)
{
    if (!ctx || !name || cap == 0) return fail("null argument");
    if (step != 1 && step != 2) return fail("step must be 1 or 2");
    if (validate(p, step)) return 1;
    CK(cudaSetDevice(ctx->device));
    GroupKernel gk;
    if (group_kernel(ctx, step, p->k, 2 * p->an + 1, p->N, p->chnls, p->tau_2D, p->tau_5D, p->useSD ? 1 : 0, gk)) return 1;
    snprintf(name, cap, "%s", gk.name);
    return 0;
}

int lfbm5d_step1_device(lfbm5d_ctx *ctx, const lfbm5d_params *p, float *d_noisy_io, const unsigned *sai_mask, float *d_basic_out)
{
    if (!ctx || !d_noisy_io || !sai_mask || !d_basic_out) return fail("null argument");
    return step_device(ctx, 1, p, d_noisy_io, nullptr, d_basic_out, sai_mask);
}
int lfbm5d_step2_device(lfbm5d_ctx *ctx, const lfbm5d_params *p, float *d_noisy_io, float *d_basic_io, const unsigned *sai_mask,
                        float *d_denoised_out)
{
    if (!ctx || !d_noisy_io || !d_basic_io || !sai_mask || !d_denoised_out) return fail("null argument");
    return step_device(ctx, 2, p, d_noisy_io, d_basic_io, d_denoised_out, sai_mask);
}

// One step through the host entry points, pipelined SAI by SAI (HostIO): uploads + colour transform on stream2 in the order of the
// static plan, early return of the colour-round-tripped inputs and of the finished SAIs on stream4, the passes on the main stream.
static int step_host(lfbm5d_ctx *ctx, int step, const lfbm5d_params *p, float *const *noisy_io, float *const *basic_io, const unsigned *sai_mask,
                     float *const *out_host)
{
    if (validate(p, step)) return 1;
    CK(cudaSetDevice(ctx->device));
    const unsigned asize = p->awidth * p->aheight;
    const size_t HW = (size_t) p->width * p->height, each = HW * p->chnls;
    if (ctx->noisy.ensure(asize * each * 4) || ctx->out.ensure(asize * each * 4) || ctx->mask.ensure(asize * 4)) return 1;
    if (step == 2 && ctx->basic.ensure(asize * each * 4)) return 1;
    const bool docolor = p->chnls == 3 && p->color_space != LFBM5D_RGB;
    if (docolor && (ctx->rt_noisy.ensure(asize * each * 4) || (step == 2 && ctx->rt_basic.ensure(asize * each * 4)))) return 1;
    // The constant tables of the step go to the device first: a change of tables needs a device-wide synchronisation (ensure_tables),
    // and from inside step_begin it would wait for every upload queued below — the first window would start after the whole light
    // field had arrived instead of after its nine SAIs. Here nothing is in flight yet; step_begin then finds the tables in place.
    if (setup_tables(ctx, step, p, p->tau_4D)) return 1;
    HostIO &io = ctx->io;
    while (io.up.size() < asize) { cudaEvent_t e; CK(cudaEventCreateWithFlags(&e, cudaEventDisableTiming)); io.up.push_back(e); }
    while (io.fin.size() < asize) { cudaEvent_t e; CK(cudaEventCreateWithFlags(&e, cudaEventDisableTiming)); io.fin.push_back(e); }
    // static plan of the step: upload order = order of first use; last_use = when an SAI becomes final
    std::vector<unsigned> plan6((size_t) (asize + 1) * 6);
    const unsigned nwin = lfbm5d_step_plan(p, sai_mask, plan6.data(), asize + 1);
    const unsigned asw = 2 * p->an + 1;
    io.plan.clear(); io.last_use.assign(asize, -1); io.done.assign(asize, 0); io.plan_ok = true; io.window = 0;
    io.h_out = out_host; io.d_out = ctx->out.as<float>();
    std::vector<unsigned> order;
    std::vector<char> queued(asize, 0);
    for (unsigned i = 0; i < nwin; i++) {
        const unsigned *e = &plan6[6 * i];
        io.plan.push_back(e[0]); io.plan.push_back(e[1]);
        for (unsigned s = e[2]; s < e[2] + asw; s++)
            for (unsigned t = e[3]; t < e[3] + asw; t++) {
                const unsigned st = sai_index(*p, s, t);
                io.last_use[st] = (int) i;
                if (sai_mask[st] && !queued[st]) { queued[st] = 1; order.push_back(st); }
            }
    }
    for (unsigned st = 0; st < asize; st++) if (sai_mask[st] && !queued[st]) order.push_back(st);
    cudaStream_t sU = ctx->stream2, sD = ctx->stream4;
    // the buffers may still be read by copies of an earlier call on these streams: they were synchronised at its end
    CK(cudaMemcpyAsync(ctx->mask.p, sai_mask, asize * 4, cudaMemcpyHostToDevice, sU));
    for (unsigned st : order) {
        float *dn = ctx->noisy.as<float>() + st * each, *db = step == 2 ? ctx->basic.as<float>() + st * each : nullptr;
        CK(cudaMemcpyAsync(dn, noisy_io[st], each * 4, cudaMemcpyHostToDevice, sU));
        if (db) CK(cudaMemcpyAsync(db, basic_io[st], each * 4, cudaMemcpyHostToDevice, sU));
        if (docolor) {
            const unsigned *m1 = ctx->mask.as<unsigned>() + st;
            // what the reference leaves in its inputs (forward then inverse transform), then the working colour space in place
            const unsigned W = p->width, H = p->height, cs = p->color_space;
            launch_color(ctx, sU, dn, ctx->rt_noisy.as<float>() + st * each, m1, 1, W, H, cs, 2, 0, H);
            launch_color(ctx, sU, dn, dn, m1, 1, W, H, cs, 1, 0, H);
            if (db) {
                launch_color(ctx, sU, db, ctx->rt_basic.as<float>() + st * each, m1, 1, W, H, cs, 2, 0, H);
                launch_color(ctx, sU, db, db, m1, 1, W, H, cs, 1, 0, H);
            }
        }
        CK(cudaEventRecord(io.up[st], sU));
        if (docolor) {
            CK(cudaStreamWaitEvent(sD, io.up[st], 0));
            CK(cudaMemcpyAsync(noisy_io[st], ctx->rt_noisy.as<float>() + st * each, each * 4, cudaMemcpyDeviceToHost, sD));
            if (db) CK(cudaMemcpyAsync(basic_io[st], ctx->rt_basic.as<float>() + st * each, each * 4, cudaMemcpyDeviceToHost, sD));
        }
    }
    io.on = true;
    const int rc = step_device(ctx, step, p, ctx->noisy.as<float>(), step == 2 ? ctx->basic.as<float>() : nullptr, ctx->out.as<float>(), sai_mask);
    io.on = false;
    cudaStreamSynchronize(sU);
    cudaStreamSynchronize(sD);
    if (rc) return 1;
    CK(cudaGetLastError());
    return 0;
}

int lfbm5d_step1(lfbm5d_ctx *ctx, const lfbm5d_params *p, float *const *noisy_io, const unsigned *sai_mask, float *const *basic_out)
{
    if (!ctx || !noisy_io || !sai_mask || !basic_out) return fail("null argument");
    return step_host(ctx, 1, p, noisy_io, nullptr, sai_mask, basic_out);
}

int lfbm5d_step2(lfbm5d_ctx *ctx, const lfbm5d_params *p, float *const *noisy_io, float *const *basic_io, const unsigned *sai_mask,
                 float *const *denoised_out)
{
    if (!ctx || !noisy_io || !basic_io || !sai_mask || !denoised_out) return fail("null argument");
    return step_host(ctx, 2, p, noisy_io, basic_io, sai_mask, denoised_out);
}

int lfbm3d_run(lfbm5d_ctx *ctx, const lfbm3d_params *p, float *const *noisy_io, const unsigned *sai_mask, float *const *basic_out,
               float *const *denoised_out)
{
    if (!ctx || !noisy_io || !sai_mask || !basic_out || !denoised_out) return fail("null argument");
    if (validate_bm3d(p)) return 1;
    CK(cudaSetDevice(ctx->device));
    const size_t each = (size_t) p->width * p->height * p->chnls;
    if (upload_lf(ctx, ctx->noisy, noisy_io, sai_mask, p->asize, each) || ctx->basic.ensure(p->asize * each * 4) ||
        ctx->out.ensure(p->asize * each * 4)) return 1;
    if (bm3d_device(ctx, p, ctx->noisy.as<float>(), sai_mask, ctx->basic.as<float>(), ctx->out.as<float>())) return 1;
    if (download_lf(ctx, ctx->noisy, noisy_io, sai_mask, p->asize, each) || download_lf(ctx, ctx->basic, basic_out, sai_mask, p->asize, each))
        return 1;
    return download_lf(ctx, ctx->out, denoised_out, sai_mask, p->asize, each);
}

int lfbm3d_run_device(lfbm5d_ctx *ctx, const lfbm3d_params *p, float *d_noisy_io, const unsigned *sai_mask, float *d_basic_out,
                      float *d_denoised_out)
{
    if (!ctx || !d_noisy_io || !sai_mask || !d_basic_out || !d_denoised_out) return fail("null argument");
    return bm3d_device(ctx, p, d_noisy_io, sai_mask, d_basic_out, d_denoised_out);
}

unsigned lfbm5d_step_plan(const lfbm5d_params *p, const unsigned *sai_mask, unsigned *out, unsigned max_entries)
{
    // Static form of the reference's window selection (bm5d.cpp:182-202): every SAI of a finished window is marked processed
    // (:370-382 or the end of the inner loop), so an unprocessed SAI has never been aggregated into, all of them tie on the
    // number of zero weights and the `>=` scan keeps the highest index. Entries: (ps, pt, min_s, min_t, level, sadct) where
    // level = longest chain of earlier windows sharing an SAI (same-level windows commute) and sadct = 1 once a window with
    // an empty SAI has been seen in sequential order (:276-280 is sticky).
    if (!p || !sai_mask || !out) return 0;
    const unsigned aw = p->awidth, ah = p->aheight, asize = aw * ah, asw = 2 * p->an + 1;
    if (asw > aw || asw > ah) return 0;
    std::vector<unsigned> proc(asize);
    unsigned remaining = 0;
    for (unsigned st = 0; st < asize; st++) { proc[st] = !sai_mask[st]; remaining += proc[st] == 0; }
    const unsigned max_proc = remaining;
    const unsigned cst = sai_index(*p, ah / 2, aw / 2);
    std::vector<int> last_level(asize, -1);
    unsigned n = 0, sticky = 0;
    while (remaining && n < max_entries) {
        unsigned pst_g = cst, ps, pt;
        if (remaining != max_proc || !sai_mask[cst])
            for (unsigned st = 0; st < asize; st++) if (!proc[st]) pst_g = st;
        sai_coords(*p, pst_g, ps, pt);
        int c_s, min_s, max_s, c_t, min_t, max_t;
        angular_search_window(c_s, min_s, max_s, ps, ah, p->an);
        angular_search_window(c_t, min_t, max_t, pt, aw, p->an);
        int level = 0;
        unsigned nmasked = 0;
        for (int s = min_s; s <= max_s; s++)
            for (int t2 = min_t; t2 <= max_t; t2++) {
                const unsigned st = sai_index(*p, s, t2);
                level = std::max(level, last_level[st] + 1);
                nmasked += sai_mask[st] == 0;
            }
        if (nmasked && p->tau_4D == LFBM5D_DCT) sticky = 1;
        for (int s = min_s; s <= max_s; s++)
            for (int t2 = min_t; t2 <= max_t; t2++) {
                const unsigned st = sai_index(*p, s, t2);
                last_level[st] = level;
                if (!proc[st]) proc[st] = 1;
            }
        unsigned *e = out + 6 * n;
        e[0] = ps; e[1] = pt; e[2] = (unsigned) min_s; e[3] = (unsigned) min_t; e[4] = (unsigned) level; e[5] = sticky;
        n++;
        remaining = 0;
        for (unsigned st = 0; st < asize; st++) remaining += proc[st] == 0;
    }
    return n;
}

unsigned lfbm5d_debug_schedule(lfbm5d_ctx *ctx, unsigned *out, unsigned max_entries)
{
    if (!ctx) return 0;
    const unsigned n = (unsigned) (ctx->sched.size() / 4);
    for (unsigned i = 0; i < n && i < max_entries; i++)
        for (int j = 0; j < 4; j++) out[4 * i + j] = ctx->sched[4 * i + j];
    return n;
}

// Set-up shared by the two debug exports: the parameters are validated as one window of (2 an + 1)^2 SAIs, the tables and buffers of
// a pass are made ready, and `win` becomes the identity window (window SAI a is plane a); the caller sets its mask and proc flags.
static int debug_setup(lfbm5d_ctx *ctx, int step, const lfbm5d_params *p, PassCfg &pc, LfWindow &win)
{
    lfbm5d_params q = *p;
    if (q.awidth < 2 * q.an + 1) q.awidth = 2 * q.an + 1;
    if (q.aheight < 2 * q.an + 1) q.aheight = 2 * q.an + 1;
    if (validate(&q, step)) return 1;
    CK(cudaSetDevice(ctx->device));
    if (make_passcfg(pc, step, p, p->tau_4D) || setup_tables(ctx, step, p, p->tau_4D) || ensure_pass_buffers(ctx, pc) || upload_grid(ctx, pc))
        return 1;
    win.A = (int) pc.A;
    for (unsigned a = 0; a < pc.A; a++) win.st[a] = (int) a;
    return 0;
}

// Read-back shared by the two debug exports, after the stream has drained: the match lists scattered onto the padded positions of
// their reference patches, and the disparity argmin and shape flags of the first `nplanes` planes.
static int debug_readback(lfbm5d_ctx *ctx, const PassCfg &pc, unsigned nplanes, unsigned *out_count, unsigned *out_idx, unsigned *out_first,
                          unsigned *out_shape)
{
    CK(cudaStreamSynchronize(ctx->stream));
    const size_t plane = (size_t) pc.wb * pc.hb;
    const size_t R = pc.rows.size() * pc.cols.size(), nc = pc.cols.size();
    if (out_count && out_idx) {
        std::vector<unsigned> cnt(R), idx(R * (pc.N + 1));
        CK(cudaMemcpy(cnt.data(), ctx->bmcount.p, R * 4, cudaMemcpyDeviceToHost));
        CK(cudaMemcpy(idx.data(), ctx->bmidx.p, R * (pc.N + 1) * 4, cudaMemcpyDeviceToHost));
        memset(out_count, 0, plane * 4);
        for (size_t r = 0; r < R; r++) {
            const size_t k_r = (size_t) pc.rows[r / nc] * pc.wb + pc.cols[r % nc];
            out_count[k_r] = cnt[r];
            for (unsigned n = 0; n < cnt[r]; n++) out_idx[k_r * (pc.N + 1) + n] = idx[r * (pc.N + 1) + n];
        }
    }
    if (out_first) CK(cudaMemcpy(out_first, ctx->first.p, nplanes * plane * 4, cudaMemcpyDeviceToHost));
    if (out_shape) {
        std::vector<unsigned char> sh(nplanes * plane);
        CK(cudaMemcpy(sh.data(), ctx->shape.p, nplanes * plane, cudaMemcpyDeviceToHost));
        for (size_t i = 0; i < sh.size(); i++) out_shape[i] = sh[i];
    }
    return 0;
}

int lfbm5d_debug_pass(lfbm5d_ctx *ctx, int step, const lfbm5d_params *p, const float *noisy_sym, const float *basic_sym,
                      float *num_sym_io, float *den_sym_io, const unsigned *mask_asw, const unsigned *procSAI_asw, unsigned pst,
                      unsigned *out_count, unsigned *out_idx, unsigned *out_first, unsigned *out_shape)
{
    return lfbm5d_debug_pass_ex(ctx, step, p, noisy_sym, basic_sym, num_sym_io, den_sym_io, mask_asw, procSAI_asw, pst, pst, out_count, out_idx,
                                out_first, out_shape);
}

int lfbm5d_debug_pass_ex(lfbm5d_ctx *ctx, int step, const lfbm5d_params *p, const float *noisy_sym, const float *basic_sym,
                         float *num_sym_io, float *den_sym_io, const unsigned *mask_asw, const unsigned *procSAI_asw, unsigned cst, unsigned pst,
                         unsigned *out_count, unsigned *out_idx, unsigned *out_first, unsigned *out_shape)
{
    if (!ctx || !noisy_sym || !num_sym_io || !den_sym_io || !mask_asw || !procSAI_asw) return fail("null argument");
    if (step != 1 && step != 2) return fail("step must be 1 or 2");
    if (step == 2 && !basic_sym) return fail("step 2 needs the basic estimate");
    PassCfg pc;
    LfWindow win{};
    if (debug_setup(ctx, step, p, pc, win)) return 1;
    if (pst >= pc.A) return fail("pst out of range");
    const size_t plane = (size_t) pc.wb * pc.hb, bytes = pc.A * pc.C * plane * 4;
    for (unsigned a = 0; a < pc.A; a++) { win.mask[a] = mask_asw[a]; win.proc[a] = procSAI_asw[a]; }
    CK(cudaMemcpyAsync(ctx->nsym.p, noisy_sym, bytes, cudaMemcpyHostToDevice, ctx->stream));
    if (step == 2) CK(cudaMemcpyAsync(ctx->bsym.p, basic_sym, bytes, cudaMemcpyHostToDevice, ctx->stream));
    CK(cudaMemcpyAsync(ctx->numsym.p, num_sym_io, bytes, cudaMemcpyHostToDevice, ctx->stream));
    CK(cudaMemcpyAsync(ctx->densym.p, den_sym_io, bytes, cudaMemcpyHostToDevice, ctx->stream));
    CK(cudaMemsetAsync(ctx->first.p, 0xFF, pc.A * plane * 4, ctx->stream));
    CK(cudaMemsetAsync(ctx->shape.p, 0, pc.A * plane, ctx->stream));
    launch_est0(ctx, pc, win, 0, (int) pc.hb);
    if (cst >= pc.A) return fail("cst out of range");
    if (run_pass(ctx, pc, win, (int) pst, (int) cst)) return 1;
    CK(cudaMemcpyAsync(num_sym_io, ctx->numsym.p, bytes, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaMemcpyAsync(den_sym_io, ctx->densym.p, bytes, cudaMemcpyDeviceToHost, ctx->stream));
    return debug_readback(ctx, pc, pc.A, out_count, out_idx, out_first, out_shape);
}


int lfbm5d_debug_block_matching(lfbm5d_ctx *ctx, int step, const lfbm5d_params *p, const float *planes, unsigned nplanes,
                                unsigned *out_count, unsigned *out_idx, unsigned *out_first, unsigned *out_shape)
{
    if (!ctx || !p || !planes) return fail("null argument");
    if (step != 1 && step != 2) return fail("step must be 1 or 2");
    PassCfg pc;
    LfWindow win{};
    if (debug_setup(ctx, step, p, pc, win)) return 1;
    if (nplanes < 1 || nplanes > pc.A) return fail("1 <= nplanes <= (2*an+1)^2");
    const size_t plane = (size_t) pc.wb * pc.hb;
    for (unsigned a = 0; a < pc.A; a++) { win.mask[a] = a < nplanes; win.proc[a] = a >= nplanes; }
    CK(cudaMemcpyAsync(ctx->est0.p, planes, nplanes * plane * 4, cudaMemcpyHostToDevice, ctx->stream));
    CK(cudaMemsetAsync(ctx->first.p, 0xFF, pc.A * plane * 4, ctx->stream));
    CK(cudaMemsetAsync(ctx->shape.p, 0, pc.A * plane, ctx->stream));
    ctx->bm_only = true;
    const int rc = run_pass(ctx, pc, win, 0, 0);
    ctx->bm_only = false;
    if (rc) return 1;
    return debug_readback(ctx, pc, nplanes, out_count, out_idx, out_first, out_shape);
}

} // extern "C"

#include "team.cuh"
