/* lfbm5d_cuda.h — C ABI of the B200-native LFBM5D denoising hot path.
 *
 * This is the drop-in boundary: plain pointers and sizes, no C++ or torch types. The C++
 * adapters in lfbm5d_b200/csrc/lfbm5d_host.{h,cpp} wrap it with the reference's own signatures
 * (run_bm5d_1st_step / run_bm5d_2nd_step, bm5d.h:11-62; run_bm3d_LF, bm3d_LF.h:10-35) and
 * INTEGRATION.md shows the binding a maintainer of the reference would add.
 *
 * Semantics follow the reference with nb_threads == 1 (see DESIGN.md): results do not depend on
 * nb_threads, which is accepted and ignored. All functions return 0 (EXIT_SUCCESS) or 1
 * (EXIT_FAILURE) like the reference's drivers; lfbm5d_last_error() gives the reason.
 * There is no CPU fallback: without a CUDA device every call fails.
 */
#ifndef LFBM5D_CUDA_H
#define LFBM5D_CUDA_H
#include <stddef.h>
#ifdef __cplusplus
extern "C" {
#endif

/* enum values = the reference's #defines (main.cpp:20-32) */
enum { LFBM5D_YUV = 0, LFBM5D_YCBCR = 1, LFBM5D_OPP = 2, LFBM5D_RGB = 3, LFBM5D_ID = 4, LFBM5D_DCT = 5, LFBM5D_SADCT = 6,
       LFBM5D_BIOR = 7, LFBM5D_HADAMARD = 8, LFBM5D_HAAR = 9, LFBM5D_NONE = 10, LFBM5D_ROWMAJOR = 11, LFBM5D_COLMAJOR = 12 };

typedef struct lfbm5d_ctx lfbm5d_ctx;

/* POD mirror of the argument list of run_bm5d_1st_step / run_bm5d_2nd_step (bm5d.h:11-62). */
typedef struct lfbm5d_params {
    float    sigma;
    float    lambda;        /* lambdaHard5D; ignored by step 2 */
    unsigned ang_major;     /* LFBM5D_ROWMAJOR / LFBM5D_COLMAJOR */
    unsigned awidth, aheight;
    unsigned an;            /* anHard / anWien: half size of the angular search window, 0, 1 or 2 ((2an+1)^2 SAIs per group).
                             * an = 2 needs N * k^2 <= 2048 in step 1 and 2 * N * k^2 <= 2048 in step 2 (one channel of the
                             * 25-SAI group in the shared memory of one CTA): k = 16 with N <= 8 / N <= 4, k = 8 with N <= 32 / N <= 16 */
    unsigned width, height, chnls;
    unsigned N;             /* NHard / NWien: a power of two <= 32. At k = 16 and an <= 1, groups whose channel does not fit into the
                             * shared memory of one CTA (N = 32 in step 1, N >= 16 in step 2) run on 2- or 4-CTA clusters
                             * (lfbm5d_group_cluster tells which) */
    unsigned nSim;          /* half size of the self search window */
    unsigned nDisp;         /* half size of the disparity search window, <= 16 ((2nDisp+1)^2 offsets per SAI of the window).
                             * The SAIs must be at least nSim + nDisp pixels high and wide (mirror padding) */
    unsigned k;             /* kHard / kWien: patch side, 8, 12 or 16 (k = 16: N <= 32 at an <= 1 in both steps). k = 12 takes tau_2D = id or dct (bior needs a power of two),
                             * an = 0 or 1, and N * A * k * (k + 1) * 4 B <= 220 KB (twice that in step 2; A = (2an+1)^2):
                             * at an = 1, N <= 32 in step 1 and N <= 16 in step 2 */
    unsigned p;             /* pHard / pWien */
    unsigned useSD;
    unsigned tau_2D, tau_4D, tau_5D;
    unsigned color_space;
    unsigned nb_threads;    /* accepted, ignored (always nb_threads == 1 semantics) */
} lfbm5d_params;

/* POD mirror of run_bm3d_LF's argument list (bm3d_LF.h:10-35). */
typedef struct lfbm3d_params {
    float    sigma;
    unsigned asize;         /* number of SAIs */
    unsigned width, height, chnls;
    unsigned nHard, nWien, kHard, kWien, NHard, NWien, pHard, pWien;     /* kHard, kWien: 8, 12 or 16; 12 with dct only */
    unsigned useSD_h, useSD_w;
    unsigned tau_2D_hard, tau_2D_wien;
    float    lambdaHard3D;
    unsigned color_space;
    unsigned nb_threads;
} lfbm3d_params;

typedef struct lfbm5d_stats {
    unsigned long long kernel_launches;   /* kernels of this library launched since the last reset */
    unsigned           window_passes;     /* core calls (bm5d_{1st,2nd}_step equivalents) since the last reset */
    float              ms_block_matching; /* device time (CUDA events) since the last reset, when timing is enabled */
    float              ms_groups;         /* gather + transforms + shrinkage (+ staging of the filtered patches) */
    float              ms_aggregate;      /* ordered weighted aggregation */
    float              ms_other;
    float              ms_sat;            /* summed-area kernel alone (dominant block-matching kernel) */
} lfbm5d_stats;

int  lfbm5d_create(lfbm5d_ctx **out, int device);
void lfbm5d_destroy(lfbm5d_ctx *ctx);
const char *lfbm5d_last_error(void);
void lfbm5d_reset_stats(lfbm5d_ctx *ctx);
void lfbm5d_get_stats(lfbm5d_ctx *ctx, lfbm5d_stats *out);
void lfbm5d_enable_timing(lfbm5d_ctx *ctx, int on);   /* per-phase CUDA-event timing (adds synchronisation) */
/* cudaStream_t the library launches on, as void* (for callers that time with their own events) */
void *lfbm5d_stream(lfbm5d_ctx *ctx);

/* ---- reference-facing entry points: HOST buffers, copies inside ---------------------------------
 * noisy[st] / basic[st] / denoised[st]: asize caller-owned host arrays of width*height*chnls floats,
 * planar (c*W*H + i*W + j), st ordered per ang_major, like the reference's vector<vector<float>>.
 * Side effects as in the reference: noisy (and basic in step 2) come back colour-round-tripped
 * (bm5d.cpp:133, 711-714, 827-830, 1414-1419). Entries of masked-out SAIs are not touched. */
int lfbm5d_step1(lfbm5d_ctx *ctx, const lfbm5d_params *p, float *const *noisy_io, const unsigned *sai_mask,
                 float *const *basic_out);
int lfbm5d_step2(lfbm5d_ctx *ctx, const lfbm5d_params *p, float *const *noisy_io, float *const *basic_io,
                 const unsigned *sai_mask, float *const *denoised_out);
int lfbm3d_run(lfbm5d_ctx *ctx, const lfbm3d_params *p, float *const *noisy_io, const unsigned *sai_mask,
               float *const *basic_out, float *const *denoised_out);

/* ---- device-resident variants: d_* are device pointers to [asize][chnls][height][width] floats --- */
int lfbm5d_step1_device(lfbm5d_ctx *ctx, const lfbm5d_params *p, float *d_noisy_io, const unsigned *sai_mask, float *d_basic_out);
int lfbm5d_step2_device(lfbm5d_ctx *ctx, const lfbm5d_params *p, float *d_noisy_io, float *d_basic_io,
                        const unsigned *sai_mask, float *d_denoised_out);
int lfbm3d_run_device(lfbm5d_ctx *ctx, const lfbm3d_params *p, float *d_noisy_io, const unsigned *sai_mask, float *d_basic_out,
                      float *d_denoised_out);
/* stop after this many window passes per step (0 = run to completion); for bounded measurements only */
void lfbm5d_set_max_passes(lfbm5d_ctx *ctx, unsigned max_passes);
/* How the group kernel of `step` runs with these parameters on the context's device: *cluster_size = 1 when one CTA holds a
 * group, else the CTAs of the thread-block cluster that share it through distributed shared memory (2 or 4; k = 16 groups of
 * 3x3 windows over the opt-in shared memory of one CTA), with *max_active_clusters = cudaOccupancyMaxActiveClusters of that
 * configuration (0 for cluster_size 1). Fails, naming the cluster size and the bytes per CTA, if the device cannot run it. */
int lfbm5d_group_cluster(lfbm5d_ctx *ctx, int step, const lfbm5d_params *p, int *cluster_size, int *max_active_clusters);
/* Debug: the name of the group kernel a window pass of `step` launches with these parameters on the context's device, as
 * "k_groups<2,3>", "k_groups_w8<1>", "k_groups_cl<2,4>", ..., written NUL-terminated into name[cap] (truncated to fit).
 * Fails like lfbm5d_group_cluster on parameters the library rejects. */
int lfbm5d_group_kernel(lfbm5d_ctx *ctx, int step, const lfbm5d_params *p, char *name, unsigned cap);

/* ---- static window schedule ----------------------------------------------------------------------
 * The angular windows of a step (bm5d.cpp:171-402) in the order of the reference's schedule; windows that share no SAI commute.
 * out[6 * i + ...] = (ps, pt, first s of the window, first t, level, sadct) of window i: windows of one level share no SAI, and
 * sadct = 1 once a window with an empty SAI has turned tau_4D = dct into sadct (bm5d.cpp:276-280). Returns the number of windows. */
unsigned lfbm5d_step_plan(const lfbm5d_params *p, const unsigned *sai_mask, unsigned *out, unsigned max_entries);

/* ---- one light field on several GPUs: a team of ranks that split every window pass (lfbm5d_b200/csrc/team.cuh) ----
 * Reference rows of the pass grid, and the pixel rows they aggregate into, are dealt out in bands (north_star's row-band partition,
 * halo = search radius + patch size); the offset planes of the block matching are dealt out whole. Results are bit-identical to the
 * single-GPU entry points. One process per GPU: every rank creates its context, rank 0 draws lfbm5d_team_unique_id and ships the
 * 128 bytes to the others (e.g. torch.distributed / MPI broadcast), every rank calls lfbm5d_team_create_nccl (NCCL is loaded with
 * dlopen at that point). lfbm5d_team_create_emulated puts `world` ranks as contexts on ONE device and replaces the exchanges by
 * device copies (how the band logic is tested on a single GPU). */
typedef struct lfbm5d_team lfbm5d_team;
int  lfbm5d_team_create_emulated(lfbm5d_team **out, int device, int world);
int  lfbm5d_team_unique_id(char *id128);
int  lfbm5d_team_create_nccl(lfbm5d_team **out, lfbm5d_ctx *ctx, int rank, int world, const char *id128);
void lfbm5d_team_destroy(lfbm5d_team *team);
int  lfbm5d_team_local_ranks(lfbm5d_team *team);      /* emulated: world; NCCL: 1 */
/* Lanes (>= 1, default 1): the windows of a step form a static plan whose levels hold windows that share no SAI (lfbm5d_step_plan);
 * with n lanes up to n windows of a level run concurrently, each on its own contexts (pass buffers) and exchange state but on the
 * same light field, so that the latency-bound parts of one window pass hide behind the bandwidth-bound parts of another. Results
 * do not change (windows of a level commute). */
int  lfbm5d_team_set_lanes(lfbm5d_team *team, int nlanes);
unsigned long long lfbm5d_team_launches(lfbm5d_team *team);   /* kernels launched by all contexts of the team since their stats were reset */
/* One step (1 or 2) of ONE light field on the whole team. d_*: arrays of lfbm5d_team_local_ranks() device pointers, one replica of the
 * light field per local rank ([asize][chnls][height][width] floats, as for lfbm5d_step{1,2}_device). A rank reads and colour-transforms
 * only the rows of its band (+ halo) of d_noisy_io / d_basic_io; on return d_out[l] holds the rows [row_lo, keep_hi) of lfbm5d_team_band
 * (d_basic_io of step 2 may be the d_out of step 1 as it is: when the bands of step 2 read rows a rank did not keep from step 1 —
 * other patch size / step, another number of ranks with rows — the team first sends the step-1 bands around), or, with gather != 0,
 * the complete result on every rank. */
int  lfbm5d_team_step(lfbm5d_team *team, int step, const lfbm5d_params *p, float *const *d_noisy_io, float *const *d_basic_io,
                      const unsigned *sai_mask, float *const *d_out, int gather);
int  lfbm5d_team_band(lfbm5d_team *team, int rank, int *row_lo, int *row_hi, int *keep_hi);
/* the same bands from the parameters alone (before a step runs): what a host driver uploads to rank `rank` is [row_lo, keep_hi) */
int  lfbm5d_team_plan_band(int world, int rank, int step, const lfbm5d_params *p, int *row_lo, int *row_hi, int *keep_hi);
/* rows [row_lo, row_hi) of every plane of every non-masked SAI between host arrays (asize pointers, as for lfbm5d_step1) and a device
 * light field, asynchronously on the context's stream (lfbm5d_sync waits): the band-wise upload / download of a team's ranks */
int  lfbm5d_copy_rows(lfbm5d_ctx *ctx, float *const *host, float *d_lf, const unsigned *sai_mask, unsigned asize, unsigned chnls,
                      unsigned width, unsigned height, unsigned row_lo, unsigned row_hi, int to_device);
int  lfbm5d_sync(lfbm5d_ctx *ctx);
/* bytes this process sent so far; passes whose selection was redone from exchanged sums (fallback without peer view); reference
 * patches whose exact distance ties were resolved through the peer view; whether the peer view (cudaIpc / NVLink loads) is in use */
void lfbm5d_team_stats(lfbm5d_team *team, unsigned long long *bytes_exchanged, unsigned *passes_redone, unsigned long long *tie_patches,
                       int *peer_view);
/* per-phase device time (CUDA events on the first local rank): returns in out12 the ms accumulated since timing was switched on for
 * pad, est0 exchange, block matching, match exchange, selection + groups + aggregation 1, border exchange, aggregation 2, border + counter
 * exchange, and inside block matching: self planes, partial selection, disparity planes, disparity argmin */
void lfbm5d_team_timing(lfbm5d_team *team, int on, float *out12);
void lfbm5d_team_disable_peer_view(lfbm5d_team *team);   /* tests: force the exchange-and-redo fallback */
/* NCCL teams map each other's buffers with cudaIpc and exchange by storing straight into peer memory over NVLink (one copy kernel +
 * flag per exchange); on = 0 keeps the mappings for the exact-tie path but sends the exchanges through NCCL send / recv (comparison) */
void lfbm5d_team_use_peer_exchange(lfbm5d_team *team, int on);

/* ---- parity/debug exports (used by tests only) ---------------------------------------------------
 * One window pass (the reference's bm5d_1st_step / bm5d_2nd_step, `pst == cst` branch) on HOST padded
 * buffers [A][chnls][h_b][w_b], A = (2*an+1)^2, h_b = height + 2*(nSim+nDisp); p->width/height are the
 * UNPADDED sizes. num/den are updated in place. Optional outputs (may be NULL): self matches of the
 * reference SAI as count[h_b*w_b], idx[h_b*w_b*(N+1)]; stereo results first[A][h_b*w_b], shape[A][h_b*w_b]
 * in the layout of oracle/lfbm5d_oracle.h: orc_pass. */
int lfbm5d_debug_pass(lfbm5d_ctx *ctx, int step, const lfbm5d_params *p, const float *noisy_sym, const float *basic_sym,
                      float *num_sym_io, float *den_sym_io, const unsigned *mask_asw, const unsigned *procSAI_asw,
                      unsigned pst, unsigned *out_count, unsigned *out_idx, unsigned *out_first, unsigned *out_shape);
/* Same with the slot the window was centred on: pst != cst runs the partial-window branch (bm5d_core_processing.cpp:531-821 /
 * :1332-1658; only the grid patches of SAI pst that still hold a pixel without weight are processed). */
int lfbm5d_debug_pass_ex(lfbm5d_ctx *ctx, int step, const lfbm5d_params *p, const float *noisy_sym, const float *basic_sym,
                         float *num_sym_io, float *den_sym_io, const unsigned *mask_asw, const unsigned *procSAI_asw, unsigned cst,
                         unsigned pst, unsigned *out_count, unsigned *out_idx, unsigned *out_first, unsigned *out_shape);
/* Block matching alone (precompute_BM, bm5d_core_processing.cpp:3301-3461, and precompute_BM_stereo, :3479-3611) on HOST channel-0
 * planes [nplanes][h_b*w_b]: plane 0 is the reference SAI, planes 1.. are matched against it. Outputs as in lfbm5d_debug_pass
 * (count / idx of plane 0; first / shape [nplanes][h_b*w_b], rows of plane 0 unused). For parity tests at full plane sizes. */
int lfbm5d_debug_block_matching(lfbm5d_ctx *ctx, int step, const lfbm5d_params *p, const float *planes, unsigned nplanes,
                                unsigned *out_count, unsigned *out_idx, unsigned *out_first, unsigned *out_shape);
/* Window schedule of the last step call: (processed st, min_s, min_t, core calls) per window pass. */
unsigned lfbm5d_debug_schedule(lfbm5d_ctx *ctx, unsigned *out, unsigned max_entries);

#ifdef __cplusplus
}
#endif
#endif
