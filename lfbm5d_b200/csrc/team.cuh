// One light field on G GPUs — parallelism INSIDE a window pass (SURVEY.md 8(e), north_star's row-band partition).
//
// Rank g of a team owns the reference rows rows[a0_g .. a1_g) of the pass grid and the pixel rows P_g = [y0_g, y1_g) of the padded
// planes (y0_g = rows[a0_g] - n: the first row its groups can touch). Its groups write into C_g = [y0_g, c1_g), c1_g =
// rows[a1_g - 1] + n + k, which reaches O_g = [y1_g, c1_g) rows into the next rank's band ("search radius plus patch size").
// Per pass:
//   1. every rank builds the padded working set on C_g and the running estimate (channel 0) on P_g; the est0 rows are exchanged,
//      so that every rank holds the complete planes block matching reads;
//   2. block matching is PLANE parallel (the float32 summed-area recurrences run from the top-left corner of a plane: a plane is
//      not split): the 703 self planes and the 8 x 169 disparity planes are dealt out; disparity results (argmin / shape maps of a
//      SAI) go to everybody, the self candidates as per-rank top-(N+1) lists to the owner of the reference row, who merges them;
//   3. groups (transforms, shrinkage) for the own reference rows; aggregation, still in the reference's order: on O_g the sums of
//      rank g come BEFORE those of rank g + 1 (lower reference rows first), so rank g adds its patches on [c1_{g-1}, c1_g) first
//      and sends the rows O_g to rank g + 1, which continues the very same float sums with its own patches and returns the final
//      rows (rank g keeps them as a replica: it needs them to start the next pass that touches these SAIs).
// No float operation changes its operands or its order: num / den, and therefore every later match list, are BIT-IDENTICAL to
// the single-GPU run (tests/test_team_gpu.py). Exchanges are NCCL send/recv groups on the compute stream, or device copies
// between G contexts on ONE device (emulated team: how the band logic is tested on a single GPU).
#pragma once
#include "team_kernels.cuh"
#include <dlfcn.h>

namespace {

struct Band {
    int a0 = 0, a1 = 0;          // own reference rows
    int r0 = 0, r1 = 0;          // = a0 * nc, a1 * nc
    int y0 = 0, y1 = 0;          // owned pixel rows (padded coordinates)
    int c1 = 0;                  // own groups touch [y0, c1)
    int pc1 = 0;                 // c1 of the previous rank (y0 for rank 0): rows [y0, pc1) continue the previous rank's sums
    int i0 = 0, i1 = 0;          // interior (unpadded) rows of [y0, y1)
    int j0 = 0, j1 = 0;          // interior rows of [y0, c1): what the rank keeps up to date of num / den
};

struct PlaneShare { int s0, s1, sg0, sg1, pl0, pl1; };      // disparity slots, self groups and self planes of a rank in a pass

enum TeamBuf { TB_EST0, TB_FIRST, TB_SHAPE, TB_PKEY_SEND, TB_PKEY_ALL, TB_PCNT_SEND, TB_PCNT_ALL, TB_NUMSYM, TB_DENSYM, TB_COUNTERS,
               TB_S_AT, TB_S_MIR, TB_GSEND, TB_GRECV, TB_NBUF };

struct TeamSeg { int src, dst; int sbuf, dbuf; size_t soff, doff, bytes; };      // dst < 0: to every other rank, same place
#define TSLOT 2048           // bytes per rank in the counter buffers (two halves, used alternately: a peer can be one exchange ahead)
#define TSLOT_U64 256

// ---- NCCL through dlopen: the library has no link-time dependency on it (single-GPU users never load it) ----
struct NcclId { char internal[128]; };
struct NcclApi {
    void *h = nullptr;
    int (*GetUniqueId)(void *) = nullptr;
    int (*CommInitRank)(void **, int, NcclId, int) = nullptr;
    int (*CommDestroy)(void *) = nullptr;
    int (*Send)(const void *, size_t, int, int, void *, cudaStream_t) = nullptr;
    int (*Recv)(void *, size_t, int, int, void *, cudaStream_t) = nullptr;
    int (*GroupStart)() = nullptr;
    int (*GroupEnd)() = nullptr;
    const char *(*GetErrorString)(int) = nullptr;
};
NcclApi g_nccl;

int nccl_load()
{
    if (g_nccl.h) return 0;
    const char *names[] = { getenv("LFBM5D_NCCL_LIB"), "libnccl.so.2", "libnccl.so" };
    for (const char *nm : names) {
        if (!nm) continue;
        g_nccl.h = dlopen(nm, RTLD_NOW | RTLD_GLOBAL);
        if (g_nccl.h) break;
    }
    if (!g_nccl.h) return fail("libnccl.so.2 not found (set LFBM5D_NCCL_LIB, or import torch first: it brings its own)");
#define NCCL_SYM(field, name) *(void **) (&g_nccl.field) = dlsym(g_nccl.h, name); if (!g_nccl.field) return fail(std::string("NCCL symbol missing: ") + name)
    NCCL_SYM(GetUniqueId, "ncclGetUniqueId"); NCCL_SYM(CommInitRank, "ncclCommInitRank"); NCCL_SYM(CommDestroy, "ncclCommDestroy");
    NCCL_SYM(Send, "ncclSend"); NCCL_SYM(Recv, "ncclRecv"); NCCL_SYM(GroupStart, "ncclGroupStart"); NCCL_SYM(GroupEnd, "ncclGroupEnd");
    NCCL_SYM(GetErrorString, "ncclGetErrorString");
#undef NCCL_SYM
    return 0;
}
#define NCK(x) do { int r_ = (x); if (r_ != 0) return fail(std::string(#x) + ": " + g_nccl.GetErrorString(r_)); } while (0)

} // namespace

struct lfbm5d_team {
    int world = 1;
    std::vector<lfbm5d_ctx *> local;       // contexts of the ranks living in this process (emulated: all of them; NCCL: one)
    std::vector<int> local_rank;
    bool owns_ctx = false;
    void *comm = nullptr;                  // ncclComm_t (NCCL teams)
    // step state shared by all ranks (every rank takes the same decisions from the same exchanged counts)
    StepState ss;
    std::vector<Band> bands;
    std::vector<Band> held;                // bands of a step 1 that ended without a gather: rank g holds the rows [i0, j1) of LF_basic
    std::vector<float *> d_noisy, d_basic; // per local rank
    unsigned long long bytes_exchanged = 0;
    unsigned passes_redone = 0;
    // peer view of the other ranks' buffers (emulated: the other contexts' buffers; NCCL teams: cudaIpc mappings, NVLink): the
    // sampled self sums for the exact-tie selection, and every exchanged buffer for the direct peer-memory exchanges
    bool peer_ready = false, peer_ok = true;
    const float *peer_at[LF_MAXRANKS] = {}, *peer_mir[LF_MAXRANKS] = {};
    char *peer_buf[LF_MAXRANKS][TB_NBUF] = {};
    std::vector<void *> peer_opened;               // mappings to close
    std::vector<std::vector<size_t>> peer_keys;    // geometries whose buffers have been allocated and mapped
    unsigned xepoch = 0;                           // exchange counter (peer-memory exchanges)
    unsigned cparity = 0;                          // which half of the counter buffers the next counter exchange uses
    DevBuf xsegs, xflags, xdone, xflagptrs;
    bool use_peer_exchange = true;
    struct { LfWindow win; int pst = 0, cst = 0; bool partial = false; std::vector<PlaneShare> share; } pw;      // pass in flight
    WindowRun wf;                                 // window in flight
    std::vector<lfbm5d_team *> lanes;             // further lanes of this team: own contexts and exchange state, the same light field
    bool is_lane = false;
    unsigned long long tie_patches = 0;
    // per-phase device time of local rank 0 (lfbm5d_team_timing): events at the phase boundaries of a pass
    bool timing = false;
    cudaEvent_t tev[12] = {}, bev[6] = {};
    float phase_ms[12] = {};
};

namespace {

struct TeamCtxBufs { DevBuf pkey_send, pkey_all, pcnt_send, pcnt_all, counters, gsend, grecv; };
std::vector<std::pair<lfbm5d_ctx *, TeamCtxBufs *>> g_team_bufs;
TeamCtxBufs *team_bufs(lfbm5d_ctx *ctx)
{
    for (auto &e : g_team_bufs) if (e.first == ctx) return e.second;
    g_team_bufs.emplace_back(ctx, new TeamCtxBufs());
    return g_team_bufs.back().second;
}
void team_bufs_release(lfbm5d_ctx *ctx)
{
    for (size_t i = 0; i < g_team_bufs.size(); i++)
        if (g_team_bufs[i].first == ctx) {
            TeamCtxBufs *b = g_team_bufs[i].second;
            DevBuf *all[] = { &b->pkey_send, &b->pkey_all, &b->pcnt_send, &b->pcnt_all, &b->counters, &b->gsend, &b->grecv };
            for (auto d : all) d->release();
            delete b;
            g_team_bufs.erase(g_team_bufs.begin() + i);
            return;
        }
}

char *team_ptr(lfbm5d_ctx *ctx, int id)
{
    TeamCtxBufs *b = team_bufs(ctx);
    switch (id) {
        case TB_EST0: return ctx->est0.as<char>();
        case TB_FIRST: return ctx->first.as<char>();
        case TB_SHAPE: return ctx->shape.as<char>();
        case TB_PKEY_SEND: return b->pkey_send.as<char>();
        case TB_PKEY_ALL: return b->pkey_all.as<char>();
        case TB_PCNT_SEND: return b->pcnt_send.as<char>();
        case TB_PCNT_ALL: return b->pcnt_all.as<char>();
        case TB_NUMSYM: return ctx->numsym.as<char>();
        case TB_DENSYM: return ctx->densym.as<char>();
        case TB_COUNTERS: return b->counters.as<char>();
        case TB_S_AT: return ctx->s_at.as<char>();
        case TB_S_MIR: return ctx->s_mir.as<char>();
        case TB_GSEND: return b->gsend.as<char>();
        case TB_GRECV: return b->grecv.as<char>();
        default: return nullptr;
    }
}

// Exchange over peer memory (NCCL teams whose buffers are mapped into each other with cudaIpc): ONE kernel stores this rank's
// outgoing segments straight into the receivers' buffers over NVLink and then raises this exchange's number in every peer's flag
// slot; a one-warp kernel waits for the peers' numbers. Every exchange is a barrier of the team, so a rank is at most one exchange
// ahead of another: what exchange e + 1 writes never overlaps what a receiver still uses between e and e + 1 (team.cuh header:
// disjoint rows / planes / slots per exchange; the counter buffers alternate between two halves).
int team_exchange_peer(lfbm5d_team *T, const std::vector<TeamSeg> &segs)
{
    lfbm5d_ctx *ctx = T->local[0];
    const int me = T->local_rank[0], G = T->world;
    std::vector<PeerSegD> d;
    unsigned long long chunks = 0;
    for (const TeamSeg &s : segs) {
        if (!s.bytes || s.src != me) continue;
        for (int q = 0; q < G; q++) {
            if (s.dst >= 0 ? q != s.dst : q == me) continue;
            PeerSegD e;
            e.src = team_ptr(ctx, s.sbuf) + s.soff;
            e.dst = (q == me ? team_ptr(ctx, s.dbuf) : T->peer_buf[q][s.dbuf]) + s.doff;
            e.bytes = s.bytes; e.first_chunk = chunks;
            chunks += (s.bytes + PEER_CHUNK - 1) / PEER_CHUNK;
            d.push_back(e);
            if (q != me) T->bytes_exchanged += s.bytes;
        }
    }
    if (!d.empty()) {
        if (T->xsegs.ensure(d.size() * sizeof(PeerSegD))) return 1;
        CK(cudaMemcpyAsync(T->xsegs.p, d.data(), d.size() * sizeof(PeerSegD), cudaMemcpyHostToDevice, ctx->stream));      // pageable: staged before the call returns
    }
    const unsigned epoch = ++T->xepoch;
    const unsigned grid = (unsigned) std::max<unsigned long long>(1, std::min<unsigned long long>(chunks, (unsigned long long) ctx->num_sms * 8));
    k_peer_copy<<<grid, 256, 0, ctx->stream>>>(T->xsegs.as<PeerSegD>(), (int) d.size(), (unsigned) chunks, T->xdone.as<unsigned>(),
                                               T->xflagptrs.as<unsigned *>(), me, G, epoch);
    k_peer_wait<<<1, 32, 0, ctx->stream>>>(T->xflags.as<unsigned>(), me, G, epoch, T->xdone.as<unsigned>() + 8);
    ctx->stats.kernel_launches += 2;
    CK(cudaGetLastError());
    return 0;
}

// Execute a list of segments. NCCL team: one group of sends / receives on the compute stream of the (single) local rank.
// Emulated team: device copies between the contexts, fenced by device-wide synchronisations (test path).
int team_exchange(lfbm5d_team *T, const std::vector<TeamSeg> &segs)
{
    if (segs.empty()) return 0;
    if (T->comm && T->peer_ready && T->use_peer_exchange) return team_exchange_peer(T, segs);
    if (T->comm) {
        lfbm5d_ctx *ctx = T->local[0];
        const int me = T->local_rank[0];
        bool any = false;
        for (const TeamSeg &s : segs) if (s.bytes && (s.src == me || s.dst == me || s.dst < 0)) { any = true; break; }
        if (!any) return 0;
        NCK(g_nccl.GroupStart());
        for (const TeamSeg &s : segs) {
            if (!s.bytes) continue;
            if (s.dst < 0) {
                if (s.src == me) { for (int d = 0; d < T->world; d++) if (d != me) NCK(g_nccl.Send(team_ptr(ctx, s.sbuf) + s.soff, s.bytes, 0, d, T->comm, ctx->stream)); }
                else NCK(g_nccl.Recv(team_ptr(ctx, s.dbuf) + s.doff, s.bytes, 0, s.src, T->comm, ctx->stream));
                if (s.src == me) T->bytes_exchanged += s.bytes * (T->world - 1);
            } else if (s.src == s.dst) {
                if (s.src == me) CK(cudaMemcpyAsync(team_ptr(ctx, s.dbuf) + s.doff, team_ptr(ctx, s.sbuf) + s.soff, s.bytes, cudaMemcpyDeviceToDevice, ctx->stream));
            } else {
                if (s.src == me) { NCK(g_nccl.Send(team_ptr(ctx, s.sbuf) + s.soff, s.bytes, 0, s.dst, T->comm, ctx->stream)); T->bytes_exchanged += s.bytes; }
                if (s.dst == me) NCK(g_nccl.Recv(team_ptr(ctx, s.dbuf) + s.doff, s.bytes, 0, s.src, T->comm, ctx->stream));
            }
        }
        NCK(g_nccl.GroupEnd());
        return 0;
    }
    CK(cudaDeviceSynchronize());
    cudaStream_t st = T->local[0]->stream;
    for (const TeamSeg &s : segs) {
        if (!s.bytes) continue;
        for (int d = 0; d < T->world; d++) {
            if (s.dst >= 0 ? d != s.dst : d == s.src) continue;
            CK(cudaMemcpyAsync(team_ptr(T->local[d], s.dbuf) + s.doff, team_ptr(T->local[s.src], s.sbuf) + s.soff, s.bytes, cudaMemcpyDeviceToDevice, st));
            if (d != s.src) T->bytes_exchanged += s.bytes;
        }
    }
    CK(cudaDeviceSynchronize());
    return 0;
}

// Row bands of a pass grid for G ranks. Only as many ranks get rows as the no-triple-overlap rule allows (c1_g <= y0_{g+2}: a pixel
// row sees the groups of at most two ranks); the others own nothing and only take part in the block matching.
std::vector<Band> team_bands(const PassCfg &pc, int G)
{
    const int nr = (int) pc.rows.size(), nc = (int) pc.cols.size(), n = (int) pc.n, k = (int) pc.k, hb = (int) pc.hb, H = (int) pc.H;
    int Ge = G;
    std::vector<int> a0;
    for (; Ge >= 1; Ge--) {
        a0.assign(Ge + 1, 0);
        for (int g = 0; g <= Ge; g++) a0[g] = (int) ((long long) nr * g / Ge);
        bool ok = true;
        for (int g = 0; g < Ge; g++) if (a0[g + 1] <= a0[g]) ok = false;
        for (int g = 0; ok && g + 2 < Ge; g++)
            if (pc.rows[a0[g + 1] - 1] + n + k > pc.rows[a0[g + 2]] - n) ok = false;
        if (ok || Ge == 1) break;
    }
    std::vector<Band> B(G);
    for (int g = 0; g < G; g++) {
        Band &b = B[g];
        if (g < Ge) {
            b.a0 = a0[g]; b.a1 = a0[g + 1];
            b.y0 = g == 0 ? 0 : pc.rows[b.a0] - n;
            b.y1 = g == Ge - 1 ? hb : pc.rows[a0[g + 1]] - n;
            b.c1 = g == Ge - 1 ? hb : std::min(hb, pc.rows[b.a1 - 1] + n + k);
            b.pc1 = g == 0 ? 0 : B[g - 1].c1;
        } else { b.a0 = b.a1 = nr; b.y0 = b.y1 = b.c1 = b.pc1 = hb; }
        b.r0 = b.a0 * nc; b.r1 = b.a1 * nc;
        b.i0 = std::min(std::max(b.y0 - n, 0), H); b.i1 = std::min(std::max(b.y1 - n, 0), H);
        b.j0 = b.i0; b.j1 = std::min(std::max(b.c1 - n, 0), H);
        if (g == 0) { b.i0 = 0; b.j0 = 0; }
    }
    return B;
}

// Deal the offset planes of a pass out: disparity slots evenly (whole SAIs: their argmin needs all (2 nDisp + 1)^2 planes), then the self
// groups in contiguous runs so that every rank ends up with about the same number of planes.
std::vector<PlaneShare> team_planes(const SatPlan &P, int G)
{
    std::vector<PlaneShare> S(G);
    const int per_slot = P.planes_per_slot;
    const double total = (double) P.nself_planes + (double) P.nslots * per_slot;
    int sg = 0;
    double cum = 0.0;
    for (int g = 0; g < G; g++) {
        PlaneShare &s = S[g];
        s.s0 = (int) ((long long) P.nslots * g / G); s.s1 = (int) ((long long) P.nslots * (g + 1) / G);
        s.sg0 = sg;
        cum += (double) (s.s1 - s.s0) * per_slot;
        const double goal = total * (g + 1) / G;          // cumulative: rounding does not pile up on the last rank
        if (g == G - 1) sg = P.nself_groups;
        else
            while (sg < P.nself_groups && cum + P.groups[sg].nplanes / 2.0 <= goal) { cum += P.groups[sg].nplanes; sg++; }
        s.sg1 = sg;
        s.pl0 = s.sg0 < P.nself_groups ? P.groups[s.sg0].first_plane : P.nself_planes;
        s.pl1 = s.sg1 < P.nself_groups ? P.groups[s.sg1].first_plane : P.nself_planes;
    }
    return S;
}

int team_ensure(lfbm5d_team *T, lfbm5d_ctx *ctx, const PassCfg &pc)
{
    const PassGeom pg = pass_geom(pc);
    TeamCtxBufs *b = team_bufs(ctx);
    const size_t NM = pc.N + 1, G = (size_t) T->world;
    if (pg.nself > 0 && (b->pkey_send.ensure((size_t) pg.R * NM * 8) || b->pkey_all.ensure(G * pg.R * NM * 8) || b->pcnt_send.ensure((size_t) pg.R * 4) ||
                         b->pcnt_all.ensure(G * pg.R * 4))) return 1;
    if (b->counters.ensure(2 * G * TSLOT)) return 1;
    return 0;
}

// byte offset of rank g's slot in the half of the counter buffers the current counter exchange uses
size_t cslot(const lfbm5d_team *T, int g) { return ((size_t) T->cparity * T->world + g) * TSLOT; }

#define TMARK(i) do { if (T->timing) CK(cudaEventRecord(T->tev[i], T->local[0]->stream)); } while (0)

// ---- one core call of the team, in pieces (a lane enqueues bm + body and reads the counters later) ----
// block matching of the own planes + exchange of the match tables
int team_pass_bm(lfbm5d_team *T, const PassCfg &pc, const LfWindow &win, int pst, int cst)
{
    const bool partial = cst >= 0 && cst != pst;
    T->pw.win = win; T->pw.pst = pst; T->pw.cst = cst; T->pw.partial = partial;
    const int G = T->world, nl = (int) T->local.size();
    const PassGeom pg = pass_geom(pc);
    const size_t plane = pg.plane, NM = pc.N + 1;
    const int C = (int) pc.C, wb = (int) pc.wb;
    std::vector<SatPlan *> plans(nl);
    std::vector<PlaneShare> &share = T->pw.share;
    share.clear();
    TMARK(2);
    // ---- block matching: own planes ----
    for (int l = 0; l < nl; l++) {
        lfbm5d_ctx *ctx = T->local[l];
        const int g = T->local_rank[l];
        CK(cudaSetDevice(ctx->device));
        if (ensure_tables(ctx)) return 1;
        if (partial) {      // active reference patches of the own rows; block matching keeps its full extents in the team path
            unsigned *cnt = nullptr;
            if (launch_active_refs(ctx, pc, pst, &cnt)) return 1;
        }
        SatPlan *Pp = sat_plan(ctx, pc, win, pst, false, -1, -1);
        if (!Pp) return 1;
        plans[l] = Pp;
        const SatPlan &P = *Pp;
        if (share.empty()) share = team_planes(P, G);
        const PlaneShare &sh = share[g];
        if (next_sat_epoch(ctx)) return 1;
        cudaStream_t sB = ctx->stream3;
        CK(cudaEventRecord(ctx->ev_fork, ctx->stream));
        CK(cudaStreamWaitEvent(sB, ctx->ev_fork, 0));
        const bool tm = T->timing && l == 0;
        if (tm) CK(cudaEventRecord(T->bev[0], ctx->stream));
        // own disparity slots in chunks of the sums buffer, counted from sh.s0 (slot s still sits at s % nbuf)
        if (launch_stereo(ctx, pc, P, sh.s0, sh.s1, sB, tm ? T->bev[3] : nullptr, [&]() -> int {
                if (pg.nself > 0 && sh.pl1 > sh.pl0) {
                    LAUNCH(ctx, k_fill, grid_for(ctx, (size_t) (sh.pl1 - sh.pl0) * pg.R), 256, 0, ctx->s_mir.as<float>() + (size_t) sh.pl0 * pg.R,
                           2 * pg.threshold, (size_t) (sh.pl1 - sh.pl0) * pg.R);   // core:3317
                    if (launch_sat_self(ctx, pc, P, sh.sg0, sh.sg1, ctx->stream)) return 1;
                }
                if (tm) CK(cudaEventRecord(T->bev[1], ctx->stream));
                if (pg.nself > 0) {
                    TeamCtxBufs *b = team_bufs(ctx);
                    void (*kp)(SelGeom, const float *, const float *, int, int, unsigned *, unsigned long long *) = nullptr;
                    switch (pc.N) {
                        case 2: kp = k_bm_partial<3>; break;
                        case 4: kp = k_bm_partial<5>; break;
                        case 8: kp = k_bm_partial<9>; break;
                        case 16: kp = k_bm_partial<17>; break;
                        default: kp = k_bm_partial<33>; break;
                    }
                    LAUNCH(ctx, kp, (pg.R + 127) / 128, 128, 0, sel_geom(ctx, pc), ctx->s_at.as<float>(), ctx->s_mir.as<float>(), sh.pl0, sh.pl1,
                           b->pcnt_send.as<unsigned>(), b->pkey_send.as<unsigned long long>());
                }
                if (tm) CK(cudaEventRecord(T->bev[2], ctx->stream));
                return 0;
            })) return 1;
        if (tm) CK(cudaEventRecord(T->bev[4], sB));
        CK(cudaEventRecord(ctx->ev_join, sB));
        CK(cudaStreamWaitEvent(ctx->stream, ctx->ev_join, 0));
        if (tm) CK(cudaEventRecord(T->tev[3], ctx->stream));
        if (!T->comm && T->timing) CK(cudaDeviceSynchronize());      // emulated team under timing: one rank at a time on the device
    }
    const SatPlan &P0 = *plans[0];
    if (T->comm) TMARK(3);
    {   // ---- exchange: disparity maps to everybody, partial candidate lists to the owners of the reference rows ----
        std::vector<TeamSeg> segs;
        // a rank reads the disparity maps at the self matches of its own reference rows only: rows within nSim of them
        for (int g = 0; g < G; g++)
            for (int s = share[g].s0; s < share[g].s1; s++) {
                const int st = P0.stereo_sai[s];
                for (int h = 0; h < G; h++) {
                    const Band &bh = T->bands[h];
                    if (h == g || bh.a1 <= bh.a0) continue;
                    const int ylo = std::max(0, pc.rows[bh.a0] - (int) pc.nSim), yhi = std::min((int) pc.hb, pc.rows[bh.a1 - 1] + (int) pc.nSim + 1);
                    const size_t o = (size_t) st * plane + (size_t) ylo * wb, nb = (size_t) (yhi - ylo) * wb;
                    segs.push_back({ g, h, TB_FIRST, TB_FIRST, o * 4, o * 4, nb * 4 });
                    segs.push_back({ g, h, TB_SHAPE, TB_SHAPE, o, o, nb });
                }
            }
        if (pg.nself > 0)
            for (int g = 0; g < G; g++)
                for (int h = 0; h < G; h++) {
                    const Band &bh = T->bands[h];
                    const size_t nrp = (size_t) (bh.r1 - bh.r0);
                    segs.push_back({ g, h, TB_PKEY_SEND, TB_PKEY_ALL, (size_t) bh.r0 * NM * 8, ((size_t) g * pg.R + bh.r0) * NM * 8, nrp * NM * 8 });
                    segs.push_back({ g, h, TB_PCNT_SEND, TB_PCNT_ALL, (size_t) bh.r0 * 4, ((size_t) g * pg.R + bh.r0) * 4, nrp * 4 });
                }
        if (team_exchange(T, segs)) return 1;
    }
    return 0;
}

// merged selection, groups, both parts of the aggregation and the border exchanges of a pass (enqueue only, no host sync)
int team_pass_body(lfbm5d_team *T, const PassCfg &pc, bool redo)
{
    const LfWindow &win = T->pw.win;
    const int pst = T->pw.pst;
    const bool partial = T->pw.partial;
    const std::vector<PlaneShare> &share = T->pw.share;
    const int G = T->world, nl = (int) T->local.size();
    const PassGeom pg = pass_geom(pc);
    const size_t plane = pg.plane;
    const int C = (int) pc.C, wb = (int) pc.wb;
    TMARK(4);
    // ---- merged selection, groups and the first part of the aggregation: rows [pc1, c1) ----
    for (int l = 0; l < nl; l++) {
        lfbm5d_ctx *ctx = T->local[l];
        const int g = T->local_rank[l];
        const Band &bd = T->bands[g];
        TeamCtxBufs *b = team_bufs(ctx);
        CK(cudaSetDevice(ctx->device));
        unsigned long long *cnts = reinterpret_cast<unsigned long long *>(b->counters.as<char>() + cslot(T, g));
        CK(cudaMemsetAsync(cnts, 0, 64, ctx->stream));
        const int nown = bd.r1 - bd.r0;
        if (nown > 0) {
            if (pg.nself > 0 && !redo) {
                const SelGeom sg = sel_geom(ctx, pc);
                void (*km)(SelGeom, int, int, int, const unsigned *, const unsigned long long *, unsigned *, unsigned *, unsigned *, unsigned *) = nullptr;
                switch (pc.N) {
                    case 2: km = k_bm_merge<3>; break;
                    case 4: km = k_bm_merge<5>; break;
                    case 8: km = k_bm_merge<9>; break;
                    case 16: km = k_bm_merge<17>; break;
                    default: km = k_bm_merge<33>; break;
                }
                if (ctx->tielist.ensure(((size_t) pg.R + 1) * 4)) return 1;
                unsigned *tl = ctx->tielist.as<unsigned>();
                // with the peer view the tied patches are redone right here; without it they are only counted (cnts[1]) and the
                // team falls back to exchanging the complete sums and redoing the pass
                unsigned *tcount = T->peer_ready ? reinterpret_cast<unsigned *>(cnts + 2) : reinterpret_cast<unsigned *>(cnts + 1);
                LAUNCH(ctx, km, (nown + 127) / 128, 128, 0, sg, G, bd.r0, bd.r1, b->pcnt_all.as<unsigned>(), b->pkey_all.as<unsigned long long>(),
                       ctx->bmcount.as<unsigned>(), ctx->bmidx.as<unsigned>(), T->peer_ready ? tl : (unsigned *) nullptr, tcount);
                if (T->peer_ready) {
                    PeerTable pt{};
                    pt.G = G;
                    for (int q = 0; q < G; q++) { pt.s_at[q] = T->peer_at[q]; pt.s_mir[q] = T->peer_mir[q]; pt.pl0[q] = share[q].pl0; }
                    pt.pl0[G] = share[G - 1].pl1;
                    LAUNCH(ctx, k_bm_select, std::min<size_t>(nown, (size_t) ctx->num_sms * 16), 32, (size_t) pg.Ns * pg.Ns * 8, sg, ctx->s_at.as<float>(),
                           ctx->s_mir.as<float>(), ctx->bmcount.as<unsigned>(), ctx->bmidx.as<unsigned>(), (const unsigned *) tl,
                           (const unsigned *) reinterpret_cast<unsigned *>(cnts + 2), pt);
                }
            } else if (pg.nself > 0) {      // ties somewhere: every rank now holds the complete sums, the reference's selection as on one GPU
                if (launch_self_select(ctx, pc, ctx->stream)) return 1;
            } else
                LAUNCH(ctx, k_bm_identity, (nown + 255) / 256, 256, 0, ctx->rows.as<int>(), ctx->cols.as<int>(), pg.nc, wb, bd.r0, bd.r1, (int) pc.N,
                       ctx->bmcount.as<unsigned>(), ctx->bmidx.as<unsigned>());
            if (launch_group_masks(ctx, pc, win, pst, bd.r0, bd.r1)) return 1;
            if (clear_zero_blocks(ctx, pc) || launch_groups(ctx, pc, win, pst, partial, bd.r0, bd.r1)) return 1;
            if (launch_aggregate(ctx, pc, win, bd.pc1, bd.c1, bd.a0, bd.a1)) return 1;
        }
    }
    TMARK(5);
    {   // rows O_g = [y1, c1) go to the next rank, which continues the sums
        std::vector<TeamSeg> segs;
        for (int g = 0; g + 1 < G; g++) {
            const Band &bd = T->bands[g];
            if (bd.c1 <= bd.y1) continue;
            for (int a = 0; a < (int) pc.A; a++) {
                if (!win.mask[a] || win.proc[a]) continue;
                for (int c = 0; c < C; c++) {
                    const size_t off = (((size_t) a * C + c) * plane + (size_t) bd.y1 * wb) * 4, bytes = (size_t) (bd.c1 - bd.y1) * wb * 4;
                    segs.push_back({ g, g + 1, TB_NUMSYM, TB_NUMSYM, off, off, bytes });
                    segs.push_back({ g, g + 1, TB_DENSYM, TB_DENSYM, off, off, bytes });
                }
            }
        }
        if (team_exchange(T, segs)) return 1;
    }
    TMARK(6);
    // ---- second part of the aggregation: rows [y0, pc1) on top of the previous rank's sums; coverage and tie counts ----
    for (int l = 0; l < nl; l++) {
        lfbm5d_ctx *ctx = T->local[l];
        const int g = T->local_rank[l];
        const Band &bd = T->bands[g];
        TeamCtxBufs *b = team_bufs(ctx);
        CK(cudaSetDevice(ctx->device));
        if (bd.r1 > bd.r0 && launch_aggregate(ctx, pc, win, bd.y0, bd.pc1, bd.a0, bd.a1)) return 1;
        unsigned long long *cnts = reinterpret_cast<unsigned long long *>(b->counters.as<char>() + cslot(T, g));
        if (bd.i1 > bd.i0)
            LAUNCH(ctx, k_count_cov_rows, grid_for(ctx, (size_t) pc.A * C * (bd.i1 - bd.i0) * pc.W), 256, 0, ctx->densym.as<float>(), win, (int) pc.W, (int) pc.H,
                   C, (int) pc.n, (int) pc.k, bd.i0, bd.i1 - bd.i0, cnts);
    }
    TMARK(7);
    {   // final rows [y0, pc1) back to the previous rank (its replica of O_{g-1}); counters to everybody
        std::vector<TeamSeg> segs;
        for (int g = 1; g < G; g++) {
            const Band &bd = T->bands[g];
            if (bd.pc1 <= bd.y0) continue;
            for (int a = 0; a < (int) pc.A; a++) {
                if (!win.mask[a] || win.proc[a]) continue;
                for (int c = 0; c < C; c++) {
                    const size_t off = (((size_t) a * C + c) * plane + (size_t) bd.y0 * wb) * 4, bytes = (size_t) (bd.pc1 - bd.y0) * wb * 4;
                    segs.push_back({ g, g - 1, TB_NUMSYM, TB_NUMSYM, off, off, bytes });
                    segs.push_back({ g, g - 1, TB_DENSYM, TB_DENSYM, off, off, bytes });
                }
            }
        }
        for (int g = 0; g < G; g++) segs.push_back({ g, -1, TB_COUNTERS, TB_COUNTERS, cslot(T, g), cslot(T, g), 24 });
        if (team_exchange(T, segs)) return 1;
    }
    TMARK(8);
    return 0;
}

// every rank reads the same counters (host sync) and takes the same decisions from them
int team_pass_read(lfbm5d_team *T, unsigned long long *cov, unsigned long long *ties)
{
    const int G = T->world, nl = (int) T->local.size();
    // ---- every rank reads the same counters and takes the same decision ----
    unsigned long long total_cov = 0, total_ties = 0;
    for (int l = 0; l < nl; l++) {
        lfbm5d_ctx *ctx = T->local[l];
        CK(cudaSetDevice(ctx->device));
        std::vector<unsigned long long> h((size_t) G * TSLOT_U64);
        CK(cudaMemcpyAsync(h.data(), team_bufs(ctx)->counters.as<char>() + cslot(T, 0), h.size() * 8, cudaMemcpyDeviceToHost, ctx->stream));
        CK(cudaStreamSynchronize(ctx->stream));
        if (l == 0)
            for (int g = 0; g < G; g++) {
                total_cov += h[(size_t) g * TSLOT_U64]; total_ties += h[(size_t) g * TSLOT_U64 + 1] & 0xffffffffull;
                T->tie_patches += h[(size_t) g * TSLOT_U64 + 2] & 0xffffffffull;
            }
        ctx->stats.window_passes++;
    }
    T->cparity ^= 1u;
    *cov = total_cov; *ties = total_ties;
    if (T->timing) {    // phases 2..8: block matching, exchange, selection + groups + aggregation, exchange, aggregation 2, exchange
        for (int i = 2; i < 8; i++) { float ms = 0.f; if (cudaEventElapsedTime(&ms, T->tev[i], T->tev[i + 1]) == cudaSuccess) T->phase_ms[i] += ms; }
        // inside block matching: self planes, partial selection (main stream); disparity planes, argmin (second stream)
        const int pairs[4][2] = { { 0, 1 }, { 1, 2 }, { 0, 3 }, { 3, 4 } };
        for (int i = 0; i < 4; i++) { float ms = 0.f; if (cudaEventElapsedTime(&ms, T->bev[pairs[i][0]], T->bev[pairs[i][1]]) == cudaSuccess) T->phase_ms[8 + i] += ms; }
    }
    return 0;
}

// One core call of the team (all ranks in lockstep; `pst == cst` or the partial-window branch), synchronous.
// Returns through *cov the number of covered entries of LF_denoised_percent (summed over the ranks).
int team_pass_finish(lfbm5d_team *T, const PassCfg &pc, unsigned long long *cov)
{
    unsigned long long ties = 0;
    if (team_pass_read(T, cov, &ties)) return 1;
    if (ties == 0) return 0;
    // Exact float ties among the selected distances of some reference patch while the ranks cannot read each other's sums (no
    // peer view): the reference's result then depends on its heap algorithm over the complete candidate sequence. Redo the pass
    // from the padded accumulators with the complete sums on every rank (the planes are still there: only their exchange, the
    // selection, the groups and the aggregation run again).
    const int G = T->world, nl = (int) T->local.size();
    const PassGeom pg = pass_geom(pc);
    const std::vector<PlaneShare> &share = T->pw.share;
    const LfWindow &win = T->pw.win;
    T->passes_redone++;
    std::vector<TeamSeg> segs;
    for (int g = 0; g < G; g++) {
        const size_t off = (size_t) share[g].pl0 * pg.R * 4, bytes = (size_t) (share[g].pl1 - share[g].pl0) * pg.R * 4;
        segs.push_back({ g, -1, TB_S_AT, TB_S_AT, off, off, bytes });
        segs.push_back({ g, -1, TB_S_MIR, TB_S_MIR, off, off, bytes });
    }
    if (team_exchange(T, segs)) return 1;
    for (int l = 0; l < nl; l++) {      // restore the accumulators of the window on the rows the pass wrote
        lfbm5d_ctx *ctx = T->local[l];
        const Band &bd = T->bands[T->local_rank[l]];
        CK(cudaSetDevice(ctx->device));
        launch_pad(ctx, pc, win, T->d_noisy[l], pc.step == 2 ? T->d_basic[l] : nullptr, bd.y0, bd.c1, bd.y1);
    }
    if (team_pass_body(T, pc, true) || team_pass_read(T, cov, &ties)) return 1;
    return 0;
}

// running estimate of the window on the own rows + its exchange (every rank then holds the complete channel-0 planes)
int team_est0_exchange(lfbm5d_team *T, const PassCfg &pc, const LfWindow &win)
{
    const size_t plane = (size_t) pc.wb * pc.hb;
    std::vector<TeamSeg> segs;
    for (int g = 0; g < T->world; g++) {
        const Band &bd = T->bands[g];
        if (bd.y1 <= bd.y0) continue;
        for (int a = 0; a < (int) pc.A; a++)
            if (win.mask[a]) {
                const size_t off = ((size_t) a * plane + (size_t) bd.y0 * pc.wb) * 4;
                segs.push_back({ g, -1, TB_EST0, TB_EST0, off, off, (size_t) (bd.y1 - bd.y0) * pc.wb * 4 });
            }
    }
    return team_exchange(T, segs);
}

// per-SAI counts of zero weights, summed over the ranks (window / SAI selection, bm5d.cpp:189-202, :318-333)
int team_count_zero(lfbm5d_team *T, const std::vector<unsigned> &items, bool padded, const PassCfg &pc, std::vector<unsigned long long> &out)
{
    const int G = T->world, nl = (int) T->local.size();
    const int nit = (int) items.size();
    if (nit > 60) return fail("too many SAIs in one count");
    for (int l = 0; l < nl; l++) {
        lfbm5d_ctx *ctx = T->local[l];
        const int g = T->local_rank[l];
        const Band &bd = T->bands[g];
        CK(cudaSetDevice(ctx->device));
        unsigned long long *cnts = reinterpret_cast<unsigned long long *>(team_bufs(ctx)->counters.as<char>() + cslot(T, g));
        CK(cudaMemsetAsync(cnts, 0, 64 * 8, ctx->stream));
        for (int i = 0; i < nit; i++) {
            if (padded)      // padded weights of window slot items[i], all channels, own rows [y0, y1)
                launch_count_zero(ctx, ctx->densym.as<float>() + (size_t) items[i] * pc.C * pc.wb * pc.hb, (int) pc.C, (int) pc.wb, (int) pc.hb, bd.y0, bd.y1, cnts + i);
            else
                launch_count_zero(ctx, ctx->den.as<float>() + (size_t) items[i] * pc.C * pc.W * pc.H, (int) pc.C, (int) pc.W, (int) pc.H, bd.i0, bd.i1, cnts + i);
        }
    }
    std::vector<TeamSeg> segs;
    for (int g = 0; g < G; g++) segs.push_back({ g, -1, TB_COUNTERS, TB_COUNTERS, cslot(T, g), cslot(T, g), (size_t) nit * 8 });
    if (team_exchange(T, segs)) return 1;
    out.assign(nit, 0);
    for (int l = 0; l < nl; l++) {
        lfbm5d_ctx *ctx = T->local[l];
        CK(cudaSetDevice(ctx->device));
        std::vector<unsigned long long> h((size_t) G * TSLOT_U64);
        CK(cudaMemcpyAsync(h.data(), team_bufs(ctx)->counters.as<char>() + cslot(T, 0), h.size() * 8, cudaMemcpyDeviceToHost, ctx->stream));
        CK(cudaStreamSynchronize(ctx->stream));
        if (l == 0) for (int g = 0; g < G; g++) for (int i = 0; i < nit; i++) out[i] += h[(size_t) g * TSLOT_U64 + i];
    }
    T->cparity ^= 1u;
    return 0;
}

// tiny all-to-all of host values through the counter slots (also a barrier: a rank has everybody's value only after everybody
// reached this point): slot g = 64 x 8 bytes
int team_host_allgather(lfbm5d_team *T, const void *mine_per_local, size_t bytes, std::vector<unsigned char> &all)
{
    const int G = T->world, nl = (int) T->local.size();
    for (int l = 0; l < nl; l++) {
        lfbm5d_ctx *ctx = T->local[l];
        CK(cudaSetDevice(ctx->device));
        TeamCtxBufs *b = team_bufs(ctx);
        if (bytes > TSLOT) return fail("host all-gather: value too large");
        if (b->counters.ensure((size_t) 2 * G * TSLOT)) return 1;
        CK(cudaMemcpyAsync(b->counters.as<char>() + cslot(T, T->local_rank[l]), (const char *) mine_per_local + (size_t) l * bytes, bytes,
                           cudaMemcpyHostToDevice, ctx->stream));
    }
    std::vector<TeamSeg> segs;
    for (int g = 0; g < G; g++) segs.push_back({ g, -1, TB_COUNTERS, TB_COUNTERS, cslot(T, g), cslot(T, g), bytes });
    if (team_exchange(T, segs)) return 1;
    all.assign((size_t) G * bytes, 0);
    for (int l = 0; l < nl; l++) {
        lfbm5d_ctx *ctx = T->local[l];
        CK(cudaSetDevice(ctx->device));
        std::vector<unsigned char> h((size_t) G * TSLOT);
        CK(cudaMemcpyAsync(h.data(), team_bufs(ctx)->counters.as<char>() + cslot(T, 0), h.size(), cudaMemcpyDeviceToHost, ctx->stream));
        CK(cudaStreamSynchronize(ctx->stream));
        if (l == 0) for (int g = 0; g < G; g++) memcpy(all.data() + (size_t) g * bytes, h.data() + (size_t) g * TSLOT, bytes);
    }
    T->cparity ^= 1u;
    return 0;
}

void team_peer_close(lfbm5d_team *T)
{
    for (void *p : T->peer_opened) cudaIpcCloseMemHandle(p);
    T->peer_opened.clear();
    T->peer_ready = false;
}

// Allocate every buffer a step with geometry pc needs and make the exchanged ones addressable from every rank. DevBufs only grow,
// and every rank sees the same sequence of geometries: a geometry that was set up before needs nothing. For a new one all peer
// mappings are closed first (an exported allocation must not be freed while it is mapped elsewhere), the buffers are (re)allocated,
// and everything is exported / imported again.
int team_peer_setup(lfbm5d_team *T, const PassCfg &pc, int step)
{
    const PassGeom pg = pass_geom(pc);
    const int G = T->world, nl = (int) T->local.size();
    auto ensure_all = [&](lfbm5d_ctx *ctx) -> int {
        CK(cudaSetDevice(ctx->device));
        if (ensure_pass_buffers(ctx, pc) || team_ensure(T, ctx, pc)) return 1;
        // gather buffers of team_step_end
        size_t maxrows = 0;
        for (int g = 0; g < G; g++) maxrows = std::max<size_t>(maxrows, (size_t) (T->bands[g].i1 - T->bands[g].i0));
        for (const Band &hb : T->held) maxrows = std::max<size_t>(maxrows, (size_t) (hb.i1 - hb.i0));      // step 1 of this team: already allocated
        const size_t blk = (size_t) T->ss.asize() * pc.C * maxrows * pc.W * 4;
        TeamCtxBufs *b = team_bufs(ctx);
        if (!T->is_lane && (b->gsend.ensure(blk) || b->grecv.ensure(blk * G))) return 1;
        return 0;
    };
    if (!T->comm) {      // emulated: all contexts live here
        for (int l = 0; l < nl; l++) if (ensure_all(T->local[l])) return 1;
        for (int l = 0; l < nl; l++) { T->peer_at[T->local_rank[l]] = T->local[l]->s_at.as<float>(); T->peer_mir[T->local_rank[l]] = T->local[l]->s_mir.as<float>(); }
        T->peer_ready = T->peer_ok;
        return 0;
    }
    lfbm5d_ctx *ctx = T->local[0];
    const int me = T->local_rank[0];
    const std::vector<size_t> key = { (size_t) step, (size_t) pc.wb, (size_t) pc.hb, (size_t) pc.k, (size_t) pc.N, (size_t) pc.A, (size_t) pc.C, (size_t) pc.nSim,
                                      (size_t) pc.nDisp, (size_t) pg.R, (size_t) T->ss.asize() };
    for (auto &k : T->peer_keys) if (k == key) return ensure_all(ctx);      // nothing grows: no reallocation, mappings stay valid
    T->peer_keys.push_back(key);
    team_peer_close(T);
    std::vector<unsigned char> all;
    unsigned long long z = 0;
    if (team_host_allgather(T, &z, 8, all)) return 1;        // barrier (over NCCL: the mappings are gone): everything is closed before anybody frees
    if (ensure_all(ctx)) return 1;
    CK(cudaSetDevice(ctx->device));
    if (T->xflags.ensure(LF_MAXRANKS * 4 * 2) == 0 && T->xflags.cap && T->xepoch == 0) CK(cudaMemsetAsync(T->xflags.p, 0, T->xflags.cap, ctx->stream));
    if (T->xdone.ensure(64)) return 1;
    CK(cudaMemsetAsync(T->xdone.p, 0, 64, ctx->stream));
    if (T->xflagptrs.ensure(LF_MAXRANKS * sizeof(void *))) return 1;
    if (!T->peer_ok) return 0;
    // export: TB_NBUF buffers + the flag slots
    struct Exp { cudaIpcMemHandle_t h[TB_NBUF + 1]; unsigned char have[TB_NBUF + 1]; unsigned char ok; };
    static_assert(sizeof(Exp) <= TSLOT, "handles do not fit the counter slot");
    Exp mine;
    memset(&mine, 0, sizeof(mine));
    mine.ok = 1;
    for (int b = 0; b <= TB_NBUF; b++) {
        void *p = b < TB_NBUF ? (void *) team_ptr(ctx, b) : T->xflags.p;
        if (!p) continue;
        if (cudaIpcGetMemHandle(&mine.h[b], p) == cudaSuccess) mine.have[b] = 1; else { mine.ok = 0; cudaGetLastError(); }
    }
    if (team_host_allgather(T, &mine, sizeof(mine), all)) return 1;
    bool ok = true;
    for (int g = 0; g < G; g++) ok = ok && reinterpret_cast<Exp *>(all.data() + (size_t) g * sizeof(Exp))->ok != 0;
    std::vector<unsigned *> flagptrs(LF_MAXRANKS, nullptr);
    if (ok)
        for (int g = 0; g < G && ok; g++) {
            const Exp *e = reinterpret_cast<Exp *>(all.data() + (size_t) g * sizeof(Exp));
            for (int b = 0; b <= TB_NBUF && ok; b++) {
                void *p = nullptr;
                if (g == me) p = b < TB_NBUF ? (void *) team_ptr(ctx, b) : T->xflags.p;
                else if (e->have[b]) {
                    if (cudaIpcOpenMemHandle(&p, e->h[b], cudaIpcMemLazyEnablePeerAccess) != cudaSuccess) { ok = false; cudaGetLastError(); break; }
                    T->peer_opened.push_back(p);
                }
                if (b < TB_NBUF) T->peer_buf[g][b] = (char *) p; else flagptrs[g] = (unsigned *) p;
            }
            T->peer_at[g] = (const float *) T->peer_buf[g][TB_S_AT]; T->peer_mir[g] = (const float *) T->peer_buf[g][TB_S_MIR];
        }
    // everybody must agree (a rank that could not map its peers makes the whole team fall back to NCCL exchanges)
    unsigned long long okf = ok ? 1 : 0;
    if (team_host_allgather(T, &okf, 8, all)) return 1;
    for (int g = 0; g < G; g++) ok = ok && *reinterpret_cast<unsigned long long *>(all.data() + (size_t) g * 8) != 0;
    if (!ok) { team_peer_close(T); T->peer_ok = false; return 0; }
    CK(cudaMemcpyAsync(T->xflagptrs.p, flagptrs.data(), LF_MAXRANKS * sizeof(void *), cudaMemcpyHostToDevice, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    T->peer_ready = true;
    return 0;
}

// The interior rows [i0, i1) of every rank's band of the light field d_lf (one pointer per local rank), sent to every other rank:
// afterwards every rank holds all rows. Staged through the gather buffers (packed rows of all planes).
int team_gather_bands(lfbm5d_team *T, const std::vector<Band> &bands, float *const *d_lf)
{
    StepState &S = T->ss;
    const lfbm5d_params *p = &S.p;
    const int nl = (int) T->local.size(), G = T->world;
    const int W = (int) p->width, H = (int) p->height;
    const size_t nplanes = (size_t) S.asize() * p->chnls;
    size_t maxrows = 0;
    for (int g = 0; g < G; g++) maxrows = std::max<size_t>(maxrows, (size_t) (bands[g].i1 - bands[g].i0));
    const size_t blk = nplanes * maxrows * W * 4;
    for (int l = 0; l < nl; l++) {
        lfbm5d_ctx *ctx = T->local[l];
        const Band &bd = bands[T->local_rank[l]];
        TeamCtxBufs *b = team_bufs(ctx);
        CK(cudaSetDevice(ctx->device));
        if (b->gsend.ensure(blk) || b->grecv.ensure(blk * G)) return 1;      // sized by team_peer_setup: nothing grows here
        if (bd.i1 > bd.i0)
            LAUNCH(ctx, k_pack_rows, grid_for(ctx, nplanes * (bd.i1 - bd.i0) * W), 256, 0, d_lf[l], b->gsend.as<float>(), nplanes, W, H, bd.i0, bd.i1 - bd.i0, 0);
    }
    std::vector<TeamSeg> segs;
    for (int g = 0; g < G; g++) {
        const Band &bd = bands[g];
        for (int h = 0; h < G; h++)
            if (h != g) segs.push_back({ g, h, TB_GSEND, TB_GRECV, 0, (size_t) g * blk, nplanes * (size_t) (bd.i1 - bd.i0) * W * 4 });
    }
    if (team_exchange(T, segs)) return 1;
    for (int l = 0; l < nl; l++) {
        lfbm5d_ctx *ctx = T->local[l];
        TeamCtxBufs *b = team_bufs(ctx);
        CK(cudaSetDevice(ctx->device));
        for (int g = 0; g < G; g++) {
            const Band &bd = bands[g];
            if (g == T->local_rank[l] || bd.i1 <= bd.i0) continue;
            LAUNCH(ctx, k_pack_rows, grid_for(ctx, nplanes * (bd.i1 - bd.i0) * W), 256, 0, d_lf[l], b->grecv.as<float>() + (size_t) g * (blk / 4), nplanes, W, H,
                   bd.i0, bd.i1 - bd.i0, 1);
        }
    }
    return 0;
}

int team_step_begin(lfbm5d_team *T, int step, const lfbm5d_params *p_, float *const *d_noisy, float *const *d_basic, const unsigned *mask_)
{
    if (validate(p_, step)) return 1;
    const int nl = (int) T->local.size();
    StepState &S = T->ss;
    if (step_state_init(S, step, p_, mask_)) return 1;
    const lfbm5d_params *p = &S.p;
    const unsigned asize = S.asize();
    T->bands = team_bands(S.pc, T->world);
    // Step 1 of this team left LF_basic band-resident (no gather) and the bands of this step read rows some rank does not hold (other
    // patch size / step: other bands, possibly another number of ranks with rows): the owners send their rows around first. Every
    // rank takes the same decision from the same two band tables. (Config 3: the step-2 bands lie inside the step-1 bands, nothing moves.)
    bool late_gather = false;
    if (step == 2 && (int) T->held.size() == T->world)
        for (int g = 0; g < T->world; g++) {
            const Band &nb = T->bands[g], &hb = T->held[g];
            if (nb.j1 > nb.j0 && (nb.j0 < hb.i0 || nb.j1 > hb.j1)) late_gather = true;
        }
    if (step == 1 || !late_gather) T->held.clear();
    T->d_noisy.assign(d_noisy, d_noisy + nl);
    T->d_basic.assign(nl, nullptr);
    if (step == 2) T->d_basic.assign(d_basic, d_basic + nl);
    const size_t each = S.each();
    for (int l = 0; l < nl; l++) {
        lfbm5d_ctx *ctx = T->local[l];
        const Band &bd = T->bands[T->local_rank[l]];
        CK(cudaSetDevice(ctx->device));
        ctx->sched.clear();
        if (ctx->mask.ensure(asize * 4) || ctx->num.ensure(asize * each * 4) || ctx->den.ensure(asize * each * 4)) return 1;
        CK(cudaMemcpyAsync(ctx->mask.p, S.mask.data(), asize * 4, cudaMemcpyHostToDevice, ctx->stream));
        if (S.docolor) {      // only the rows this rank's groups read (own band + the rows it shares with the next rank)
            launch_color(ctx, ctx->stream, T->d_noisy[l], T->d_noisy[l], ctx->mask.as<unsigned>(), asize, p->width, p->height, p->color_space, 1, bd.j0, bd.j1);
            if (step == 2 && !late_gather)
                launch_color(ctx, ctx->stream, T->d_basic[l], T->d_basic[l], ctx->mask.as<unsigned>(), asize, p->width, p->height, p->color_space, 1, bd.j0, bd.j1);
        }
        CK(cudaMemsetAsync(ctx->num.p, 0, asize * each * 4, ctx->stream));
        CK(cudaMemsetAsync(ctx->den.p, 0, asize * each * 4, ctx->stream));
    }
    if (team_peer_setup(T, S.pc, step)) return 1;       // allocates the pass buffers (under the export protocol of NCCL teams)
    if (late_gather) {
        if (team_gather_bands(T, T->held, T->d_basic.data())) return 1;
        T->held.clear();
        for (int l = 0; l < nl; l++) {
            lfbm5d_ctx *ctx = T->local[l];
            const Band &bd = T->bands[T->local_rank[l]];
            CK(cudaSetDevice(ctx->device));
            if (S.docolor)
                launch_color(ctx, ctx->stream, T->d_basic[l], T->d_basic[l], ctx->mask.as<unsigned>(), asize, p->width, p->height, p->color_space, 1, bd.j0, bd.j1);
        }
    }
    for (int l = 0; l < nl; l++) {
        lfbm5d_ctx *ctx = T->local[l];
        CK(cudaSetDevice(ctx->device));
        if (setup_tables(ctx, step, p, S.tau_4D) || upload_grid(ctx, S.pc)) return 1;
    }
    // further lanes: the same step on their own contexts, the accumulators (and the mask) of lane 0
    for (lfbm5d_team *Tl : T->lanes) {
        Tl->ss = T->ss;
        Tl->bands = T->bands; Tl->d_noisy = T->d_noisy; Tl->d_basic = T->d_basic;
        for (int l = 0; l < nl; l++) {
            lfbm5d_ctx *cl = Tl->local[l], *c0 = T->local[l];
            CK(cudaSetDevice(cl->device));
            cl->num.borrow(c0->num); cl->den.borrow(c0->den); cl->mask.borrow(c0->mask);
            cl->sched.clear();
        }
        if (team_peer_setup(Tl, Tl->ss.pc, step)) return 1;
        for (int l = 0; l < nl; l++) {
            lfbm5d_ctx *cl = Tl->local[l];
            CK(cudaSetDevice(cl->device));
            if (setup_tables(cl, step, p, S.tau_4D) || upload_grid(cl, Tl->ss.pc)) return 1;
        }
    }
    if (!T->lanes.empty())      // the colour transform / the cleared accumulators of lane 0's stream, before any lane reads them
        for (int l = 0; l < nl; l++) { CK(cudaSetDevice(T->local[l]->device)); CK(cudaStreamSynchronize(T->local[l]->stream)); }
    return 0;
}

// window selection of the team: the counts of zero weights are summed over the bands
int team_select(lfbm5d_team *T, unsigned &ps, unsigned &pt)
{
    return select_window(T->ss, ps, pt, [&](const std::vector<unsigned> &sais, std::vector<unsigned long long> &zeros) {
        zeros.clear();
        for (size_t b0 = 0; b0 < sais.size(); b0 += 48) {
            std::vector<unsigned> chunk(sais.begin() + b0, sais.begin() + std::min(sais.size(), b0 + 48));
            std::vector<unsigned long long> h;
            if (team_count_zero(T, chunk, false, T->ss.pc, h)) return 1;
            zeros.insert(zeros.end(), h.begin(), h.end());
        }
        return 0;
    });
}

// ---- one angular window (bm5d.cpp:204-402), all ranks in lockstep, in two halves: team_window_begin enqueues everything up to and
// including the first core call, team_window_finish reads its counters (host sync) and takes the window to its end. A driver
// with several lanes begins independent windows on all of them before it finishes the first.

// everything of a core call that comes before the counters: choice of pst, running estimate, block matching, groups, aggregation
int team_window_prepass(lfbm5d_team *T)
{
    StepState &S = T->ss;
    const int nl = (int) T->local.size();
    const PassCfg &pc = S.pc;
    WindowRun &wf = T->wf;
    const LfWindow &win = wf.win;
    if (window_next(wf, [&](const std::vector<unsigned> &slots, std::vector<unsigned long long> &zeros) {
            return team_count_zero(T, slots, true, pc, zeros);
        })) return 1;
    if (wf.calls > 0)      // the running estimate of the window after the previous core call (core:169 / :937), own rows
        for (int l = 0; l < nl; l++) {
            lfbm5d_ctx *ctx = T->local[l];
            const Band &bd = T->bands[T->local_rank[l]];
            CK(cudaSetDevice(ctx->device));
            launch_est0(ctx, pc, win, bd.y0, bd.y1);
        }
    TMARK(1);
    if (team_est0_exchange(T, pc, win)) return 1;
    return team_pass_bm(T, pc, win, (int) wf.pst_asw, (int) wf.cst_asw) || team_pass_body(T, pc, false);
}

// force_sadct: -1 = sequential rule; 0 / 1 = the plan's value for this window (window_open)
int team_window_begin(lfbm5d_team *T, unsigned ps, unsigned pt, int force_sadct)
{
    StepState &S = T->ss;
    const lfbm5d_params *p = &S.p;
    const int step = S.step, nl = (int) T->local.size();
    const PassCfg &pc = S.pc;
    if (window_open(S, T->wf, ps, pt, force_sadct))
        for (int l = 0; l < nl; l++) { CK(cudaSetDevice(T->local[l]->device)); if (setup_tables(T->local[l], step, p, S.tau_4D)) return 1; }
    const LfWindow &win = T->wf.win;
    TMARK(0);
    for (int l = 0; l < nl; l++) {      // padded working set on the rows the own groups touch; running estimate on the own rows
        lfbm5d_ctx *ctx = T->local[l];
        const Band &bd = T->bands[T->local_rank[l]];
        CK(cudaSetDevice(ctx->device));
        launch_pad(ctx, pc, win, T->d_noisy[l], step == 2 ? T->d_basic[l] : nullptr, bd.y0, bd.c1, bd.y1);
    }
    if (!T->wf.n_unproc) return 0;
    return team_window_prepass(T);
}

int team_window_finish(lfbm5d_team *T, lfbm5d_team *sched_to)
{
    StepState &S = T->ss;
    const int nl = (int) T->local.size();
    const PassCfg &pc = S.pc;
    WindowRun &wf = T->wf;
    const LfWindow &win = wf.win;
    while (wf.n_unproc) {
        unsigned long long cnt = 0;
        if (team_pass_finish(T, pc, &cnt)) return 1;
        if (T->timing && wf.calls == 0)
            for (int i = 0; i < 2; i++) { float ms = 0.f; if (cudaEventElapsedTime(&ms, T->tev[i], T->tev[i + 1]) == cudaSuccess) T->phase_ms[i] += ms; }
        for (int l = 0; l < nl; l++) {      // crop the accumulators back: the own band and the replica rows shared with the next rank
            lfbm5d_ctx *ctx = T->local[l];
            const Band &bd = T->bands[T->local_rank[l]];
            CK(cudaSetDevice(ctx->device));
            launch_unpad(ctx, pc, win, bd.j0, bd.j1, nullptr);
        }
        if (!window_after_call(S, wf, cnt)) break;
        if (team_window_prepass(T)) return 1;
    }
    const std::array<unsigned, 4> e = window_close(S, wf);
    for (int l = 0; l < nl; l++) sched_to->local[l]->sched.insert(sched_to->local[l]->sched.end(), e.begin(), e.end());
    // lanes: the unpadding kernels of the window must be through before another lane (or the final estimate) reads num / den
    if (sched_to != T || !T->lanes.empty())
        for (int l = 0; l < nl; l++) { CK(cudaSetDevice(T->local[l]->device)); CK(cudaStreamSynchronize(T->local[l]->stream)); }
    return 0;
}

int team_window(lfbm5d_team *T, unsigned ps, unsigned pt)
{
    return team_window_begin(T, ps, pt, -1) || team_window_finish(T, T);
}

// Final estimate on the rows each rank holds; gather != 0: the bands of `out` are then exchanged so that every rank has all of it
int team_step_end(lfbm5d_team *T, float *const *d_out, int gather)
{
    StepState &S = T->ss;
    const lfbm5d_params *p = &S.p;
    const int nl = (int) T->local.size(), G = T->world;
    const unsigned asize = S.asize();
    const int W = (int) p->width, H = (int) p->height;
    for (int l = 0; l < nl; l++) {
        lfbm5d_ctx *ctx = T->local[l];
        const Band &bd = T->bands[T->local_rank[l]];
        CK(cudaSetDevice(ctx->device));
        launch_final(ctx, S, T->d_noisy[l], T->d_basic[l], d_out[l], 0, asize, 1, bd.j0, bd.j1);
        if (S.docolor) {      // rows this rank never transformed: leave them as the reference leaves its inputs (colour round trip)
            const int lo[2] = { 0, bd.j1 }, hi[2] = { bd.j0, H };
            for (int q = 0; q < 2; q++) {
                launch_color(ctx, ctx->stream, T->d_noisy[l], T->d_noisy[l], ctx->mask.as<unsigned>(), asize, W, H, p->color_space, 2, lo[q], hi[q]);
                if (S.step == 2)
                    launch_color(ctx, ctx->stream, T->d_basic[l], T->d_basic[l], ctx->mask.as<unsigned>(), asize, W, H, p->color_space, 2, lo[q], hi[q]);
            }
        }
        CK(cudaGetLastError());
    }
    if (gather && G > 1 && team_gather_bands(T, T->bands, d_out)) return 1;
    // no gather: step 2 on this team finds the rows of LF_basic where this step left them (team_step_begin)
    T->held.clear();
    if (!gather && G > 1 && S.step == 1) T->held = T->bands;
    for (int l = 0; l < nl; l++) { CK(cudaSetDevice(T->local[l]->device)); CK(cudaStreamSynchronize(T->local[l]->stream)); }
    return 0;
}

} // namespace

extern "C" {

int lfbm5d_team_create_emulated(lfbm5d_team **out, int device, int world)
{
    if (!out || world < 1 || world > LF_MAXRANKS) return fail("bad team arguments (1 <= world <= 16)");
    lfbm5d_team *T = new lfbm5d_team();
    T->world = world; T->owns_ctx = true;
    for (int g = 0; g < world; g++) {
        lfbm5d_ctx *c = nullptr;
        if (lfbm5d_create(&c, device)) { for (auto q : T->local) lfbm5d_destroy(q); delete T; return 1; }
        T->local.push_back(c); T->local_rank.push_back(g);
    }
    *out = T;
    return 0;
}

int lfbm5d_team_unique_id(char *id128)
{
    if (!id128) return fail("null argument");
    if (nccl_load()) return 1;
    NcclId id;
    NCK(g_nccl.GetUniqueId(&id));
    memcpy(id128, id.internal, 128);
    return 0;
}

int lfbm5d_team_create_nccl(lfbm5d_team **out, lfbm5d_ctx *ctx, int rank, int world, const char *id128)
{
    if (!out || !ctx || !id128 || world < 1 || world > LF_MAXRANKS || rank < 0 || rank >= world) return fail("bad team arguments (1 <= world <= 16)");
    if (nccl_load()) return 1;
    CK(cudaSetDevice(ctx->device));
    lfbm5d_team *T = new lfbm5d_team();
    T->world = world;
    T->local.push_back(ctx); T->local_rank.push_back(rank);
    NcclId id;
    memcpy(id.internal, id128, 128);
    const int rc = g_nccl.CommInitRank(&T->comm, world, id, rank);
    if (rc != 0) { delete T; return fail(std::string("ncclCommInitRank: ") + g_nccl.GetErrorString(rc)); }
    *out = T;
    return 0;
}

void lfbm5d_team_destroy(lfbm5d_team *T)
{
    if (!T) return;
    for (auto Tl : T->lanes) lfbm5d_team_destroy(Tl);
    T->lanes.clear();
    for (auto c : T->local) { cudaSetDevice(c->device); cudaStreamSynchronize(c->stream); }
    if (T->comm && T->peer_ready) {      // nobody frees its buffers while they are mapped elsewhere
        team_peer_close(T);
        unsigned long long z = 0;
        std::vector<unsigned char> all;
        team_host_allgather(T, &z, 8, all);
        for (auto c : T->local) { cudaSetDevice(c->device); cudaStreamSynchronize(c->stream); }
    }
    T->xsegs.release(); T->xflags.release(); T->xdone.release(); T->xflagptrs.release();
    for (auto c : T->local) team_bufs_release(c);
    if (T->comm && !T->is_lane) g_nccl.CommDestroy(T->comm);
    if (T->owns_ctx) for (auto c : T->local) lfbm5d_destroy(c);
    delete T;
}

int lfbm5d_team_local_ranks(lfbm5d_team *T) { return T ? (int) T->local.size() : 0; }

/* Number of lanes of the team (>= 1): independent windows of a step (same level of the static plan) run concurrently, one per lane.
 * Every further lane has its own contexts (pass buffers: ~22 GB per lane at 17x17x1024^2 with an = 1, about three times that with
 * an = 2) and exchange state. Buffers are allocated at a lane's first pass; one that does not fit fails the step with the
 * cudaMalloc error and its size. */
int lfbm5d_team_set_lanes(lfbm5d_team *T, int nlanes)
{
    if (!T || nlanes < 1 || nlanes > 8 || T->is_lane) return fail("bad lane count (1 .. 8)");
    while ((int) T->lanes.size() + 1 > nlanes) { lfbm5d_team_destroy(T->lanes.back()); T->lanes.pop_back(); }
    while ((int) T->lanes.size() + 1 < nlanes) {
        lfbm5d_team *Tl = new lfbm5d_team();
        Tl->world = T->world; Tl->owns_ctx = true; Tl->is_lane = true; Tl->comm = T->comm;
        Tl->use_peer_exchange = T->use_peer_exchange; Tl->peer_ok = T->peer_ok;
        for (size_t l = 0; l < T->local.size(); l++) {
            lfbm5d_ctx *c = nullptr;
            if (lfbm5d_create(&c, T->local[l]->device)) { lfbm5d_team_destroy(Tl); return 1; }
            Tl->local.push_back(c); Tl->local_rank.push_back(T->local_rank[l]);
        }
        T->lanes.push_back(Tl);
    }
    return 0;
}

/* kernels launched by all contexts of the team (all lanes) since the last lfbm5d_reset_stats of each */
unsigned long long lfbm5d_team_launches(lfbm5d_team *T)
{
    if (!T) return 0;
    unsigned long long n = 0;
    for (auto c : T->local) n += c->stats.kernel_launches;
    for (auto Tl : T->lanes) for (auto c : Tl->local) n += c->stats.kernel_launches;
    return n;
}

/* one LFBM5D step of ONE light field on the whole team; d_* are arrays of lfbm5d_team_local_ranks() device pointers (one copy of the
 * light field per local rank, [asize][chnls][height][width] floats) */
int lfbm5d_team_step(lfbm5d_team *T, int step, const lfbm5d_params *p, float *const *d_noisy_io, float *const *d_basic_io, const unsigned *sai_mask,
                     float *const *d_out, int gather)
{
    if (!T || !p || !d_noisy_io || !sai_mask || !d_out || (step == 2 && !d_basic_io)) return fail("null argument");
    if (step != 1 && step != 2) return fail("step must be 1 or 2");
    if (team_step_begin(T, step, p, d_noisy_io, d_basic_io, sai_mask)) return 1;
    const unsigned max_passes = T->local[0]->max_passes;
    if (T->lanes.empty()) {
        while (T->ss.remaining) {
            unsigned ps = 0, pt = 0;
            if (team_select(T, ps, pt) || team_window(T, ps, pt)) return 1;
            if (max_passes && T->ss.passes >= max_passes) break;
        }
    } else {
        // Several lanes: the windows of a step form a static plan (lfbm5d_step_plan); the windows of one plan level share no SAI and
        // commute, so they run concurrently, one per lane — the latency-bound parts of a pass (the strip chains of the summed-area
        // planes, the exchanges, the host's counter read) of one window hide behind the bandwidth-bound parts of the others.
        const unsigned asize = p->awidth * p->aheight;
        std::vector<unsigned> plan((size_t) (asize + 1) * 6);
        const unsigned nwin = lfbm5d_step_plan(p, sai_mask, plan.data(), asize + 1);
        std::vector<lfbm5d_team *> L;
        L.push_back(T);
        for (lfbm5d_team *Tl : T->lanes) L.push_back(Tl);
        // Software pipeline over the plan sorted by level: window i goes to lane i mod L; before it begins, every earlier window
        // that shares an SAI with it — and the lane's previous window — is finished (counters read, accumulators written back).
        // Up to L windows are in flight; only true dependencies stall. Every rank walks the same deterministic sequence.
        const unsigned asw = 2 * p->an + 1;
        std::vector<unsigned> order;
        unsigned maxlevel = 0;
        for (unsigned i = 0; i < nwin; i++) maxlevel = std::max(maxlevel, plan[6 * i + 4]);
        for (unsigned lev = 0; lev <= maxlevel; lev++)
            for (unsigned i = 0; i < nwin; i++) if (plan[6 * i + 4] == lev) order.push_back(i);
        if (max_passes && order.size() > max_passes) order.resize(max_passes);
        auto overlap = [&](unsigned a_, unsigned b_) {
            const unsigned *x = &plan[6 * a_], *y = &plan[6 * b_];
            return !(x[2] + asw <= y[2] || y[2] + asw <= x[2] || x[3] + asw <= y[3] || y[3] + asw <= x[3]);
        };
        const size_t nL = L.size();
        std::vector<int> state(order.size(), 0);          // 0 not begun, 1 in flight, 2 finished
        auto finish = [&](size_t q) -> int {
            if (state[q] != 1) return 0;
            state[q] = 2;
            return team_window_finish(L[q % nL], T);
        };
        for (size_t q = 0; q < order.size(); q++) {
            if (q >= nL && finish(q - nL)) return 1;        // the lane's previous window
            for (size_t d = 0; d < q; d++)
                if (state[d] == 1 && overlap(order[d], order[q]) && finish(d)) return 1;
            const unsigned *e = &plan[6 * order[q]];
            if (team_window_begin(L[q % nL], e[0], e[1], (int) e[5])) return 1;
            state[q] = 1;
        }
        for (size_t q = 0; q < order.size(); q++) if (finish(q)) return 1;
    }
    return team_step_end(T, d_out, gather);
}

/* interior rows [*row_lo, *row_hi) of every SAI that rank `rank` owns in the step that ran last (its band of the output), and the
 * rows [*row_lo, *keep_hi) it holds valid results for (its band + the rows shared with the next rank) */
int lfbm5d_team_band(lfbm5d_team *T, int rank, int *row_lo, int *row_hi, int *keep_hi)
{
    if (!T || rank < 0 || rank >= (int) T->bands.size()) return fail("no band: run a step first");
    const Band &b = T->bands[rank];
    if (row_lo) *row_lo = b.i0;
    if (row_hi) *row_hi = b.i1;
    if (keep_hi) *keep_hi = b.j1;
    return 0;
}

/* Bands a step with parameters p would use on a team of `world` ranks, without running it: interior rows [*row_lo, *row_hi) owned by
 * `rank`, and [*row_lo, *keep_hi) = every row of the inputs the rank reads (what a host driver has to upload to it). */
int lfbm5d_team_plan_band(int world, int rank, int step, const lfbm5d_params *p, int *row_lo, int *row_hi, int *keep_hi)
{
    if (!p || world < 1 || world > LF_MAXRANKS || rank < 0 || rank >= world) return fail("bad arguments");
    if (validate(p, step)) return 1;
    PassCfg pc;
    if (make_passcfg(pc, step, p, p->tau_4D)) return 1;
    const std::vector<Band> B = team_bands(pc, world);
    if (row_lo) *row_lo = B[rank].i0;
    if (row_hi) *row_hi = B[rank].i1;
    if (keep_hi) *keep_hi = B[rank].j1;
    return 0;
}

/* Copy the rows [row_lo, row_hi) of every plane of every non-masked SAI between caller-owned host arrays (asize pointers, planar
 * width*height*chnls floats each, as for lfbm5d_step1) and a device light field [asize][chnls][height][width], on the context's
 * stream (asynchronous: pinned host memory makes it overlap; lfbm5d_sync waits). One strided copy per SAI. */
int lfbm5d_copy_rows(lfbm5d_ctx *ctx, float *const *host, float *d_lf, const unsigned *sai_mask, unsigned asize, unsigned chnls, unsigned width,
                     unsigned height, unsigned row_lo, unsigned row_hi, int to_device)
{
    if (!ctx || !host || !d_lf || !sai_mask) return fail("null argument");
    if (row_hi > height || row_lo >= row_hi) return row_lo == row_hi ? 0 : fail("bad row range");
    CK(cudaSetDevice(ctx->device));
    const size_t plane = (size_t) width * height, rowbytes = (size_t) (row_hi - row_lo) * width * 4;
    for (unsigned st = 0; st < asize; st++) {
        if (!sai_mask[st]) continue;
        float *d = d_lf + (size_t) st * chnls * plane + (size_t) row_lo * width;
        float *hp = host[st] + (size_t) row_lo * width;
        if (to_device) CK(cudaMemcpy2DAsync(d, plane * 4, hp, plane * 4, rowbytes, chnls, cudaMemcpyHostToDevice, ctx->stream));
        else CK(cudaMemcpy2DAsync(hp, plane * 4, d, plane * 4, rowbytes, chnls, cudaMemcpyDeviceToHost, ctx->stream));
    }
    return 0;
}

int lfbm5d_sync(lfbm5d_ctx *ctx)
{
    if (!ctx) return fail("null argument");
    CK(cudaSetDevice(ctx->device));
    CK(cudaStreamSynchronize(ctx->stream));
    return 0;
}

void lfbm5d_team_stats(lfbm5d_team *T, unsigned long long *bytes_exchanged, unsigned *passes_redone, unsigned long long *tie_patches, int *peer_view)
{
    if (!T) return;
    unsigned long long b = T->bytes_exchanged, tp = T->tie_patches;
    unsigned pr = T->passes_redone;
    for (auto Tl : T->lanes) { b += Tl->bytes_exchanged; tp += Tl->tie_patches; pr += Tl->passes_redone; }
    if (bytes_exchanged) *bytes_exchanged = b;
    if (passes_redone) *passes_redone = pr;
    if (tie_patches) *tie_patches = tp;
    if (peer_view) *peer_view = T->peer_ready ? 1 : 0;
}

/* per-phase device time of the first local rank: out[0..7] = pad, est0 exchange, block matching, match exchange, selection + groups +
 * aggregation 1, border exchange, aggregation 2, border + counter exchange; out[8..11] = inside block matching: self planes, partial
 * selection, disparity planes, disparity argmin (ms since timing was switched on) */
void lfbm5d_team_timing(lfbm5d_team *T, int on, float *out12)
{
    if (!T) return;
    if (out12) for (int i = 0; i < 12; i++) out12[i] = T->phase_ms[i];
    if (on && !T->tev[0]) { cudaSetDevice(T->local[0]->device); for (auto &e : T->tev) cudaEventCreate(&e); for (auto &e : T->bev) cudaEventCreate(&e); }
    if (on != (T->timing ? 1 : 0)) for (auto &m : T->phase_ms) m = 0.f;
    T->timing = on != 0;
}

/* tests: give up the peer view of the self sums, so that exact ties take the exchange-and-redo fallback */
void lfbm5d_team_disable_peer_view(lfbm5d_team *T)
{
    if (!T) return;
    if (T->comm) team_peer_close(T);
    T->peer_ready = false; T->peer_ok = false;
    for (auto Tl : T->lanes) lfbm5d_team_disable_peer_view(Tl);
}

/* 0: exchanges of an NCCL team go through NCCL send / recv even when the buffers are peer-mapped (comparison runs) */
void lfbm5d_team_use_peer_exchange(lfbm5d_team *T, int on)
{
    if (!T) return;
    T->use_peer_exchange = on != 0;
    for (auto Tl : T->lanes) Tl->use_peer_exchange = on != 0;
}

} // extern "C"
