// capi.cu — the C-ABI of include/stlcalib.h: context, pack upload, batched evaluation.
// Host orchestration only; every number comes from the CUDA kernels.  No CPU fallback:
// stl_create fails without an sm_100 device.
#include <algorithm>
#include <cfloat>
#include <climits>
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <mutex>
#include <string>
#include <vector>

#include <nccl.h>

#include "../../include/stlcalib.h"
#include "gprfit.hpp"
#include "hostmath.hpp"
#include "kernels.h"
#include "lm.h"
#include "packlayout.hpp"

using namespace stl;

struct stl_ctx {
    int device = 0;
    stl_params_t params;
    DevParams dpr;
    cudaStream_t own_stream = nullptr;   // created by the context
    cudaStream_t stream = nullptr;       // default stream of calls without an explicit one (stl_set_stream)
    cudaStream_t last_stream = nullptr;  // stream of the previous call: a change inserts an event dependency
    cudaEvent_t handoff = nullptr;
    // stl_step_batch: BuildProblem + linearisation run on a stream of their own beside the evaluation's 3-D stage
    cudaStream_t aux_stream = nullptr;
    cudaEvent_t ev_k1 = nullptr, ev_k2a = nullptr, ev_k3 = nullptr, ev_aux = nullptr;
    long long overlapped_steps = 0;
    long long launches = 0;
    std::mutex mu;
    std::string err;
    bool has_pack = false;
    float adj_r2 = 0.f;  // squared radius of the leaf adjacency lists, rounded up (0: none)
    DevPack pk;
    int n_sm = 0;
    // the pack's layout and K1 routing (packlayout.hpp, DESIGN §3 "Oversize keyframes"): the one-kernel K1 (assoc2d.cu) runs
    // the fitting keyframes, the banded three-kernel K1 (assoc2d_split.cu) the oversize ones (pk.ov)
    PackLayout lay;
    bool allow_oversize = false;  // stl_allow_oversize_keyframes: read by the next upload
    OvKf *d_ov = nullptr;         // [n_ov]
    // the current keyframe list (every keyframe after an upload, stl_select_keyframes) and the device copies of the routes of
    // the whole pack (its K1 lists) and of the last selection: pk.sel / sel_mp / ov_sel point into the current one's
    KfRoute route;
    struct DevRoute {
        int *lists = nullptr;    // [2][n_kf] KfRoute::lists (only with oversize keyframes)
        int *sel = nullptr;      // [cap]
        int2 *sel_mp = nullptr;  // [cap + 1]
        int cap = 0;
    } d_all, d_sel;
    double *d_frames = nullptr;           // stl_eval_frames: [Bc][n_kf][13] of one workspace chunk
    // workspace
    DevWork wk;
    int wk_cap = 0;
    bool dbg_alloc = false;
    double *d_sums = nullptr;
    int d_sums_cap = 0;
    DevCand *h_cand = nullptr;  // pinned
    double *h_sums = nullptr;   // pinned
    int h_cap = 0;
    cudaEvent_t h2d_done = nullptr;  // pinned candidate staging is reused only after its copies completed
    std::vector<double> last_x;
    int dbg_b = -1;
    // which candidates' K1 results (correspondences, query lists) the workspace holds right now: rows of x, in slot order
    std::vector<double> wk_x;
    bool wk_has_nn = false;  // ... and the 1-NN positions of their 3-D queries (K2a)
    long long assoc_reused = 0;
    // multi-GPU: keyframes sharded over the ranks of this communicator (owned)
    ncclComm_t comm = nullptr;
    int comm_rank = 0, comm_size = 1;
    // the record exchange inside the last kernel of a call, over cudaIpc-mapped peer memory (p2p.cuh)
    bool p2p_on = false;
    unsigned p2p_seq = 0;
    P2pView p2p;  // data / flag pointers of every rank, rank, n, err
    double *p2p_data = nullptr;
    unsigned *p2p_flag = nullptr;
    long long p2p_exchanges = 0, nccl_exchanges = 0;
    // LM path
    LmState lm;
    double *d_lin = nullptr;
    double *h_lin = nullptr;
    long long lin_cap = 0;  // doubles
    // profiling
    bool profiling = false;
    struct Ev { cudaEvent_t a, b; int stage; bool count; };
    std::vector<Ev> evs;
    std::vector<cudaEvent_t> ev_pool;
    double stage_ms[STL_NSTAGES] = {0};
    long long stage_n[STL_NSTAGES] = {0};
    double counters[8] = {0};
};

namespace {

stl_status_t fail(stl_ctx *c, stl_status_t code, const char *fmt, ...) {
    char buf[512];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof(buf), fmt, ap);
    va_end(ap);
    if (c) c->err = buf;
    return code;
}

// Every call of a context runs on ONE stream at a time (they share the workspace): when the
// stream changes, the new one waits for the work already queued on the previous one.
cudaStream_t acquire_stream(stl_ctx *c, void *requested) {
    cudaStream_t st = requested ? (cudaStream_t)requested : c->stream;
    if (st != c->last_stream) {
        if (c->last_stream) {
            cudaEventRecord(c->handoff, c->last_stream);
            cudaStreamWaitEvent(st, c->handoff, 0);
        }
        c->last_stream = st;
    }
    return st;
}

#define CK(call)                                                                                          \
    do {                                                                                                  \
        cudaError_t e_ = (call);                                                                          \
        if (e_ != cudaSuccess) return fail(ctx, STL_ERR_CUDA, "%s: %s (%s:%d)", #call, cudaGetErrorString(e_), __FILE__, __LINE__); \
    } while (0)

template <class T> void dfree(T *&p) { if (p) { cudaFree(p); p = nullptr; } }

void free_pack(stl_ctx *c) {
    DevPack &p = c->pk;
    dfree(p.kf); dfree(p.px); dfree(p.py); dfree(p.pz); dfree(p.orig); dfree(p.node_lo); dfree(p.node_hi); dfree(p.adj); dfree(p.adj_cov);
    dfree(p.pl_rec); dfree(p.pl_m);
    dfree(p.k1tab); dfree(p.bitmap); dfree(p.grid_start); dfree(p.grid_kp); dfree(p.kp_xy); dfree(p.kp_xyd); dfree(p.kp_mp); dfree(p.Tcw);
    dfree(p.relpose); dfree(p.covis_valid); dfree(p.covis_uv); dfree(p.he_Tc); dfree(p.he_Tl);
    p = DevPack();
    dfree(c->d_frames); dfree(c->d_ov);
    for (stl_ctx::DevRoute *d : {&c->d_all, &c->d_sel}) { dfree(d->lists); dfree(d->sel); dfree(d->sel_mp); *d = stl_ctx::DevRoute(); }
    c->lay = PackLayout();
    c->route = KfRoute();
    c->has_pack = false;
}
void free_work(stl_ctx *c) {
    DevWork &w = c->wk;
    dfree(w.cand); dfree(w.corr_kp); dfree(w.corr_pt); dfree(w.corr_sp); dfree(w.q_corr); dfree(w.q_kpsp); dfree(w.n_corr); dfree(w.n_q);
    dfree(w.k1_ticket); dfree(w.k1_rec); dfree(w.k1_match); dfree(w.k1_ov_match); dfree(w.k1_surv); dfree(w.k1_cnt); dfree(w.k1_best_d2); dfree(w.k1_best_key);
    dfree(w.frame); dfree(w.align); dfree(w.nn_pos); dfree(w.nn_g2); dfree(w.nb); dfree(w.nbx); dfree(w.nb_m); dfree(w.nb_last); dfree(w.dbg_nn); dfree(w.dbg_m); dfree(w.dbg_plane); dfree(w.dbg_dist); dfree(w.dbg_knn); dfree(w.dbg_stats);
    dfree(w.overflow); dfree(w.k1_clk);
    w = DevWork();
    dfree(c->d_frames);  // sized by the chunk
    c->wk_cap = 0;
    c->dbg_alloc = false;
}

void set_dev_params(stl_ctx *c) {
    const stl_params_t &p = c->params;
    DevParams &d = c->dpr;
    d.max_pixel_dist2 = p.max_pixel_dist * p.max_pixel_dist;
    d.thr2d = p.corr_3d_2d_threshold;
    d.thr3d = p.corr_3d_3d_threshold;
    d.radius2 = p.norm_radius * p.norm_radius;
    d.reg_thr = p.norm_reg_threshold;
    d.min_diff2 = p.min_diff_dist * p.min_diff_dist;
    d.max_3d_dist2 = p.max_3d_dist * p.max_3d_dist;
    d.delta2d = p.robust_kernel_delta;
    d.delta3d = p.robust_kernel_3ddelta;
    d.w0 = p.err_weight[0];
    d.w1 = p.err_weight[1];
    d.num_min_corr = p.num_min_corr;
    d.k = p.norm_max_pts;
    d.min_pts = p.norm_min_pts;
    d.use_plane = p.use_plane;
    d.use_gpr = p.use_gpr; d.plane_index = p.plane_index;
    d.variant = p.variant; d.min_diff = p.min_diff_dist;
    // leaf adjacency lists cover norm_radius (the k-NN searches never look farther); STL_NO_ADJ=1 keeps the plain descent
    c->adj_r2 = 0.f; d.adj_r = 0.f;
    if (!getenv("STL_NO_ADJ") && p.use_plane && p.norm_radius > 0 && p.norm_radius < 1e3) {
        c->adj_r2 = nextafterf((float)d.radius2, INFINITY);
        d.adj_r = nextafterf((float)sqrt(d.radius2), 0.f);
    }
    d.gpr_sigma = p.gpr_sigma; d.gpr_l = p.gpr_l; d.gpr_noise = p.gpr_sigma_noise;
}

struct StageTimer {
    stl_ctx *c; int stage; cudaStream_t st; cudaEvent_t a = nullptr, b = nullptr; bool count;
    // count = false: the time is added to the stage, the launch count is not (second half of a stage split around a wait)
    StageTimer(stl_ctx *c_, int s, cudaStream_t st_, bool count_ = true) : c(c_), stage(s), st(st_), count(count_) {
        if (!c->profiling) return;
        auto get = [&]() { cudaEvent_t e; if (c->ev_pool.empty()) cudaEventCreate(&e); else { e = c->ev_pool.back(); c->ev_pool.pop_back(); } return e; };
        a = get(); b = get();
        cudaEventRecord(a, st);
    }
    ~StageTimer() {
        if (!a) return;
        cudaEventRecord(b, st);
        c->evs.push_back({a, b, stage, count});
    }
};

void drain_events(stl_ctx *c) {
    for (auto &e : c->evs) {
        cudaEventSynchronize(e.b);
        float ms = 0;
        if (cudaEventElapsedTime(&ms, e.a, e.b) == cudaSuccess) { c->stage_ms[e.stage] += ms; c->stage_n[e.stage] += e.count ? 1 : 0; }
        c->ev_pool.push_back(e.a);
        c->ev_pool.push_back(e.b);
    }
    c->evs.clear();
}

// The exchange folded into the kernel that finishes the record (p2p.cuh): a view for ONE exchange of B candidates, or a
// disabled view (n = 0) when the peer path cannot take it — the caller then runs allreduce_record (NCCL) instead.
P2pView p2p_view(stl_ctx *ctx, int B, int off, int width) {
    P2pView v;
    if (!ctx->p2p_on || B > kP2pMaxB || width > kP2pWidth) return v;
    v = ctx->p2p;
    v.seq = ++ctx->p2p_seq;
    v.off = off; v.width = width;
    ctx->p2p_exchanges += 1;
    return v;
}

// Workspace of one candidate chunk.  Allocation is all-or-nothing: a failure midway frees what was
// obtained and leaves wk_cap == 0, so the next call starts over instead of using half a workspace.
// The counters are cleared on the stream the context last used (any later stream waits for it).
stl_status_t ensure_work(stl_ctx *ctx, int B, bool debug) {
    const DevPack &pk = ctx->pk;
    if (ctx->wk_cap == 0) {
        size_t free_b = 0, total_b = 0;
        CK(cudaMemGetInfo(&free_b, &total_b));
        // (the three-kernel K1's survivors and matches: only those of the oversize keyframes)
        const size_t per_cand = (size_t)pk.n_kp_total * 24 + (size_t)pk.n_mp_total * (20 * kMaxK + 16) + (size_t)pk.n_kf * (sizeof(FrameRec) + 4 * sizeof(AlignRec) + 24) + (size_t)pk.n_ov_match * sizeof(ulonglong2) + (size_t)pk.n_ov_surv * 4 + (size_t)pk.n_kp_total * 16 + sizeof(DevCand);
        size_t budget = std::min<size_t>((size_t)12 << 30, free_b / 4);
        int cap = (int)std::max<size_t>(1, std::min<size_t>(budget / std::max<size_t>(per_cand, 1), 256));
        if (const char *e = getenv("STL_MAX_CHUNK")) cap = std::max(1, std::min(cap, atoi(e)));  // tests: force the multi-chunk path
        DevWork &w = ctx->wk;
        w.Bc = cap;
        // CTAs per (candidate, keyframe) of the query kernels: a function of the keyframe count ONLY (never of the batch size:
        // the sub-block partials are summed in sub order, and a batch must give the bits its candidates give one by one)
        // (4 / 8 / 16 measured on a 188-keyframe shard: 0.319 / 0.316 / 0.329 ms per step — the small-shard kernels are bound
        // by the latency of their longest query, not by the number of CTAs)
        w.sub = 4;
        if (getenv("STL_SUB")) w.sub = std::max(1, std::min(16, atoi(getenv("STL_SUB"))));
        const size_t nk = (size_t)std::max<long long>(pk.n_kp_total, 1) * cap, nf = (size_t)pk.n_kf * cap;
        const size_t nm = (size_t)std::max<long long>(pk.n_mp_total, 1) * cap;
        auto alloc_all = [&]() -> cudaError_t {
            cudaError_t e;
#define A_(p, bytes) do { e = cudaMalloc(&(p), (bytes)); if (e != cudaSuccess) return e; } while (0)
            A_(w.cand, sizeof(DevCand) * cap);
            A_(w.corr_kp, 4 * nk); A_(w.corr_pt, 4 * nk); A_(w.corr_sp, 4 * nk); A_(w.q_corr, 4 * nk); A_(w.q_kpsp, 8 * nk);
            A_(w.n_corr, 4 * nf); A_(w.n_q, 4 * nf);
            if (ctx->lay.n_fit > 0) {  // persistent K1: scratch per resident CTA, not per unit
                w.k1_slots = 2 * std::max(ctx->n_sm, 1);
                A_(w.k1_match, sizeof(ulonglong2) * kK1MatchCap * (size_t)w.k1_slots);
                A_(w.k1_rec, sizeof(float4) * kK1SurvCap * (size_t)w.k1_slots);
                A_(w.k1_ticket, 8);
                e = cudaMemsetAsync(w.k1_ticket, 0, 8, ctx->last_stream); if (e != cudaSuccess) return e;
            }
            if (pk.n_ov > 0) {  // three-kernel K1: per (candidate, oversize keyframe)
                const size_t c = (size_t)cap;
                A_(w.k1_ov_match, sizeof(ulonglong2) * (size_t)pk.n_ov_match * c); A_(w.k1_surv, 4 * (size_t)pk.n_ov_surv * c);
                A_(w.k1_cnt, 16 * (size_t)pk.n_ov * c);
                A_(w.k1_best_d2, 8 * (size_t)std::max<long long>(pk.n_ov_kp, 1) * c); A_(w.k1_best_key, 8 * (size_t)std::max<long long>(pk.n_ov_kp, 1) * c);
            }
            A_(w.frame, sizeof(FrameRec) * nf); A_(w.align, sizeof(AlignRec) * nf * w.sub);
            A_(w.nn_pos, 4 * nm); A_(w.nn_g2, 4 * nm); A_(w.nb, 4 * nm * kMaxK); A_(w.nbx, sizeof(float4) * nm * kMaxK); A_(w.nb_m, 4 * nm); A_(w.nb_last, 8 * nm);
            w.nbx_stride = (long long)nm;
            if (getenv("STL_K1_CLK")) { A_(w.k1_clk, 64 * nf); e = cudaMemsetAsync(w.k1_clk, 0, 64 * nf, ctx->last_stream); if (e != cudaSuccess) return e; }
            A_(w.overflow, 4);
#undef A_
            return cudaMemsetAsync(w.overflow, 0, 4, ctx->last_stream);
        };
        const cudaError_t e = alloc_all();
        if (e != cudaSuccess) {
            free_work(ctx);
            return fail(ctx, STL_ERR_CUDA, "workspace allocation: %s", cudaGetErrorString(e));
        }
        ctx->wk_cap = cap;
    }
    if (debug && !ctx->dbg_alloc) {
        DevWork &w = ctx->wk;
        const size_t nk = (size_t)std::max<long long>(pk.n_kp_total, 1);
        cudaError_t e = cudaMalloc(&w.dbg_nn, 4 * nk);
        if (e == cudaSuccess) e = cudaMalloc(&w.dbg_m, 4 * nk);
        if (e == cudaSuccess) e = cudaMalloc(&w.dbg_plane, 4 * nk);
        if (e == cudaSuccess) e = cudaMalloc(&w.dbg_dist, 8 * nk);
        if (e == cudaSuccess) e = cudaMalloc(&w.dbg_knn, 4 * nk * kMaxK);
        if (e == cudaSuccess) e = cudaMalloc(&w.dbg_stats, 64);
        if (e == cudaSuccess) e = cudaMemsetAsync(w.dbg_stats, 0, 64, ctx->last_stream);
        if (e != cudaSuccess) {
            dfree(w.dbg_nn); dfree(w.dbg_m); dfree(w.dbg_plane); dfree(w.dbg_dist); dfree(w.dbg_knn); dfree(w.dbg_stats);
            return fail(ctx, STL_ERR_CUDA, "debug workspace allocation: %s", cudaGetErrorString(e));
        }
        ctx->dbg_alloc = true;
    }
    if (B > ctx->h_cap) {
        if (ctx->h_cand) cudaFreeHost(ctx->h_cand);
        if (ctx->h_sums) cudaFreeHost(ctx->h_sums);
        ctx->h_cand = nullptr; ctx->h_sums = nullptr;
        ctx->h_cap = 0;
        CK(cudaMallocHost(&ctx->h_cand, sizeof(DevCand) * B));
        CK(cudaMallocHost(&ctx->h_sums, sizeof(double) * STL_EVAL_NSUMS * B));
        ctx->h_cap = B;
    }
    if (B > ctx->d_sums_cap) {
        dfree(ctx->d_sums);
        ctx->d_sums_cap = 0;
        CK(cudaMalloc(&ctx->d_sums, sizeof(double) * STL_EVAL_NSUMS * B));
        ctx->d_sums_cap = B;
    }
    return STL_OK;
}

// K1 kernels one pass launches (work counter [5]): the one-kernel K1 when the pack has a fitting keyframe, the three of the
// banded K1 when it has an oversize one
int k1_launches(const stl_ctx *c) { return (c->lay.n_fit > 0 ? 1 : 0) + (c->pk.n_ov > 0 ? 3 : 0); }

// K1 over the selected keyframes of nb candidates: the one-kernel K1 over the fitting ones (the pack's own selection when no
// keyframe is oversize), the banded three-kernel K1 over the oversize ones; both write the same per-keyframe records
stl_status_t launch_k1(stl_ctx *ctx, int nb, cudaStream_t st, int with_terms) {
    const PackLayout &L = ctx->lay;
    if (L.n_fit > 0) {
        DevPack fit = ctx->pk;
        if (fit.n_ov > 0) { fit.sel = (ctx->route.all ? ctx->d_all : ctx->d_sel).lists; fit.n_sel = ctx->route.n_fit; }
        CK(launch_assoc2d(fit, ctx->wk, ctx->dpr, nb, L.k1_smem, L.max_kp, L.max_tab, L.max_groups, st, with_terms));
    }
    if (ctx->pk.n_ov > 0)
        CK(launch_assoc2d_split(ctx->pk, ctx->wk, ctx->dpr, nb, L.k1_split_smem, L.ov_max_bands, L.ov_max_surv, st, with_terms));
    return STL_OK;
}

// scan points and keypoints an evaluation of B candidates walks (those of the selected keyframes)
void set_eval_counters(stl_ctx *ctx, int B) {
    ctx->counters[0] = (double)ctx->route.pts * B;
    ctx->counters[1] = (double)ctx->route.kp * B;
    ctx->counters[4] = ((double)ctx->route.pts * 12.0 + (double)ctx->route.kp * 16.0) * B;
}

// 3-D 1-NN / k-NN queries of an evaluation whose records count q3 3-D terms (cnt_3d3d summed over the candidates)
void set_query_counters(stl_ctx *ctx, double q3) {
    ctx->counters[2] = ctx->params.err_weight[1] > 1e-10 ? q3 : 0.0;
    ctx->counters[3] = (ctx->params.use_plane && ctx->params.err_weight[1] > 1e-10) ? q3 : 0.0;
}

// Enqueues the evaluation of B candidates; d_out [B][STL_EVAL_NSUMS] device.
// exchange: the record of this call is complete after K3 (stl_eval_batch): K3 sums it over the ranks, chunk by chunk, when
// the peer path is up; *exchanged tells the caller whether that happened (else it runs the NCCL all-reduce)
// marks: record ev_k1 / ev_k2a / ev_k3 behind K1 / K2a / K3 (single-chunk batches only: the overlapped step)
stl_status_t enqueue_eval(stl_ctx *ctx, const double *x, int B, double *d_out, cudaStream_t st, bool debug, int out_stride = STL_EVAL_NSUMS,
                          bool exchange = false, bool *exchanged = nullptr, bool marks = false) {
    stl_status_t s = ensure_work(ctx, B, debug);
    if (s != STL_OK) return s;
    if (!ctx->h2d_done) CK(cudaEventCreateWithFlags(&ctx->h2d_done, cudaEventDisableTiming));
    CK(cudaEventSynchronize(ctx->h2d_done));
    for (int b = 0; b < B; ++b) make_candidate(x + (size_t)b * 7, ctx->h_cand + b);
    const int Bc = ctx->wk.Bc;
    for (int c0 = 0; c0 < B; c0 += Bc) {
        const int nb = std::min(Bc, B - c0);
        CK(cudaMemcpyAsync(ctx->wk.cand, ctx->h_cand + c0, sizeof(DevCand) * nb, cudaMemcpyHostToDevice, st));
        { StageTimer t(ctx, STL_STAGE_ASSOC2D, st); s = launch_k1(ctx, nb, st, 1); if (s != STL_OK) return s; }
        ctx->launches += k1_launches(ctx) - 1;
        if (marks) CK(cudaEventRecord(ctx->ev_k1, st));
        { StageTimer t(ctx, STL_STAGE_KNN3D, st); CK(launch_align3d(ctx->pk, ctx->wk, ctx->dpr, nb, debug ? 1 : 0, st, marks ? ctx->ev_k2a : nullptr,
                                                                            marks ? ctx->lm.nnb_pos : nullptr, marks ? ctx->lm.nbb_m : nullptr)); }
        {
            StageTimer t(ctx, STL_STAGE_REDUCE, st);
            const P2pView pv = exchange ? p2p_view(ctx, nb, 0, STL_EVAL_NSUMS) : P2pView();
            if (exchanged) *exchanged = pv.n > 1;
            CK(launch_reduce(ctx->pk, ctx->wk, ctx->dpr, nb, d_out + (size_t)c0 * out_stride, st, out_stride, &pv));
        }
        if (marks) CK(cudaEventRecord(ctx->ev_k3, st));
        ctx->launches += 4;  // K1, K2a, K2b, K3
        ctx->wk_x.assign(x + (size_t)c0 * 7, x + (size_t)(c0 + nb) * 7);
        ctx->wk_has_nn = true;  // K2a runs for every query of a kept frame and writes its nn_pos
    }
    CK(cudaEventRecord(ctx->h2d_done, st));
    set_eval_counters(ctx, B);
    ctx->last_x.assign(x, x + (size_t)B * 7);
    ctx->dbg_b = -1;
    return STL_OK;
}

// The one exchange of the path: fp64 sum of the per-candidate record over the keyframe shards, in place, on the
// compute stream (iba_global.cpp:239-251,274-275,318-326 are the sums it completes).
stl_status_t allreduce_record(stl_ctx *ctx, double *d_buf, size_t count, cudaStream_t st) {
    if (!ctx->comm || ctx->comm_size <= 1) return STL_OK;
    StageTimer t(ctx, STL_STAGE_ALLREDUCE, st);
    ctx->nccl_exchanges += 1;
    const ncclResult_t r = ncclAllReduce(d_buf, d_buf, count, ncclDouble, ncclSum, ctx->comm, st);
    if (r != ncclSuccess) return fail(ctx, STL_ERR_CUDA, "ncclAllReduce: %s", ncclGetErrorString(r));
    return STL_OK;
}

// Enqueues BuildProblem at x0[p] for the problems p < P flagged in `rebuild` (null: all, as a new set of P problems) on `st`.
// The 2-D association (FindProjectCorrespondences) of a chunk of up to wk.Bc problems is taken from the workspace when the
// preceding evaluation left the correspondences of exactly those x0 there, else K1 runs (without the cost terms) over the
// chunk's starts.  Every chunk's problems are associated by the same launches, one lane each.
// hint_ready (single problem only): the association runs on a stream of its own beside the evaluation that (a) answers its
// map-point 1-NN itself (K2a with lm_pos / lm_m: k_lm_knn_b is not launched) and (b) signals hint_ready behind K2a
// [lo, hi) (hi < 0: P): only the problems of that range are handled by this call — the set is begun when lo = 0 and completed
// when hi = P, so that a caller can put an evaluation of each chunk of starts in front of its association (stl_step_multi)
stl_status_t enqueue_associate(stl_ctx *ctx, const double *x0, int P, const uint8_t *rebuild, cudaStream_t st, cudaEvent_t hint_ready = nullptr,
                               int lo = 0, int hi = -1) {
    const DevPack &pk = ctx->pk;
    LmState &lm = ctx->lm;
    if (hi < 0) hi = P;
    int n_all = 0;
    std::vector<int> todo;
    for (int p = 0; p < P; ++p)
        if (!rebuild || rebuild[p]) { ++n_all; if (p >= lo && p < hi) todo.push_back(p); }
    const int n = (int)todo.size(), Bc = ctx->wk.Bc;
    stl_status_t s = ensure_work(ctx, std::max(1, std::min(n, Bc)), false);  // pinned staging for a chunk of starts
    if (s != STL_OK) return s;
    cudaError_t e = cudaSuccess;
    if (lo == 0) e = lm_begin(pk, ctx->dpr, lm, P, rebuild != nullptr, std::max(1, std::min(n_all, Bc)), st);
    if (e != cudaSuccess) return fail(ctx, STL_ERR_CUDA, "association buffers: %s", cudaGetErrorString(e));
    const bool cert = !getenv("STL_NO_NN_CERT");
    std::vector<int2> lanes;
    for (int c0 = 0; c0 < n; c0 += Bc) {
        const int nb = std::min(Bc, n - c0);
        lanes.assign(nb, make_int2(0, 0));
        bool reuse = !getenv("STL_NO_ASSOC_REUSE");
        for (int j = 0; j < nb && reuse; ++j) {
            const double *xp = x0 + (size_t)todo[c0 + j] * 7;
            int slot = -1;
            for (size_t k = 0; k * 7 + 7 <= ctx->wk_x.size(); ++k)
                if (memcmp(&ctx->wk_x[k * 7], xp, 7 * sizeof(double)) == 0) { slot = (int)k; break; }
            lanes[j] = make_int2(slot, todo[c0 + j]);
            reuse = slot >= 0;
        }
        const bool hints = reuse && ctx->wk_has_nn;  // K2a's 1-NN of the same map points at these x
        if (reuse) {
            ctx->assoc_reused += nb;
        } else {
            if (hint_ready) return fail(ctx, STL_ERR_STATE, "overlapped step: the evaluation's correspondences are not in the workspace");
            DevCand *hc = ctx->h_cand;
            if (!ctx->h2d_done) CK(cudaEventCreateWithFlags(&ctx->h2d_done, cudaEventDisableTiming));
            CK(cudaEventSynchronize(ctx->h2d_done));
            ctx->wk_x.resize((size_t)nb * 7);
            for (int j = 0; j < nb; ++j) {
                const double *xp = x0 + (size_t)todo[c0 + j] * 7;
                make_candidate(xp, hc + j);
                memcpy(&ctx->wk_x[(size_t)j * 7], xp, 7 * sizeof(double));
                lanes[j] = make_int2(j, todo[c0 + j]);
            }
            CK(cudaMemcpyAsync(ctx->wk.cand, hc, sizeof(DevCand) * nb, cudaMemcpyHostToDevice, st));
            CK(cudaEventRecord(ctx->h2d_done, st));
            // 2-D association at x0 (FindProjectCorrespondences, iba_local.cpp:191): K1 without the cost terms
            { StageTimer t(ctx, STL_STAGE_ASSOC2D, st); s = launch_k1(ctx, nb, st, 0); if (s != STL_OK) return s; }
            ctx->launches += k1_launches(ctx);
            ctx->wk_has_nn = false;
        }
        e = lm_set_lanes(lm, lanes.data(), nb, st);
        if (e == cudaSuccess && hint_ready) {  // on a stream of its own: the part that needs K2a's answer waits for it, outside the stage timers
            { StageTimer t(ctx, STL_STAGE_ASSOC_LM, st); e = lm_associate(pk, ctx->wk, ctx->dpr, lm, nb, st, hints, cert, 1);
              if (e == cudaSuccess) e = lm_compact2d(lm, st); }
            if (e == cudaSuccess) e = cudaStreamWaitEvent(st, hint_ready, 0);
            if (e == cudaSuccess) { StageTimer t(ctx, STL_STAGE_ASSOC_LM, st, false); e = lm_associate(pk, ctx->wk, ctx->dpr, lm, nb, st, hints, cert, 2, true); }
        } else if (e == cudaSuccess) {
            StageTimer t(ctx, STL_STAGE_ASSOC_LM, st); e = lm_associate(pk, ctx->wk, ctx->dpr, lm, nb, st, hints, cert);
        }
        if (e != cudaSuccess) return fail(ctx, STL_ERR_CUDA, "associate: %s", cudaGetErrorString(e));
        ctx->launches += (ctx->dpr.plane_index && !ctx->dpr.use_gpr) ? 3 : 4;  // the association kernels (cub select kernels not counted)
    }
    if (hi < P) return STL_OK;
    if (!hint_ready) { StageTimer t(ctx, STL_STAGE_ASSOC_LM, st, false); e = lm_compact2d(lm, st); }
    if (e == cudaSuccess) e = lm_finish_associate(lm, ctx->dpr.use_gpr != 0, st);
    if (e == cudaSuccess && !hint_ready) e = lm_copy_counts(lm, st);  // the overlapped step reads them back after its linearisation
    if (e != cudaSuccess) return fail(ctx, STL_ERR_CUDA, "associate: %s", cudaGetErrorString(e));
    if (ctx->params.use_gpr && ctx->params.gpr_optimize && n_all > 0) {  // GPR::fit per factor (IBACalib2.hpp:460-461), host side, per rebuilt problem
        DevCand *d_c0 = nullptr;
        e = cudaMalloc(&d_c0, sizeof(DevCand));
        for (int p = 0; p < P && e == cudaSuccess; ++p) {
            if (rebuild && !rebuild[p]) continue;
            DevCand hc;
            make_candidate(x0 + (size_t)p * 7, &hc);
            e = cudaMemcpyAsync(d_c0, &hc, sizeof(DevCand), cudaMemcpyHostToDevice, st);
            if (e == cudaSuccess) e = lm_fit_gpr_hyper(pk, d_c0, ctx->dpr, lm, p, st, ctx->params.gpr_grad_flavour);
            ctx->launches += 2;
        }
        cudaFree(d_c0);
        if (e != cudaSuccess) return fail(ctx, STL_ERR_CUDA, "GPR hyper-parameter fit: %s", cudaGetErrorString(e));
    }
    ctx->dbg_b = -1;
    ctx->last_x.clear();
    return STL_OK;
}

// The calls that read ONE frozen problem (stl_linearize_batch, stl_block_counts, stl_eval_blocks, stl_gpr_hyper, stl_step_batch
// without re-association) refuse a set of several.
stl_status_t need_single(stl_ctx *ctx, const char *call, const char *multi) {
    if (ctx->lm.ready && ctx->lm.P > 1)
        return fail(ctx, STL_ERR_STATE, "%s: the frozen set holds %d problems; use %s (or stl_associate to freeze one)", call, ctx->lm.P, multi);
    return STL_OK;
}

// Makes r the current keyframe list, whose device copy is complete (d_all for every keyframe, else d_sel).  Every keyframe
// (the state of a new pack): no selection array, the kernels' grids are those of the whole pack.
void use_route(stl_ctx *c, KfRoute &&r) {
    const stl_ctx::DevRoute &d = r.all ? c->d_all : c->d_sel;
    DevPack &pk = c->pk;
    pk.sel = r.all ? nullptr : d.sel; pk.sel_mp = r.all ? nullptr : d.sel_mp;
    pk.n_sel = r.n_sel; pk.n_sel_mp = r.n_sel_mp;
    pk.ov_sel = d.lists ? d.lists + pk.n_kf : nullptr; pk.n_ov_sel = r.n_ov;
    c->route = std::move(r);
}

// A new selection invalidates what was computed over the previous one: the frozen problem set (the linearise calls refuse until
// the next association), the 2-D association reuse and the debug re-evaluation
void drop_selection_state(stl_ctx *c) {
    c->lm.ready = false;
    c->wk_x.clear();
    c->wk_has_nn = false;
    c->last_x.clear();
    c->dbg_b = -1;
}

// the debug getters read an unselected keyframe as empty
bool kf_selected(const stl_ctx *c, int kf) { return c->route.mask[(size_t)kf] != 0; }

stl_status_t run_debug(stl_ctx *ctx, int b) {
    if (!ctx->has_pack) return fail(ctx, STL_ERR_STATE, "no pack uploaded");
    if (b < 0 || (size_t)b * 7 + 7 > ctx->last_x.size()) return fail(ctx, STL_ERR_INVALID, "candidate %d was not part of the last batch", b);
    if (ctx->dbg_b == b) return STL_OK;
    std::vector<double> keep = ctx->last_x;
    double xb[7];
    memcpy(xb, &keep[(size_t)b * 7], sizeof(xb));
    stl_status_t s = ensure_work(ctx, 1, true);
    if (s != STL_OK) return s;
    cudaStream_t st = acquire_stream(ctx, nullptr);
    s = enqueue_eval(ctx, xb, 1, ctx->d_sums, st, true);
    ctx->last_x = keep;
    if (s != STL_OK) return s;
    CK(cudaStreamSynchronize(st));
    ctx->dbg_b = b;
    return STL_OK;
}

}  // namespace

extern "C" {

int32_t stl_abi_version(void) { return STL_ABI_VERSION; }

void stl_default_params(stl_params_t *p) {
    memset(p, 0, sizeof(*p));
    p->max_pixel_dist = 1.5; p->corr_3d_2d_threshold = 40.0; p->corr_3d_3d_threshold = 10.0;
    p->norm_radius = 0.6; p->norm_reg_threshold = 0.02; p->min_diff_dist = 0.2;
    p->err_weight[0] = 1.0; p->err_weight[1] = 1.0;
    p->he_threshold = 0.094; p->valid_rate = 0.95;
    p->max_3d_dist = 1.0; p->robust_kernel_delta = 2.98; p->robust_kernel_3ddelta = 1.0;
    p->num_min_corr = 30; p->norm_max_pts = 30; p->norm_min_pts = 5; p->use_plane = 1;
    p->use_gpr = 0; p->gpr_sigma = 10.0; p->gpr_l = 10.0; p->gpr_sigma_noise = 1e-10;
    p->plane_index = 1; p->variant = 0;
    p->gpr_optimize = 0; p->gpr_grad_flavour = 0;
}

stl_status_t stl_create(const stl_params_t *params, int32_t device, stl_ctx_t **out) {
    if (!out || !params) return STL_ERR_INVALID;
    *out = nullptr;
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess || n <= 0 || device < 0 || device >= n) { cudaGetLastError(); return STL_ERR_NO_DEVICE; }
    cudaDeviceProp prop;
    if (cudaGetDeviceProperties(&prop, device) != cudaSuccess) return STL_ERR_NO_DEVICE;
    if (prop.major != 10 || prop.minor != 0) return STL_ERR_NO_DEVICE;  // only sm_100a SASS is embedded (no PTX): a 10.3 part cannot run it
    if (params->norm_max_pts < 1 || params->norm_max_pts > kMaxK) return STL_ERR_CAPACITY;
    if (params->variant != 0 && params->variant != 1) return STL_ERR_INVALID;
    if (cudaSetDevice(device) != cudaSuccess) return STL_ERR_CUDA;
    stl_ctx *c = new stl_ctx();
    c->device = device;
    c->params = *params;
    set_dev_params(c);
    if (cudaStreamCreateWithFlags(&c->own_stream, cudaStreamNonBlocking) != cudaSuccess) { delete c; return STL_ERR_CUDA; }
    c->stream = c->own_stream;
    c->last_stream = c->own_stream;
    cudaEventCreateWithFlags(&c->handoff, cudaEventDisableTiming);
    *out = c;
    return STL_OK;
}

void stl_destroy(stl_ctx_t *c) {
    if (!c) return;
    cudaSetDevice(c->device);
    cudaDeviceSynchronize();
    for (int q = 0; q < kP2pMaxRanks; ++q) {
        if (q != c->comm_rank && c->p2p.data[q]) cudaIpcCloseMemHandle(c->p2p.data[q]);
        if (q != c->comm_rank && c->p2p.flag[q]) cudaIpcCloseMemHandle(c->p2p.flag[q]);
    }
    dfree(c->p2p_data); dfree(c->p2p_flag); dfree(c->p2p.err);
    if (c->comm) { ncclCommDestroy(c->comm); c->comm = nullptr; }
    drain_events(c);
    for (auto e : c->ev_pool) cudaEventDestroy(e);
    free_work(c);
    free_pack(c);
    lm_free(c->lm);
    dfree(c->d_sums); dfree(c->d_lin);
    if (c->h_cand) cudaFreeHost(c->h_cand);
    if (c->h_sums) cudaFreeHost(c->h_sums);
    if (c->h_lin) cudaFreeHost(c->h_lin);
    if (c->h2d_done) cudaEventDestroy(c->h2d_done);
    if (c->handoff) cudaEventDestroy(c->handoff);
    if (c->aux_stream) cudaStreamDestroy(c->aux_stream);
    for (cudaEvent_t e : {c->ev_k1, c->ev_k2a, c->ev_k3, c->ev_aux}) if (e) cudaEventDestroy(e);
    if (c->own_stream) cudaStreamDestroy(c->own_stream);
    delete c;
}

const char *stl_last_error(const stl_ctx_t *c) { return c ? c->err.c_str() : "null context"; }

stl_status_t stl_upload_pack(stl_ctx_t *ctx, const stl_pack_t *p) {
    if (!ctx || !p) return STL_ERR_INVALID;
    std::lock_guard<std::mutex> lk(ctx->mu);
    CK(cudaSetDevice(ctx->device));
    // ---- validation, layout and K1 routing (host, packlayout.hpp): a rejected pack leaves the context as it was
    K1Limits lim;
    CK(cudaDeviceGetAttribute(&lim.smem_optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, ctx->device));
    lim.k1_smem = assoc2d_smem_bytes;
    lim.split_smem = assoc2d_split_smem_bytes;
    lim.allow_oversize = ctx->allow_oversize;
    const char *route_env = getenv("STL_K1_OVERSIZE");
    lim.route_all = (route_env && strcmp(route_env, "all") == 0) || getenv("STL_K1_SPLIT");  // diagnostic: every keyframe on the banded K1
    PackLayout lay;
    const stl_status_t s = layout_pack(p, lim, lay, ctx->err);
    if (s != STL_OK) return s;
    if (lay.n_fit > 0) CK(assoc2d_configure(lay.k1_smem));
    if (!lay.ov.empty()) CK(assoc2d_split_configure(lay.k1_split_smem));

    // ---- from here on the previous state is gone
    free_work(ctx);
    free_pack(ctx);
    lm_free(ctx->lm);
    ctx->lay = std::move(lay);
    const PackLayout &L = ctx->lay;
    std::vector<DevKf> &hk = ctx->lay.kf;
    const int F = L.n_kf, C = L.n_covis;
    const long long NK = L.n_kp_total;
    CK(cudaDeviceGetAttribute(&ctx->n_sm, cudaDevAttrMultiProcessorCount, ctx->device));
    cudaStream_t st = acquire_stream(ctx, nullptr);
    struct Scope {  // events and the raw-scan scratch are released on every exit path
        cudaEvent_t ev0 = nullptr, ev1 = nullptr; float *d_raw = nullptr; BuildScratch scr;
        ~Scope() { if (ev0) cudaEventDestroy(ev0); if (ev1) cudaEventDestroy(ev1); if (d_raw) cudaFree(d_raw); scr.release(); }
    } scope;
    CK(cudaEventCreate(&scope.ev0)); CK(cudaEventCreate(&scope.ev1));
    cudaEvent_t ev0 = scope.ev0, ev1 = scope.ev1;
    CK(cudaEventRecord(ev0, st));
    PackTables tab;
    build_tables(p, L, ctx->params.variant, ctx->params.max_pixel_dist, tab);
    KfRoute all = route_keyframes(L, nullptr, 0);

    // ---- device allocation + small uploads
    DevPack &pk = ctx->pk;
    pk.n_kf = F; pk.n_covis = C; pk.n_pad_total = L.n_pad_total; pk.n_nodes_total = L.n_nodes_total; pk.n_kp_total = NK; pk.n_mp_total = L.n_mp_total;
    const long long nodes = L.n_nodes_total;
    const size_t npt = (size_t)std::max<long long>(L.n_pad_total, 4), nkk = (size_t)std::max<long long>(NK, 1);
    CK(cudaMalloc(&pk.kf, sizeof(DevKf) * F));
    CK(cudaMalloc(&pk.px, 4 * npt)); CK(cudaMalloc(&pk.py, 4 * npt)); CK(cudaMalloc(&pk.pz, 4 * npt)); CK(cudaMalloc(&pk.orig, 4 * npt));
    CK(cudaMalloc(&pk.node_lo, sizeof(float4) * nodes)); CK(cudaMalloc(&pk.node_hi, sizeof(float4) * nodes));
    if (ctx->adj_r2 > 0.f) { CK(cudaMalloc(&pk.adj, sizeof(uint16_t) * 32 * (size_t)nodes)); CK(cudaMalloc(&pk.adj_cov, sizeof(float) * (size_t)nodes)); }
    CK(cudaMalloc(&pk.k1tab, tab.k1tab.size()));
    CK(cudaMemcpyAsync(pk.k1tab, tab.k1tab.data(), tab.k1tab.size(), cudaMemcpyHostToDevice, st));
    CK(cudaMalloc(&pk.bitmap, 4 * (size_t)L.bm_words)); CK(cudaMalloc(&pk.grid_start, 4 * (size_t)L.grid_cells)); CK(cudaMalloc(&pk.grid_kp, 4 * nkk));
    CK(cudaMalloc(&pk.kp_xy, sizeof(float2) * nkk)); CK(cudaMalloc(&pk.kp_mp, 12 * nkk));
    CK(cudaMalloc(&pk.Tcw, 48 * (size_t)F)); CK(cudaMalloc(&pk.relpose, 48 * (size_t)std::max(F * C, 1)));
    CK(cudaMalloc(&pk.covis_valid, (size_t)std::max(F * C, 1))); CK(cudaMalloc(&pk.covis_uv, sizeof(float2) * std::max<size_t>(nkk * C, 1)));
    CK(cudaMalloc(&pk.he_Tc, 48 * (size_t)F)); CK(cudaMalloc(&pk.he_Tl, 96 * (size_t)F));
    CK(cudaMemcpyAsync(pk.kf, hk.data(), sizeof(DevKf) * F, cudaMemcpyHostToDevice, st));
    CK(cudaMemcpyAsync(pk.bitmap, tab.bitmap.data(), 4 * (size_t)L.bm_words, cudaMemcpyHostToDevice, st));
    CK(cudaMemcpyAsync(pk.grid_start, tab.grid_start.data(), 4 * (size_t)L.grid_cells, cudaMemcpyHostToDevice, st));
    if (NK > 0) {
        CK(cudaMemcpyAsync(pk.grid_kp, tab.grid_kp.data(), 4 * (size_t)NK, cudaMemcpyHostToDevice, st));
        CK(cudaMemcpyAsync(pk.kp_xy, tab.kp_xy, 8 * (size_t)NK, cudaMemcpyHostToDevice, st));
        if (ctx->params.variant == 1) {
            CK(cudaMalloc(&pk.kp_xyd, sizeof(double2) * nkk));
            CK(cudaMemcpyAsync(pk.kp_xyd, tab.kp_xyd.data(), 16 * (size_t)NK, cudaMemcpyHostToDevice, st));
        }
        CK(cudaMemcpyAsync(pk.kp_mp, p->kp_mappoint, 12 * (size_t)NK, cudaMemcpyHostToDevice, st));
        if (C > 0) CK(cudaMemcpyAsync(pk.covis_uv, p->covis_uv, 8 * (size_t)NK * C, cudaMemcpyHostToDevice, st));
    }
    CK(cudaMemcpyAsync(pk.Tcw, p->Tcw, 48 * (size_t)F, cudaMemcpyHostToDevice, st));
    if (C > 0) {
        CK(cudaMemcpyAsync(pk.relpose, p->covis_relpose, 48 * (size_t)F * C, cudaMemcpyHostToDevice, st));
        CK(cudaMemcpyAsync(pk.covis_valid, p->covis_valid, (size_t)F * C, cudaMemcpyHostToDevice, st));
    }
    CK(cudaMemcpyAsync(pk.he_Tc, p->he_Tc, 48 * (size_t)F, cudaMemcpyHostToDevice, st));
    CK(cudaMemcpyAsync(pk.he_Tl, p->he_Tl, 96 * (size_t)F, cudaMemcpyHostToDevice, st));
    if (!L.ov.empty()) {  // the oversize descriptors and the K1 lists of the whole pack (and room for those of a selection)
        const int n_ov = (int)L.ov.size();
        pk.n_ov = n_ov; pk.n_ov_kp = L.n_ov_kp; pk.n_ov_surv = L.n_ov_surv; pk.n_ov_match = L.n_ov_match;
        CK(cudaMalloc(&ctx->d_ov, sizeof(OvKf) * (size_t)n_ov));
        CK(cudaMemcpyAsync(ctx->d_ov, L.ov.data(), sizeof(OvKf) * (size_t)n_ov, cudaMemcpyHostToDevice, st));
        pk.ov = ctx->d_ov;
        CK(cudaMalloc(&ctx->d_all.lists, sizeof(int) * 2 * (size_t)F));
        CK(cudaMalloc(&ctx->d_sel.lists, sizeof(int) * 2 * (size_t)F));
        CK(cudaMemcpyAsync(ctx->d_all.lists, all.lists.data(), sizeof(int) * 2 * (size_t)F, cudaMemcpyHostToDevice, st));
    }
    CK(cudaStreamSynchronize(st));

    // ---- scans: chunked upload + index build
    {
        const long long chunk_pts = 32ll << 20;
        float *&d_raw = scope.d_raw;
        float k0_ms = 0.f;
        long long raw_cap = 0;
        int f0 = 0;
        while (f0 < F) {
            int f1 = f0 + 1;
            while (f1 < F && p->scan_offset[f1 + 1] - p->scan_offset[f0] <= chunk_pts && f1 - f0 < 32768) ++f1;
            const long long n = p->scan_offset[f1] - p->scan_offset[f0];
            if (n > raw_cap) { dfree(d_raw); raw_cap = std::max(n, std::min(chunk_pts, (long long)p->scan_offset[F])); CK(cudaMalloc(&d_raw, 12 * (size_t)std::max<long long>(raw_cap, 1))); }
            if (n > 0) CK(cudaMemcpyAsync(d_raw, p->scan_xyz + p->scan_offset[f0] * 3, 12 * (size_t)n, cudaMemcpyHostToDevice, st));
            std::vector<long long> off(f1 - f0 + 1);
            for (int f = f0; f <= f1; ++f) off[f - f0] = p->scan_offset[f];
            cudaError_t e = build_scan_index(d_raw, off.data(), f1 - f0, f0, hk.data(), pk, ctx->adj_r2, st, scope.scr, &k0_ms);
            if (e != cudaSuccess) return fail(ctx, STL_ERR_CUDA, "index build: %s", cudaGetErrorString(e));
            f0 = f1;
        }
        dfree(d_raw);
        // K0's own device time (kernels only); the wall time of the whole upload is the caller's to measure
        ctx->stage_ms[STL_STAGE_BUILD] += k0_ms;
        ctx->stage_n[STL_STAGE_BUILD] += 1;
    }
    CK(cudaMemcpy(hk.data(), pk.kf, sizeof(DevKf) * F, cudaMemcpyDeviceToHost));  // pmax filled by the build
    if (pk.adj && getenv("STL_DEBUG_STATS")) {  // how many real leaves got no adjacency row (> 32 neighbours)?
        long long real = 0, empty = 0, entries = 0, partial = 0;
        double cov_sum = 0;
        std::vector<uint16_t> row;
        std::vector<float> cov;
        for (int f = 0; f < F; f += std::max(1, F / 16)) {
            const int nl = (hk[f].n_pts + kLeaf - 1) / kLeaf;
            row.resize((size_t)nl * 32);
            CK(cudaMemcpy(row.data(), pk.adj + hk[f].node_off * 32, row.size() * 2, cudaMemcpyDeviceToHost));
            cov.resize((size_t)nl);
            CK(cudaMemcpy(cov.data(), pk.adj_cov + hk[f].node_off, cov.size() * 4, cudaMemcpyDeviceToHost));
            for (int l = 0; l < nl; ++l) if (cov[l] >= 0 && cov[l] < 1e30f) { ++partial; cov_sum += std::sqrt((double)cov[l]); }
            for (int l = 0; l < nl; ++l) {
                int c = 0;
                for (int t = 0; t < 32; ++t) c += row[(size_t)l * 32 + t] != 0xffffu;
                ++real; empty += c == 0; entries += c;
            }
        }
        fprintf(stderr, "[stl] leaf adjacency (sampled keyframes): %lld leaves, %.2f%% without a row, %.1f neighbours per row, %.1f%% truncated (mean coverage %.3f m)\n", real,
                100.0 * empty / std::max<long long>(real, 1), (double)entries / std::max<long long>(real - empty, 1),
                100.0 * partial / std::max<long long>(real, 1), cov_sum / std::max<long long>(partial, 1));
    }
    if (ctx->params.plane_index) {
        CK(cudaMalloc(&pk.pl_rec, sizeof(PlaneRec) * npt));
        CK(cudaMalloc(&pk.pl_m, 4 * npt));
        CK(cudaEventRecord(ev0, st));
        for (int f0 = 0; f0 < F;) {  // bounded scratch: a few million points at a time
            int f1 = f0 + 1;
            long long pts = hk[f0].n_pad;
            while (f1 < F && pts + hk[f1].n_pad <= (4ll << 20)) pts += hk[f1++].n_pad;
            cudaError_t e = build_plane_index(pk, hk.data(), f0, f1 - f0, ctx->dpr, st, scope.scr);
            if (e != cudaSuccess) return fail(ctx, STL_ERR_CUDA, "plane index: %s", cudaGetErrorString(e));
            f0 = f1;
        }
        CK(cudaEventRecord(ev1, st));
        CK(cudaStreamSynchronize(st));
        float ms = 0;
        CK(cudaEventElapsedTime(&ms, ev0, ev1));
        ctx->stage_ms[STL_STAGE_PLANE_INDEX] += ms;
        ctx->stage_n[STL_STAGE_PLANE_INDEX] += 1;
    }
    use_route(ctx, std::move(all));
    ctx->has_pack = true;
    return STL_OK;
}

stl_status_t stl_eval_batch_device(stl_ctx_t *ctx, const double *x, int32_t B, double *d_sums, void *stream) {
    if (!ctx || !x || !d_sums || B <= 0) return STL_ERR_INVALID;
    std::lock_guard<std::mutex> lk(ctx->mu);
    if (!ctx->has_pack) return fail(ctx, STL_ERR_STATE, "stl_upload_pack has not been called");
    CK(cudaSetDevice(ctx->device));
    cudaStream_t st = acquire_stream(ctx, stream);
    bool done = false;
    stl_status_t s = enqueue_eval(ctx, x, B, d_sums, st, false, STL_EVAL_NSUMS, true, &done);
    if (s != STL_OK || done) return s;
    return allreduce_record(ctx, d_sums, (size_t)B * STL_EVAL_NSUMS, st);
}

stl_status_t stl_eval_batch(stl_ctx_t *ctx, const double *x, int32_t B, stl_eval_sums_t *sums) {
    if (!ctx || !x || !sums || B <= 0) return STL_ERR_INVALID;
    std::lock_guard<std::mutex> lk(ctx->mu);
    if (!ctx->has_pack) return fail(ctx, STL_ERR_STATE, "stl_upload_pack has not been called");
    CK(cudaSetDevice(ctx->device));
    stl_status_t s = ensure_work(ctx, B, false);
    if (s != STL_OK) return s;
    cudaStream_t st = acquire_stream(ctx, nullptr);
    bool done = false;
    s = enqueue_eval(ctx, x, B, ctx->d_sums, st, false, STL_EVAL_NSUMS, true, &done);
    if (s != STL_OK) return s;
    if (!done) s = allreduce_record(ctx, ctx->d_sums, (size_t)B * STL_EVAL_NSUMS, st);
    if (s != STL_OK) return s;
    CK(cudaMemcpyAsync(ctx->h_sums, ctx->d_sums, sizeof(double) * STL_EVAL_NSUMS * B, cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    memcpy(sums, ctx->h_sums, sizeof(double) * STL_EVAL_NSUMS * B);
    double q3 = 0;
    for (int b = 0; b < B; ++b) q3 += sums[b].cnt_3d3d;
    set_query_counters(ctx, q3);
    return STL_OK;
}

void stl_finalize(const stl_params_t *pr, const stl_eval_sums_t *s, stl_ba_error_t *o) {
    // iba_global.cpp:330-343
    if (s->valid_3d2d == 0 && pr->err_weight[0] > 1e-10) o->f1 = DBL_MAX; else o->f1 = s->sum_3d2d / s->valid_3d2d;
    if (s->valid_3d3d == 0 && pr->err_weight[1] > 1e-10) o->f2 = DBL_MAX; else o->f2 = s->sum_3d3d / s->valid_3d3d;
    o->C = s->sum_he / s->cnt_he;
    o->valid_cnt_3d_2d = (int32_t)s->valid_3d2d;
    o->cnt_3d_2d = (int32_t)s->cnt_3d2d;
}

void stl_bbo(const stl_params_t *pr, const stl_ba_error_t *e, double bbo[4]) {
    // iba_global.cpp:386-388
    bbo[0] = e->f1 * pr->err_weight[0] + e->f2 * pr->err_weight[1];
    bbo[1] = e->C - pr->he_threshold;
    bbo[2] = -e->C - pr->he_threshold;
    bbo[3] = pr->valid_rate - (double)e->valid_cnt_3d_2d / (e->cnt_3d_2d + 1);
}

stl_status_t stl_debug_corrset(stl_ctx_t *ctx, int32_t b, int32_t kf, uint32_t *kp_idx, uint32_t *pt_idx, int32_t cap, int32_t *n) {
    if (!ctx || !n) return STL_ERR_INVALID;
    std::lock_guard<std::mutex> lk(ctx->mu);
    CK(cudaSetDevice(ctx->device));
    stl_status_t s = run_debug(ctx, b);
    if (s != STL_OK) return s;
    if (kf < 0 || kf >= ctx->pk.n_kf) return fail(ctx, STL_ERR_INVALID, "keyframe out of range");
    if (!kf_selected(ctx, kf)) { *n = 0; return STL_OK; }
    int nc = 0;
    CK(cudaMemcpy(&nc, ctx->wk.n_corr + kf, 4, cudaMemcpyDeviceToHost));
    *n = nc;
    const int m = std::min(nc, cap);
    if (m > 0 && kp_idx) CK(cudaMemcpy(kp_idx, ctx->wk.corr_kp + ctx->lay.kf[kf].kp_off, 4 * (size_t)m, cudaMemcpyDeviceToHost));
    if (m > 0 && pt_idx) CK(cudaMemcpy(pt_idx, ctx->wk.corr_pt + ctx->lay.kf[kf].kp_off, 4 * (size_t)m, cudaMemcpyDeviceToHost));
    return STL_OK;
}

stl_status_t stl_debug_align(stl_ctx_t *ctx, int32_t b, int32_t kf, uint32_t *kp_idx, uint32_t *nn_idx, int32_t *n_neigh, int32_t *is_plane,
                             double *dist, uint32_t *knn_idx, int32_t cap, int32_t *n) {
    if (!ctx || !n) return STL_ERR_INVALID;
    std::lock_guard<std::mutex> lk(ctx->mu);
    CK(cudaSetDevice(ctx->device));
    stl_status_t s = run_debug(ctx, b);
    if (s != STL_OK) return s;
    if (kf < 0 || kf >= ctx->pk.n_kf) return fail(ctx, STL_ERR_INVALID, "keyframe out of range");
    if (!kf_selected(ctx, kf)) { *n = 0; return STL_OK; }
    int nq = 0;
    CK(cudaMemcpy(&nq, ctx->wk.n_q + kf, 4, cudaMemcpyDeviceToHost));
    *n = nq;
    const int m = std::min(nq, cap);
    if (m <= 0) return STL_OK;
    const long long off = ctx->lay.kf[kf].kp_off;
    if (kp_idx) {
        int nc = 0;
        CK(cudaMemcpy(&nc, ctx->wk.n_corr + kf, 4, cudaMemcpyDeviceToHost));
        std::vector<uint32_t> qc(m), ck(std::max(nc, 1));
        CK(cudaMemcpy(qc.data(), ctx->wk.q_corr + off, 4 * (size_t)m, cudaMemcpyDeviceToHost));
        CK(cudaMemcpy(ck.data(), ctx->wk.corr_kp + off, 4 * (size_t)nc, cudaMemcpyDeviceToHost));
        for (int i = 0; i < m; ++i) kp_idx[i] = ck[qc[i]];
    }
    if (nn_idx) CK(cudaMemcpy(nn_idx, ctx->wk.dbg_nn + off, 4 * (size_t)m, cudaMemcpyDeviceToHost));
    if (n_neigh) CK(cudaMemcpy(n_neigh, ctx->wk.dbg_m + off, 4 * (size_t)m, cudaMemcpyDeviceToHost));
    if (is_plane) CK(cudaMemcpy(is_plane, ctx->wk.dbg_plane + off, 4 * (size_t)m, cudaMemcpyDeviceToHost));
    if (dist) CK(cudaMemcpy(dist, ctx->wk.dbg_dist + off, 8 * (size_t)m, cudaMemcpyDeviceToHost));
    if (knn_idx) CK(cudaMemcpy(knn_idx, ctx->wk.dbg_knn + off * kMaxK, 4 * (size_t)m * kMaxK, cudaMemcpyDeviceToHost));
    return STL_OK;
}

stl_status_t stl_debug_frame(stl_ctx_t *ctx, int32_t b, int32_t kf, double out[13]) {
    if (!ctx || !out) return STL_ERR_INVALID;
    std::lock_guard<std::mutex> lk(ctx->mu);
    CK(cudaSetDevice(ctx->device));
    stl_status_t s = run_debug(ctx, b);
    if (s != STL_OK) return s;
    if (kf < 0 || kf >= ctx->pk.n_kf) return fail(ctx, STL_ERR_INVALID, "keyframe out of range");
    if (!kf_selected(ctx, kf)) { for (int i = 0; i < 13; ++i) out[i] = 0; return STL_OK; }
    FrameRec r;
    CK(cudaMemcpy(&r, ctx->wk.frame + kf, sizeof(r), cudaMemcpyDeviceToHost));
    std::vector<AlignRec> a(ctx->wk.sub);
    CK(cudaMemcpy(a.data(), ctx->wk.align + (size_t)kf * ctx->wk.sub, sizeof(AlignRec) * ctx->wk.sub, cudaMemcpyDeviceToHost));
    out[0] = r.s2d; out[1] = r.v2d; out[2] = r.c2d; out[3] = r.she; out[4] = r.che; out[5] = r.kept; out[6] = r.ncorr; out[7] = r.nq;
    for (int i = 8; i < 13; ++i) out[i] = 0;
    if (ctx->wk.k1_clk) {
        std::vector<long long> h((size_t)ctx->pk.n_kf * 8);
        cudaMemcpy(h.data(), ctx->wk.k1_clk, 64 * (size_t)ctx->pk.n_kf, cudaMemcpyDeviceToHost);
        double a[8] = {0};
        for (int f = 0; f < ctx->pk.n_kf; ++f) for (int i = 0; i < 8; ++i) a[i] += (double)h[(size_t)f * 8 + i] / ctx->pk.n_kf;
        fprintf(stderr, "[stl] K1 mean clocks/unit: prologue %.0f | cells + table wait %.0f | stream %.0f | exact-1 %.0f | tie pass %.0f | corrset + covisible term %.0f | reduction %.0f | epilogue %.0f\n", a[7], a[0], a[1], a[2], a[3], a[4], a[5], a[6]);
    }
    if (getenv("STL_DEBUG_STATS")) {
        unsigned long long st[8];
        cudaMemcpy(st, ctx->wk.dbg_stats, 64, cudaMemcpyDeviceToHost);
        if (st[0] + st[4]) fprintf(stderr, "[stl] K2a search paths (cumulative): k-NN %llu = adjacency %.1f%% + restart %.1f%% + no row %.1f%% | 1-NN %llu = adjacency %.1f%% + descent after scan %.1f%% + no row %.1f%%\n",
                st[0], 100.0 * st[1] / std::max(st[0], 1ull), 100.0 * st[2] / std::max(st[0], 1ull), 100.0 * st[3] / std::max(st[0], 1ull),
                st[4], 100.0 * st[5] / std::max(st[4], 1ull), 100.0 * st[6] / std::max(st[4], 1ull), 100.0 * st[7] / std::max(st[4], 1ull));
    }
    for (auto &x : a) { out[8] += x.s3d; out[9] += x.v3d; out[10] += x.c3d; out[11] += x.vpl; out[12] += x.vpt; }
    return STL_OK;
}

stl_status_t stl_select_keyframes(stl_ctx_t *ctx, const int32_t *kf, int32_t n) {
    if (!ctx) return STL_ERR_INVALID;
    std::lock_guard<std::mutex> lk(ctx->mu);
    if (!ctx->has_pack) return fail(ctx, STL_ERR_STATE, "stl_upload_pack has not been called");
    const int F = ctx->pk.n_kf;
    if (kf) {  // validated completely before anything changes
        if (n < 0 || n > F) return fail(ctx, STL_ERR_INVALID, "stl_select_keyframes: n = %d is outside [0, n_kf = %d]", n, F);
        for (int i = 0; i < n; ++i) {
            if (kf[i] < 0 || kf[i] >= F) return fail(ctx, STL_ERR_INVALID, "stl_select_keyframes: kf[%d] = %d is outside [0, %d)", i, kf[i], F);
            if (i > 0 && kf[i] <= kf[i - 1]) return fail(ctx, STL_ERR_INVALID, "stl_select_keyframes: the list is not strictly increasing at %d", i);
        }
    }
    CK(cudaSetDevice(ctx->device));
    cudaStream_t st = acquire_stream(ctx, nullptr);
    CK(cudaStreamSynchronize(st));  // the kernels already queued read the previous selection arrays
    drop_selection_state(ctx);
    // from here on the context selects every keyframe until the new selection is complete on the device: a CUDA failure on the
    // way leaves it there (never half-switched between two lists)
    use_route(ctx, route_keyframes(ctx->lay, nullptr, 0));
    if (!kf) return STL_OK;
    KfRoute r = route_keyframes(ctx->lay, kf, n);
    stl_ctx::DevRoute &d = ctx->d_sel;
    cudaError_t e = cudaSuccess;
    if (n > d.cap || !d.sel) {
        dfree(d.sel); dfree(d.sel_mp);
        d.cap = 0;
        const size_t cap = (size_t)std::max(n, 1);
        e = cudaMalloc(&d.sel, sizeof(int) * cap);
        if (e == cudaSuccess) e = cudaMalloc(&d.sel_mp, sizeof(int2) * (cap + 1));
        if (e == cudaSuccess) d.cap = (int)cap;
        else { dfree(d.sel); dfree(d.sel_mp); }
    }
    if (e == cudaSuccess && n > 0) e = cudaMemcpyAsync(d.sel, r.sel.data(), sizeof(int) * (size_t)n, cudaMemcpyHostToDevice, st);
    if (e == cudaSuccess) e = cudaMemcpyAsync(d.sel_mp, r.sel_mp.data(), sizeof(int2) * ((size_t)n + 1), cudaMemcpyHostToDevice, st);
    if (e == cudaSuccess && d.lists) e = cudaMemcpyAsync(d.lists, r.lists.data(), sizeof(int) * 2 * (size_t)F, cudaMemcpyHostToDevice, st);
    if (e == cudaSuccess) e = cudaStreamSynchronize(st);
    if (e != cudaSuccess) return fail(ctx, STL_ERR_CUDA, "stl_select_keyframes: %s (every keyframe stays selected)", cudaGetErrorString(e));
    use_route(ctx, std::move(r));
    return STL_OK;
}

stl_status_t stl_allow_oversize_keyframes(stl_ctx_t *ctx, int32_t allow) {
    if (!ctx) return STL_ERR_INVALID;
    std::lock_guard<std::mutex> lk(ctx->mu);
    if (allow != 0 && allow != 1) return fail(ctx, STL_ERR_INVALID, "stl_allow_oversize_keyframes: allow = %d is neither 0 nor 1", allow);
    ctx->allow_oversize = allow != 0;
    return STL_OK;
}

stl_status_t stl_oversize_keyframes(stl_ctx_t *ctx, int32_t *kf, int32_t cap, int32_t *n) {
    if (!ctx || !n || cap < 0) return STL_ERR_INVALID;
    std::lock_guard<std::mutex> lk(ctx->mu);
    if (!ctx->has_pack) return fail(ctx, STL_ERR_STATE, "stl_upload_pack has not been called");
    *n = (int32_t)ctx->lay.ov.size();
    const int m = std::min(*n, cap);
    if (kf) for (int i = 0; i < m; ++i) kf[i] = ctx->lay.ov[(size_t)i].f;
    return STL_OK;
}

stl_status_t stl_eval_frames(stl_ctx_t *ctx, const double *x, int32_t B, double *out) {
    if (!ctx || !x || !out || B <= 0) return STL_ERR_INVALID;
    std::lock_guard<std::mutex> lk(ctx->mu);
    if (!ctx->has_pack) return fail(ctx, STL_ERR_STATE, "stl_upload_pack has not been called");
    CK(cudaSetDevice(ctx->device));
    stl_status_t s = ensure_work(ctx, B, false);
    if (s != STL_OK) return s;
    const int F = ctx->pk.n_kf, Bc = ctx->wk.Bc;
    const size_t row = (size_t)F * 13;
    if (!ctx->d_frames) CK(cudaMalloc(&ctx->d_frames, sizeof(double) * row * Bc));
    cudaStream_t st = acquire_stream(ctx, nullptr);
    // one workspace chunk at a time: evaluation (no exchange: each rank returns its own keyframes), then the gather of its records
    for (int c0 = 0; c0 < B; c0 += Bc) {
        const int nb = std::min(Bc, B - c0);
        s = enqueue_eval(ctx, x + (size_t)c0 * 7, nb, ctx->d_sums, st, false);
        if (s != STL_OK) return s;
        CK(cudaMemsetAsync(ctx->d_frames, 0, sizeof(double) * row * nb, st));
        CK(launch_frames(ctx->pk, ctx->wk, ctx->dpr, nb, ctx->d_frames, st));
        ctx->launches += 1;
        CK(cudaMemcpyAsync(out + row * c0, ctx->d_frames, sizeof(double) * row * nb, cudaMemcpyDeviceToHost, st));
    }
    CK(cudaStreamSynchronize(st));
    set_eval_counters(ctx, B);
    double q3 = 0;  // cnt_3d3d of the rows: the record's count, exactly (integers)
    for (size_t r = 0; r < (size_t)B * F; ++r) q3 += out[r * 13 + 10];
    set_query_counters(ctx, q3);
    ctx->last_x.assign(x, x + (size_t)B * 7);  // as stl_eval_batch: the debug getters and the 2-D association reuse see this batch
    return STL_OK;
}

stl_status_t stl_knn3d(stl_ctx_t *ctx, int32_t kf, const double *q, int32_t nq, int32_t k, double radius2, uint32_t *out_idx, double *out_d2,
                       int32_t *out_count) {
    if (!ctx || !q || nq < 0 || k < 1 || k > kMaxK) return STL_ERR_INVALID;
    std::lock_guard<std::mutex> lk(ctx->mu);
    if (!ctx->has_pack) return fail(ctx, STL_ERR_STATE, "no pack uploaded");
    if (kf < 0 || kf >= ctx->pk.n_kf) return fail(ctx, STL_ERR_INVALID, "keyframe out of range");
    if (nq == 0) return STL_OK;
    CK(cudaSetDevice(ctx->device));
    double *dq = nullptr, *dd = nullptr; uint32_t *di = nullptr; int *dc = nullptr;
    CK(cudaMalloc(&dq, 24 * (size_t)nq)); CK(cudaMalloc(&dd, 8 * (size_t)nq * k)); CK(cudaMalloc(&di, 4 * (size_t)nq * k)); CK(cudaMalloc(&dc, 4 * (size_t)nq));
    cudaStream_t st = acquire_stream(ctx, nullptr);
    CK(cudaMemcpyAsync(dq, q, 24 * (size_t)nq, cudaMemcpyHostToDevice, st));
    cudaError_t e = launch_knn3d(ctx->pk, kf, dq, nq, k, radius2, di, dd, dc, st);
    if (e == cudaSuccess && out_idx) e = cudaMemcpyAsync(out_idx, di, 4 * (size_t)nq * k, cudaMemcpyDeviceToHost, st);
    if (e == cudaSuccess && out_d2) e = cudaMemcpyAsync(out_d2, dd, 8 * (size_t)nq * k, cudaMemcpyDeviceToHost, st);
    if (e == cudaSuccess && out_count) e = cudaMemcpyAsync(out_count, dc, 4 * (size_t)nq, cudaMemcpyDeviceToHost, st);
    if (e == cudaSuccess) e = cudaStreamSynchronize(st);
    cudaFree(dq); cudaFree(dd); cudaFree(di); cudaFree(dc);
    if (e != cudaSuccess) return fail(ctx, STL_ERR_CUDA, "knn3d: %s", cudaGetErrorString(e));
    return STL_OK;
}

stl_status_t stl_debug_trig(stl_ctx_t *ctx, const double *x, int32_t n, double *acos_out, double *cos_out) {
    if (!ctx || !x || !acos_out || !cos_out || n < 0) return STL_ERR_INVALID;
    std::lock_guard<std::mutex> lk(ctx->mu);
    CK(cudaSetDevice(ctx->device));
    if (n == 0) return STL_OK;
    double *d = nullptr;
    CK(cudaMalloc(&d, 24 * (size_t)n));
    cudaStream_t st = acquire_stream(ctx, nullptr);
    cudaError_t e = cudaMemcpyAsync(d, x, 8 * (size_t)n, cudaMemcpyHostToDevice, st);
    if (e == cudaSuccess) e = launch_debug_trig(d, n, d + n, d + 2 * (size_t)n, st);
    if (e == cudaSuccess) e = cudaMemcpyAsync(acos_out, d + n, 8 * (size_t)n, cudaMemcpyDeviceToHost, st);
    if (e == cudaSuccess) e = cudaMemcpyAsync(cos_out, d + 2 * (size_t)n, 8 * (size_t)n, cudaMemcpyDeviceToHost, st);
    if (e == cudaSuccess) e = cudaStreamSynchronize(st);
    cudaFree(d);
    if (e != cudaSuccess) return fail(ctx, STL_ERR_CUDA, "debug_trig: %s", cudaGetErrorString(e));
    return STL_OK;
}

// ---- LM path -------------------------------------------------------------------

// Arguments of the calls that (re)build a problem set: P in [1, STL_MAX_PROBLEMS], a rebuild mask only for the current set
static stl_status_t check_set_args(stl_ctx *ctx, const char *call, int P, const uint8_t *rebuild) {
    if (P < 1) return fail(ctx, STL_ERR_INVALID, "%s: P = %d", call, P);
    if (P > STL_MAX_PROBLEMS) return fail(ctx, STL_ERR_CAPACITY, "%s: P = %d exceeds STL_MAX_PROBLEMS = %d", call, P, STL_MAX_PROBLEMS);
    if (rebuild && (!ctx->lm.ready || ctx->lm.P != P))
        return fail(ctx, STL_ERR_INVALID, "%s: a rebuild mask needs P equal to the size of the frozen set (%d)", call, ctx->lm.ready ? ctx->lm.P : 0);
    if (!ctx->has_pack) return fail(ctx, STL_ERR_STATE, "stl_upload_pack has not been called");
    if (ctx->params.variant != 0)
        return fail(ctx, STL_ERR_STATE, "%s follows iba_local.cpp, which has no iba_global_stable variant: create the context with variant = 0", call);
    const long long ns = std::max<long long>(ctx->pk.n_mp_total, 1);
    if ((long long)P * ((ns + 15) / 16 * 16) > INT_MAX) return fail(ctx, STL_ERR_CAPACITY, "%s: %d problems of %lld block slots", call, P, ns);
    return STL_OK;
}

// Validates the problem of every candidate (null: B == P, candidate b on problem b) and returns the host list to stage
static stl_status_t check_problems(stl_ctx *ctx, int B, const int32_t *problem, std::vector<int> &out) {
    if (!ctx->lm.ready) return fail(ctx, STL_ERR_STATE, "stl_associate_multi has not been called");
    const int P = ctx->lm.P;
    if (!problem && B != P) return fail(ctx, STL_ERR_INVALID, "problem = NULL needs B = P (B = %d, P = %d)", B, P);
    out.resize(B);
    for (int b = 0; b < B; ++b) {
        out[b] = problem ? problem[b] : b;
        if (out[b] < 0 || out[b] >= P) return fail(ctx, STL_ERR_INVALID, "problem[%d] = %d is outside [0, %d)", b, out[b], P);
    }
    return STL_OK;
}

stl_status_t stl_associate_multi(stl_ctx_t *ctx, const double *x0, int32_t P, const uint8_t *rebuild, int64_t *n_blocks) {
    if (!ctx || !x0) return STL_ERR_INVALID;
    std::lock_guard<std::mutex> lk(ctx->mu);
    stl_status_t s = check_set_args(ctx, P == 1 && !rebuild ? "stl_associate" : "stl_associate_multi", P, rebuild);
    if (s != STL_OK) return s;
    CK(cudaSetDevice(ctx->device));
    s = ensure_work(ctx, 1, false);
    if (s != STL_OK) return s;
    cudaStream_t st = acquire_stream(ctx, nullptr);
    s = enqueue_associate(ctx, x0, P, rebuild, st);
    if (s != STL_OK) return s;
    if (n_blocks) {  // BuildProblem returns the block counts: the one host round trip of the association
        const cudaError_t e = lm_block_counts(ctx->lm);
        if (e != cudaSuccess) return fail(ctx, STL_ERR_CUDA, "associate: %s", cudaGetErrorString(e));
        for (int i = 0; i < 4 * P; ++i) n_blocks[i] = ctx->lm.n_blocks[i];
    }
    return STL_OK;
}

stl_status_t stl_associate(stl_ctx_t *ctx, const double *x0, int64_t n_blocks[4]) { return stl_associate_multi(ctx, x0, 1, nullptr, n_blocks); }

static stl_status_t block_counts_locked(stl_ctx *ctx, int64_t *n_blocks, int cap_problems) {
    if (!ctx->lm.ready) return fail(ctx, STL_ERR_STATE, "stl_associate has not been called");
    if (cap_problems < ctx->lm.P) return fail(ctx, STL_ERR_CAPACITY, "%d problems, room for %d", ctx->lm.P, cap_problems);
    CK(cudaSetDevice(ctx->device));
    const cudaError_t e = lm_block_counts(ctx->lm);
    if (e != cudaSuccess) return fail(ctx, STL_ERR_CUDA, "block counts: %s", cudaGetErrorString(e));
    for (int i = 0; i < 4 * ctx->lm.P; ++i) n_blocks[i] = ctx->lm.n_blocks[i];
    return STL_OK;
}

stl_status_t stl_block_counts_multi(stl_ctx_t *ctx, int64_t *n_blocks, int32_t cap_problems) {
    if (!ctx || !n_blocks) return STL_ERR_INVALID;
    std::lock_guard<std::mutex> lk(ctx->mu);
    return block_counts_locked(ctx, n_blocks, cap_problems);
}

stl_status_t stl_block_counts(stl_ctx_t *ctx, int64_t n_blocks[4]) {
    if (!ctx || !n_blocks) return STL_ERR_INVALID;
    std::lock_guard<std::mutex> lk(ctx->mu);
    const stl_status_t s = need_single(ctx, "stl_block_counts", "stl_block_counts_multi");
    return s != STL_OK ? s : block_counts_locked(ctx, n_blocks, 1);
}

// exch_off / exch_width: the record k_lin_finish completes starts exch_off doubles from its own output row and is exch_width
// long (0: no exchange); *exchanged as in enqueue_eval
// problem (optional, host [B]): the problem of each candidate (null: problem 0)
static stl_status_t lin_enqueue(stl_ctx *ctx, const double *x, const int *problem, int B, double *d_out, cudaStream_t st, int out_stride = STL_LIN_NSUMS,
                                int exch_off = 0, int exch_width = 0, bool *exchanged = nullptr, cudaEvent_t before_finish = nullptr, bool cand_staged = false) {
    if (!ctx->lm.ready) return fail(ctx, STL_ERR_STATE, "stl_associate has not been called");
    cudaError_t e;
    const P2pView pv = exch_width > 0 ? p2p_view(ctx, B, exch_off, exch_width) : P2pView();
    if (exchanged) *exchanged = pv.n > 1;
    { StageTimer t(ctx, STL_STAGE_LINEARIZE, st); e = lm_linearize(ctx->pk, ctx->dpr, ctx->lm, x, problem, B, d_out, st, nullptr, out_stride, &pv, before_finish, cand_staged); }
    if (e != cudaSuccess) return fail(ctx, STL_ERR_CUDA, "linearize: %s", cudaGetErrorString(e));
    ctx->launches += 2 + (ctx->lm.use_gpr ? 1 : 0);  // k_linearize, (k_linearize_gpr,) k_lin_finish
    return STL_OK;
}

static stl_status_t ensure_lin(stl_ctx *ctx, int B, int width) {
    if ((long long)B * width > ctx->lin_cap) {
        dfree(ctx->d_lin);
        if (ctx->h_lin) cudaFreeHost(ctx->h_lin);
        ctx->h_lin = nullptr;
        ctx->lin_cap = 0;
        CK(cudaMalloc(&ctx->d_lin, sizeof(double) * width * B));
        CK(cudaMallocHost(&ctx->h_lin, sizeof(double) * width * B));
        ctx->lin_cap = (long long)B * width;
    }
    return STL_OK;
}

static stl_status_t step_enqueue(stl_ctx *ctx, const double *x, int B, int reassociate, double *d_out, cudaStream_t st) {
    stl_status_t s = ensure_work(ctx, B, false);
    if (s != STL_OK) return s;
    // One LM iteration at x with the plane index: BuildProblem needs K1's correspondences and (for its map-point 1-NN) K2a's
    // answer, the linearisation needs BuildProblem, and nothing of that needs K2b / K3 — so the association chain runs on a
    // second stream beside K2a / K2b / K3 (plane look-ups are bound by scattered sectors, the traversal by issue slots) and
    // the two meet again in front of the kernel that finishes the record.
    const bool overlap = reassociate && B <= ctx->wk.Bc && ctx->dpr.plane_index && !ctx->dpr.use_gpr &&
                         !getenv("STL_NO_ASSOC_REUSE") && !getenv("STL_NO_OVERLAP");
    if (overlap) {
        if (!ctx->aux_stream) {
            CK(cudaStreamCreateWithFlags(&ctx->aux_stream, cudaStreamNonBlocking));
            CK(cudaEventCreateWithFlags(&ctx->ev_k1, cudaEventDisableTiming)); CK(cudaEventCreateWithFlags(&ctx->ev_k2a, cudaEventDisableTiming));
            CK(cudaEventCreateWithFlags(&ctx->ev_k3, cudaEventDisableTiming)); CK(cudaEventCreateWithFlags(&ctx->ev_aux, cudaEventDisableTiming));
        }
        cudaStream_t ax = ctx->aux_stream;
        {   // K2a fills the association's 1-NN buffers: they must exist before it is launched
            const cudaError_t e = lm_reserve(ctx->pk, ctx->dpr, ctx->lm, 1, 1, st);
            if (e != cudaSuccess) return fail(ctx, STL_ERR_CUDA, "association buffers: %s", cudaGetErrorString(e));
        }
        s = enqueue_eval(ctx, x, B, d_out, st, false, STL_STEP_NSUMS, false, nullptr, true);
        if (s != STL_OK) return s;
        CK(cudaStreamWaitEvent(ax, ctx->ev_k1, 0));
        {   // the candidates' duals go to the device now, not between the association and the linearisation
            const cudaError_t e = lm_stage_candidates(ctx->lm, x, nullptr, B, ax);
            if (e != cudaSuccess) return fail(ctx, STL_ERR_CUDA, "candidate staging: %s", cudaGetErrorString(e));
        }
        s = enqueue_associate(ctx, x, 1, nullptr, ax, ctx->ev_k2a);
        bool done = false;
        if (s == STL_OK) s = lin_enqueue(ctx, x, nullptr, B, d_out + STL_EVAL_NSUMS, ax, STL_STEP_NSUMS, -STL_EVAL_NSUMS, STL_STEP_NSUMS, &done, ctx->ev_k3, true);
        if (s == STL_OK && lm_copy_counts(ctx->lm, ax) != cudaSuccess) s = fail(ctx, STL_ERR_CUDA, "block-count read-back");  // deferred by the association
        // whatever happened, the caller's stream is not released before the second stream has drained
        cudaEventRecord(ctx->ev_aux, ax);
        cudaStreamWaitEvent(st, ctx->ev_aux, 0);
        if (s != STL_OK) return s;
        ctx->overlapped_steps += 1;
        ctx->last_x.assign(x, x + (size_t)B * 7);
        return done ? STL_OK : allreduce_record(ctx, d_out, (size_t)B * STL_STEP_NSUMS, st);
    }
    s = enqueue_eval(ctx, x, B, d_out, st, false, STL_STEP_NSUMS);
    if (s != STL_OK) return s;
    if (reassociate) {
        s = enqueue_associate(ctx, x, 1, nullptr, st);
        if (s != STL_OK) return s;
    }
    bool done = false;
    s = lin_enqueue(ctx, x, nullptr, B, d_out + STL_EVAL_NSUMS, st, STL_STEP_NSUMS, -STL_EVAL_NSUMS, STL_STEP_NSUMS, &done);
    if (s != STL_OK) return s;
    ctx->last_x.assign(x, x + (size_t)B * 7);  // the evaluation part stays inspectable through the debug getters
    return done ? STL_OK : allreduce_record(ctx, d_out, (size_t)B * STL_STEP_NSUMS, st);
}

stl_status_t stl_step_batch_device(stl_ctx_t *ctx, const double *x, int32_t B, int32_t reassociate, double *d_out, void *stream) {
    if (!ctx || !x || !d_out || B <= 0) return STL_ERR_INVALID;
    std::lock_guard<std::mutex> lk(ctx->mu);
    if (!ctx->has_pack) return fail(ctx, STL_ERR_STATE, "stl_upload_pack has not been called");
    if (ctx->params.variant != 0) return fail(ctx, STL_ERR_STATE, "stl_step_batch needs variant = 0 (iba_local.cpp has no iba_global_stable variant)");
    if (!reassociate && !ctx->lm.ready) return fail(ctx, STL_ERR_STATE, "stl_step_batch without reassociate needs a previous association");
    if (!reassociate && need_single(ctx, "stl_step_batch", "stl_step_multi") != STL_OK) return STL_ERR_STATE;
    CK(cudaSetDevice(ctx->device));
    return step_enqueue(ctx, x, B, reassociate, d_out, acquire_stream(ctx, stream));
}

stl_status_t stl_step_batch(stl_ctx_t *ctx, const double *x, int32_t B, int32_t reassociate, stl_step_sums_t *out) {
    if (!ctx || !x || !out || B <= 0) return STL_ERR_INVALID;
    std::lock_guard<std::mutex> lk(ctx->mu);
    if (!ctx->has_pack) return fail(ctx, STL_ERR_STATE, "stl_upload_pack has not been called");
    if (ctx->params.variant != 0) return fail(ctx, STL_ERR_STATE, "stl_step_batch needs variant = 0 (iba_local.cpp has no iba_global_stable variant)");
    if (!reassociate && !ctx->lm.ready) return fail(ctx, STL_ERR_STATE, "stl_step_batch without reassociate needs a previous association");
    if (!reassociate && need_single(ctx, "stl_step_batch", "stl_step_multi") != STL_OK) return STL_ERR_STATE;
    CK(cudaSetDevice(ctx->device));
    stl_status_t s = ensure_lin(ctx, B, STL_STEP_NSUMS);
    if (s != STL_OK) return s;
    cudaStream_t st = acquire_stream(ctx, nullptr);
    s = step_enqueue(ctx, x, B, reassociate, ctx->d_lin, st);
    if (s != STL_OK) return s;
    CK(cudaMemcpyAsync(ctx->h_lin, ctx->d_lin, sizeof(double) * STL_STEP_NSUMS * B, cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    memcpy(out, ctx->h_lin, sizeof(double) * STL_STEP_NSUMS * B);
    return STL_OK;
}

stl_status_t stl_linearize_batch_device(stl_ctx_t *ctx, const double *x, int32_t B, double *d_out, void *stream) {
    if (!ctx || !x || !d_out || B <= 0) return STL_ERR_INVALID;
    std::lock_guard<std::mutex> lk(ctx->mu);
    if (need_single(ctx, "stl_linearize_batch_device", "stl_linearize_multi_device") != STL_OK) return STL_ERR_STATE;
    CK(cudaSetDevice(ctx->device));
    cudaStream_t st = acquire_stream(ctx, stream);
    bool done = false;
    stl_status_t s = lin_enqueue(ctx, x, nullptr, B, d_out, st, STL_LIN_NSUMS, 0, STL_LIN_NSUMS, &done);
    if (s != STL_OK || done) return s;
    return allreduce_record(ctx, d_out, (size_t)B * STL_LIN_NSUMS, st);
}

stl_status_t stl_linearize_batch(stl_ctx_t *ctx, const double *x, int32_t B, stl_lin_sums_t *out) {
    if (!ctx || !x || !out || B <= 0) return STL_ERR_INVALID;
    std::lock_guard<std::mutex> lk(ctx->mu);
    if (need_single(ctx, "stl_linearize_batch", "stl_linearize_multi") != STL_OK) return STL_ERR_STATE;
    CK(cudaSetDevice(ctx->device));
    stl_status_t s = ensure_lin(ctx, B, STL_LIN_NSUMS);
    if (s != STL_OK) return s;
    cudaStream_t st = acquire_stream(ctx, nullptr);
    bool done = false;
    s = lin_enqueue(ctx, x, nullptr, B, ctx->d_lin, st, STL_LIN_NSUMS, 0, STL_LIN_NSUMS, &done);
    if (s != STL_OK) return s;
    if (!done) s = allreduce_record(ctx, ctx->d_lin, (size_t)B * STL_LIN_NSUMS, st);
    if (s != STL_OK) return s;
    CK(cudaMemcpyAsync(ctx->h_lin, ctx->d_lin, sizeof(double) * STL_LIN_NSUMS * B, cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    memcpy(out, ctx->h_lin, sizeof(double) * STL_LIN_NSUMS * B);
    return STL_OK;
}

stl_status_t stl_linearize_multi_device(stl_ctx_t *ctx, const double *x, int32_t B, const int32_t *problem, double *d_out, void *stream) {
    if (!ctx || !x || !d_out || B <= 0) return STL_ERR_INVALID;
    std::lock_guard<std::mutex> lk(ctx->mu);
    std::vector<int> prob;
    stl_status_t s = check_problems(ctx, B, problem, prob);
    if (s != STL_OK) return s;
    CK(cudaSetDevice(ctx->device));
    cudaStream_t st = acquire_stream(ctx, stream);
    bool done = false;
    s = lin_enqueue(ctx, x, prob.data(), B, d_out, st, STL_LIN_NSUMS, 0, STL_LIN_NSUMS, &done);
    if (s != STL_OK || done) return s;
    return allreduce_record(ctx, d_out, (size_t)B * STL_LIN_NSUMS, st);
}

stl_status_t stl_linearize_multi(stl_ctx_t *ctx, const double *x, int32_t B, const int32_t *problem, stl_lin_sums_t *out) {
    if (!ctx || !x || !out || B <= 0) return STL_ERR_INVALID;
    std::lock_guard<std::mutex> lk(ctx->mu);
    std::vector<int> prob;
    stl_status_t s = check_problems(ctx, B, problem, prob);
    if (s != STL_OK) return s;
    CK(cudaSetDevice(ctx->device));
    s = ensure_lin(ctx, B, STL_LIN_NSUMS);
    if (s != STL_OK) return s;
    cudaStream_t st = acquire_stream(ctx, nullptr);
    bool done = false;
    s = lin_enqueue(ctx, x, prob.data(), B, ctx->d_lin, st, STL_LIN_NSUMS, 0, STL_LIN_NSUMS, &done);
    if (s != STL_OK) return s;
    if (!done) s = allreduce_record(ctx, ctx->d_lin, (size_t)B * STL_LIN_NSUMS, st);
    if (s != STL_OK) return s;
    CK(cudaMemcpyAsync(ctx->h_lin, ctx->d_lin, sizeof(double) * STL_LIN_NSUMS * B, cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    memcpy(out, ctx->h_lin, sizeof(double) * STL_LIN_NSUMS * B);
    return STL_OK;
}

// One LM iteration for each of P starts.  P = 1 is stl_step_batch(x, 1, rebuild ? rebuild[0] : 1) (overlapped); a larger set runs
// the stages one after another on the caller's stream, chunk by chunk of the workspace: evaluation of the chunk's starts, then
// BuildProblem of its flagged problems, reusing the correspondences and the 1-NN the evaluation has just left in the workspace;
// finally the linearisation of problem p at x[p] for all P.
static stl_status_t step_multi_enqueue(stl_ctx *ctx, const double *x, int P, const uint8_t *rebuild, double *d_out, cudaStream_t st) {
    if (P == 1) return step_enqueue(ctx, x, 1, rebuild ? rebuild[0] : 1, d_out, st);
    stl_status_t s = STL_OK;
    for (int c0 = 0; c0 < P && s == STL_OK; c0 += ctx->wk.Bc) {
        const int nb = std::min(ctx->wk.Bc, P - c0);
        s = enqueue_eval(ctx, x + (size_t)c0 * 7, nb, d_out + (size_t)c0 * STL_STEP_NSUMS, st, false, STL_STEP_NSUMS);
        if (s == STL_OK) s = enqueue_associate(ctx, x, P, rebuild, st, nullptr, c0, c0 + nb);
    }
    if (s != STL_OK) return s;
    std::vector<int> prob(P);
    for (int p = 0; p < P; ++p) prob[p] = p;
    bool done = false;
    s = lin_enqueue(ctx, x, prob.data(), P, d_out + STL_EVAL_NSUMS, st, STL_STEP_NSUMS, -STL_EVAL_NSUMS, STL_STEP_NSUMS, &done);
    if (s != STL_OK) return s;
    ctx->last_x.assign(x, x + (size_t)P * 7);
    return done ? STL_OK : allreduce_record(ctx, d_out, (size_t)P * STL_STEP_NSUMS, st);
}

stl_status_t stl_step_multi_device(stl_ctx_t *ctx, const double *x, int32_t P, const uint8_t *rebuild, double *d_out, void *stream) {
    if (!ctx || !x || !d_out) return STL_ERR_INVALID;
    std::lock_guard<std::mutex> lk(ctx->mu);
    stl_status_t s = check_set_args(ctx, "stl_step_multi", P, rebuild);
    if (s != STL_OK) return s;
    CK(cudaSetDevice(ctx->device));
    s = ensure_work(ctx, P, false);
    if (s != STL_OK) return s;
    return step_multi_enqueue(ctx, x, P, rebuild, d_out, acquire_stream(ctx, stream));
}

stl_status_t stl_step_multi(stl_ctx_t *ctx, const double *x, int32_t P, const uint8_t *rebuild, stl_step_sums_t *out) {
    if (!ctx || !x || !out) return STL_ERR_INVALID;
    std::lock_guard<std::mutex> lk(ctx->mu);
    stl_status_t s = check_set_args(ctx, "stl_step_multi", P, rebuild);
    if (s != STL_OK) return s;
    CK(cudaSetDevice(ctx->device));
    s = ensure_work(ctx, P, false);
    if (s == STL_OK) s = ensure_lin(ctx, P, STL_STEP_NSUMS);
    if (s != STL_OK) return s;
    cudaStream_t st = acquire_stream(ctx, nullptr);
    s = step_multi_enqueue(ctx, x, P, rebuild, ctx->d_lin, st);
    if (s != STL_OK) return s;
    CK(cudaMemcpyAsync(ctx->h_lin, ctx->d_lin, sizeof(double) * STL_STEP_NSUMS * P, cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    memcpy(out, ctx->h_lin, sizeof(double) * STL_STEP_NSUMS * P);
    return STL_OK;
}

stl_status_t stl_eval_blocks(stl_ctx_t *ctx, const double *x, int32_t rmax, int64_t cap_blocks, int32_t *type, int32_t *kf, int32_t *kp,
                             int32_t *n_res, double *residuals, double *jacobians, int64_t *n_blocks_out) {
    if (!ctx || !x || !type || !kf || !kp || !n_res || !residuals || !jacobians) return STL_ERR_INVALID;
    std::lock_guard<std::mutex> lk(ctx->mu);
    if (!ctx->lm.ready) return fail(ctx, STL_ERR_STATE, "stl_associate has not been called");
    if (need_single(ctx, "stl_eval_blocks", "stl_associate") != STL_OK) return STL_ERR_STATE;
    if (rmax < 3 || rmax < 2 * ctx->pk.n_covis) return fail(ctx, STL_ERR_INVALID, "rmax = %d is smaller than max(3, 2 * n_covis = %d)", rmax, 2 * ctx->pk.n_covis);
    CK(cudaSetDevice(ctx->device));
    CK(lm_block_counts(ctx->lm));
    const long long nb = ctx->lm.n_blocks[0] + ctx->lm.n_blocks[1] + ctx->lm.n_blocks[2] + ctx->lm.n_blocks[3];
    if (n_blocks_out) *n_blocks_out = nb;
    if (nb > cap_blocks) return fail(ctx, STL_ERR_CAPACITY, "%lld residual blocks, room for %lld", nb, (long long)cap_blocks);
    if (nb == 0) return STL_OK;
    CK(cudaSetDevice(ctx->device));
    BlockOut bo;
    bo.rmax = rmax;
    int32_t *d_i = nullptr;
    double *d_d = nullptr, *d_sums = nullptr;
    const size_t nbs = (size_t)nb;
    cudaError_t e = cudaMalloc(&d_i, 4 * 4 * nbs);
    if (e == cudaSuccess) e = cudaMalloc(&d_d, 8 * nbs * rmax * 8);
    if (e == cudaSuccess) e = cudaMalloc(&d_sums, sizeof(double) * STL_LIN_NSUMS);
    stl_status_t s = STL_OK;
    cudaStream_t st = acquire_stream(ctx, nullptr);
    // rows past n_res stay zero (g2o's zero padding, IBACalib.hpp:133-137); cleared on the stream the kernel runs on
    if (e == cudaSuccess) e = cudaMemsetAsync(d_d, 0, 8 * nbs * rmax * 8, st);
    if (e == cudaSuccess) {
        bo.type = d_i; bo.kf = d_i + nbs; bo.kp = d_i + 2 * nbs; bo.nres = d_i + 3 * nbs;
        bo.res = d_d; bo.jac = d_d + nbs * rmax;
        e = lm_linearize(ctx->pk, ctx->dpr, ctx->lm, x, nullptr, 1, d_sums, st, &bo);
        ctx->launches += 2 + (ctx->lm.use_gpr ? 1 : 0);
        if (e == cudaSuccess) e = cudaStreamSynchronize(st);
        if (e == cudaSuccess) e = cudaMemcpy(type, bo.type, 4 * nbs, cudaMemcpyDeviceToHost);
        if (e == cudaSuccess) e = cudaMemcpy(kf, bo.kf, 4 * nbs, cudaMemcpyDeviceToHost);
        if (e == cudaSuccess) e = cudaMemcpy(kp, bo.kp, 4 * nbs, cudaMemcpyDeviceToHost);
        if (e == cudaSuccess) e = cudaMemcpy(n_res, bo.nres, 4 * nbs, cudaMemcpyDeviceToHost);
        if (e == cudaSuccess) e = cudaMemcpy(residuals, bo.res, 8 * nbs * rmax, cudaMemcpyDeviceToHost);
        if (e == cudaSuccess) e = cudaMemcpy(jacobians, bo.jac, 8 * nbs * rmax * 7, cudaMemcpyDeviceToHost);
    }
    cudaFree(d_i); cudaFree(d_d); cudaFree(d_sums);
    if (e != cudaSuccess) s = fail(ctx, STL_ERR_CUDA, "eval_blocks: %s", cudaGetErrorString(e));
    return s;
}

// ---- measurement -----------------------------------------------------------------

stl_status_t stl_set_stream(stl_ctx_t *ctx, void *stream) {
    if (!ctx) return STL_ERR_INVALID;
    std::lock_guard<std::mutex> lk(ctx->mu);
    ctx->stream = stream ? (cudaStream_t)stream : ctx->own_stream;
    return STL_OK;
}

stl_status_t stl_set_profiling(stl_ctx_t *ctx, int32_t enabled) {
    if (!ctx) return STL_ERR_INVALID;
    std::lock_guard<std::mutex> lk(ctx->mu);
    ctx->profiling = enabled != 0;
    return STL_OK;
}

stl_status_t stl_stage_stats(stl_ctx_t *ctx, double ms[STL_NSTAGES], int64_t launches[STL_NSTAGES]) {
    if (!ctx) return STL_ERR_INVALID;
    std::lock_guard<std::mutex> lk(ctx->mu);
    cudaSetDevice(ctx->device);
    drain_events(ctx);
    for (int i = 0; i < STL_NSTAGES; ++i) {
        if (ms) ms[i] = ctx->stage_ms[i];
        if (launches) launches[i] = ctx->stage_n[i];
        ctx->stage_ms[i] = 0;
        ctx->stage_n[i] = 0;
    }
    return STL_OK;
}

stl_status_t stl_work_counters(stl_ctx_t *ctx, double out[8]) {
    if (!ctx || !out) return STL_ERR_INVALID;
    std::lock_guard<std::mutex> lk(ctx->mu);
    ctx->counters[5] = (double)ctx->launches;
    if (ctx->wk.overflow) {  // units whose survivor list overflowed and took the exact-over-all-points path (cumulative)
        int ov = 0;
        cudaSetDevice(ctx->device);
        if (cudaMemcpy(&ov, ctx->wk.overflow, sizeof(int), cudaMemcpyDeviceToHost) == cudaSuccess) ctx->counters[6] = (double)ov;
    }
    ctx->counters[7] = (double)ctx->assoc_reused;
    memcpy(out, ctx->counters, sizeof(ctx->counters));
    return STL_OK;
}

// ---- GPR hyper-parameters (host) -----------------------------------------------------------

stl_status_t stl_gpr_nlml(const double *x, const double *y, int32_t n, double sigma_noise, double sigma, double l, int32_t flavour,
                          double *cost, double grad[2]) {
    if (!x || !y || n <= 0 || n > 4096) return STL_ERR_INVALID;
    std::vector<double> D;
    gpr_self_pdist(x, n, D);
    return gpr_nlml(D, y, n, sigma_noise, sigma, l, flavour, cost, grad) ? STL_OK : STL_ERR_INVALID;
}

stl_status_t stl_gpr_fit(const double *x, const double *y, int32_t n, double sigma_noise, double sigma0, double l0, int32_t max_iter,
                         int32_t flavour, double out[6]) {
    if (!x || !y || !out || n <= 0 || n > 4096 || max_iter < 0) return STL_ERR_INVALID;
    const GprFitResult r = gpr_fit(x, y, n, sigma_noise, sigma0, l0, max_iter, flavour);
    out[0] = r.sigma; out[1] = r.l; out[2] = r.cost0; out[3] = r.cost; out[4] = r.iterations; out[5] = r.evaluations;
    return r.ok ? STL_OK : STL_ERR_INVALID;
}

stl_status_t stl_gpr_hyper(stl_ctx_t *ctx, double *sigma_l, int64_t cap_blocks) {
    if (!ctx || !sigma_l) return STL_ERR_INVALID;
    std::lock_guard<std::mutex> lk(ctx->mu);
    if (!ctx->lm.ready) return fail(ctx, STL_ERR_STATE, "stl_associate has not been called");
    if (need_single(ctx, "stl_gpr_hyper", "stl_associate") != STL_OK) return STL_ERR_STATE;
    CK(cudaSetDevice(ctx->device));
    CK(lm_block_counts(ctx->lm));
    if (ctx->lm.n_blocks[3] > cap_blocks) return fail(ctx, STL_ERR_CAPACITY, "%lld GPR blocks, room for %lld", ctx->lm.n_blocks[3], (long long)cap_blocks);
    CK(lm_get_gpr_hyper(ctx->dpr, ctx->lm, sigma_l, acquire_stream(ctx, nullptr)));
    return STL_OK;
}

// ---- N4: hand-eye initialisation and calibration BA on the same parameter block ---------------------

stl_status_t stl_he_linearize(stl_ctx_t *ctx, const stl_he_edges_t *edges, const double *x, int32_t B, stl_lin_sums_t *out, double *chi2) {
    if (!ctx || !edges || !x || !out || B <= 0 || edges->n < 0) return STL_ERR_INVALID;
    if (edges->n > 0 && (!edges->Ta || !edges->Tb)) return STL_ERR_INVALID;
    std::lock_guard<std::mutex> lk(ctx->mu);
    CK(cudaSetDevice(ctx->device));
    CK(he_linearize(*edges, x, B, reinterpret_cast<double *>(out), chi2, acquire_stream(ctx, nullptr)));
    ctx->launches += 2;
    return STL_OK;
}

stl_status_t stl_calib_linearize(stl_ctx_t *ctx, const stl_calib_edges_t *edges, const double *x, int32_t B, stl_lin_sums_t *out, double *chi2) {
    if (!ctx || !edges || !x || !out || B <= 0 || edges->n_kf < 0 || edges->n_edges < 0) return STL_ERR_INVALID;
    if (edges->n_edges > 0 && (!edges->edge_offset || !edges->Tlw_quat || !edges->intrinsics || !edges->Xw || !edges->obs || !edges->inv_sigma2))
        return fail(ctx, STL_ERR_INVALID, "null member of stl_calib_edges_t");
    if (edges->n_kf > 0 && (edges->edge_offset[0] != 0 || edges->edge_offset[edges->n_kf] != edges->n_edges))
        return fail(ctx, STL_ERR_INVALID, "edge_offset must run from 0 to n_edges");
    std::lock_guard<std::mutex> lk(ctx->mu);
    CK(cudaSetDevice(ctx->device));
    CK(calib_linearize(*edges, x, B, reinterpret_cast<double *>(out), chi2, acquire_stream(ctx, nullptr)));
    ctx->launches += 2;
    return STL_OK;
}

// ---- multi-GPU ---------------------------------------------------------------------

stl_status_t stl_comm_unique_id(uint8_t id[STL_COMM_ID_BYTES]) {
    if (!id) return STL_ERR_INVALID;
    static_assert(sizeof(ncclUniqueId) <= STL_COMM_ID_BYTES, "ncclUniqueId does not fit STL_COMM_ID_BYTES");
    ncclUniqueId u;
    if (ncclGetUniqueId(&u) != ncclSuccess) return STL_ERR_CUDA;
    memset(id, 0, STL_COMM_ID_BYTES);
    memcpy(id, &u, sizeof(u));
    return STL_OK;
}

stl_status_t stl_comm_init(stl_ctx_t *ctx, const uint8_t id[STL_COMM_ID_BYTES], int32_t rank, int32_t n_ranks) {
    if (!ctx || !id || n_ranks < 1 || rank < 0 || rank >= n_ranks) return STL_ERR_INVALID;
    std::lock_guard<std::mutex> lk(ctx->mu);
    if (ctx->comm) return fail(ctx, STL_ERR_STATE, "a communicator is already attached");
    CK(cudaSetDevice(ctx->device));
    ncclUniqueId u;
    memcpy(&u, id, sizeof(u));
    const ncclResult_t r = ncclCommInitRank(&ctx->comm, n_ranks, u, rank);
    if (r != ncclSuccess) { ctx->comm = nullptr; return fail(ctx, STL_ERR_CUDA, "ncclCommInitRank: %s", ncclGetErrorString(r)); }
    ctx->comm_rank = rank; ctx->comm_size = n_ranks;
    // peer-memory exchange (p2p.cuh): every rank maps every other rank's receive buffer; enabled only if ALL ranks succeed
    int ok = 0;
    if (!getenv("STL_NO_P2P") && n_ranks > 1 && n_ranks <= kP2pMaxRanks) {
        const size_t db = sizeof(double) * 2 * n_ranks * kP2pMaxB * kP2pWidth, fb = sizeof(unsigned) * 2 * n_ranks * kP2pMaxB;
        cudaIpcMemHandle_t mine[2], *all = new cudaIpcMemHandle_t[2 * n_ranks];
        char *d_send = nullptr, *d_recv = nullptr;
        cudaStream_t st = acquire_stream(ctx, nullptr);
        bool good = cudaMalloc(&ctx->p2p_data, db) == cudaSuccess && cudaMalloc(&ctx->p2p_flag, fb) == cudaSuccess &&
                    cudaMalloc(&ctx->p2p.err, sizeof(int)) == cudaSuccess && cudaMemset(ctx->p2p_data, 0, db) == cudaSuccess &&
                    cudaMemset(ctx->p2p_flag, 0, fb) == cudaSuccess && cudaMemset(ctx->p2p.err, 0, sizeof(int)) == cudaSuccess &&
                    cudaIpcGetMemHandle(&mine[0], ctx->p2p_data) == cudaSuccess && cudaIpcGetMemHandle(&mine[1], ctx->p2p_flag) == cudaSuccess &&
                    cudaMalloc(&d_send, sizeof(mine)) == cudaSuccess && cudaMalloc(&d_recv, sizeof(mine) * n_ranks) == cudaSuccess &&
                    cudaMemcpy(d_send, mine, sizeof(mine), cudaMemcpyHostToDevice) == cudaSuccess;
        // the handles travel through the communicator itself; the collective is issued even on a rank whose setup failed
        if (!good) { cudaGetLastError(); if (!d_send) cudaMalloc(&d_send, sizeof(mine)); if (!d_recv) cudaMalloc(&d_recv, sizeof(mine) * n_ranks); }
        if (d_send && d_recv && ncclAllGather(d_send, d_recv, sizeof(mine), ncclChar, ctx->comm, st) == ncclSuccess && cudaStreamSynchronize(st) == cudaSuccess &&
            cudaMemcpy(all, d_recv, sizeof(mine) * n_ranks, cudaMemcpyDeviceToHost) == cudaSuccess && good) {
            ok = 1;
            for (int q = 0; q < n_ranks && ok; ++q) {
                if (q == rank) { ctx->p2p.data[q] = ctx->p2p_data; ctx->p2p.flag[q] = ctx->p2p_flag; continue; }
                void *pd = nullptr, *pf = nullptr;
                if (cudaIpcOpenMemHandle(&pd, all[2 * q], cudaIpcMemLazyEnablePeerAccess) != cudaSuccess ||
                    cudaIpcOpenMemHandle(&pf, all[2 * q + 1], cudaIpcMemLazyEnablePeerAccess) != cudaSuccess) { ok = 0; cudaGetLastError(); break; }
                ctx->p2p.data[q] = (double *)pd; ctx->p2p.flag[q] = (unsigned *)pf;
            }
        }
        // agreement: one rank without the mapping and all fall back to NCCL
        int *d_ok = nullptr;
        if (cudaMalloc(&d_ok, sizeof(int)) == cudaSuccess && cudaMemcpy(d_ok, &ok, sizeof(int), cudaMemcpyHostToDevice) == cudaSuccess &&
            ncclAllReduce(d_ok, d_ok, 1, ncclInt, ncclMin, ctx->comm, st) == ncclSuccess && cudaStreamSynchronize(st) == cudaSuccess)
            cudaMemcpy(&ok, d_ok, sizeof(int), cudaMemcpyDeviceToHost);
        else ok = 0;
        cudaFree(d_ok); cudaFree(d_send); cudaFree(d_recv);
        delete[] all;
        ctx->p2p.n = n_ranks; ctx->p2p.rank = rank;
        ctx->p2p_on = ok == 1;
    }
    return STL_OK;
}

stl_status_t stl_comm_stats(stl_ctx_t *ctx, int64_t out[3]) {
    if (!ctx || !out) return STL_ERR_INVALID;
    std::lock_guard<std::mutex> lk(ctx->mu);
    out[0] = ctx->p2p_on ? 1 : 0; out[1] = ctx->p2p_exchanges; out[2] = ctx->nccl_exchanges;
    return STL_OK;
}

stl_status_t stl_comm_info(stl_ctx_t *ctx, int32_t *rank, int32_t *n_ranks) {
    if (!ctx) return STL_ERR_INVALID;
    std::lock_guard<std::mutex> lk(ctx->mu);
    if (rank) *rank = ctx->comm ? ctx->comm_rank : 0;
    if (n_ranks) *n_ranks = ctx->comm ? ctx->comm_size : 1;
    return STL_OK;
}

}  // extern "C"
