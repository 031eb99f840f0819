// stlcalib_host.hpp — C++ host adapters above the C-ABI (header-only, no third-party headers).
//
// Mirrors, name for name, the call shapes the reference's optimisers use, so that a reference
// maintainer replaces the body of the function and nothing above it:
//
//   stl::BAError(xvec, ctx)        <- BAError(xvec, PointClouds, KdTrees, vTwl, KFIdMap, KeyFrames,
//                                     iba_params, multiprocessing, verborse)
//                                     src/examples/iba_global.cpp:169-173, iba_func.cpp:179-183
//                                     returns {f1, f2, C, valid_cnt_3d_2d, cnt_3d_2d}; DBL_MAX sentinels
//   stl::BALoss::eval_x            <- BALoss::eval_x(NOMAD::EvalPoint&, const NOMAD::Double&, bool&)
//                                     src/examples/iba_global.cpp:377-396  (BBO "f C1 C2 C3")
//   stl::BALoss::eval_block        <- Nomad 4 Evaluator::eval_block (a whole poll batch per device call)
//   stl::LMProblem                 <- BuildProblem + ceres::Problem::Evaluate / g2o linearizeOplus
//                                     src/examples/iba_local.cpp:145-323,434-446; include/IBACalib.hpp:74-155
//
// Error behaviour: the reference signals nothing but the values (infeasible points go through the
// PB constraints); here a failed device call throws std::runtime_error with stl_last_error().
#pragma once
#include <array>
#include <cstdio>
#include <stdexcept>
#include <string>
#include <tuple>
#include <vector>

#include "stlcalib.h"

namespace stl {

class Context {
  public:
    explicit Context(const stl_params_t &params, int device = 0) : params_(params) {
        const stl_status_t s = stl_create(&params_, device, &ctx_);
        if (s != STL_OK) throw std::runtime_error("stl_create failed (status " + std::to_string((int)s) + "): an sm_100 GPU is required");
    }
    Context(const Context &) = delete;
    Context &operator=(const Context &) = delete;
    ~Context() { stl_destroy(ctx_); }

    // BALoss constructor state: scans, keyframes, per-scan index (iba_global.cpp:349-367)
    void upload(const stl_pack_t &pack) { check(stl_upload_pack(ctx_, &pack), "stl_upload_pack"); }

    std::vector<stl_eval_sums_t> eval_sums(const double *x, int B) {
        std::vector<stl_eval_sums_t> out((size_t)B);
        check(stl_eval_batch(ctx_, x, B, out.data()), "stl_eval_batch");
        return out;
    }
    std::array<int64_t, 4> associate(const double *x0) {
        std::array<int64_t, 4> n{};
        check(stl_associate(ctx_, x0, n.data()), "stl_associate");
        return n;
    }
    // per-block residuals / Jacobians of the frozen problem (stl_eval_blocks); n = blocks from associate()
    struct Blocks {
        int rmax = 0;
        std::vector<int32_t> type, kf, kp, n_res;
        std::vector<double> residuals, jacobians;  // [n][rmax], [n][rmax][7]
        size_t size() const { return type.size(); }
    };
    Blocks eval_blocks(const double *x, int64_t n, int rmax) {
        Blocks b;
        b.rmax = rmax;
        const size_t cap = (size_t)(n > 0 ? n : 1);
        b.type.resize(cap); b.kf.resize(cap); b.kp.resize(cap); b.n_res.resize(cap);
        b.residuals.resize(cap * rmax); b.jacobians.resize(cap * rmax * 7);
        int64_t got = 0;
        check(stl_eval_blocks(ctx_, x, rmax, (int64_t)cap, b.type.data(), b.kf.data(), b.kp.data(), b.n_res.data(), b.residuals.data(),
                              b.jacobians.data(), &got),
              "stl_eval_blocks");
        b.type.resize((size_t)got); b.kf.resize((size_t)got); b.kp.resize((size_t)got); b.n_res.resize((size_t)got);
        b.residuals.resize((size_t)got * rmax); b.jacobians.resize((size_t)got * rmax * 7);
        return b;
    }
    std::vector<stl_lin_sums_t> linearize(const double *x, int B) {
        std::vector<stl_lin_sums_t> out((size_t)B);
        check(stl_linearize_batch(ctx_, x, B, out.data()), "stl_linearize_batch");
        return out;
    }
    // BAError sums + (BuildProblem at x[0]) + linearisation in one device round (one LM iteration, or a NOMAD poll on the
    // frozen association): [B] records of {eval sums, linearisation}
    std::vector<stl_step_sums_t> step(const double *x, int B, bool reassociate) {
        std::vector<stl_step_sums_t> out((size_t)B);
        check(stl_step_batch(ctx_, x, B, reassociate ? 1 : 0, out.data()), "stl_step_batch");
        return out;
    }
    // several starts on one context (a problem set): BuildProblem at x0[p] for p < P ([P][7]); rebuild (optional [P]) re-associates
    // only the flagged problems of the current set of P.  Block counts [P][4].
    std::vector<std::array<int64_t, 4>> associate_multi(const double *x0, int P, const uint8_t *rebuild = nullptr) {
        std::vector<std::array<int64_t, 4>> n((size_t)P);
        check(stl_associate_multi(ctx_, x0, P, rebuild, n[0].data()), "stl_associate_multi");
        return n;
    }
    // candidate b (x [B][7]) on problem problem[b] (null: B == P, candidate b on problem b)
    std::vector<stl_lin_sums_t> linearize_multi(const double *x, int B, const int32_t *problem = nullptr) {
        std::vector<stl_lin_sums_t> out((size_t)B);
        check(stl_linearize_multi(ctx_, x, B, problem, out.data()), "stl_linearize_multi");
        return out;
    }
    // normal equations per keyframe: [B][n_kf] rows (n_kf = the pack's), row f of candidate b = keyframe f's blocks alone on
    // problem problem[b] (null: every candidate on problem 0, a set of one); zero rows for unselected keyframes
    std::vector<stl_lin_sums_t> linearize_frames(const double *x, int B, int n_kf, const int32_t *problem = nullptr) {
        std::vector<stl_lin_sums_t> out((size_t)B * (size_t)n_kf);
        check(stl_linearize_frames(ctx_, x, B, problem, out.data()), "stl_linearize_frames");
        return out;
    }
    // one LM iteration of P starts: {eval sums, linearisation} of problem p at x[p], BuildProblem of the flagged problems first
    std::vector<stl_step_sums_t> step_multi(const double *x, int P, const uint8_t *rebuild = nullptr) {
        std::vector<stl_step_sums_t> out((size_t)P);
        check(stl_step_multi(ctx_, x, P, rebuild, out.data()), "stl_step_multi");
        return out;
    }
    // keyframe selection on the resident pack (stl_select_keyframes): every later call walks only the local keyframes kf (strictly
    // increasing; an empty list selects none) as a pack of only those would; select_all() restores the whole pack.  Both drop
    // the frozen problem set (associate again before linearising).
    // (an empty vector may have a null data(), which the C-ABI reads as "all keyframes": it is passed a non-null pointer instead)
    void select_keyframes(const std::vector<int32_t> &kf) {
        static const int32_t none = 0;
        check(stl_select_keyframes(ctx_, kf.empty() ? &none : kf.data(), (int32_t)kf.size()), "stl_select_keyframes");
    }
    void select_all() { check(stl_select_keyframes(ctx_, nullptr, 0), "stl_select_keyframes"); }
    // oversize keyframes (stl_allow_oversize_keyframes): read by the next upload; the resident pack is not touched
    void allow_oversize_keyframes(bool allow) { check(stl_allow_oversize_keyframes(ctx_, allow ? 1 : 0), "stl_allow_oversize_keyframes"); }
    // local keyframes of the resident pack on the oversize path, increasing
    std::vector<int32_t> oversize_keyframes() {
        int32_t n = 0;
        check(stl_oversize_keyframes(ctx_, nullptr, 0, &n), "stl_oversize_keyframes");
        std::vector<int32_t> kf((size_t)n);
        if (n > 0) check(stl_oversize_keyframes(ctx_, kf.data(), n, &n), "stl_oversize_keyframes");
        return kf;
    }
    // BAError per keyframe: [B][n_kf][13] records of stl_debug_frame's layout (zero rows for unselected keyframes); n_kf = the pack's
    std::vector<double> eval_frames(const double *x, int B, int n_kf) {
        std::vector<double> out((size_t)B * (size_t)n_kf * 13);
        check(stl_eval_frames(ctx_, x, B, out.data()), "stl_eval_frames");
        return out;
    }
    // keyframes sharded over several GPUs: this context holds shard `rank` of `n_ranks`; `id` comes from
    // stl_comm_unique_id on one rank (handed over by the host program).  Afterwards every call returns the totals.
    void comm_init(const uint8_t id[STL_COMM_ID_BYTES], int rank, int n_ranks) { check(stl_comm_init(ctx_, id, rank, n_ranks), "stl_comm_init"); }
    const stl_params_t &params() const { return params_; }
    stl_ctx_t *raw() { return ctx_; }

  private:
    void check(stl_status_t s, const char *what) {
        if (s != STL_OK) throw std::runtime_error(std::string(what) + ": " + stl_last_error(ctx_));
    }
    stl_params_t params_;
    stl_ctx_t *ctx_ = nullptr;
};

// f1, f2, C, valid_cnt_3d_2d, cnt_3d_2d — BAError's return tuple (iba_global.cpp:343)
inline std::tuple<double, double, double, int, int> BAError(const double *xvec, Context &ctx, bool verborse = false) {
    const stl_eval_sums_t s = ctx.eval_sums(xvec, 1)[0];
    stl_ba_error_t e;
    stl_finalize(&ctx.params(), &s, &e);
    if (verborse) std::printf("plane: %d, point: %d 3d-2d: %d\n", (int)s.valid_pl, (int)s.valid_pt, (int)s.valid_3d2d);  // iba_global.cpp:341-342
    return {e.f1, e.f2, e.C, e.valid_cnt_3d_2d, e.cnt_3d_2d};
}

// Shaped like `class BALoss : public NOMAD::Evaluator` (iba_global.cpp:346-405) without the Nomad
// base class (Nomad is not vendored); see INTEGRATION.md for the three-line derived class.
class BALoss {
  public:
    explicit BALoss(Context &ctx) : ctx_(ctx) {}
    // x[7] in, bbo[4] = {f, C1, C2, C3} out; countEval = true; returns true (iba_global.cpp:377-396)
    bool eval_x(const double x[7], double bbo[4], bool &countEval) const {
        const stl_eval_sums_t s = ctx_.eval_sums(x, 1)[0];
        stl_ba_error_t e;
        stl_finalize(&ctx_.params(), &s, &e);
        stl_bbo(&ctx_.params(), &e, bbo);
        countEval = true;
        return true;
    }
    // the string handed to EvalPoint::setBBO (iba_global.cpp:389-393)
    static std::string bbo_string(const double bbo[4]) {
        char buf[160];
        std::snprintf(buf, sizeof(buf), "%.17g %.17g %.17g %.17g", bbo[0], bbo[1], bbo[2], bbo[3]);
        return buf;
    }
    // a block of poll candidates in one device call; out[b] = {f, C1, C2, C3}
    void eval_block(const double *x, int B, double *bbo, std::vector<bool> &countEval) const {
        const std::vector<stl_eval_sums_t> s = ctx_.eval_sums(x, B);
        countEval.assign((size_t)B, true);
        for (int b = 0; b < B; ++b) {
            stl_ba_error_t e;
            stl_finalize(&ctx_.params(), &s[(size_t)b], &e);
            stl_bbo(&ctx_.params(), &e, bbo + 4 * b);
        }
    }

  private:
    Context &ctx_;
};

// One 7-double parameter block; build() = BuildProblem (iba_local.cpp:443), evaluate() = the cost,
// gradient and Gauss-Newton matrix Ceres/g2o assemble from the residual blocks (Huber applied).
class LMProblem {
  public:
    explicit LMProblem(Context &ctx) : ctx_(ctx) {}
    std::array<int64_t, 4> build(const double x0[7]) { return n_ = ctx_.associate(x0); }
    stl_lin_sums_t evaluate(const double x[7]) { return ctx_.linearize(x, 1)[0]; }
    // block by block (raw residuals + Jacobian rows): what each CostFunction::Evaluate / g2o edge returns
    Context::Blocks blocks(const double x[7], int rmax) { return ctx_.eval_blocks(x, n_[0] + n_[1] + n_[2] + n_[3], rmax); }

  private:
    Context &ctx_;
    std::array<int64_t, 4> n_{};
};

// P LMProblems on one context (multi-start refinement): problem p is frozen at its own start.
class LMProblemSet {
  public:
    explicit LMProblemSet(Context &ctx) : ctx_(ctx) {}
    // X0 [P][7]; rebuild (optional [P]): re-associate only the flagged problems of the current set
    std::vector<std::array<int64_t, 4>> build(const double *X0, int P, const uint8_t *rebuild = nullptr) {
        return n_ = ctx_.associate_multi(X0, P, rebuild);
    }
    // candidate b (X [B][7]) on problem problem[b] (null: B == P, candidate p on problem p)
    std::vector<stl_lin_sums_t> evaluate(const double *X, int B, const int32_t *problem = nullptr) { return ctx_.linearize_multi(X, B, problem); }
    int size() const { return (int)n_.size(); }

  private:
    Context &ctx_;
    std::vector<std::array<int64_t, 4>> n_;
};

}  // namespace stl
