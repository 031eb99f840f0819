// reduce.cu — K3: per-candidate reduction of the per-keyframe partial records into the
// accumulators of BAError (src/examples/iba_global.cpp:175-186,239-251,318-326).
// fp64, fixed order (strided partials per thread, then a fixed shuffle tree): the
// result is bit-reproducible run to run.  One CTA per candidate.
#include "../../include/stlcalib.h"
#include "kernels.h"
#include "p2p.cuh"

namespace stl {
namespace {

constexpr int kT = 256;

__global__ void __launch_bounds__(kT) k_reduce(const DevPack pk, const DevWork wk, const DevParams pr, double *__restrict__ out, const int out_stride, const P2pView P) {
    const int b = blockIdx.x;
    const int F = pk.n_kf, sub = wk.sub;
    double v[STL_EVAL_NSUMS];
#pragma unroll
    for (int i = 0; i < STL_EVAL_NSUMS; ++i) v[i] = 0;
    // selection positions: the partial sums have the order of a pack holding only the selected keyframes
    for (int i = threadIdx.x; i < pk.n_sel; i += kT) {
        const int f = sel_kf(pk, i);
        const FrameRec r = wk.frame[(long long)b * F + f];
        v[0] += r.s2d; v[2] += r.she; v[3] += r.che; v[4] += r.c2d; v[5] += r.v2d; v[10] += r.kept; v[11] += r.ncorr;
        if (pr.w1 <= 1e-10) {  // iba_global.cpp:214-219: no 3-D term, one "valid" count per kept frame
            v[6] += r.kept; v[7] += r.kept;
        } else {
            for (int j = 0; j < sub; ++j) {
                const AlignRec a = wk.align[((long long)b * F + f) * sub + j];
                v[1] += a.s3d; v[6] += a.c3d; v[7] += a.v3d; v[8] += a.vpl; v[9] += a.vpt;
            }
        }
    }
    __shared__ double red[STL_EVAL_NSUMS][kT / 32];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
    for (int i = 0; i < STL_EVAL_NSUMS; ++i) {
        double x = v[i];
        for (int o = 16; o; o >>= 1) x += __shfl_down_sync(0xffffffffu, x, o);
        if (lane == 0) red[i][warp] = x;
    }
    __syncthreads();
    if (threadIdx.x < STL_EVAL_NSUMS) {
        double x = 0;
        for (int w = 0; w < kT / 32; ++w) x += red[threadIdx.x][w];
        out[(long long)b * out_stride + threadIdx.x] = x;
    }
    if (P.n > 1) p2p_allreduce_record(P, b, out + (long long)b * out_stride + P.off);  // keyframes sharded over GPUs: sum the shards here
}

// stl_eval_frames: one thread per selected (keyframe, candidate) folds FrameRec + AlignRec[sub] into the 13 values of
// stl_debug_frame, in its order; with err_weight[1] <= 1e-10 the 3-D columns take k_reduce's "one valid count per kept frame"
// instead, so that the rows of a candidate sum to its record.  out: [B][n_kf][13]; rows of unselected keyframes are not written.
__global__ void __launch_bounds__(kT) k_frames(const DevPack pk, const DevWork wk, const DevParams pr, const int B, double *__restrict__ out) {
    const long long t = (long long)blockIdx.x * kT + threadIdx.x;
    if (t >= (long long)pk.n_sel * B) return;
    const int i = (int)(t / B), b = (int)(t - (long long)i * B);
    const long long rec = (long long)b * pk.n_kf + sel_kf(pk, i);
    const FrameRec r = wk.frame[rec];
    double *o = out + rec * 13;
    o[0] = r.s2d; o[1] = r.v2d; o[2] = r.c2d; o[3] = r.she; o[4] = r.che; o[5] = r.kept; o[6] = r.ncorr; o[7] = r.nq;
    double s3d = 0, v3d = 0, c3d = 0, vpl = 0, vpt = 0;
    if (pr.w1 <= 1e-10) {
        v3d = r.kept; c3d = r.kept;
    } else {
        for (int j = 0; j < wk.sub; ++j) {
            const AlignRec a = wk.align[rec * wk.sub + j];
            s3d += a.s3d; v3d += a.v3d; c3d += a.c3d; vpl += a.vpl; vpt += a.vpt;
        }
    }
    o[8] = s3d; o[9] = v3d; o[10] = c3d; o[11] = vpl; o[12] = vpt;
}

}  // namespace

cudaError_t launch_reduce(const DevPack &pk, const DevWork &wk, const DevParams &pr, int B, double *d_out, cudaStream_t st, int out_stride,
                          const P2pView *p2p) {
    if (B <= 0) return cudaSuccess;
    k_reduce<<<B, kT, 0, st>>>(pk, wk, pr, d_out, out_stride > 0 ? out_stride : STL_EVAL_NSUMS, p2p ? *p2p : P2pView());
    return cudaGetLastError();
}

cudaError_t launch_frames(const DevPack &pk, const DevWork &wk, const DevParams &pr, int B, double *d_out, cudaStream_t st) {
    const long long n = (long long)pk.n_sel * B;
    if (n <= 0) return cudaSuccess;
    k_frames<<<(unsigned)((n + kT - 1) / kT), kT, 0, st>>>(pk, wk, pr, B, d_out);
    return cudaGetLastError();
}

}  // namespace stl
