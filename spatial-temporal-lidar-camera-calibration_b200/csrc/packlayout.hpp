// packlayout.hpp — the host decisions of a pack upload, without a device: validation of stl_pack_t, the per-keyframe
// layout (DevKf), the K1 routing between the one-kernel and the banded K1, the candidate-independent K1 tables, and the
// routing of a keyframe list.  No kernel and no CUDA runtime call; compiled by nvcc only because common.cuh defines
// device helpers beside its layout structs.
#pragma once
#include <cstddef>
#include <cstdint>
#include <string>
#include <vector>

#include "../../include/stlcalib.h"
#include "kernels.h"

namespace stl {

// What the K1 routing is given: the device's opt-in shared memory per block, the shared memory the one-kernel K1
// (assoc2d_smem_bytes) and the banded K1's stream kernel (assoc2d_split_smem_bytes) need, and the two switches
struct K1Limits {
    int smem_optin = 0;
    size_t (*k1_smem)(int max_kp, int max_tab_bytes, int max_groups) = nullptr;
    size_t (*split_smem)(int max_band_words, int max_groups) = nullptr;
    bool allow_oversize = false;  // stl_allow_oversize_keyframes
    bool route_all = false;       // every keyframe on the banded K1 (STL_K1_OVERSIZE=all / STL_K1_SPLIT=1)
};

struct PackLayout {
    int n_kf = 0, n_covis = 0;
    std::vector<DevKf> kf;  // [n_kf]; pmax is filled by the index build
    long long n_pad_total = 0, n_nodes_total = 0, n_kp_total = 0, n_mp_total = 0;
    long long bm_words = 0, grid_cells = 0, tab_bytes = 0;  // sizes of the bitmap, grid_start and k1tab arrays
    // K1 routing (DESIGN §3 "Oversize keyframes"): keyframes leave the one-kernel K1's set largest-first (by their own
    // shared memory, ties: lower index first) until the maxima of the rest fit the opt-in limit
    int n_fit = 0;                        // keyframes of the one-kernel K1
    int max_kp = 0, max_tab = 0, max_groups = 0;  // their maxima
    size_t k1_smem = 0;                   // the one-kernel K1's shared memory (0: no fitting keyframe)
    std::vector<OvKf> ov;                 // the oversize keyframes, increasing, with their workspace slices
    std::vector<int> ov_ord;              // [n_kf] oversize ordinal of each keyframe (-1: fitting)
    long long n_ov_kp = 0, n_ov_surv = 0, n_ov_match = 0;
    int ov_max_bands = 0, ov_max_surv = 0;
    size_t k1_split_smem = 0;             // the banded K1's stream kernel shared memory (0: no oversize keyframe)
};

// Validates the pack and lays it out.  On failure returns the status and sets err; `out` is then unspecified.
stl_status_t layout_pack(const stl_pack_t *p, const K1Limits &lim, PackLayout &out, std::string &err);

// The candidate-independent K1 tables of a laid-out pack (common.cuh, DevPack)
struct PackTables {
    // variant 1 (iba_global_stable.cpp:67-80): the query pixel of a keypoint is its map point re-projected with the SLAM
    // pose, in fp64 (NaN: no map point, not queried); the float32 copy drives the coarse tables
    std::vector<double> kp_xyd;
    std::vector<float> kp_xyf;
    const float *kp_xy = nullptr;  // the query pixels of the coarse tables: the pack's kp_xy, or kp_xyf under variant 1
    std::vector<uint32_t> bitmap, grid_start, grid_kp;
    std::vector<uint8_t> k1tab;
};
void build_tables(const stl_pack_t *p, const PackLayout &L, int variant, double max_pixel_dist, PackTables &t);

// What a launch over one keyframe list needs: every keyframe (kf == nullptr) or a strictly increasing selection
struct KfRoute {
    bool all = true;            // every keyframe: the kernels read no selection list
    int n_sel = 0;
    std::vector<int> sel;       // [n_sel] (a selection only)
    std::vector<int2> sel_mp;   // [n_sel + 1] (first compacted map-point slot of position i, mp_off - that) (a selection only)
    long long n_sel_mp = 0;
    // [2][n_kf]: the selected fitting keyframes, then the ordinals of the selected oversize ones (the K1 launches read them
    // only when the pack has oversize keyframes)
    std::vector<int> lists;
    int n_fit = 0, n_ov = 0;
    std::vector<uint8_t> mask;  // [n_kf] 1 = selected
    long long pts = 0, kp = 0;  // scan points / keypoints of the selected keyframes
};
KfRoute route_keyframes(const PackLayout &L, const int *kf, int n);

}  // namespace stl
