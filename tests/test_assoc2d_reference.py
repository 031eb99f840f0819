"""The oracle's 2-D association (FindProjectCorrespondences, iba_global.cpp:55-96) against a plain numpy brute force, at the
camera shapes the GPU tests use beyond KITTI-00: fx != fy, other image sizes, and keypoints on the 8 px grid cells, the 2 px
bitmap cells, the image border and just outside it.  The GPU parity tests rest on the oracle, so the oracle is checked first.

The brute force is the reference's rule written out: project every scan point with fx for BOTH pixel rows
(u = (fx x + cx z) / z, v = (fx y + cy z) / z), keep z > 0, 0 <= u < W, 0 <= v < H, and give each keypoint the projected point
nearest by (squared distance, original index) if that distance is within max_pixel_dist."""
import numpy as np
import pytest

SIZES = [(1241, 376), (1226, 370), (1242, 375), (1210, 376), (1212, 376), (640, 480), (376, 1241), (1920, 1080)]


def camera_for(W, H):
    """Intrinsics that fit a W x H image: KITTI-00's focal length scaled to the longer side, principal point near the centre
    (KITTI-00's own values at 1241 x 376)."""
    if (W, H) == (1241, 376):
        return 718.856, 718.856, 607.1928, 185.2157
    f = float(np.float32(718.856 * max(W, H) / 1241))
    return f, f, float(np.float32(W / 2 - 0.35)), float(np.float32(H / 2 + 0.15))


def border_keypoints(pack, x, kf, seed=0):
    """Overwrites keypoints of keyframe `kf` (in place) with pixels on the edges the GPU tables are built on: exactly on 8 px
    grid-cell and 2 px bitmap-cell boundaries next to a projected point, on the image border (0, W - 1e-3) and just outside it
    (-0.5, W + 0.5), in both axes.  The projection is the reference's (fx for both rows) at extrinsic x."""
    rng = np.random.default_rng(seed)
    W, H = (int(v) for v in pack.image_wh[kf])
    u, v, _ = project(pack, x, kf)
    ok = (u >= 0) & (u < W) & (v >= 0) & (v < H)
    u, v = u[ok], v[ok]
    k0, k1 = int(pack.kp_offset[kf]), int(pack.kp_offset[kf + 1])
    xy = []
    for cell in (8.0, 2.0):                                    # grid and bitmap cell boundaries, each axis
        for _ in range(12):
            i = rng.integers(len(u))
            xy.append((np.round(u[i] / cell) * cell, v[i]))
            xy.append((u[i], np.round(v[i] / cell) * cell))
    near_l, near_r = np.argsort(u)[:12], np.argsort(-u)[:12]   # points closest to the left and right borders
    near_t, near_b = np.argsort(v)[:12], np.argsort(-v)[:12]
    for i in near_l:
        xy += [(0.0, v[i]), (-0.5, v[i])]
    for i in near_r:
        xy += [(W - 1e-3, v[i]), (W + 0.5, v[i])]
    for i in near_t:
        xy += [(u[i], 0.0), (u[i], -0.5)]
    for i in near_b:
        xy += [(u[i], H - 1e-3), (u[i], H + 0.5)]
    xy += [(0.0, 0.0), (-0.5, -0.5), (W - 1e-3, H - 1e-3), (W + 0.5, H + 0.5)]
    xy = np.asarray(xy, np.float32)
    n = min(len(xy), k1 - k0)
    pack.kp_xy[k0:k0 + n] = xy[:n]
    return n


def project(pack, x, kf):
    """(u, v, original index) of every scan point of keyframe kf with z > 0, in fp64 and the oracle's operation order
    (pointcloud.h:82-86, iba_global.cpp:71-74)."""
    from oracle import oracle as O
    R, t, _ = O.sim3exp(np.asarray(x, np.float64))
    s0, s1 = int(pack.scan_offset[kf]), int(pack.scan_offset[kf + 1])
    P = pack.scan_xyz[s0:s1].astype(np.float64)
    q = [t[i] + ((R[i, 0] * P[:, 0] + R[i, 1] * P[:, 1]) + R[i, 2] * P[:, 2]) for i in range(3)]
    fx, _, cx, cy = (float(v) for v in pack.intrinsics[kf])
    z = q[2]
    keep = z > 0
    idx = np.flatnonzero(keep)
    z = z[keep]
    u = (fx * q[0][keep] + cx * z) / z
    v = (fx * q[1][keep] + cy * z) / z                          # fx, not fy: the reference's quirk
    return u, v, idx


def brute_corrset(pack, x, kf, max_pixel_dist):
    W, H = (float(v) for v in pack.image_wh[kf])
    u, v, idx = project(pack, x, kf)
    ok = (u >= 0) & (u < W) & (v >= 0) & (v < H)
    u, v, idx = u[ok], v[ok], idx[ok]
    k0, k1 = int(pack.kp_offset[kf]), int(pack.kp_offset[kf + 1])
    kp = pack.kp_xy[k0:k1].astype(np.float64)
    out_kp, out_pt = [], []
    if len(idx) == 0:
        return np.zeros(0, np.uint32), np.zeros(0, np.uint32)
    for k in range(k1 - k0):
        du, dv = u - kp[k, 0], v - kp[k, 1]
        d2 = du * du + dv * dv
        j = int(np.argmin(d2))                                 # first minimum = lowest original index among exact ties
        if d2[j] <= max_pixel_dist * max_pixel_dist:
            out_kp.append(k); out_pt.append(idx[j])
    return np.asarray(out_kp, np.uint32), np.asarray(out_pt, np.uint32)


def _small(synth, W=1241, H=376, fx=None, fy=None, cx=None, cy=None, seed=3, n_kp=400):
    cfx, cfy, ccx, ccy = camera_for(W, H)
    pack, x_gt, _ = synth.generate(n_kf=2, beams=32, az_steps=700, n_kp=n_kp, width=W, height=H,
                                   fx=fx or cfx, fy=fy or cfy, cx=cx if cx is not None else ccx, cy=cy if cy is not None else ccy, seed=seed)
    return pack, x_gt


def _compare(oracle_mod, pkg, pack, X, min_corr=30):
    p = pkg.default_params()
    orc = oracle_mod.Oracle(pack, params=p, kind="port")
    total = 0
    for x in X:
        for kf in range(pack.n_kf):
            d = orc.frame_debug(x, kf)
            kp, pt = brute_corrset(pack, x, kf, p.max_pixel_dist)
            assert np.array_equal(d["corr_kp"], kp) and np.array_equal(d["corr_pt"], pt), (kf, len(kp), len(d["corr_kp"]))
            total += len(kp)
    assert total >= min_corr
    orc.close()
    return total


@pytest.mark.parametrize("fy_scale", [0.97, 1.03])
def test_fx_ne_fy_uses_fx_for_both_rows(oracle_mod, pkg, synth, fy_scale):
    pack, x_gt = _small(synth)
    X = synth.candidates(x_gt, 2, 0.3, seed=5)
    base = _compare(oracle_mod, pkg, pack, X)
    pack.intrinsics = pack.intrinsics.copy()
    pack.intrinsics[:, 1] = np.float32(pack.intrinsics[:, 0] * fy_scale)
    assert _compare(oracle_mod, pkg, pack, X) == base          # fy plays no part in the association


@pytest.mark.parametrize("W,H", SIZES, ids=[f"{w}x{h}" for w, h in SIZES])
def test_image_sizes(oracle_mod, pkg, synth, W, H):
    pack, x_gt = _small(synth, W, H)
    assert (pack.image_wh == [W, H]).all()
    _compare(oracle_mod, pkg, pack, synth.candidates(x_gt, 2, 0.3, seed=6))


def test_principal_point_off_centre(oracle_mod, pkg, synth):
    pack, x_gt = _small(synth, cx=607.1928 + 37.5, cy=185.2157 - 21.25)
    _compare(oracle_mod, pkg, pack, synth.candidates(x_gt, 2, 0.3, seed=7))


@pytest.mark.parametrize("W,H", [(1241, 376), (1210, 376), (376, 1241)], ids=["1241x376", "1210x376", "376x1241"])
def test_keypoints_on_cell_edges_and_image_border(oracle_mod, pkg, synth, W, H):
    """Keypoints exactly on 8 px / 2 px boundaries, on the border and half a pixel outside it.  The ones outside the image still
    match points inside it (the reference bounds the projected points, not the keypoints)."""
    pack, x_gt = _small(synth, W, H)
    X = synth.candidates(x_gt, 2, 0.3, seed=8)
    for kf in range(pack.n_kf):
        border_keypoints(pack, X[0], kf, seed=kf)
    _compare(oracle_mod, pkg, pack, X)
    kp, _ = brute_corrset(pack, X[0], 0, 1.5)
    xy = pack.kp_xy[kp.astype(np.int64)]
    outside = (xy[:, 0] < 0) | (xy[:, 0] >= W) | (xy[:, 1] < 0) | (xy[:, 1] >= H)
    assert outside.any(), "no keypoint outside the image found a match: the case would not test the border"
