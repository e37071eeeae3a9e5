"""Pins the CPU oracle (oracle/gsx_oracle.py) against
  (1) the reference's own golden vectors and known-answer tests for the path, and
  (2) outputs of the unmodified reference frozen by tests/golden/make_golden.py.
CPU only; runs in the `-m "not gpu"` suite."""
import math
import os

import numpy as np
import pytest
import torch

import gsx_oracle as oracle
from frozen import PIXEL_STRIDE, assert_rows_close, load  # tests/golden is on sys.path, see conftest.py
from gradslam_b200.synthetic import make_sequence

GOLD = os.path.join(os.path.dirname(__file__), "golden")


@pytest.fixture(scope="module")
def msrd():
    return {k: torch.from_numpy(v) for k, v in load("msrd_b2s3.npz").items()}


@pytest.fixture(scope="module")
def ref():
    return load("ref_slam.npz")


# ---------------------------------------------------------------------------------------------------------
# K1 — the reference's golden .npy vectors (reference tests/structures/test_rgbdimages.py:105-165)
# ---------------------------------------------------------------------------------------------------------
def test_vertex_maps_match_reference_golden(msrd):
    maps = oracle.frame_maps(msrd["depths"], msrd["intrinsics"], msrd["poses"])
    for name, key, atol in (("vertex", "vertex_map", 1e-6), ("gvertex", "global_vertex_map", 2e-6)):
        got = maps[name].reshape(-1, 3)
        # reference tolerance: sum of squared differences < 1e-2 (test_rgbdimages.py:105-113); we are far inside
        assert ((got[::PIXEL_STRIDE] - msrd[key + "/sample"]) ** 2).sum() < 1e-6
        assert_rows_close(got, msrd, key, rtol=1e-5, atol=atol, stride=PIXEL_STRIDE)


def test_normal_maps_match_reference_golden(msrd):
    maps = oracle.frame_maps(msrd["depths"], msrd["intrinsics"], msrd["poses"])
    for got, key in ((maps["normal"], "normal_map"), (maps["gnormal"], "global_normal_map")):
        # reference criterion: >= 99 % of elements within squared error 1e-5 (test_rgbdimages.py:118-120, 152-165).
        # The .npy vectors were produced by a build that evaluates the cross product without FMA (exactly 0 where a
        # pixel's right and lower neighbours are both missing); the reference's CPU build in the build container
        # contracts it (rounding residue there), which is what the oracle follows - the frozen run of THAT build is
        # compared bit for bit in test_frame_maps_equal_frozen_reference_run.
        frac = (((got.reshape(-1, 3)[::PIXEL_STRIDE] - msrd[key + "/sample"]) ** 2) < 1e-5).float().mean().item()
        assert frac > 0.99, frac
    # away from those pixels the agreement is tight
    d = msrd["depths"][..., 0]
    right = torch.zeros_like(d, dtype=torch.bool)
    below = torch.zeros_like(d, dtype=torch.bool)
    right[..., :, :-1] = d[..., :, 1:] <= 0
    right[..., :, -1] = right[..., :, -2]
    below[..., :-1, :] = d[..., 1:, :] <= 0
    below[..., -1, :] = below[..., -2, :]
    regular = ~(right & below)
    close = ((maps["normal"].reshape(-1, 3)[::PIXEL_STRIDE] - msrd["normal_map/sample"]) ** 2) < 1e-5
    assert close[regular.reshape(-1)[::PIXEL_STRIDE]].float().mean() > 0.999
    # normals are zero exactly where the depth is missing (test_rgbdimages.py:137-140)
    invalid = ~(msrd["depths"][..., 0] > 0)
    assert maps["normal"][invalid].abs().max() == 0


def test_vertex_map_reprojects_to_pixel_grid(msrd):
    """Re-projecting the local vertex map with K recovers the pixel grid within 1e-4 (test_rgbdimages.py:90-103)."""
    depth, K = msrd["depths"], msrd["intrinsics"]
    v = oracle.frame_maps(depth, K, None)["vertex"]
    B, L, H, W, _ = v.shape
    fx, fy, cx, cy = K[:, 0, 0, 0], K[:, 0, 1, 1], K[:, 0, 0, 2], K[:, 0, 1, 2]
    valid = depth[..., 0] > 0
    z = torch.where(valid, v[..., 2], torch.ones_like(v[..., 2]))
    u = v[..., 0] / z * fx.view(B, 1, 1, 1) + cx.view(B, 1, 1, 1)
    w = v[..., 1] / z * fy.view(B, 1, 1, 1) + cy.view(B, 1, 1, 1)
    uu = torch.arange(W, dtype=torch.float32).view(1, 1, 1, W).expand(B, L, H, W)
    vv = torch.arange(H, dtype=torch.float32).view(1, 1, H, 1).expand(B, L, H, W)
    assert (u - uu)[valid].abs().max() < 1e-3
    assert (w - vv)[valid].abs().max() < 1e-3


def test_inverse_intrinsics_known_answer():
    """reference tests/geometry/test_projutils.py:271-354 style closed form."""
    K = torch.eye(4)
    K[0, 0], K[1, 1], K[0, 2], K[1, 2] = 120.3, -120.0, 79.875, 59.875
    Kinv = oracle.inverse_intrinsics(K)
    torch.testing.assert_close(Kinv @ K, torch.eye(4), rtol=1e-5, atol=1e-5)


# ---------------------------------------------------------------------------------------------------------
# fusion known answers restated from the reference's tests/slam/test_fusionutils.py
# ---------------------------------------------------------------------------------------------------------
def test_get_alpha_known_answer():
    """The reference's known answers (tests/slam/test_fusionutils.py:27-53): sigma=0.6, eps=1e-20."""
    pts = torch.tensor([[5.0, 5.0, 5.0], [3.0, 3.0, 3.0], [1.0, 2.0, 3.0], [3.0, 2.0, 1.0], [-1.0, 0.0, 1.0],
                        [0.0, 0.0, 0.0]])
    a = oracle.get_alpha(pts, 0.6, eps=1e-20)[:, 0]
    want = torch.tensor([1e-20, 5.17e-17, 3.5924e-09, 3.5924e-09, 6.2177e-02, 1.0])
    torch.testing.assert_close(a, want, rtol=1e-3, atol=1e-20)
    assert (a > 0).all()


def _tiny_map(points, normals, ccounts):
    return oracle.SurfelMap([points], [normals], [torch.zeros_like(points)], [ccounts])


def test_best_unique_ordering_known_answer():
    """Restates test_fusionutils.py:672-750: among candidates of one pixel keep the largest ccount, then the
    smallest ray distance, then the smallest index; output sorted by (b, h, w)."""
    # 6 map points; frame vertex map 2x2, all at z=1
    gv = torch.zeros(1, 2, 2, 3)
    gv[..., 2] = 1.0
    pts = torch.tensor([[0, 0, 1.00], [0, 0, 1.01], [0, 0, 1.02], [0, 0, 0.99], [0, 0, 1.00], [0, 0, 1.03]])
    cc = torch.tensor([[2.0], [5.0], [5.0], [1.0], [1.0], [7.0]])
    smap = _tiny_map(pts, torch.zeros_like(pts), cc)
    #            b  n  h  w
    table = torch.tensor([[0, 0, 0, 0], [0, 1, 0, 0], [0, 2, 0, 0],  # pixel (0,0): cc 2,5,5 -> n=1 (closer than 2)
                          [0, 3, 1, 1], [0, 4, 1, 1],                # pixel (1,1): cc 1,1 -> n=4 (ray 0 < 1e-4)
                          [0, 5, 0, 1]])                             # pixel (0,1): single
    got = oracle.find_best_unique_correspondences(smap, gv, table)
    assert got.tolist() == [[0, 1, 0, 0], [0, 5, 0, 1], [0, 4, 1, 1]]
    # identical keys fall back to the smallest index
    cc2 = torch.tensor([[3.0], [3.0], [3.0], [1.0], [1.0], [7.0]])
    pts2 = pts.clone()
    pts2[:3, 2] = 1.01
    got = oracle.find_best_unique_correspondences(_tiny_map(pts2, torch.zeros_like(pts), cc2), gv, table)
    assert got.tolist()[0] == [0, 0, 0, 0]


def test_fuse_known_answer():
    """Restates the structure of test_fusionutils.py:918-986: 2x2 frame, 3 matches + 1 append; the merged colour
    is the confidence-weighted mean and the new point is appended last."""
    H = W = 2
    depth = torch.ones(1, 1, H, W, 1)
    K = torch.eye(4).view(1, 1, 4, 4).clone()
    K[0, 0, 0, 2] = K[0, 0, 1, 2] = 0.5
    maps = oracle.frame_maps(depth, K, torch.eye(4).view(1, 1, 4, 4))
    rgb = torch.tensor([[1.0, 0, 0], [0, 1.0, 0], [0, 0, 1.0], [1.0, 1.0, 1.0]]).view(1, 1, H, W, 3)
    gv = maps["gvertex"][0, 0].reshape(-1, 3)
    smap = oracle.SurfelMap([gv[:3].clone()], [maps["gnormal"][0, 0].reshape(-1, 3)[:3].clone()],
                            [torch.full((3, 3), 0.5)], [torch.tensor([[1.0], [2.0], [3.0]])])
    table = torch.tensor([[0, 0, 0, 0], [0, 1, 0, 1], [0, 2, 1, 0]])
    out = oracle.fuse_with_map(smap, maps, rgb, table, sigma=0.6)
    alpha = oracle.get_alpha(maps["vertex"][0, 0], 0.6).reshape(-1)
    assert out.counts() == [4]
    for n, cc in enumerate((1.0, 2.0, 3.0)):
        want = (cc * 0.5 + alpha[n] * rgb.view(-1, 3)[n]) / (cc + alpha[n])
        torch.testing.assert_close(out.colors[0][n], want, rtol=1e-6, atol=1e-7)
        torch.testing.assert_close(out.ccounts[0][n, 0], cc + alpha[n], rtol=1e-6, atol=1e-7)
        torch.testing.assert_close(out.points[0][n], gv[n], rtol=1e-6, atol=1e-7)  # same position stays put
    torch.testing.assert_close(out.points[0][3], gv[3])
    torch.testing.assert_close(out.colors[0][3], torch.ones(3))
    torch.testing.assert_close(out.ccounts[0][3, 0], alpha[3])


def test_active_points_recover_every_valid_pixel():
    """test_fusionutils.py:305-333: projecting the frame-0 map back into frame 0 hits every valid pixel once."""
    rgb, depth, K, poses = make_sequence(2, 1, 32, 40, seed=11)
    maps = oracle.frame_maps(depth, K, poses)
    smap = oracle.update_map_fusion(oracle.SurfelMap(), maps, rgb, poses[:, 0], K[:, 0], 0.05, math.cos(math.radians(20)), 0.6)
    table = oracle.find_active_map_points(smap, poses[:, 0], K[:, 0], 32, 40)
    valid = maps["valid"][:, 0]
    assert table.shape[0] == int(valid.sum())
    hit = torch.zeros_like(valid)
    hit[table[:, 0], table[:, 2], table[:, 3]] = True
    assert torch.equal(hit, valid)
    # correspondences = valid pixels minus valid-depth-but-zero-normal pixels (test_fusionutils.py:879-913)
    corr = oracle.find_correspondences(smap, maps, poses[:, 0], K[:, 0], 0.05, math.cos(math.radians(20)))
    zero_n = (maps["gnormal"][:, 0].abs().sum(-1) == 0) & valid
    assert corr.shape[0] == int(valid.sum()) - int(zero_n.sum())


def test_solve_linear_system_known_answer():
    """tests/odometry/test_icputils.py:18-49: the damped normal equations reproduce x on a consistent system."""
    torch.manual_seed(0)
    A = torch.randn(5, 4)
    x = torch.randn(4, 1)
    got = oracle.solve_linear_system(A, A @ x, damp=1e-8)
    torch.testing.assert_close(got, x, rtol=1e-3, atol=1e-3)


def test_se3_exp_small_angle_branch():
    T = oracle.se3_exp(torch.tensor([0.1, 0.2, 0.3, 1e-8, -2e-8, 3e-8]))
    assert T[3].tolist() == [0, 0, 0, 1]
    torch.testing.assert_close(T[:3, 3], torch.tensor([0.1, 0.2, 0.3]), rtol=1e-6, atol=1e-7)
    T = oracle.se3_exp(torch.tensor([0.0, 0.0, 0.0, 0.0, 0.0, math.pi / 2]))
    torch.testing.assert_close(T[:3, :3], torch.tensor([[0.0, -1, 0], [1, 0, 0], [0, 0, 1]]), rtol=1e-6, atol=1e-6)


def test_knn1_ties_take_lowest_index():
    tgt = torch.tensor([[1.0, 0, 0], [0, 1.0, 0], [1.0, 0, 0], [0, 0, 5.0]])
    src = torch.tensor([[1.0, 0, 0], [0, 0.9, 0], [0, 0, 9.0]])
    d, i = oracle.knn1(src, tgt)
    assert i.tolist() == [0, 1, 3]
    torch.testing.assert_close(d, torch.tensor([0.0, 0.01, 16.0]), rtol=1e-5, atol=1e-7)


# ---------------------------------------------------------------------------------------------------------
# frozen outputs of the unmodified reference (tests/golden/make_golden.py)
# ---------------------------------------------------------------------------------------------------------
CASES = [
    ("pf_gt_64", "pointfusion", 2, 4, 64, 64, 0, dict(odom="gt")),
    ("pf_gt_120", "pointfusion", 1, 4, 120, 160, 1, dict(odom="gt")),
    ("pf_icp_64", "pointfusion", 1, 3, 64, 64, 0, dict(odom="icp", numiters=10)),
    ("pf_gradicp_64", "pointfusion", 2, 3, 64, 64, 2, dict(odom="gradicp", numiters=10)),
    ("icpslam_gradicp_64", "aggregate", 2, 3, 64, 64, 0, dict(odom="gradicp", numiters=5)),
    ("icpslam_icp_64", "aggregate", 1, 2, 64, 64, 3, dict(odom="icp", numiters=8)),
]


@pytest.mark.parametrize("case", CASES, ids=[c[0] for c in CASES])
def test_slam_runs_match_frozen_reference(ref, case):
    name, mode, B, L, H, W, seed, kw = case
    rgb, depth, K, poses = make_sequence(B, L, H, W, seed=seed)
    res = oracle.run_slam(rgb, depth, K, poses, mode=mode, **kw)
    assert res.map.counts() == ref[name + "/counts"].tolist()
    # north_star tolerances: 1e-4 on poses, 1e-3 on fused point coordinates.  Ground-truth odometry is ~100x inside;
    # the ICP loops amplify the 1-ulp differences of the reference's BLAS-ordered sums (LM accept / reject, 8-10
    # iterations), measured up to 3.6e-5 on a pose and 9e-5 on a point, so they are held to half the north_star bounds.
    ptol, xtol = (1e-5, 2e-5) if kw["odom"] == "gt" else (5e-5, 5e-4)
    torch.testing.assert_close(res.poses, torch.from_numpy(ref[name + "/poses"]), rtol=0, atol=ptol)
    for b in range(B):
        assert_rows_close(res.map.points[b], ref, "%s/points/%d" % (name, b), rtol=0, atol=xtol)
        assert_rows_close(res.map.normals[b], ref, "%s/normals/%d" % (name, b), rtol=0, atol=xtol)
        assert_rows_close(res.map.colors[b], ref, "%s/colors/%d" % (name, b), rtol=0, atol=2e-6)
        if mode == "pointfusion":
            assert_rows_close(res.map.ccounts[b], ref, "%s/ccounts/%d" % (name, b), rtol=1e-6, atol=1e-7)


def test_frame_maps_equal_frozen_reference_run(ref):
    """K1 on the bench's input distribution (random holes, so pixels whose right and lower neighbours are both missing
    occur): local vertex and normal maps are BIT-identical to the reference's CPU run (the normal's cross product and
    length follow its FMA rounding); the global maps go through the reference's einsum (BLAS order) and agree to
    an ulp."""
    rgb, depth, K, poses = make_sequence(2, 2, 60, 80, seed=6)
    maps = oracle.frame_maps(depth, K, poses)
    assert torch.equal(maps["vertex"], torch.from_numpy(ref["k1/vertex"]))
    assert torch.equal(maps["normal"], torch.from_numpy(ref["k1/normal"]))
    torch.testing.assert_close(maps["gvertex"], torch.from_numpy(ref["k1/gvertex"]), rtol=0, atol=1e-6)
    torch.testing.assert_close(maps["gnormal"], torch.from_numpy(ref["k1/gnormal"]), rtol=0, atol=2.5e-7)
    # the degenerate pixels exist in this input and their normals are NOT zero (neither here nor in the reference)
    d = depth[..., 0]
    deg = (d[:, :, :-1, :-1] > 0) & (d[:, :, :-1, 1:] <= 0) & (d[:, :, 1:, :-1] <= 0)
    assert deg.sum() > 0


def test_full_size_run_matches_frozen_reference(ref):
    """640x480, B=1, L=6, odom=gt on the bench's input distribution against the unmodified reference: map sizes after
    every frame, checksums and a 1-in-53 sample of the final surfels (tests/golden/fullsize.py states the bounds)."""
    from golden.fullsize import FULL_L, check_against_frozen_reference

    rgb, depth, K, poses = make_sequence(1, FULL_L, 480, 640, seed=0)
    dot_th = math.cos(20 * math.pi / 180)
    smap = oracle.SurfelMap()
    sizes = []
    for s in range(FULL_L):
        maps = oracle.frame_maps(depth[:, s:s + 1], K, poses[:, s:s + 1])
        smap = oracle.update_map_fusion(smap, maps, rgb[:, s:s + 1], poses[:, s], K[:, 0], 0.05, dot_th, 0.6)
        sizes.append(smap.counts()[0])
    check_against_frozen_reference(ref, sizes, smap.points[0], smap.normals[0], smap.colors[0], smap.ccounts[0])


def test_correspondence_tables_match_frozen_reference(ref):
    """Index work: the three tables of one fusion step are identical, row for row, to the reference's."""
    rgb, depth, K, poses = make_sequence(2, 3, 64, 64, seed=4)
    dot_th = math.cos(20 * math.pi / 180)
    smap = oracle.SurfelMap()
    for s in range(2):
        maps = oracle.frame_maps(depth[:, s:s + 1], K, poses[:, s:s + 1])
        smap = oracle.update_map_fusion(smap, maps, rgb[:, s:s + 1], poses[:, s], K[:, 0], 0.05, dot_th, 0.6)
    assert smap.counts() == ref["tables/map_before/counts"].tolist()
    maps = oracle.frame_maps(depth[:, 2:3], K, poses[:, 2:3])
    gv, gn = maps["gvertex"][:, 0], maps["gnormal"][:, 0]
    active = oracle.find_active_map_points(smap, poses[:, 2], K[:, 0], 64, 64)
    assert torch.equal(active, torch.from_numpy(ref["tables/active"]))
    similar, mask = oracle.find_similar_map_points(smap, gv, gn, active, 0.05, dot_th)
    assert torch.equal(similar, torch.from_numpy(ref["tables/similar"]))
    assert torch.equal(mask, torch.from_numpy(ref["tables/similar_mask"]))
    unique = oracle.find_best_unique_correspondences(smap, gv, similar)
    assert torch.equal(unique, torch.from_numpy(ref["tables/unique"]))
    fused = oracle.fuse_with_map(smap, maps, rgb[:, 2:3], unique, 0.6)
    assert fused.counts() == ref["tables/map_after/counts"].tolist()
    for b in range(2):
        assert_rows_close(fused.points[b], ref, "tables/map_after/points/%d" % b, rtol=0, atol=2e-6)
        assert_rows_close(fused.ccounts[b], ref, "tables/map_after/ccounts/%d" % b, rtol=1e-6, atol=1e-7)


def test_icp_transform_recovery_matches_frozen_reference(ref):
    rgb, depth, K, poses = make_sequence(1, 1, 48, 64, seed=5, hole_fraction=0.0)
    maps = oracle.frame_maps(depth, K, poses)
    tgt = maps["gvertex"][0, 0].reshape(-1, 3)
    tgt_n = maps["gnormal"][0, 0].reshape(-1, 3)
    T_true = torch.from_numpy(ref["icp/T_true"])
    src = tgt @ T_true[:3, :3].t() + T_true[:3, 3]
    T_icp, _ = oracle.point_to_plane_icp(src, tgt, tgt_n, torch.eye(4), numiters=12)
    T_grad, _ = oracle.point_to_plane_gradicp(src, tgt, tgt_n, torch.eye(4), numiters=12)
    torch.testing.assert_close(T_icp, torch.from_numpy(ref["icp/T_icp"]), rtol=0, atol=1e-4)
    torch.testing.assert_close(T_grad, torch.from_numpy(ref["icp/T_gradicp"]), rtol=0, atol=1e-4)


# ---------------------------------------------------------------------------------------------------------
# the reference's two hand-built known-answer cases, restated verbatim as data
# ---------------------------------------------------------------------------------------------------------
REF_PTS = [[5.0, 5.0, 5.0], [3.0, 3.0, 3.0], [1.0, 2.0, 3.0], [3.0, 2.0, 1.0], [-1.0, 0.0, 1.0], [0.0, 0.0, 0.0]]
REF_IMAGE = [[[0.0, 1.0, 0.0], [0.0, 2.0, 0.0]], [[0.0, 5.0, 1.0], [8.0, 8.0, 8.0]]]


def test_reference_sorting_known_answer():
    """tests/slam/test_fusionutils.py:672-750 (test_sorting_correspondences)."""
    pts = torch.tensor(REF_PTS)
    pts[3] = torch.tensor([-0.5, -0.5, 1.0])
    table = torch.tensor([[0, 4, 0, 0], [0, 0, 1, 1], [0, 5, 1, 0], [0, 1, 0, 0], [0, 2, 1, 1], [0, 3, 0, 0]])
    cc = oracle.get_alpha(pts, 0.6)
    cc[3] = 1e-12
    K = torch.tensor([[2.0, 0, 1, 0], [0, 2.0, 1, 0], [0, 0, 1, 0], [0, 0, 0, 1]]).view(1, 1, 4, 4)
    maps = oracle.frame_maps(torch.ones(1, 1, 2, 2, 1), K, None)
    torch.testing.assert_close(maps["vertex"][0, 0], torch.tensor([[[-0.5, -0.5, 1.0], [0.0, -0.5, 1.0]],
                                                                  [[-0.5, 0.0, 1.0], [0.0, 0.0, 1.0]]]),
                               rtol=1e-5, atol=1e-6)
    smap = oracle.SurfelMap([pts], [torch.zeros_like(pts)], [torch.zeros_like(pts)], [cc])
    got = oracle.find_best_unique_correspondences(smap, maps["gvertex"][:, 0], table)
    assert got.tolist() == [[0, 4, 0, 0], [0, 5, 1, 0], [0, 2, 1, 1]]


def test_reference_fuse_known_answer():
    """tests/slam/test_fusionutils.py:918-986 (test_fuse_with_map): depth 1e-20 makes alpha == 1 for every pixel."""
    pts = torch.tensor(REF_PTS)
    table = torch.tensor([[0, 1, 0, 0], [0, 2, 0, 1], [0, 5, 1, 0]])
    image = torch.tensor(REF_IMAGE).view(1, 1, 2, 2, 3)
    torch.manual_seed(0)
    K = torch.rand(4, 4).view(1, 1, 4, 4)
    maps = oracle.frame_maps(torch.ones(1, 1, 2, 2, 1) * 1e-20, K, torch.eye(4).view(1, 1, 4, 4))
    smap = oracle.SurfelMap([pts.clone()], [pts.clone()], [pts.clone()], [torch.ones(6, 1)])
    out = oracle.fuse_with_map(smap, maps, image, table, 0.6)
    want = torch.tensor([[5.0, 5, 5], [1.5, 2, 1.5], [0.5, 2, 1.5], [3, 2, 1], [-1, 0, 1], [0, 2.5, 0.5], [8, 8, 8]])
    torch.testing.assert_close(out.colors[0], want, rtol=1e-5, atol=1e-6)


# ---------------------------------------------------------------------------------------------------------------
# backward passes: the oracle's autograd against gradients recorded from the reference (tests/golden/ref_grad.npz,
# written by tests/golden/make_golden_grad.py).  The CUDA backward kernels are compared with the oracle's autograd on
# the GPU (tests/test_gpu_backward.py), so this closes the chain reference -> oracle -> kernels for d/d inputs too.
# ---------------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def ref_grad():
    return np.load(os.path.join(GOLD, "ref_grad.npz"))


def _close_grad(got, want, rtol, atol_rel):
    want = torch.from_numpy(np.asarray(want))
    assert torch.isfinite(got).all()
    torch.testing.assert_close(got, want, rtol=rtol, atol=atol_rel * want.abs().max().item())


def test_oracle_pointfusion_gradients_match_reference(ref_grad):
    rgb, depth, K, poses = make_sequence(1, 2, 24, 32, seed=41, yaw0=0.6)
    d, c = depth.clone().requires_grad_(True), rgb.clone().requires_grad_(True)
    res = oracle.run_slam(c, d, K, poses, odom="gt")
    n = res.map.counts()[0]
    assert n == int(ref_grad["pf_gt/count"][0])
    g = torch.Generator().manual_seed(5)
    wp, wc, wf = torch.randn(n, 3, generator=g), torch.randn(n, 3, generator=g), torch.randn(n, 1, generator=g)
    ((res.map.points[0] * wp).sum() + (res.map.colors[0] * wc).sum() + (res.map.ccounts[0] * wf).sum()).backward()
    _close_grad(d.grad, ref_grad["pf_gt/d_depth"], 1e-3, 1e-4)
    _close_grad(c.grad, ref_grad["pf_gt/d_rgb"], 1e-4, 1e-6)


@pytest.mark.parametrize("name", ["gradicp", "icp"])
def test_oracle_icp_gradients_match_reference(ref_grad, name):
    rgb, depth, K, poses = make_sequence(1, 1, 40, 56, seed=31, hole_fraction=0.0, yaw0=0.6)
    m = oracle.frame_maps(depth, K, poses)
    tgt = m["gvertex"][0, 0].reshape(-1, 3).contiguous()
    tgt_n = m["gnormal"][0, 0].reshape(-1, 3).contiguous()
    T_true = oracle.se3_exp(torch.tensor([0.01, -0.005, 0.008, 0.01, -0.01, 0.005]))
    s = oracle.rigid_apply(T_true, tgt).clone().requires_grad_(True)
    fn = oracle.point_to_plane_gradicp if name == "gradicp" else oracle.point_to_plane_icp
    T, _ = fn(s, tgt, tgt_n, torch.eye(4), numiters=4)
    torch.testing.assert_close(T.detach(), torch.from_numpy(ref_grad[name + "/T"]), rtol=0, atol=1e-5)
    w = torch.randn(4, 4, generator=torch.Generator().manual_seed(1))
    (T * w).sum().backward()
    _close_grad(s.grad, ref_grad[name + "/d_src"], 2e-2, 2e-3)


def test_oracle_icpslam_pose_gradient_matches_reference(ref_grad):
    rgb, depth, K, poses = make_sequence(1, 2, 32, 40, seed=17, yaw0=0.6)
    d = depth.clone().requires_grad_(True)
    res = oracle.run_slam(rgb, d, K, poses, mode="aggregate", odom="gradicp", numiters=3, dsratio=2)
    torch.testing.assert_close(res.poses.detach(), torch.from_numpy(ref_grad["icpslam/poses"]), rtol=0, atol=1e-5)
    w = torch.randn(res.poses.shape, generator=torch.Generator().manual_seed(9))
    (res.poses * w).sum().backward()
    _close_grad(d.grad, ref_grad["icpslam/d_depth"], 5e-2, 5e-3)


# ---------------------------------------------------------------------------------------------------------------
# non-default parameters (tests/golden/make_golden_params.py): thresholds / sigma of the fusion, ICP down-sampling,
# damping, distance threshold, gradLM gate parameters, a non-square image, a first pose that is not the identity
# ---------------------------------------------------------------------------------------------------------------
PARAM_CASES = [
    ("pf_gt_tight", "pointfusion", 2, 4, 64, 64, 11, dict(), dict(odom="gt", dist_th=0.02, angle_th=10, sigma=0.3)),
    ("pf_gt_loose", "pointfusion", 1, 4, 48, 80, 12, dict(), dict(odom="gt", dist_th=0.2, angle_th=45, sigma=1.5)),
    ("pf_gt_yaw", "pointfusion", 2, 3, 64, 64, 13, dict(yaw0=0.6), dict(odom="gt")),
    ("pf_icp_ds2", "pointfusion", 1, 3, 64, 64, 14, dict(yaw0=0.6), dict(odom="icp", numiters=6, dsratio=2, damp=1e-4)),
    ("pf_gradicp_gates", "pointfusion", 1, 3, 64, 64, 15, dict(yaw0=0.6),
     dict(odom="gradicp", numiters=6, dsratio=2, lambda_max=4.0, B=2.0, B2=0.5, nu=50.0)),
    ("icpslam_gradicp_thresh", "aggregate", 1, 3, 64, 64, 16, dict(yaw0=0.6),
     dict(odom="gradicp", numiters=5, dsratio=2, dist_thresh=0.5)),
]


@pytest.fixture(scope="module")
def ref_params():
    return load("ref_slam_params.npz")


@pytest.mark.parametrize("case", PARAM_CASES, ids=[c[0] for c in PARAM_CASES])
def test_slam_runs_with_other_parameters_match_frozen_reference(ref_params, case):
    name, mode, B, L, H, W, seed, seq_kw, kw = case
    rgb, depth, K, poses = make_sequence(B, L, H, W, seed=seed, **seq_kw)
    res = oracle.run_slam(rgb, depth, K, poses, mode=mode, **kw)
    assert res.map.counts() == ref_params[name + "/counts"].tolist()
    torch.testing.assert_close(res.poses, torch.from_numpy(ref_params[name + "/poses"]), rtol=0, atol=1e-5)
    for b in range(B):
        for attr, tol in (("points", 2e-5), ("normals", 2e-5), ("colors", 2e-6)):
            assert_rows_close(getattr(res.map, attr)[b], ref_params, "%s/%s/%d" % (name, attr, b), rtol=0, atol=tol)
        if mode == "pointfusion":
            assert_rows_close(res.map.ccounts[b], ref_params, "%s/ccounts/%d" % (name, b), rtol=1e-6, atol=1e-7)


# edge cases: all-invalid frames, an empty sequence, partial frames, a frame without any correspondence
from edge_cases import EDGE_CASES, edge_inputs  # noqa: E402  (tests/golden is on sys.path, see conftest.py)


@pytest.mark.parametrize("name", EDGE_CASES)
def test_edge_cases_match_frozen_reference(ref_params, name):
    rgb, depth, K, poses = edge_inputs(name)
    res = oracle.run_slam(rgb, depth, K, poses, odom="gt")
    counts = ref_params[name + "/counts"].tolist()
    assert res.map.counts() == counts
    for b, n in enumerate(counts):
        if n == 0:
            assert res.map.points[b].shape[0] == 0
            continue
        assert_rows_close(res.map.points[b], ref_params, "%s/points/%d" % (name, b), rtol=0, atol=2e-5)
        assert_rows_close(res.map.ccounts[b], ref_params, "%s/ccounts/%d" % (name, b), rtol=1e-6, atol=1e-7)
