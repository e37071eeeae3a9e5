"""GPU parity for NON-DEFAULT parameters: the CUDA path against the CPU oracle on the same seeded inputs and against the
outputs frozen from the unmodified reference (tests/golden/ref_slam_params.npz, made by
tests/golden/make_golden_params.py).  Ground-truth-odometry cases are index / IEEE work end to end and must match the
oracle bit for bit; ICP cases are held to north_star's tolerances (1e-4 on poses, 1e-3 on fused points)."""
import pytest
import torch

import gsx_oracle as oracle
from frozen import assert_rows_close, load  # tests/golden is on sys.path, see conftest.py
from gradslam_b200.synthetic import make_sequence

pytestmark = pytest.mark.gpu
DEV = torch.device("cuda:0")

# (name, class, mode, B, L, H, W, seed, make_sequence kwargs, slam kwargs) - the cases of make_golden_params.py
PARAM_CASES = [
    ("pf_gt_tight", "PointFusion", "pointfusion", 2, 4, 64, 64, 11, dict(),
     dict(odom="gt", dist_th=0.02, angle_th=10, sigma=0.3)),
    ("pf_gt_loose", "PointFusion", "pointfusion", 1, 4, 48, 80, 12, dict(),
     dict(odom="gt", dist_th=0.2, angle_th=45, sigma=1.5)),
    ("pf_gt_yaw", "PointFusion", "pointfusion", 2, 3, 64, 64, 13, dict(yaw0=0.6), dict(odom="gt")),
    ("pf_icp_ds2", "PointFusion", "pointfusion", 1, 3, 64, 64, 14, dict(yaw0=0.6),
     dict(odom="icp", numiters=6, dsratio=2, damp=1e-4)),
    ("pf_gradicp_gates", "PointFusion", "pointfusion", 1, 3, 64, 64, 15, dict(yaw0=0.6),
     dict(odom="gradicp", numiters=6, dsratio=2, lambda_max=4.0, B=2.0, B2=0.5, nu=50.0)),
    ("icpslam_gradicp_thresh", "ICPSLAM", "aggregate", 1, 3, 64, 64, 16, dict(yaw0=0.6),
     dict(odom="gradicp", numiters=5, dsratio=2, dist_thresh=0.5)),
]


@pytest.fixture(scope="module")
def frozen():
    return load("ref_slam_params.npz")


def _nn_dist(a, b):
    return oracle.knn1(a, b)[0].sqrt()


@pytest.mark.parametrize("case", PARAM_CASES, ids=[c[0] for c in PARAM_CASES])
def test_slam_with_other_parameters(frozen, case):
    import gradslam_b200 as gs

    name, cls, mode, B, L, H, W, seed, seq_kw, kw = case
    rgb, depth, K, poses = make_sequence(B, L, H, W, seed=seed, **seq_kw)
    slam = getattr(gs, cls)(device=DEV, **kw)
    pc, rec = slam(gs.RGBDImages(rgb.to(DEV), depth.to(DEV), K.to(DEV), poses.to(DEV)))
    ref = oracle.run_slam(rgb, depth, K, poses, mode=mode, **kw)
    got = [int(c) for c in pc.num_points_per_pointcloud.tolist()]
    if kw["odom"] == "gt":
        # bit-exact against the oracle ...
        assert got == ref.map.counts()
        assert torch.equal(rec.cpu(), poses)
        for b in range(B):
            assert torch.equal(pc.points_list[b].cpu(), ref.map.points[b])
            assert torch.equal(pc.normals_list[b].cpu(), ref.map.normals[b])
            assert torch.equal(pc.colors_list[b].cpu(), ref.map.colors[b])
            assert torch.equal(pc.features_list[b].cpu(), ref.map.ccounts[b])
        # ... and within the golden-test tolerances of the frozen reference outputs
        assert got == frozen[name + "/counts"].tolist()
        for b in range(B):
            assert_rows_close(pc.points_list[b], frozen, "%s/points/%d" % (name, b), rtol=0, atol=2e-5)
            assert_rows_close(pc.features_list[b], frozen, "%s/ccounts/%d" % (name, b), rtol=1e-6, atol=1e-7)
        return
    # ICP odometry: north_star tolerances, against the oracle and against the frozen reference poses
    torch.testing.assert_close(rec.cpu(), ref.poses, rtol=0, atol=1e-4)
    torch.testing.assert_close(rec.cpu(), torch.from_numpy(frozen[name + "/poses"]), rtol=0, atol=1e-4)
    for b in range(B):
        want = ref.map.counts()[b]
        # a pose difference of ~1e-6 can flip a borderline match, so sizes may differ by a handful of points
        assert abs(got[b] - want) <= max(3, want // 500), (got, ref.map.counts())
        mine = pc.points_list[b].cpu()
        if got[b] == want:
            torch.testing.assert_close(mine, ref.map.points[b], rtol=0, atol=1e-3)
        else:  # set comparison: every point has a counterpart within 1e-3
            assert _nn_dist(mine, ref.map.points[b]).quantile(0.999) < 1e-3
            assert _nn_dist(ref.map.points[b], mine).quantile(0.999) < 1e-3


from edge_cases import EDGE_CASES, edge_inputs  # noqa: E402  (tests/golden is on sys.path, see conftest.py)


@pytest.mark.parametrize("name", EDGE_CASES)
def test_edge_cases(frozen, name):
    """All-invalid frames, an empty sequence, partial frames, a frame without any correspondence: bit-exact against the
    oracle, golden-test tolerances against the frozen reference outputs; through the whole-sequence driver AND through
    the per-frame step API."""
    import gradslam_b200 as gs

    rgb, depth, K, poses = edge_inputs(name)
    ref = oracle.run_slam(rgb, depth, K, poses, odom="gt")
    counts = frozen[name + "/counts"].tolist()
    assert ref.map.counts() == counts
    slam = gs.PointFusion(odom="gt", device=DEV)
    frames = gs.RGBDImages(rgb.to(DEV), depth.to(DEV), K.to(DEV), poses.to(DEV))
    pc_seq, _ = slam(frames)
    pc_step = gs.Pointclouds(device=DEV)
    for s in range(frames.shape[1]):
        pc_step, _ = slam.step(pc_step, frames[:, s], None, inplace=True)
    for pc in (pc_seq, pc_step):
        assert [int(c) for c in pc.num_points_per_pointcloud.tolist()] == counts
        for b, n in enumerate(counts):
            assert torch.equal(pc.points_list[b].cpu(), ref.map.points[b])
            assert torch.equal(pc.normals_list[b].cpu(), ref.map.normals[b])
            assert torch.equal(pc.colors_list[b].cpu(), ref.map.colors[b])
            assert torch.equal(pc.features_list[b].cpu(), ref.map.ccounts[b])
            if n:
                assert_rows_close(pc.points_list[b], frozen, "%s/points/%d" % (name, b), rtol=0, atol=2e-5)
