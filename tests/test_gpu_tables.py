"""GPU parity for the table-returning association API (index work: bit-exact against the oracle and against the
tables frozen from the unmodified reference), plus the reference's hand-built known-answer cases."""
import math

import pytest
import torch

import gsx_oracle as oracle
from frozen import load  # tests/golden is on sys.path, see conftest.py
from gradslam_b200.synthetic import make_sequence

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
DOT_TH = math.cos(20 * math.pi / 180)


def _scenario():
    import gradslam_b200 as gs
    from gradslam_b200.slam import fusionutils

    rgb, depth, K, poses = make_sequence(2, 3, 64, 64, seed=4)
    frames = gs.RGBDImages(rgb.to(DEV), depth.to(DEV), K.to(DEV), poses.to(DEV))
    pc = gs.Pointclouds(device=DEV)
    smap = oracle.SurfelMap()
    for s in range(2):
        pc = fusionutils.update_map_fusion(pc, frames[:, s], 0.05, DOT_TH, 0.6, inplace=True)
        m = oracle.frame_maps(depth[:, s:s + 1], K, poses[:, s:s + 1])
        smap = oracle.update_map_fusion(smap, m, rgb[:, s:s + 1], poses[:, s], K[:, 0], 0.05, DOT_TH, 0.6)
    return gs, fusionutils, (rgb, depth, K, poses), frames, pc, smap


def test_tables_match_oracle_and_frozen_reference():
    gs, fu, (rgb, depth, K, poses), frames, pc, smap = _scenario()
    live = frames[:, 2]
    maps = oracle.frame_maps(depth[:, 2:3], K, poses[:, 2:3])
    gv, gn = maps["gvertex"][:, 0], maps["gnormal"][:, 0]
    active = fu.find_active_map_points(pc, live)
    r_active = oracle.find_active_map_points(smap, poses[:, 2], K[:, 0], 64, 64)
    assert active.dtype == torch.int64 and torch.equal(active.cpu(), r_active)
    similar, mask = fu.find_similar_map_points(pc, live, active, 0.05, DOT_TH)
    r_similar, r_mask = oracle.find_similar_map_points(smap, gv, gn, r_active, 0.05, DOT_TH)
    assert torch.equal(similar.cpu(), r_similar) and torch.equal(mask.cpu(), r_mask)
    unique = fu.find_best_unique_correspondences(pc, live, similar)
    r_unique = oracle.find_best_unique_correspondences(smap, gv, r_similar)
    assert torch.equal(unique.cpu(), r_unique)
    assert torch.equal(fu.find_correspondences(pc, live, 0.05, DOT_TH).cpu(), r_unique)
    # the same tables, frozen from the unmodified reference
    ref = load("ref_slam.npz")
    assert torch.equal(active.cpu(), torch.from_numpy(ref["tables/active"]))
    assert torch.equal(similar.cpu(), torch.from_numpy(ref["tables/similar"]))
    assert torch.equal(unique.cpu(), torch.from_numpy(ref["tables/unique"]))
    # fuse_with_map from the table == fused update == oracle
    fused = fu.fuse_with_map(pc, live, unique, 0.6, inplace=False)
    direct = fu.update_map_fusion(pc, live, 0.05, DOT_TH, 0.6, inplace=False)
    r_fused = oracle.fuse_with_map(smap, maps, rgb[:, 2:3], r_unique, 0.6)
    assert fused.num_points_per_pointcloud.tolist() == r_fused.counts() == direct.num_points_per_pointcloud.tolist()
    for b in range(2):
        assert torch.equal(fused.points_list[b], direct.points_list[b])
        assert torch.equal(fused.features_list[b], direct.features_list[b])
        torch.testing.assert_close(fused.points_list[b].cpu(), r_fused.points[b], rtol=1e-6, atol=1e-6)
        torch.testing.assert_close(fused.colors_list[b].cpu(), r_fused.colors[b], rtol=1e-6, atol=1e-6)
    assert pc.num_points_per_pointcloud.tolist() == smap.counts()  # inplace=False left the input alone


def test_reference_sorting_known_answer_on_gpu():
    """tests/slam/test_fusionutils.py:672-750 through the CUDA arg-min."""
    import gradslam_b200 as gs
    from gradslam_b200.slam import fusionutils as fu

    pts = torch.tensor([[5.0, 5.0, 5.0], [3.0, 3.0, 3.0], [1.0, 2.0, 3.0], [-0.5, -0.5, 1.0], [-1.0, 0.0, 1.0],
                        [0.0, 0.0, 0.0]]).unsqueeze(0)
    table = torch.tensor([[0, 4, 0, 0], [0, 0, 1, 1], [0, 5, 1, 0], [0, 1, 0, 0], [0, 2, 1, 1], [0, 3, 0, 0]])
    feats = fu.get_alpha(pts, 0.6, keepdim=True)
    feats[0, 3] = 1e-12
    pc = gs.Pointclouds(points=pts.to(DEV), features=feats.to(DEV))
    image = torch.tensor([[[0.0, 1.0, 0.0], [0.0, 2.0, 0.0]], [[0.0, 5.0, 1.0], [8.0, 8.0, 8.0]]]).view(1, 1, 2, 2, 3)
    K = torch.tensor([[2.0, 0, 1, 0], [0, 2.0, 1, 0], [0, 0, 1, 0], [0, 0, 0, 1]]).view(1, 1, 4, 4)
    fr = gs.RGBDImages(image.to(DEV), torch.ones(1, 1, 2, 2, 1, device=DEV), K.to(DEV))
    torch.testing.assert_close(fr.vertex_map[0, 0].cpu(), torch.tensor([[[-0.5, -0.5, 1.0], [0.0, -0.5, 1.0]],
                                                                        [[-0.5, 0.0, 1.0], [0.0, 0.0, 1.0]]]),
                               rtol=1e-5, atol=1e-6)
    got = fu.find_best_unique_correspondences(pc, fr, table.to(DEV))
    assert got.cpu().tolist() == [[0, 4, 0, 0], [0, 5, 1, 0], [0, 2, 1, 1]]


def test_reference_fuse_known_answer_on_gpu():
    """tests/slam/test_fusionutils.py:918-986 through K4."""
    import gradslam_b200 as gs
    from gradslam_b200.slam import fusionutils as fu

    pts = torch.tensor([[5.0, 5.0, 5.0], [3.0, 3.0, 3.0], [1.0, 2.0, 3.0], [3.0, 2.0, 1.0], [-1.0, 0.0, 1.0],
                        [0.0, 0.0, 0.0]]).unsqueeze(0).to(DEV)
    table = torch.tensor([[0, 1, 0, 0], [0, 2, 0, 1], [0, 5, 1, 0]], device=DEV)
    image = torch.tensor([[[0.0, 1.0, 0.0], [0.0, 2.0, 0.0]], [[0.0, 5.0, 1.0], [8.0, 8.0, 8.0]]]).view(1, 1, 2, 2, 3)
    torch.manual_seed(0)
    fr = gs.RGBDImages(image.to(DEV), torch.ones(1, 1, 2, 2, 1, device=DEV) * 1e-20,
                       torch.rand(4, 4).view(1, 1, 4, 4).to(DEV), torch.eye(4).view(1, 1, 4, 4).to(DEV))
    pc = gs.Pointclouds(points=pts, normals=pts.clone(), colors=pts.clone(), features=torch.ones_like(pts[..., :1]))
    out = fu.fuse_with_map(pc, fr, table, 0.6)
    want = torch.tensor([[5.0, 5, 5], [1.5, 2, 1.5], [0.5, 2, 1.5], [3, 2, 1], [-1, 0, 1], [0, 2.5, 0.5], [8, 8, 8]])
    torch.testing.assert_close(out.colors_padded[0].cpu(), want, rtol=1e-5, atol=1e-6)


def test_table_api_errors_and_empty_cases():
    import gradslam_b200 as gs
    from gradslam_b200.slam import fusionutils as fu

    rgb, depth, K, poses = make_sequence(1, 2, 16, 16, seed=0)
    fr = gs.RGBDImages(rgb.to(DEV), depth.to(DEV), K.to(DEV), poses.to(DEV))
    empty = gs.Pointclouds(device=DEV)
    assert fu.find_active_map_points(empty, fr[:, 0]).shape == (0, 4)
    t, m = fu.find_similar_map_points(empty, fr[:, 0], torch.empty((0, 4), dtype=torch.int64, device=DEV), 0.05, 0.9)
    assert t.shape == (0, 4) and m.shape == (0,)
    with pytest.raises(TypeError):
        fu.find_active_map_points(3, fr[:, 0])
    with pytest.raises(ValueError):
        fu.find_active_map_points(empty, fr)  # sequence length 2
    with pytest.raises(TypeError):
        fu.find_similar_map_points(empty, fr[:, 0], torch.zeros((1, 4)), 0.05, 0.9)  # not int64
    with pytest.raises(ValueError):
        fu.find_best_unique_correspondences(empty, fr[:, 0], torch.zeros((3,), dtype=torch.int64))
    pc = fu.update_map_fusion(empty, fr[:, 0], 0.05, 0.9, 0.6)
    far = gs.RGBDImages(rgb[:, :1].to(DEV), depth[:, :1].to(DEV), K.to(DEV), (poses[:, :1] + 100).to(DEV))
    with pytest.warns(UserWarning):
        assert fu.find_active_map_points(pc, far).shape[0] == 0


def test_downsample_helpers_match_oracle():
    import gradslam_b200 as gs
    from gradslam_b200.odometry import icputils
    from gradslam_b200.slam import fusionutils as fu

    gs_, fu_, (rgb, depth, K, poses), frames, pc, smap = _scenario()
    live = frames[:, 2]
    got = icputils.downsample_rgbdimages(live, 4)
    maps = oracle.frame_maps(depth[:, 2:3], K, poses[:, 2:3])
    r_pts, r_nrm = oracle.downsample_frame(maps, 4)
    table = fu.find_active_map_points(pc, frames[:, 1])
    got_m = icputils.downsample_pointclouds(pc, table, 4)
    r_table = oracle.find_active_map_points(smap, poses[:, 1], K[:, 0], 64, 64)
    rm_pts, rm_nrm = oracle.downsample_map(smap, r_table, 4)
    for b in range(2):
        assert torch.equal(got.points_list[b].cpu(), r_pts[b]) and torch.equal(got.normals_list[b].cpu(), r_nrm[b])
        torch.testing.assert_close(got_m.points_list[b].cpu(), rm_pts[b], rtol=1e-6, atol=1e-6)
        assert got_m.points_list[b].shape == rm_pts[b].shape
