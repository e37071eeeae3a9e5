"""Freezes outputs of the UNMODIFIED gradslam reference as fixtures (run in the build container only).

    python tests/golden/make_golden.py

Imports the reference from /root/reference through tests/golden/ref_loader.py (four in-memory shims, see
there) and writes

  tests/golden/msrd_b2s3.npz   the reference's own test data and golden vectors (tests/data/msrd_b2s3/*.npy: colors,
                               depths, intrinsics, poses -> vertex / normal / global maps); the inputs of the
                               reference's hot-path tests (tests/common.py load_test_data), which
                               tests/test_gpu_reference_twins.py restates against this package on the GPU, are kept
                               losslessly, the four golden maps as every 17th pixel plus checksums (frozen.py)
  tests/golden/ref_slam.npz    reference outputs on seeded synthetic sequences (gradslam_b200.synthetic, the
                               bench's own input distribution: 2 % random depth holes): PointFusion / ICPSLAM
                               final maps + poses for odom in {gt, icp, gradicp}, the frame maps (K1) of one
                               sequence, the three correspondence tables of one fusion step, an ICP / gradICP
                               transform recovery case, and one FULL-SIZE run (640x480, B=1, L=6, odom=gt):
                               per-frame map sizes, float64 checksums and every 53rd surfel of the final map.
                               Final maps are stored as every 8th surfel plus float64 checksums (frozen.py).

The inputs of ref_slam.npz are NOT stored: the tests regenerate them from the recorded seeds.
"""
import os
import sys
import warnings

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, HERE)
sys.path.insert(0, ROOT)
warnings.simplefilter("ignore")

from frozen import PIXEL_STRIDE, narrow_int, pack_rows  # noqa: E402
from ref_loader import REFERENCE_ROOT, load_reference  # noqa: E402

load_reference()
from gradslam.odometry.icputils import point_to_plane_gradICP, point_to_plane_ICP  # noqa: E402
from gradslam.slam import fusionutils as ref_fu  # noqa: E402
from gradslam.slam.icpslam import ICPSLAM  # noqa: E402
from gradslam.slam.pointfusion import PointFusion  # noqa: E402
from gradslam.structures.pointclouds import Pointclouds  # noqa: E402
from gradslam.structures.rgbdimages import RGBDImages  # noqa: E402

from gradslam_b200.synthetic import make_sequence  # noqa: E402

# (name, class, B, L, H, W, seed, kwargs)
SLAM_CASES = [
    ("pf_gt_64", "PointFusion", 2, 4, 64, 64, 0, dict(odom="gt")),
    ("pf_gt_120", "PointFusion", 1, 4, 120, 160, 1, dict(odom="gt")),
    ("pf_icp_64", "PointFusion", 1, 3, 64, 64, 0, dict(odom="icp", numiters=10)),
    ("pf_gradicp_64", "PointFusion", 2, 3, 64, 64, 2, dict(odom="gradicp", numiters=10)),
    ("icpslam_gradicp_64", "ICPSLAM", 2, 3, 64, 64, 0, dict(odom="gradicp", numiters=5)),
    ("icpslam_icp_64", "ICPSLAM", 1, 2, 64, 64, 3, dict(odom="icp", numiters=8)),
]


FULL_L = 6         # frames of the full-size run
FULL_STRIDE = 53   # every 53rd surfel of its final map is stored


def pack_map(prefix, pc, out):
    out[prefix + "/counts"] = np.array([int(c) for c in pc.num_points_per_pointcloud], dtype=np.int64)
    for b in range(len(pc)):
        pack_rows(out, "%s/points/%d" % (prefix, b), pc.points_list[b].numpy())
        pack_rows(out, "%s/normals/%d" % (prefix, b), pc.normals_list[b].numpy())
        pack_rows(out, "%s/colors/%d" % (prefix, b), pc.colors_list[b].numpy())
        if pc.has_features:
            pack_rows(out, "%s/ccounts/%d" % (prefix, b), pc.features_list[b].numpy())


def main():
    # ---- the reference's own golden vectors (K1) ---------------------------------------------------------
    d = os.path.join(REFERENCE_ROOT, "tests", "data", "msrd_b2s3")
    msrd = {k: np.load(os.path.join(d, k + ".npy")) for k in
            ("colors", "depths", "intrinsics", "poses", "vertex_map", "normal_map", "global_vertex_map",
             "global_normal_map")}
    for k in ("vertex_map", "normal_map", "global_vertex_map", "global_normal_map"):
        pack_rows(msrd, k, msrd.pop(k).reshape(-1, 3), PIXEL_STRIDE)
    np.savez_compressed(os.path.join(HERE, "msrd_b2s3.npz"), **msrd)

    out = {}
    # ---- full SLAM runs ----------------------------------------------------------------------------------
    for name, cls, B, L, H, W, seed, kw in SLAM_CASES:
        rgb, depth, K, poses = make_sequence(B, L, H, W, seed=seed)
        slam = (PointFusion if cls == "PointFusion" else ICPSLAM)(**kw)
        pc, rec = slam(RGBDImages(rgb, depth, K, poses))
        pack_map(name, pc, out)
        out[name + "/poses"] = rec.numpy()
        print(name, out[name + "/counts"])

    # ---- frame maps (K1) on the bench's input distribution (holes next to holes included) --------------------
    rgb, depth, K, poses = make_sequence(2, 2, 60, 80, seed=6)
    fr = RGBDImages(rgb, depth, K, poses)
    out["k1/vertex"] = fr.vertex_map.numpy()
    out["k1/normal"] = fr.normal_map.numpy()
    out["k1/gvertex"] = fr.global_vertex_map.numpy()
    out["k1/gnormal"] = fr.global_normal_map.numpy()

    # ---- full size: BASELINE.json's headline frame size, default holes, B=1, L=6 -----------------------------
    rgb, depth, K, poses = make_sequence(1, FULL_L, 480, 640, seed=0)
    frames = RGBDImages(rgb, depth, K, poses)
    slam = PointFusion(odom="gt")
    pc = Pointclouds()
    sizes = []
    for s in range(FULL_L):
        pc, _ = slam.step(pc, frames[:, s], None, inplace=True)
        sizes.append(int(pc.num_points_per_pointcloud[0]))
    out["full480/sizes"] = np.array(sizes, dtype=np.int64)
    idx = np.arange(0, sizes[-1], FULL_STRIDE)
    for name, lst in (("points", pc.points_list), ("normals", pc.normals_list), ("colors", pc.colors_list),
                      ("ccounts", pc.features_list)):
        a = lst[0].numpy()
        out["full480/%s_sample" % name] = a[idx]
        out["full480/%s_sum" % name] = a.astype(np.float64).sum(0)
        out["full480/%s_abs_sum" % name] = np.abs(a.astype(np.float64)).sum(0)
    print("full480 sizes", sizes)

    # ---- one fusion step, table by table -----------------------------------------------------------------
    rgb, depth, K, poses = make_sequence(2, 3, 64, 64, seed=4)
    frames = RGBDImages(rgb, depth, K, poses)
    slam = PointFusion(odom="gt")
    pc = Pointclouds()
    for s in range(2):
        pc, _ = slam.step(pc, frames[:, s], None, inplace=True)
    live = frames[:, 2]
    t_active = ref_fu.find_active_map_points(pc, live)
    t_similar, mask = ref_fu.find_similar_map_points(pc, live, t_active, slam.dist_th, slam.dot_th)
    t_unique = ref_fu.find_best_unique_correspondences(pc, live, t_similar)
    out["tables/active"] = narrow_int(t_active.numpy())
    out["tables/similar"] = narrow_int(t_similar.numpy())
    out["tables/similar_mask"] = mask.numpy()
    out["tables/unique"] = narrow_int(t_unique.numpy())
    out["tables/map_before/counts"] = np.array([int(c) for c in pc.num_points_per_pointcloud], dtype=np.int64)
    fused = ref_fu.fuse_with_map(pc.clone(), live, t_unique, slam.sigma, inplace=False)
    pack_map("tables/map_after", fused, out)
    print("tables", t_active.shape, t_similar.shape, t_unique.shape)

    # ---- ICP / gradICP transform recovery (like tests/odometry/test_icp.py, smaller) ----------------------
    rgb, depth, K, poses = make_sequence(1, 1, 48, 64, seed=5, hole_fraction=0.0)
    fr = RGBDImages(rgb, depth, K, poses)
    tgt = fr.global_vertex_map[0, 0].reshape(1, -1, 3)
    tgt_n = fr.global_normal_map[0, 0].reshape(1, -1, 3)
    from gradslam.geometry.se3utils import se3_exp

    T_true = se3_exp(torch.tensor([0.02, -0.01, 0.015, 0.03, -0.02, 0.01]))
    src = (tgt[0] @ T_true[:3, :3].t() + T_true[:3, 3]).unsqueeze(0)
    T_icp, _ = point_to_plane_ICP(src, tgt, tgt_n, torch.eye(4), numiters=12, damp=1e-8, dist_thresh=None)
    T_grad, _ = point_to_plane_gradICP(src, tgt, tgt_n, torch.eye(4), numiters=12, damp=1e-8, dist_thresh=None)
    out["icp/T_true"] = T_true.numpy()
    out["icp/T_icp"] = T_icp.numpy()
    out["icp/T_gradicp"] = T_grad.numpy()
    print("icp err", (T_icp @ T_true - torch.eye(4)).abs().max().item(),
          (T_grad @ T_true - torch.eye(4)).abs().max().item())

    # ---- loader calibration contract (datasets/datautils.py:73 scale_intrinsics; icl.py:515-533 _preprocess_poses) ------
    import importlib.util

    # (gradslam.datasets imports imageio / cv2, which are not installed: load the one module the contract lives in)
    spec = importlib.util.spec_from_file_location("ref_datautils",
                                                  os.path.join(REFERENCE_ROOT, "gradslam", "datasets", "datautils.py"))
    ref_datautils = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(ref_datautils)
    scale_intrinsics = ref_datautils.scale_intrinsics
    from gradslam.geometry.geometryutils import relative_transformation

    g = torch.Generator().manual_seed(7)
    K_in = torch.eye(4).repeat(3, 1, 1)
    K_in[:, 0, 0] = 481.2 + torch.rand(3, generator=g)
    K_in[:, 1, 1] = -480.0 + torch.rand(3, generator=g)
    K_in[:, 0, 2] = 319.5
    K_in[:, 1, 2] = 239.5
    out["f2/K_in"] = K_in.numpy()
    out["f2/ratios"] = np.array([120.0 / 480.0, 160.0 / 640.0])
    out["f2/K_scaled"] = scale_intrinsics(K_in, 120.0 / 480.0, 160.0 / 640.0).numpy()
    out["f2/K3_scaled"] = scale_intrinsics(K_in[:, :3, :3].contiguous(), 0.5, 0.75).numpy()
    Bp, Lp = 2, 5
    poses_abs = torch.eye(4).repeat(Bp, Lp, 1, 1)
    for b in range(Bp):
        for l in range(Lp):
            xi = torch.randn(6, generator=g) * torch.tensor([0.5, 0.5, 0.5, 0.8, 0.8, 0.8])
            poses_abs[b, l] = se3_exp(xi)
    poses_abs[:, :, :3, :3] += 1e-3 * torch.randn(Bp, Lp, 3, 3, generator=g)  # (loader poses are not exactly orthogonal)
    out["f2/poses_abs"] = poses_abs.numpy()
    out["f2/poses_rel"] = torch.stack([
        relative_transformation(poses_abs[b, 0].unsqueeze(0).repeat(Lp, 1, 1), poses_abs[b], orthogonal_rotations=False)
        for b in range(Bp)]).numpy()

    np.savez_compressed(os.path.join(HERE, "ref_slam.npz"), **out)
    for f in ("msrd_b2s3.npz", "ref_slam.npz"):
        print(f, os.path.getsize(os.path.join(HERE, f)) // 1024, "KiB")


if __name__ == "__main__":
    main()
