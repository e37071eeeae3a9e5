"""Freezes outputs of the UNMODIFIED gradslam reference for NON-DEFAULT parameters (run in the build container only):

    python tests/golden/make_golden_params.py     ->  tests/golden/ref_slam_params.npz

Same mechanism as make_golden.py (reference imported from /root/reference through ref_loader.py); the cases vary what
the default-parameter fixtures leave untouched: distance / angle thresholds and sigma of the fusion, the ICP
down-sampling ratio, damping, distance threshold and the gradLM gate parameters, a non-square image, a sequence
whose first pose is not the identity, and five edge cases (all-invalid frames, an empty sequence, partial frames, a
frame without any correspondence).  Inputs are NOT stored: the tests regenerate them from the recorded seeds.  Maps are
stored as every 8th surfel plus float64 checksums (frozen.py).
"""
import os
import sys
import warnings

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, HERE)
sys.path.insert(0, ROOT)
warnings.simplefilter("ignore")

from ref_loader import load_reference  # noqa: E402

load_reference()
from gradslam.slam.icpslam import ICPSLAM  # noqa: E402
from gradslam.slam.pointfusion import PointFusion  # noqa: E402
from gradslam.structures.rgbdimages import RGBDImages  # noqa: E402

from gradslam_b200.synthetic import make_sequence  # noqa: E402
from edge_cases import EDGE_CASES, edge_inputs  # noqa: E402
from frozen import pack_rows  # noqa: E402
from make_golden import pack_map  # noqa: E402

# (name, class, B, L, H, W, seed, make_sequence kwargs, slam kwargs)
PARAM_CASES = [
    ("pf_gt_tight", "PointFusion", 2, 4, 64, 64, 11, dict(), dict(odom="gt", dist_th=0.02, angle_th=10, sigma=0.3)),
    ("pf_gt_loose", "PointFusion", 1, 4, 48, 80, 12, dict(), dict(odom="gt", dist_th=0.2, angle_th=45, sigma=1.5)),
    ("pf_gt_yaw", "PointFusion", 2, 3, 64, 64, 13, dict(yaw0=0.6), dict(odom="gt")),
    ("pf_icp_ds2", "PointFusion", 1, 3, 64, 64, 14, dict(yaw0=0.6), dict(odom="icp", numiters=6, dsratio=2, damp=1e-4)),
    ("pf_gradicp_gates", "PointFusion", 1, 3, 64, 64, 15, dict(yaw0=0.6),
     dict(odom="gradicp", numiters=6, dsratio=2, lambda_max=4.0, B=2.0, B2=0.5, nu=50.0)),
    ("icpslam_gradicp_thresh", "ICPSLAM", 1, 3, 64, 64, 16, dict(yaw0=0.6),
     dict(odom="gradicp", numiters=5, dsratio=2, dist_thresh=0.5)),
]


def main():
    out = {}
    for name in EDGE_CASES:
        rgb, depth, K, poses = edge_inputs(name)
        pc, rec = PointFusion(odom="gt")(RGBDImages(rgb, depth, K, poses))
        out[name + "/counts"] = np.array([int(c) for c in pc.num_points_per_pointcloud], dtype=np.int64)
        for b in range(len(pc)):
            if out[name + "/counts"][b] > 0:
                pack_rows(out, "%s/points/%d" % (name, b), pc.points_list[b].numpy())
                pack_rows(out, "%s/ccounts/%d" % (name, b), pc.features_list[b].numpy())
        print(name, out[name + "/counts"])
    for name, cls, B, L, H, W, seed, seq_kw, kw in PARAM_CASES:
        rgb, depth, K, poses = make_sequence(B, L, H, W, seed=seed, **seq_kw)
        slam = (PointFusion if cls == "PointFusion" else ICPSLAM)(**kw)
        pc, rec = slam(RGBDImages(rgb, depth, K, poses))
        pack_map(name, pc, out)
        out[name + "/poses"] = rec.numpy()
        print(name, out[name + "/counts"], "max |pose - gt| %.2e" % (rec - poses).abs().max().item())
    np.savez_compressed(os.path.join(HERE, "ref_slam_params.npz"), **out)
    print("ref_slam_params.npz", os.path.getsize(os.path.join(HERE, "ref_slam_params.npz")) // 1024, "KiB")


if __name__ == "__main__":
    main()
