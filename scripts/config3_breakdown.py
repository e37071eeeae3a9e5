"""Where the differentiable ICPSLAM forward (BASELINE.json config 3) spends its time: inputs already on the device,
phases timed with synchronisation, then a torch.profiler table of the same call."""
import os
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch

import gradslam_b200 as gs
from gradslam_b200.odometry import icp as icp_mod
from gradslam_b200.odometry import icputils
from gradslam_b200.slam import fusionutils, icpslam
from gradslam_b200.synthetic import make_sequence

B = int(sys.argv[1]) if len(sys.argv) > 1 else 8
dev = torch.device("cuda:0")
rgb, depth, K, poses = make_sequence(B, 2, 480, 640, seed=0, yaw0=0.6)
rgb_d, K_d = rgb.to(dev), K.to(dev)
d = depth.to(dev).requires_grad_(True)
p = poses.to(dev).requires_grad_(True)
slam = gs.ICPSLAM(odom="gradicp", numiters=10, dsratio=4, device=dev)
acc = {}


def wrap(mod, name, label=None):
    fn = getattr(mod, name)

    def timed(*a, **k):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        out = fn(*a, **k)
        torch.cuda.synchronize()
        acc[label or name] = acc.get(label or name, 0.0) + (time.perf_counter() - t0) * 1e3
        return out

    setattr(mod, name, timed)


def run(tag):
    acc.clear()
    d.grad = p.grad = None
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    pc, rec = slam(gs.RGBDImages(rgb_d, d, K_d, p))
    torch.cuda.synchronize()
    t1 = time.perf_counter()
    rec.sum().backward()
    torch.cuda.synchronize()
    t2 = time.perf_counter()
    print("%s: forward %.2f ms, backward %.2f ms" % (tag, (t1 - t0) * 1e3, (t2 - t1) * 1e3), flush=True)
    return rec


for i in range(3):
    run("plain run %d" % i)
with torch.no_grad():
    for i in range(3):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        slam(gs.RGBDImages(rgb_d, depth.to(dev) if i == 0 else d.detach(), K_d, p.detach()))
        torch.cuda.synchronize()
        print("fused forward (no grad, inputs resident): %.2f ms" % ((time.perf_counter() - t0) * 1e3), flush=True)

from torch.profiler import ProfilerActivity, profile

with profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as prof:
    run("profiled")
print(prof.key_averages().table(sort_by="self_cpu_time_total", row_limit=30, max_name_column_width=60))
print(prof.key_averages().table(sort_by="self_cuda_time_total", row_limit=20, max_name_column_width=60))

# phases (adds synchronisation, so the sum exceeds the plain time)
wrap(icputils, "downsample_rgbdimages")
wrap(icputils, "downsample_pointclouds")
wrap(fusionutils, "find_active_map_points")
wrap(icp_mod, "_taped_icp")
wrap(icputils, "knn1")
wrap(fusionutils, "update_map_aggregate")
wrap(icpslam, "update_map_aggregate", "update_map_aggregate(icpslam)")
run("phased")
for k, v in sorted(acc.items(), key=lambda kv: -kv[1]):
    print("  %-36s %8.2f ms" % (k, v))
