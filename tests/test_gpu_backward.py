"""Backward of K1 (depth -> vertex / normal / global maps) against PyTorch autograd of a plain fp32 torch
implementation of the same op chain (gradslam/structures/rgbdimages.py:643-762)."""
import pytest
import torch

from gradslam_b200.synthetic import make_sequence as _make_sequence, punch_lattice_holes

pytestmark = pytest.mark.gpu


def make_sequence(*args, **kw):
    """Inputs for checking gradient FORMULAS: sparse lattice holes instead of random ones, so that no pixel's normal is
    the normalised residue of a cancelling cross product (derivative ~1e7; both the kernels and the reference produce
    it, but no tolerance survives it).  Parity on the random-hole distribution is pinned by the golden fixtures
    (tests/golden/ref_grad.npz is recorded from the reference on random holes)."""
    kw.setdefault("hole_fraction", 0.0)
    rgb, depth, K, poses = _make_sequence(*args, **kw)
    return rgb, punch_lattice_holes(depth), K, poses
DEV = "cuda:0"


def _torch_maps(depth, K, poses):
    """Differentiable fp32 torch reference (einsum-free, same formulas).  depth (B,L,H,W,1)."""
    B, L, H, W, _ = depth.shape
    fx, fy, cx, cy = K[:, 0, 0, 0] + 1e-6, K[:, 0, 1, 1] + 1e-6, K[:, 0, 0, 2], K[:, 0, 1, 2]
    u = torch.arange(W, dtype=torch.float32, device=depth.device).view(1, 1, 1, W)
    v = torch.arange(H, dtype=torch.float32, device=depth.device).view(1, 1, H, 1)
    d = depth[..., 0]
    vf = (d > 0).float()
    x = ((u - cx.view(B, 1, 1, 1)) / fx.view(B, 1, 1, 1)) * d * vf
    y = ((v - cy.view(B, 1, 1, 1)) / fy.view(B, 1, 1, 1)) * d * vf
    vert = torch.stack([x.expand(B, L, H, W), y.expand(B, L, H, W), d * vf], -1)
    dh = torch.zeros_like(vert)
    dv = torch.zeros_like(vert)
    dh[..., :, :-1, :] = vert[..., :, 1:, :] - vert[..., :, :-1, :]
    dv[..., :-1, :, :] = vert[..., 1:, :, :] - vert[..., :-1, :, :]
    dh = torch.cat([dh[..., :, :-1, :], dh[..., :, -2:-1, :]], dim=-2)
    dv = torch.cat([dv[..., :-1, :, :], dv[..., -2:-1, :, :]], dim=-3)
    c = torch.cross(dh, dv, dim=-1)
    nrm = torch.linalg.norm(c, dim=-1, keepdim=True)
    n = c / torch.where(nrm == 0, torch.ones_like(nrm), nrm) * vf.unsqueeze(-1)
    R, t = poses[..., :3, :3], poses[..., :3, 3]
    gv = (torch.einsum("blij,blhwj->blhwi", R, vert) + t.view(B, L, 1, 1, 3)) * vf.unsqueeze(-1)
    gn = torch.einsum("blij,blhwj->blhwi", R, n)
    return vert, n, gv, gn


@pytest.mark.parametrize("shape", [(2, 2, 24, 40), (1, 1, 17, 23)])
def test_backproject_backward_matches_autograd(shape):
    import gradslam_b200 as gs

    B, L, H, W = shape
    rgb, depth, K, poses = make_sequence(B, L, H, W, seed=21)
    g = torch.Generator().manual_seed(3)
    ups = [torch.randn(B, L, H, W, 3, generator=g).to(DEV) for _ in range(4)]
    # engine
    d1 = depth.to(DEV).requires_grad_(True)
    p1 = poses.to(DEV).requires_grad_(True)
    fr = gs.RGBDImages(rgb.to(DEV), d1, K.to(DEV), p1)
    outs = (fr.vertex_map, fr.normal_map, fr.global_vertex_map, fr.global_normal_map)
    loss = sum((o * w).sum() for o, w in zip(outs, ups))
    loss.backward()
    # torch reference
    d2 = depth.to(DEV).requires_grad_(True)
    p2 = poses.to(DEV).requires_grad_(True)
    refs = _torch_maps(d2, K.to(DEV), p2)
    for o, r in zip(outs, refs):
        torch.testing.assert_close(o.detach(), r.detach(), rtol=1e-4, atol=1e-5)
    sum((o * w).sum() for o, w in zip(refs, ups)).backward()
    scale = d2.grad.abs().max().item()
    torch.testing.assert_close(d1.grad, d2.grad, rtol=1e-3, atol=1e-4 * scale)
    pscale = p2.grad.abs().max().item()
    torch.testing.assert_close(p1.grad[..., :3, :], p2.grad[..., :3, :], rtol=1e-3, atol=1e-4 * pscale)
    assert p1.grad[..., 3, :].abs().max() == 0


def test_backward_only_global_maps_and_no_pose_grad():
    import gradslam_b200 as gs

    rgb, depth, K, poses = make_sequence(1, 2, 20, 28, seed=22)
    d1 = depth.to(DEV).requires_grad_(True)
    fr = gs.RGBDImages(rgb.to(DEV), d1, K.to(DEV), poses.to(DEV))
    w = torch.randn(1, 2, 20, 28, 3, device=DEV)
    (fr.global_vertex_map * w).sum().backward()
    d2 = depth.to(DEV).requires_grad_(True)
    refs = _torch_maps(d2, K.to(DEV), poses.to(DEV))
    (refs[2] * w).sum().backward()
    torch.testing.assert_close(d1.grad, d2.grad, rtol=1e-3, atol=1e-5)


def test_gradicp_function_gradients_match_oracle_autograd():
    """point_to_plane_gradICP in differentiable mode (CUDA 1-NN + taped algebra): d(T)/d(src) and
    d(T)/d(initial_transform) equal the gradients PyTorch's tape gives for the oracle restatement of the reference
    (icputils.py:370-545)."""
    import gsx_oracle as oracle
    from gradslam_b200.odometry import icputils

    rgb, depth, K, poses = make_sequence(1, 1, 40, 56, seed=31, hole_fraction=0.0, yaw0=0.6)
    m = oracle.frame_maps(depth, K, poses)
    tgt = m["gvertex"][0, 0].reshape(-1, 3).contiguous()
    tgt_n = m["gnormal"][0, 0].reshape(-1, 3).contiguous()
    T_true = oracle.se3_exp(torch.tensor([0.01, -0.005, 0.008, 0.01, -0.01, 0.005]))
    src0 = oracle.rigid_apply(T_true, tgt)
    w = torch.randn(4, 4, generator=torch.Generator().manual_seed(1))
    # oracle (CPU autograd)
    s_ref, t_ref = src0.clone().requires_grad_(True), torch.eye(4).requires_grad_(True)
    T_ref, _ = oracle.point_to_plane_gradicp(s_ref, tgt, tgt_n, t_ref, numiters=4)
    (T_ref * w).sum().backward()
    # engine, differentiable mode
    s_gpu, t_gpu = src0.clone().to(DEV).requires_grad_(True), torch.eye(4, device=DEV).requires_grad_(True)
    T_gpu, _ = icputils.point_to_plane_gradICP(s_gpu[None], tgt[None].to(DEV), tgt_n[None].to(DEV), t_gpu, numiters=4)
    (T_gpu * w.to(DEV)).sum().backward()
    torch.testing.assert_close(T_gpu.detach().cpu(), T_ref.detach(), rtol=0, atol=1e-4)
    for got, want in ((s_gpu.grad, s_ref.grad), (t_gpu.grad, t_ref.grad)):
        scale = want.abs().max().item()
        torch.testing.assert_close(got.cpu(), want, rtol=2e-2, atol=2e-3 * scale)
    # the fused (non-differentiable) loop gives the same forward value
    T_fused, _ = icputils.point_to_plane_gradICP(src0[None].to(DEV), tgt[None].to(DEV), tgt_n[None].to(DEV),
                                                 torch.eye(4, device=DEV), numiters=4)
    torch.testing.assert_close(T_fused.cpu(), T_gpu.detach().cpu(), rtol=0, atol=1e-4)


def test_icpslam_pose_gradient_wrt_live_depth():
    """Config-3 style check at small size: ICPSLAM(odom='gradicp'), L=2; gradient of the recovered pose of frame 1
    w.r.t. the depth of frame 1 (through the K1 backward kernel and the taped gradLM) vs the oracle's autograd."""
    import gradslam_b200 as gs
    import gsx_oracle as oracle

    B, L, H, W = 1, 2, 32, 40
    rgb, depth, K, poses = make_sequence(B, L, H, W, seed=33, yaw0=0.6)
    w = torch.randn(4, 4, generator=torch.Generator().manual_seed(2))
    d_ref = depth.clone().requires_grad_(True)
    ref = oracle.run_slam(rgb, d_ref, K, poses, mode="aggregate", odom="gradicp", numiters=3, dsratio=2)
    (ref.poses[0, 1] * w).sum().backward()
    d_gpu = depth.clone().to(DEV).requires_grad_(True)
    slam = gs.ICPSLAM(odom="gradicp", numiters=3, dsratio=2, device=DEV)
    pc, rec = slam(gs.RGBDImages(rgb.to(DEV), d_gpu, K.to(DEV), poses.to(DEV)))
    torch.testing.assert_close(rec.detach().cpu(), ref.poses.detach(), rtol=0, atol=1e-4)
    (rec[0, 1] * w.to(DEV)).sum().backward()
    # frame 1 (the live frame) AND frame 0 (whose pixels became the map the ICP aligns to)
    for s in (1, 0):
        g_ref, g_gpu = d_ref.grad[:, s], d_gpu.grad[:, s].cpu()
        assert torch.isfinite(g_gpu).all() and g_ref.abs().max() > 0
        scale = g_ref.abs().max().item()
        torch.testing.assert_close(g_gpu, g_ref, rtol=5e-2, atol=5e-3 * scale)


@pytest.mark.parametrize("B,L", [(1, 2), (2, 3)])
def test_pointfusion_map_gradients_match_oracle_autograd(B, L):
    """PointFusion(odom='gt') in differentiable mode: d(fused map)/d(depth, colours) through the K1 backward kernel and
    the K4 backward kernel (gsx_fusion_merge_append_bwd), against PyTorch autograd of the oracle restatement
    (fusionutils.py:580-722).  L=3 chains a merge into rows that were themselves merged one frame earlier."""
    import gradslam_b200 as gs
    import gsx_oracle as oracle

    H, W = 24, 32
    rgb, depth, K, poses = make_sequence(B, L, H, W, seed=41, yaw0=0.6)
    d_ref, c_ref = depth.clone().requires_grad_(True), rgb.clone().requires_grad_(True)
    ref = oracle.run_slam(c_ref, d_ref, K, poses, odom="gt")
    g = torch.Generator().manual_seed(5)
    counts = ref.map.counts()
    # (normals are left out of the loss: the oracle's autograd of |cross| is NaN at zero-length normals; the normal
    # channel of the K4 backward is covered by test_merge_append_op_gradients_wrt_previous_map, K1's by the tests above)
    ws = [[torch.randn(n, c, generator=g) for c in (3, 3, 1)] for n in counts]
    loss = 0
    for b in range(B):
        for t, w in zip((ref.map.points[b], ref.map.colors[b], ref.map.ccounts[b]), ws[b]):
            loss = loss + (t * w).sum()
    loss.backward()

    d_gpu, c_gpu = depth.clone().to(DEV).requires_grad_(True), rgb.clone().to(DEV).requires_grad_(True)
    slam = gs.PointFusion(odom="gt", device=DEV)
    pc, _ = slam(gs.RGBDImages(c_gpu, d_gpu, K.to(DEV), poses.to(DEV)))
    assert pc.num_points_per_pointcloud.tolist() == counts
    loss = 0
    for b in range(B):
        torch.testing.assert_close(pc.points_list[b].detach().cpu(), ref.map.points[b].detach(), rtol=1e-5, atol=1e-6)
        for t, w in zip((pc.points_list[b], pc.colors_list[b], pc.features_list[b]), ws[b]):
            loss = loss + (t * w.to(DEV)).sum()
    loss.backward()
    for got, want in ((d_gpu.grad.cpu(), d_ref.grad), (c_gpu.grad.cpu(), c_ref.grad)):
        assert torch.isfinite(got).all()
        scale = want.abs().max().item()
        torch.testing.assert_close(got, want, rtol=1e-3, atol=1e-4 * scale)
    # the same call without gradients takes the fused in-place kernels and gives the same map, bit for bit
    with torch.no_grad():
        pc2, _ = slam(gs.RGBDImages(rgb.to(DEV), depth.to(DEV), K.to(DEV), poses.to(DEV)))
    assert pc2.num_points_per_pointcloud.tolist() == counts
    for b in range(B):
        assert torch.equal(pc2.points_list[b], pc.points_list[b].detach())
        assert torch.equal(pc2.normals_list[b], pc.normals_list[b].detach())
        assert torch.equal(pc2.colors_list[b], pc.colors_list[b].detach())
        assert torch.equal(pc2.features_list[b], pc.features_list[b].detach())


def test_merge_append_op_gradients_wrt_previous_map():
    """update_map_fusion with a map that requires grad: d(updated map)/d(previous map rows) through
    gsx_fusion_merge_append_bwd (matched rows are scaled by c/(c+alpha), their confidence collects the quotient-rule
    terms, untouched rows pass through), against float64 autograd of the same formulas on the kernel's association."""
    import gradslam_b200 as gs
    from gradslam_b200.slam import fusionutils as fu

    B, H, W = 2, 20, 28
    rgb, depth, K, poses = make_sequence(B, 2, H, W, seed=43, yaw0=0.6)
    frames = gs.RGBDImages(rgb.to(DEV), depth.to(DEV), K.to(DEV), poses.to(DEV))
    with torch.no_grad():
        base = fu.update_map_fusion(gs.Pointclouds(device=DEV), frames[:, 0], 0.05, 0.94, 0.6)
        table = fu.find_correspondences(base, frames[:, 1], 0.05, 0.94)
    assert table.shape[0] > 0
    n0 = base.num_points_per_pointcloud.tolist()
    leaves = {k: getattr(base, k + "_padded").clone().requires_grad_(True)
              for k in ("points", "normals", "colors", "features")}
    pc = gs.Pointclouds(leaves["points"], leaves["normals"], leaves["colors"], leaves["features"])
    pc._set_counts(n0)
    out = fu.update_map_fusion(pc, frames[:, 1], 0.05, 0.94, 0.6)
    n1 = out.num_points_per_pointcloud.tolist()
    g = torch.Generator().manual_seed(3)
    wts = {k: torch.randn(B, max(n1), c, generator=g).to(DEV) for k, c in (("points", 3), ("normals", 3), ("colors", 3),
                                                                              ("features", 1))}
    mask = out.nonpad_mask.unsqueeze(-1)
    sum((getattr(out, k + "_padded") * wts[k] * mask).sum() for k in wts).backward()

    # float64 reference on the same association (fusionutils.py:654-699)
    f1 = frames[:, 1]
    ref = {k: v.detach().double().requires_grad_(True) for k, v in leaves.items()}
    b, n, h, w = table.unbind(1)
    alpha = fu.get_alpha(f1.vertex_map[:, 0].double(), 0.6, dim=-1, keepdim=True)[b, h, w]
    cc = ref["features"][b, n]
    tot = cc + alpha
    new = {}
    for k, fmap in (("points", f1.global_vertex_map), ("normals", f1.global_normal_map), ("colors", f1.rgb_image)):
        new[k] = ref[k].index_put((b, n), (cc * ref[k][b, n] + alpha * fmap[:, 0].double()[b, h, w]) / tot)
    new["features"] = ref["features"].index_put((b, n), tot)
    live = (torch.arange(max(n0), device=DEV).view(1, -1) < torch.tensor(n0, device=DEV).view(-1, 1)).unsqueeze(-1)
    sum((new[k] * wts[k][:, :max(n0)].double() * live).sum() for k in new).backward()
    for k in leaves:
        got, want = leaves[k].grad.double() * live, ref[k].grad
        torch.testing.assert_close(got, want, rtol=1e-4, atol=1e-5 * want.abs().max().item())


def _lm_reference_functions():
    import importlib.util
    import os
    spec = importlib.util.spec_from_file_location(
        "icp_diff_ref", os.path.join(os.path.dirname(os.path.abspath(__file__)), "test_icp_diff_host.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def test_solve_update_transform_ops_forward_and_backward():
    """K7 ops on the device (gsx_icp_solve_*, gsx_icp_update_*, gsx_rigid_transform_*) against float64 autograd of the
    reference formulas (solve_linear_system icputils.py:22-90, se3_exp se3utils.py:77-115, gates icputils.py:519-543,
    transform_pointcloud geometryutils.py:737-794)."""
    from gradslam_b200.odometry import icputils as iu
    refm = _lm_reference_functions()
    g = torch.Generator().manual_seed(11)
    A = torch.randn(300, 6, dtype=torch.float64, generator=g)
    bb = torch.randn(300, dtype=torch.float64, generator=g) * 0.05
    M = A.t() @ A
    tri = torch.triu_indices(6, 6)
    sums64 = torch.cat([M[tri[0], tri[1]], A.t() @ bb, (bb * bb).sum().view(1)])
    damp64 = torch.tensor([1e-3], dtype=torch.float64)
    wo = torch.randn(22, dtype=torch.float64, generator=g)
    # solve
    s_ref, d_ref = sums64.clone().requires_grad_(True), damp64.clone().requires_grad_(True)
    o_ref = refm._solve(torch.cat([s_ref, d_ref]))
    (o_ref * wo).sum().backward()
    s_gpu, d_gpu = sums64.float().to(DEV).requires_grad_(True), damp64.float().to(DEV).requires_grad_(True)
    xi, dT = iu._SolveFn.apply(s_gpu[None], d_gpu)  # a batch of one problem
    torch.testing.assert_close(torch.cat([xi[0], dT.reshape(-1)]).detach().cpu().double(), o_ref.detach(), rtol=0, atol=2e-6)
    ((xi * wo[:6].float().to(DEV)).sum() + (dT.reshape(-1) * wo[6:].float().to(DEV)).sum()).backward()
    for got, want in ((s_gpu.grad, s_ref.grad), (d_gpu.grad, d_ref.grad)):
        torch.testing.assert_close(got.cpu().double(), want, rtol=1e-3, atol=2e-4 * s_ref.grad.abs().max().item())
    # update, both modes and both branches
    for mode, err, nerr in ((1, 0.5, 0.3), (1, 0.3, 0.5), (0, 0.5, 0.3), (0, 0.3, 0.5)):
        xi64 = torch.randn(6, dtype=torch.float64, generator=g) * 0.05
        T64 = refm._se3_exp(torch.randn(6, dtype=torch.float64, generator=g) * 0.3)
        inp = torch.cat([xi64, torch.tensor([err, nerr, 1e-3], dtype=torch.float64), T64.reshape(-1)]).requires_grad_(True)
        wu = torch.randn(33, dtype=torch.float64, generator=g)
        o_ref = refm._update(inp, mode, 2.0, 1.0, 1.0, 200.0)
        (o_ref * wu).sum().backward()
        leaf = [t.float().to(DEV).requires_grad_(True) for t in (xi64[None], torch.tensor([err]), torch.tensor([nerr]),
                                                                  torch.tensor([1e-3]), T64[None])]
        dmp, dTa, Tn = iu._UpdateFn.apply(*leaf, mode, 2.0, 1.0, 1.0, 200.0)
        got = torch.cat([dmp.reshape(-1), dTa.reshape(-1), Tn.reshape(-1)])
        torch.testing.assert_close(got.detach().cpu().double(), o_ref.detach(), rtol=0, atol=2e-6)
        (got * wu.float().to(DEV)).sum().backward()
        g_got = torch.cat([t.grad.reshape(-1) for t in leaf]).cpu().double()
        torch.testing.assert_close(g_got, inp.grad, rtol=1e-4, atol=2e-5)
    # rigid transform
    P64 = torch.randn(1000, 3, dtype=torch.float64, generator=g)
    T64 = refm._se3_exp(torch.randn(6, dtype=torch.float64, generator=g) * 0.5)
    wp = torch.randn(1000, 3, dtype=torch.float64, generator=g)
    p_ref, t_ref = P64.clone().requires_grad_(True), T64.clone().requires_grad_(True)
    ((p_ref @ t_ref[:3, :3].t() + t_ref[:3, 3]) * wp).sum().backward()
    p_gpu, t_gpu = P64[None].float().to(DEV).requires_grad_(True), T64[None].float().to(DEV).requires_grad_(True)
    out = iu._RigidTransformFn.apply(p_gpu, t_gpu, torch.tensor([1000], dtype=torch.int32, device=DEV))
    torch.testing.assert_close(out[0].detach().cpu().double(), (P64 @ T64[:3, :3].t() + T64[:3, 3]), rtol=0, atol=1e-5)
    (out[0] * wp.float().to(DEV)).sum().backward()
    torch.testing.assert_close(p_gpu.grad[0].cpu().double(), p_ref.grad, rtol=1e-4, atol=1e-5)
    torch.testing.assert_close(t_gpu.grad[0].cpu().double(), t_ref.grad, rtol=1e-4, atol=1e-3)


def test_icp_lm_function_gradients_match_oracle_autograd():
    """point_to_plane_ICP (LM accept / reject, icputils.py:235-367) in differentiable mode against the oracle's tape."""
    import gsx_oracle as oracle
    from gradslam_b200.odometry.icputils import point_to_plane_ICP

    rgb, depth, K, poses = make_sequence(1, 1, 40, 56, seed=29, hole_fraction=0.0, yaw0=0.6)
    m = oracle.frame_maps(depth, K, poses)
    tgt = m["gvertex"][0, 0].reshape(-1, 3).contiguous()
    tgt_n = m["gnormal"][0, 0].reshape(-1, 3).contiguous()
    T_true = oracle.se3_exp(torch.tensor([0.01, -0.005, 0.008, 0.01, -0.01, 0.005]))
    src0 = oracle.rigid_apply(T_true, tgt)
    s_ref = src0.clone().requires_grad_(True)
    T_ref, _ = oracle.point_to_plane_icp(s_ref, tgt, tgt_n, torch.eye(4), numiters=4)
    wT = torch.randn(4, 4, generator=torch.Generator().manual_seed(2))
    (T_ref * wT).sum().backward()
    s_gpu = src0.clone().to(DEV).requires_grad_(True)
    T_gpu, _ = point_to_plane_ICP(s_gpu.unsqueeze(0), tgt.to(DEV).unsqueeze(0), tgt_n.to(DEV).unsqueeze(0),
                                  torch.eye(4, device=DEV), numiters=4)
    torch.testing.assert_close(T_gpu.detach().cpu(), T_ref.detach(), rtol=0, atol=1e-4)
    (T_gpu * wT.to(DEV)).sum().backward()
    scale = s_ref.grad.abs().max().item()
    torch.testing.assert_close(s_gpu.grad.cpu(), s_ref.grad, rtol=2e-2, atol=2e-3 * scale)


def test_normal_equation_op_forward_and_backward():
    """K6 as an op: the 28 sums and their hand-written backward against a plain torch construction of A, b
    (icputils.py:210-230) and PyTorch autograd, including filtered rows (idx = -1) and shared targets."""
    from gradslam_b200.odometry.icputils import _NormalEqFn

    g = torch.Generator().manual_seed(7)
    ns, nt = 700, 300
    src = torch.randn(ns, 3, generator=g)
    tgt = torch.randn(nt, 3, generator=g)
    tn = torch.nn.functional.normalize(torch.randn(nt, 3, generator=g), dim=1)
    idx = torch.randint(0, nt, (ns,), generator=g)
    idx[::7] = -1
    w = torch.randn(28, generator=g)

    def ref(s, p, n):
        keep = idx >= 0
        s, pp, nn = s[keep], p[idx[keep]], n[idx[keep]]
        sx, sy, sz = s[:, 0:1], s[:, 1:2], s[:, 2:3]
        nx, ny, nz = nn[:, 0:1], nn[:, 1:2], nn[:, 2:3]
        A = torch.cat([nx, ny, nz, nz * sy - ny * sz, nx * sz - nz * sx, ny * sx - nx * sy], 1)
        b = nx * (pp[:, 0:1] - sx) + ny * (pp[:, 1:2] - sy) + nz * (pp[:, 2:3] - sz)
        AtA, Atb = A.t() @ A, A.t() @ b
        iu = torch.triu_indices(6, 6)
        return torch.cat([AtA[iu[0], iu[1]], Atb[:, 0], (b * b).sum().view(1)])

    a = [t.clone().double().requires_grad_(True) for t in (src, tgt, tn)]
    want = ref(*a)
    (want * w.double()).sum().backward()
    b_ = [t[None].clone().to(DEV).requires_grad_(True) for t in (src, tgt, tn)]  # a batch of one cloud pair
    got = _NormalEqFn.apply(b_[0], b_[1], b_[2], idx[None].to(DEV), torch.tensor([ns], dtype=torch.int32, device=DEV))
    torch.testing.assert_close(got[0].cpu().double(), want.detach(), rtol=1e-4, atol=1e-3)
    (got[0] * w.to(DEV)).sum().backward()
    for x, y in zip(b_, a):
        scale = y.grad.abs().max().item()
        torch.testing.assert_close(x.grad[0].cpu().double(), y.grad, rtol=1e-3, atol=1e-4 * scale)


def test_batched_differentiable_icp_equals_single_element_runs():
    """The differentiable op chain on a padded batch (one set of autograd ops for all elements, ragged sizes) against
    each element alone through the public point_to_plane_gradICP: transforms bit-identical, association identical,
    gradients w.r.t. the source clouds, the target clouds and the target normals equal to float32 rounding, so an
    element's result depends neither on the padding nor on the other elements; and the providers use the chain
    (ICPSLAM-style call with B=3)."""
    import gradslam_b200 as gs
    from gradslam_b200.odometry import icputils as iu
    from gradslam_b200.odometry.gradicp import GradICPOdometryProvider

    g = torch.Generator().manual_seed(5)
    Bn, sizes_s, sizes_t = 3, [700, 512, 655], [900, 1024, 640]
    Ns, Nt = max(sizes_s), max(sizes_t)
    rgb, depth, K, poses = make_sequence(1, 1, 40, 56, seed=7, hole_fraction=0.0, yaw0=0.6)
    fr = gs.RGBDImages(rgb.to(DEV), depth.to(DEV), K.to(DEV), poses.to(DEV))
    base_p = fr.global_vertex_map[0, 0].reshape(-1, 3)
    base_n = fr.global_normal_map[0, 0].reshape(-1, 3)
    T_true = [torch.tensor([[1, 0, 0, 0.01 * (b + 1)], [0, 1, 0, -0.005], [0, 0, 1, 0.004 * b], [0, 0, 0, 1.0]],
                           device=DEV) for b in range(Bn)]
    src = torch.zeros(Bn, Ns, 3, device=DEV)
    tgt = torch.zeros(Bn, Nt, 3, device=DEV)
    tgt_n = torch.zeros(Bn, Nt, 3, device=DEV)
    for b in range(Bn):
        pick_t = torch.randperm(base_p.shape[0], generator=g)[: sizes_t[b]].to(DEV)
        pick_s = torch.randperm(base_p.shape[0], generator=g)[: sizes_s[b]].to(DEV)
        tgt[b, : sizes_t[b]] = base_p[pick_t]
        tgt_n[b, : sizes_t[b]] = base_n[pick_t]
        src[b, : sizes_s[b]] = base_p[pick_s] @ T_true[b][:3, :3].t() + T_true[b][:3, 3]
    cs = torch.tensor(sizes_s, dtype=torch.int32, device=DEV)
    ct = torch.tensor(sizes_t, dtype=torch.int32, device=DEV)
    w = torch.randn(Bn, 4, 4, generator=g).to(DEV)
    leaves = [t.clone().requires_grad_(True) for t in (src, tgt, tgt_n)]
    T_b, idx_b = iu._taped_icp(leaves[0], cs, leaves[1], leaves[2], ct, None, 1, 4, 1e-8, None)
    (T_b * w).sum().backward()
    for b in range(Bn):
        l1 = [src[b:b + 1, : sizes_s[b]].clone().requires_grad_(True), tgt[b:b + 1, : sizes_t[b]].clone().requires_grad_(True),
              tgt_n[b:b + 1, : sizes_t[b]].clone().requires_grad_(True)]
        T_1, idx_1 = iu.point_to_plane_gradICP(l1[0], l1[1], l1[2], numiters=4, damp=1e-8)
        (T_1 * w[b]).sum().backward()
        assert torch.equal(T_1, T_b[b])
        assert torch.equal(idx_1, idx_b[b, : sizes_s[b]][idx_b[b, : sizes_s[b]] >= 0])
        for got, want, n in ((leaves[0].grad[b], l1[0].grad[0], sizes_s[b]), (leaves[1].grad[b], l1[1].grad[0], sizes_t[b]),
                             (leaves[2].grad[b], l1[2].grad[0], sizes_t[b])):
            scale = want.abs().max().item()
            torch.testing.assert_close(got[:n], want, rtol=1e-4, atol=1e-5 * scale)
            assert got[n:].numel() == 0 or got[n:].abs().max() == 0  # padding rows carry no gradient
    # the providers run the batched chain when a gradient is requested
    maps = gs.Pointclouds([tgt[b, : sizes_t[b]] for b in range(Bn)], [tgt_n[b, : sizes_t[b]] for b in range(Bn)])
    s_req = [src[b, : sizes_s[b]].clone().requires_grad_(True) for b in range(Bn)]
    out = GradICPOdometryProvider(numiters=4).provide(maps, gs.Pointclouds(s_req))
    assert out.shape == (Bn, 1, 4, 4) and torch.equal(out[:, 0], T_b.detach())
    (out[:, 0] * w).sum().backward()
    for b in range(Bn):
        scale = leaves[0].grad[b].abs().max().item()
        torch.testing.assert_close(s_req[b].grad, leaves[0].grad[b, : sizes_s[b]], rtol=1e-4, atol=1e-5 * scale)
