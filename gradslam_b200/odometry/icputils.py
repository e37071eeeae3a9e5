"""Point-to-plane ICP building blocks.

Host-side mirror of gradslam/odometry/icputils.py (same names, arguments, errors).  The association
(`chamferdist.knn_points` in the reference), the row build, the normal-equation reduction, the damped solve,
the SE(3) exponential and the LM / gradLM update all run in csrc/gsx_icp.cu; nothing here loops over points.
"""
from typing import Optional, Union

import torch

from .. import _C
from ..structures.pointclouds import Pointclouds
from ..structures.rgbdimages import RGBDImages, _frame_base

__all__ = ["solve_linear_system", "gauss_newton_solve", "point_to_plane_ICP", "point_to_plane_gradICP",
           "downsample_pointclouds", "downsample_rgbdimages"]


def _need_tensor(x, name):
    if not torch.is_tensor(x):
        raise TypeError("Expected {} to be of type torch.Tensor. Got {}.".format(name, type(x)))


def solve_linear_system(A: torch.Tensor, b: torch.Tensor, damp: Union[float, torch.Tensor] = 1e-8):
    """x = (A^T A + damp I)^-1 A^T b — the normal equations, not the system itself (icputils.py:22-90)."""
    _need_tensor(A, "A")
    _need_tensor(b, "b")
    if not (isinstance(damp, float) or torch.is_tensor(damp)):
        raise TypeError("Expected damp to be of type float or torch.Tensor. Got {0}.".format(type(damp)))
    if torch.is_tensor(damp) and damp.ndim != 0:
        raise ValueError("Expected torch.Tensor damp to have ndim=0 (scalar). Got {0}.".format(damp.ndim))
    if A.ndim != 2:
        raise ValueError("A should have ndim=2, but had ndim={}".format(A.ndim))
    if b.ndim != 2:
        raise ValueError("b should have ndim=2, but had ndim={}".format(b.ndim))
    if b.shape[1] != 1:
        raise ValueError("b.shape[1] should 1, but was {0}".format(b.shape[1]))
    if A.shape[0] != b.shape[0]:
        raise ValueError("A.shape[0] and b.shape[0] should be equal ({0} != {1})".format(A.shape[0], b.shape[0]))
    damp = damp if torch.is_tensor(damp) else torch.tensor(damp, dtype=A.dtype, device=A.device)
    At = A.transpose(0, 1)
    normal = At @ A + torch.eye(A.shape[1], dtype=A.dtype, device=A.device) * damp
    return torch.inverse(normal) @ (At @ b)


def _check_clouds(src_pc, tgt_pc, tgt_normals, dist_thresh):
    _need_tensor(src_pc, "src_pc")
    _need_tensor(tgt_pc, "tgt_pc")
    _need_tensor(tgt_normals, "tgt_normals")
    if not (isinstance(dist_thresh, (float, int)) or dist_thresh is None):
        raise TypeError("Expected dist_thresh to be of type float or int. Got {0}.".format(type(dist_thresh)))
    for name, t in (("src_pc", src_pc), ("tgt_pc", tgt_pc), ("tgt_normals", tgt_normals)):
        if t.ndim != 3:
            raise ValueError("{} should have ndim=3, but had ndim={}".format(name, t.ndim))
    for name, t in (("src_pc", src_pc), ("tgt_pc", tgt_pc), ("tgt_normals", tgt_normals)):
        if t.shape[0] != 1:
            raise ValueError("{}.shape[0] should be 1, but was {} instead".format(name, t.shape[0]))
    if tgt_pc.shape[1] != tgt_normals.shape[1]:
        raise ValueError("tgt_pc.shape[1] and tgt_normals.shape[1] must be equal. Got {0}!={1}".format(
            tgt_pc.shape[1], tgt_normals.shape[1]))
    for name, t in (("src_pc", src_pc), ("tgt_pc", tgt_pc), ("tgt_normals", tgt_normals)):
        if t.shape[2] != 3:
            raise ValueError("{}.shape[2] should be 3, but was {} instead".format(name, t.shape[2]))


def _counts(n, B, device):
    return torch.full((B,), n, dtype=torch.int32, device=device)


def knn1(src: torch.Tensor, tgt: torch.Tensor, src_counts=None, tgt_counts=None, target_cache: Optional[dict] = None):
    """Exact 1-NN of every row of src (B,Ns,3) in tgt (B,Nt,3) (padded clouds: optional int32 sizes (B,); rows beyond a
    source size get idx -1).  Returns (squared distances (B,Ns), idx int64 (B,Ns)); ties resolve to the lowest target
    index.  CUDA kernel k_icp_knn_linearize.
    target_cache: a dict the caller keeps while it queries the SAME, unmodified target repeatedly (the ICP loop): the
    search grid of the target is then built by the first call only."""
    _C.require_cuda(src, "src")
    _C.require_cuda(tgt, "tgt")
    src = src.contiguous()
    B, Ns, _ = src.shape
    Nt = tgt.shape[1]
    key = (tgt.data_ptr(), tuple(tgt.shape), tuple(tgt.stride()), tgt._version, Ns)
    hit = target_cache is not None and target_cache.get("key") == key
    if hit:
        tgt_c, scratch, nt_t = target_cache["tgt"], target_cache["scratch"], target_cache["nt"]
    else:
        tgt_c = tgt.contiguous()
        scratch = torch.empty(_C.lib().gsx_knn1_scratch_bytes(B, Ns, Nt), dtype=torch.uint8, device=src.device)
        nt_t = _counts(Nt, B, src.device) if tgt_counts is None else tgt_counts
        if target_cache is not None:
            target_cache.update(key=key, tgt=tgt_c, scratch=scratch, nt=nt_t)
    # (the kernel writes the rows below each source size; the padding rows keep -1 / inf)
    idx = torch.full((B, Ns), -1, dtype=torch.int64, device=src.device)
    d2 = torch.full((B, Ns), float("inf"), dtype=torch.float32, device=src.device)
    ns_t = _counts(Ns, B, src.device) if src_counts is None else src_counts  # (kept alive across the call)
    with torch.cuda.device(src.device):
        rc = _C.lib().gsx_knn1(_C.ptr(src), _C.ptr(ns_t), Ns, _C.ptr(tgt_c), _C.ptr(nt_t), Nt, B, _C.ptr(idx),
                               _C.ptr(d2), _C.ptr(scratch), scratch.numel(), 0 if hit else 1,
                               _C.stream_ptr(src.device))
    _C.check(rc, "gsx_knn1")
    return d2, idx


def gauss_newton_solve(src_pc: torch.Tensor, tgt_pc: torch.Tensor, tgt_normals: torch.Tensor,
                       dist_thresh: Union[float, int, None] = None):
    """Point-to-plane rows for one Gauss-Newton step: A (Nsf,6), b (Nsf,1), nn indices (Nsf,) (icputils.py:93-232).
    The association is the CUDA exact 1-NN; the row algebra below is differentiable torch (as in the reference)."""
    _check_clouds(src_pc, tgt_pc, tgt_normals, dist_thresh)
    src_pc, tgt_pc, tgt_normals = src_pc.contiguous(), tgt_pc.contiguous(), tgt_normals.contiguous()
    d2, idx = knn1(src_pc.detach(), tgt_pc.detach())
    keep = torch.ones_like(d2[0], dtype=torch.bool) if dist_thresh is None else d2[0] < dist_thresh
    idx = idx[0][keep]
    s = src_pc[0][keep]
    p = tgt_pc[0].index_select(0, idx)
    n = tgt_normals[0].index_select(0, idx)
    sx, sy, sz = s[:, 0:1], s[:, 1:2], s[:, 2:3]
    nx, ny, nz = n[:, 0:1], n[:, 1:2], n[:, 2:3]
    A = torch.cat([nx, ny, nz, nz * sy - ny * sz, nx * sz - nz * sx, ny * sx - nx * sy], 1)
    b = nx * (p[:, 0:1] - sx) + ny * (p[:, 1:2] - sy) + nz * (p[:, 2:3] - sz)
    return A, b, idx


def _check_icp_args(src_pc, tgt_pc, tgt_normals, initial_transform, numiters):
    _need_tensor(src_pc, "src_pc")
    _need_tensor(tgt_pc, "tgt_pc")
    _need_tensor(tgt_normals, "tgt_normals")
    if not (torch.is_tensor(initial_transform) or initial_transform is None):
        raise TypeError("Expected initial_transform to be of type torch.Tensor. Got {0}.".format(
            type(initial_transform)))
    if not isinstance(numiters, int):
        raise TypeError("Expected numiters to be of type int. Got {0}.".format(type(numiters)))
    if initial_transform is not None:
        if initial_transform.ndim != 2:
            raise ValueError("Expected initial_transform.ndim to be 2. Got {0}.".format(initial_transform.ndim))
        if not (initial_transform.shape[0] == 4 and initial_transform.shape[1] == 4):
            raise ValueError("Expected initial_transform.shape to be (4, 4). Got {0}.".format(initial_transform.shape))


def icp_align(src, src_counts, tgt, tgt_normals, tgt_counts, T0, mode, numiters, damp, dist_thresh, lambda_max=2.0,
              B=1.0, B2=1.0, nu=200.0, want_idx=False):
    """Batched ICP (mode 0) / gradICP (mode 1) on padded clouds (Bn, N, 3) with int32 sizes.  One C call."""
    for name, t in (("src", src), ("tgt", tgt), ("tgt_normals", tgt_normals)):
        _C.require_cuda(t, name)
    Bn, Ns, _ = src.shape
    Nt = tgt.shape[1]
    dev = src.device
    out = torch.empty((Bn, 4, 4), dtype=torch.float32, device=dev)
    idx = torch.empty((Bn, Ns), dtype=torch.int64, device=dev) if want_idx else None
    lib = _C.lib()
    nbytes = lib.gsx_icp_align_scratch_bytes(Bn, Ns, Nt)
    scratch = torch.empty(nbytes, dtype=torch.uint8, device=dev)
    T0c = None if T0 is None else T0.to(dev).float().contiguous()
    with torch.cuda.device(dev):
        rc = lib.gsx_icp_align(
            _C.ptr(src.contiguous()), _C.ptr(src_counts), Ns, _C.ptr(tgt.contiguous()),
            _C.ptr(tgt_normals.contiguous()), _C.ptr(tgt_counts), Nt, Bn, _C.ptr(T0c), int(mode), int(numiters),
            float(damp), 0 if dist_thresh is None else 1, 0.0 if dist_thresh is None else float(dist_thresh),
            float(lambda_max), float(B), float(B2), float(nu), _C.ptr(out), _C.ptr(idx), _C.ptr(scratch), nbytes,
            _C.stream_ptr(dev))
    _C.check(rc, "gsx_icp_align")
    return out, idx


def _wants_grad(*tensors):
    return torch.is_grad_enabled() and any(torch.is_tensor(t) and t.requires_grad for t in tensors)


# The differentiable ICP loop is a chain of the autograd ops below on padded clouds (B, N, 3) with int32 sizes (B,):
# one chain records all batch elements (the reference's providers run one chain per element, odometry/icp.py:84-97), and
# a single cloud pair is a batch of one.  Padding rows contribute exact zeros to the fixed-order sums, so an element's
# values do not depend on the padding or on the other elements.
class _NormalEqFn(torch.autograd.Function):
    """(src (B,Ns,3), tgt (B,Nt,3), tgt_normals (B,Nt,3), nn_idx (B,Ns) int64, -1 = row unused, src sizes (B,) int32)
    -> the 28 sums (B,28) of the point-to-plane normal equations.  forward = gsx_icp_normal_eq_batched_fwd,
    backward = gsx_icp_normal_eq_batched_bwd (hand-written kernels; gradients w.r.t. src, tgt and tgt_normals)."""

    @staticmethod
    def forward(ctx, src, tgt, tgt_n, idx, src_counts):
        src_c, tgt_c, tn_c = (t.detach().contiguous().float() for t in (src, tgt, tgt_n))
        idx_c = idx.contiguous()
        _C.require_cuda(src_c, "src")
        Bn, Ns, _ = src_c.shape
        Nt, dev = tgt_c.shape[1], src_c.device
        sums = torch.empty((Bn, 28), dtype=torch.float32, device=dev)
        lib = _C.lib()
        nbytes = Bn * lib.gsx_icp_normal_eq_scratch_bytes(Ns)
        scratch = torch.empty(nbytes, dtype=torch.uint8, device=dev)
        with torch.cuda.device(dev):
            rc = lib.gsx_icp_normal_eq_batched_fwd(_C.ptr(src_c), _C.ptr(src_counts), Ns, _C.ptr(tgt_c), _C.ptr(tn_c), Nt,
                                                   Bn, _C.ptr(idx_c), _C.ptr(sums), _C.ptr(scratch), nbytes,
                                                   _C.stream_ptr(dev))
        _C.check(rc, "gsx_icp_normal_eq_batched_fwd")
        ctx.saved = (src_c, tgt_c, tn_c, idx_c, src_counts)
        return sums

    @staticmethod
    def backward(ctx, g):
        src_c, tgt_c, tn_c, idx_c, src_counts = ctx.saved
        Bn, Ns, _ = src_c.shape
        Nt, dev = tgt_c.shape[1], src_c.device
        g = g.contiguous().float()
        g_src = torch.empty_like(src_c)
        rows_p, rows_n = torch.empty_like(src_c), torch.empty_like(src_c)
        with torch.cuda.device(dev):
            rc = _C.lib().gsx_icp_normal_eq_batched_bwd(_C.ptr(src_c), _C.ptr(src_counts), Ns, _C.ptr(tgt_c),
                                                        _C.ptr(tn_c), Nt, Bn, _C.ptr(idx_c), _C.ptr(g), _C.ptr(g_src),
                                                        _C.ptr(rows_p), _C.ptr(rows_n), _C.stream_ptr(dev))
        _C.check(rc, "gsx_icp_normal_eq_batched_bwd")
        # rows with idx < 0 carry zero gradients; scatter the per-source-row target gradients with the association
        flat = (idx_c.clamp(min=0) + torch.arange(Bn, device=dev).view(Bn, 1) * Nt).view(-1)
        g_tgt = torch.zeros((Bn * Nt, 3), dtype=torch.float32, device=dev).index_add_(0, flat, rows_p.view(-1, 3))
        g_tn = torch.zeros((Bn * Nt, 3), dtype=torch.float32, device=dev).index_add_(0, flat, rows_n.view(-1, 3))
        return g_src, g_tgt.view(Bn, Nt, 3), g_tn.view(Bn, Nt, 3), None, None


class _SolveFn(torch.autograd.Function):
    """(sums (B,28), damp (B,)) -> (xi (B,6), dT (B,4,4)): damped 6x6 solve + se3_exp in one kernel (K7a).
    forward = gsx_icp_solve_fwd, backward = gsx_icp_solve_bwd (dual numbers, one lane per input)."""

    @staticmethod
    def forward(ctx, sums, damp):
        s, d = sums.detach().contiguous().float(), damp.detach().contiguous().float()
        _C.require_cuda(s, "sums")
        Bn, dev = s.shape[0], s.device
        xi = torch.empty((Bn, 6), dtype=torch.float32, device=dev)
        dT = torch.empty((Bn, 4, 4), dtype=torch.float32, device=dev)
        with torch.cuda.device(dev):
            rc = _C.lib().gsx_icp_solve_fwd(_C.ptr(s), _C.ptr(d), Bn, _C.ptr(xi), _C.ptr(dT), _C.stream_ptr(dev))
        _C.check(rc, "gsx_icp_solve_fwd")
        ctx.saved = (s, d)
        return xi, dT

    @staticmethod
    def backward(ctx, g_xi, g_dT):
        s, d = ctx.saved
        dev = s.device
        g_xi = None if g_xi is None else g_xi.contiguous().float()
        g_dT = None if g_dT is None else g_dT.contiguous().float()
        g_s, g_d = torch.empty_like(s), torch.empty_like(d)
        with torch.cuda.device(dev):
            rc = _C.lib().gsx_icp_solve_bwd(_C.ptr(s), _C.ptr(d), s.shape[0], _C.ptr(g_xi), _C.ptr(g_dT), _C.ptr(g_s),
                                            _C.ptr(g_d), _C.stream_ptr(dev))
        _C.check(rc, "gsx_icp_solve_bwd")
        return g_s, g_d


class _UpdateFn(torch.autograd.Function):
    """(xi (B,6), err (B,), new_err (B,), damp (B,), T (B,4,4)) -> (new damp, applied step (B,4,4), step @ T): LM
    accept / reject (mode 0) or the gradLM gates (mode 1), the applied se3_exp and the pose accumulation in one kernel
    (K7b).  forward = gsx_icp_update_fwd, backward = gsx_icp_update_bwd."""

    @staticmethod
    def forward(ctx, xi, err, new_err, damp, T, mode, lambda_max, B, B2, nu):
        dev = xi.device
        ins = [t.detach().contiguous().float() for t in (xi, err, new_err, damp, T)]
        _C.require_cuda(ins[0], "xi")
        Bn = ins[0].shape[0]
        damp_out = torch.empty(Bn, dtype=torch.float32, device=dev)
        dT = torch.empty((Bn, 4, 4), dtype=torch.float32, device=dev)
        Tn = torch.empty((Bn, 4, 4), dtype=torch.float32, device=dev)
        par = (int(mode), float(lambda_max), float(B), float(B2), float(nu))
        with torch.cuda.device(dev):
            rc = _C.lib().gsx_icp_update_fwd(*[_C.ptr(t) for t in ins], Bn, *par, _C.ptr(damp_out), _C.ptr(dT),
                                             _C.ptr(Tn), _C.stream_ptr(dev))
        _C.check(rc, "gsx_icp_update_fwd")
        ctx.saved = (ins, par)
        return damp_out, dT, Tn

    @staticmethod
    def backward(ctx, g_damp, g_dT, g_T):
        ins, par = ctx.saved
        dev = ins[0].device
        gs = [None if g is None else g.contiguous().float() for g in (g_damp, g_dT, g_T)]
        outs = [torch.empty_like(t) for t in ins]
        with torch.cuda.device(dev):
            rc = _C.lib().gsx_icp_update_bwd(*[_C.ptr(t) for t in ins], ins[0].shape[0], *par, *[_C.ptr(g) for g in gs],
                                             *[_C.ptr(o) for o in outs], _C.stream_ptr(dev))
        _C.check(rc, "gsx_icp_update_bwd")
        return tuple(outs) + (None,) * 5


class _RigidTransformFn(torch.autograd.Function):
    """(points (B,N,3), T (B,4,4), sizes (B,) int32) -> R p + t (transform_pointcloud, geometryutils.py:737-794), zero
    on padding rows.  forward = gsx_rigid_transform_batched_fwd, backward = gsx_rigid_transform_batched_bwd
    (deterministic reduction for d/dT)."""

    @staticmethod
    def forward(ctx, points, T, counts):
        p, Tc = points.detach().contiguous().float(), T.detach().contiguous().float()
        _C.require_cuda(p, "points")
        dev = p.device
        out = torch.empty_like(p)
        with torch.cuda.device(dev):
            rc = _C.lib().gsx_rigid_transform_batched_fwd(_C.ptr(p), _C.ptr(counts), p.shape[1], p.shape[0], _C.ptr(Tc),
                                                          _C.ptr(out), _C.stream_ptr(dev))
        _C.check(rc, "gsx_rigid_transform_batched_fwd")
        ctx.saved = (p, Tc, counts)
        return out

    @staticmethod
    def backward(ctx, g):
        p, Tc, counts = ctx.saved
        dev = p.device
        Bn, n = p.shape[0], p.shape[1]
        g = g.contiguous().float()
        g_p, g_T = torch.empty_like(p), torch.empty_like(Tc)
        lib = _C.lib()
        nbytes = Bn * lib.gsx_rigid_transform_bwd_scratch_bytes(n)
        scratch = torch.empty(nbytes, dtype=torch.uint8, device=dev)
        with torch.cuda.device(dev):
            rc = lib.gsx_rigid_transform_batched_bwd(_C.ptr(p), _C.ptr(counts), n, Bn, _C.ptr(Tc), _C.ptr(g), _C.ptr(g_p),
                                                     _C.ptr(g_T), _C.ptr(scratch), nbytes, _C.stream_ptr(dev))
        _C.check(rc, "gsx_rigid_transform_batched_bwd")
        return g_p, g_T, None


def _normal_equations(src, src_counts, tgt, tgt_n, tgt_counts, dist_thresh, target_cache=None):
    """Association (CUDA exact 1-NN, index-only) + the differentiable normal-equation op -> ((B,28) sums, idx)."""
    d2, idx = knn1(src.detach(), tgt.detach(), src_counts, tgt_counts, target_cache)
    if dist_thresh is not None:
        idx = torch.where(d2 < dist_thresh, idx, torch.full_like(idx, -1))
    return _NormalEqFn.apply(src, tgt, tgt_n, idx, src_counts), idx


def _taped_icp(src, src_counts, tgt, tgt_n, tgt_counts, T0, mode, numiters, damp, dist_thresh, lambda_max=2.0, B=1.0,
               B2=1.0, nu=200.0):
    """Differentiable ICP / gradICP, used when an input requires grad: the same loop as the fused kernel sequence, as a
    chain of autograd ops that each have a hand-written forward AND backward kernel - rigid transform
    (`_RigidTransformFn`), 1-NN association (index-only, no gradient, as in the reference), normal equations
    (`_NormalEqFn`), damped solve + se3_exp (`_SolveFn`), LM / gradLM update (`_UpdateFn`).  PyTorch only records the
    tape; no ATen arithmetic runs between the ops and there is no host synchronisation (icputils.py:235-545).
    src (Bn,Ns,3), tgt / tgt_n (Bn,Nt,3), int32 sizes (Bn,), T0 (1,4,4), (Bn,4,4) or None.  Returns (T (Bn,4,4), last nn
    idx (Bn,Ns), -1 = none); per element the poses are bit-identical to the fused no-grad loop."""
    dev = src.device
    Bn = src.shape[0]
    dampt = torch.full((Bn,), float(damp), dtype=torch.float32, device=dev)
    T = (torch.eye(4, dtype=torch.float32, device=dev).repeat(Bn, 1, 1) if T0 is None
         else T0.to(torch.float32).expand(Bn, 4, 4).contiguous())
    tgt, tgt_n = tgt.contiguous(), tgt_n.contiguous()  # once (strided views of packed map rows), not per iteration
    cur = _RigidTransformFn.apply(src, T, src_counts)
    idx = None
    grid = {}  # the target's search grid: built by the first of the 2 * numiters associations
    for _ in range(numiters):
        sums, idx = _normal_equations(cur, src_counts, tgt, tgt_n, tgt_counts, dist_thresh, grid)
        xi, dT = _SolveFn.apply(sums, dampt)
        one_step = _RigidTransformFn.apply(cur, dT, src_counts)
        sums_next, _ = _normal_equations(one_step, src_counts, tgt, tgt_n, tgt_counts, dist_thresh, grid)
        dampt, dT_applied, T = _UpdateFn.apply(xi, sums[:, 27], sums_next[:, 27], dampt, T, mode, lambda_max, B, B2, nu)
        cur = _RigidTransformFn.apply(cur, dT_applied, src_counts)
    return T, idx


def _single(src_pc, tgt_pc, tgt_normals, initial_transform, mode, numiters, damp, dist_thresh, **kw):
    """One cloud pair as a batch of one: the taped op chain when an input requires grad, else the fused loop."""
    dev = src_pc.device
    T0 = None if initial_transform is None else initial_transform.view(1, 4, 4)
    args = (src_pc.contiguous(), _counts(src_pc.shape[1], 1, dev), tgt_pc.contiguous(), tgt_normals.contiguous(),
            _counts(tgt_pc.shape[1], 1, dev), T0, mode, numiters, damp, dist_thresh)
    if _wants_grad(src_pc, tgt_pc, tgt_normals, initial_transform):
        T, idx = _taped_icp(*args, **kw)
    else:
        T, idx = icp_align(*args, want_idx=True, **kw)
    idx = idx[0]
    return T[0], idx[idx >= 0]


def point_to_plane_ICP(src_pc: torch.Tensor, tgt_pc: torch.Tensor, tgt_normals: torch.Tensor,
                       initial_transform: Optional[torch.Tensor] = None, numiters: int = 20, damp: float = 1e-8,
                       dist_thresh: Union[float, int, None] = None):
    """Rigid transform aligning src to tgt with point-to-plane LM (icputils.py:235-367).  Returns (T (4,4), nn idx)."""
    _check_icp_args(src_pc, tgt_pc, tgt_normals, initial_transform, numiters)
    return _single(src_pc, tgt_pc, tgt_normals, initial_transform, 0, numiters, damp, dist_thresh)


def point_to_plane_gradICP(src_pc: torch.Tensor, tgt_pc: torch.Tensor, tgt_normals: torch.Tensor,
                           initial_transform: Optional[torch.Tensor] = None, numiters: int = 20, damp: float = 1e-8,
                           dist_thresh: Union[float, int, None] = None, lambda_max: Union[float, int] = 2.0,
                           B: Union[float, int] = 1.0, B2: Union[float, int] = 1.0, nu: Union[float, int] = 200.0):
    """Same with the gradLM solver (icputils.py:370-545)."""
    _check_icp_args(src_pc, tgt_pc, tgt_normals, initial_transform, numiters)
    for name, v in (("lambda_max", lambda_max), ("B", B), ("B2", B2), ("nu", nu)):
        if not isinstance(v, (float, int)):
            raise TypeError("Expected {} to be of type float or int; got {}".format(name, type(v)))
    return _single(src_pc, tgt_pc, tgt_normals, initial_transform, 1, numiters, damp, dist_thresh,
                   lambda_max=lambda_max, B=B, B2=B2, nu=nu)


def downsample_pointclouds(pointclouds: Pointclouds, pc2im_bnhw: torch.Tensor, ds_ratio: int) -> Pointclouds:
    """Keeps the active map points whose pixel lies on the ds lattice (icputils.py:548-620)."""
    if not isinstance(pointclouds, Pointclouds):
        raise TypeError("Expected pointclouds to be of type gradslam.Pointclouds. Got {0}.".format(type(pointclouds)))
    if not torch.is_tensor(pc2im_bnhw):
        raise TypeError("Expected pc2im_bnhw to be of type torch.Tensor. Got {0}.".format(type(pc2im_bnhw)))
    if not isinstance(ds_ratio, int):
        raise TypeError("Expected ds_ratio to be of type int. Got {0}.".format(type(ds_ratio)))
    if pc2im_bnhw.ndim != 2:
        raise ValueError("Expected pc2im_bnhw to have ndim=2. Got {0}.".format(pc2im_bnhw.ndim))
    if pc2im_bnhw.shape[1] != 4:
        raise ValueError("pc2im_bnhw.shape[1] must be 4, but was {0}.".format(pc2im_bnhw.shape[1]))
    B = len(pointclouds)
    dev = pc2im_bnhw.device
    t = pc2im_bnhw[(pc2im_bnhw[:, 2] % ds_ratio == 0) & (pc2im_bnhw[:, 3] % ds_ratio == 0)]
    # all elements at once (the reference loops over b, icputils.py:604-617): element b keeps its rows in table order
    order = torch.sort(t[:, 0], stable=True).indices
    b_of, n_of = t[order, 0], t[order, 1]
    counts_t = torch.bincount(b_of, minlength=B)[:B]
    counts = [int(c) for c in counts_t.tolist()]  # (the one host synchronisation: the ragged sizes)
    nmax = max(counts) if counts else 0
    starts = torch.cumsum(counts_t, 0) - counts_t
    pos = torch.arange(b_of.numel(), device=dev) - starts[b_of]
    idx = torch.zeros((B, nmax), dtype=torch.int64, device=dev)
    idx[b_of, pos] = n_of
    keep = (torch.arange(nmax, device=dev).unsqueeze(0) < counts_t.unsqueeze(1)).unsqueeze(-1)

    def pick(padded):
        if padded is None:
            return None
        g = torch.gather(padded, 1, idx.unsqueeze(-1).expand(-1, -1, padded.shape[-1]))
        return torch.where(keep, g, torch.zeros((), dtype=g.dtype, device=g.device))

    out = Pointclouds(points=pick(pointclouds.points_padded), normals=pick(pointclouds.normals_padded),
                      colors=pick(pointclouds.colors_padded))
    out._set_counts(counts)
    return out


def _compact_rows(mask: torch.Tensor, values):
    """mask (B, n) bool, values: tensors (B, n, C).  Per element the selected rows, in their original order, moved to
    the front of a (B, max count, C) tensor, zeros behind them; returns (tensors, sizes as a host list)."""
    B, n = mask.shape
    counts_t = mask.sum(1)
    counts = [int(c) for c in counts_t.tolist()]  # (the one host synchronisation: the ragged sizes)
    nmax = max(counts) if counts else 0
    order = torch.sort((~mask).to(torch.uint8), dim=1, stable=True).indices[:, :nmax]  # selected rows first, in order
    keep = (torch.arange(nmax, device=mask.device).unsqueeze(0) < counts_t.unsqueeze(1)).unsqueeze(-1)
    outs = []
    for v in values:
        g = torch.gather(v, 1, order.unsqueeze(-1).expand(-1, -1, v.shape[-1]))
        outs.append(torch.where(keep, g, torch.zeros((), dtype=g.dtype, device=g.device)))
    return outs, counts


def downsample_rgbdimages(rgbdimages: RGBDImages, ds_ratio: int) -> Pointclouds:
    """Strided subsample of the global maps + valid mask -> Pointclouds (icputils.py:623-669)."""
    if not isinstance(rgbdimages, RGBDImages):
        raise TypeError("Expected rgbdimages to be of type gradslam.RGBDImages. Got {0}.".format(type(rgbdimages)))
    if not isinstance(ds_ratio, int):
        raise TypeError("Expected ds_ratio to be of type int. Got {0}.".format(type(ds_ratio)))
    if rgbdimages.shape[1] != 1:
        raise ValueError("Sequence length of rgbdimages must be 1, but was {0}.".format(rgbdimages.shape[1]))
    fr = rgbdimages.to_channels_last()
    B = len(fr)
    mask = fr.valid_depth_mask.squeeze(-1)[:, 0, ::ds_ratio, ::ds_ratio].reshape(B, -1)
    sub = lambda m: m[:, 0, ::ds_ratio, ::ds_ratio].reshape(B, -1, m.shape[-1])
    # all elements at once (the reference indexes element by element, icputils.py:655-667)
    (pts, nrm, col), counts = _compact_rows(mask, [sub(fr.global_vertex_map), sub(fr.global_normal_map),
                                                    sub(fr.rgb_image)])
    out = Pointclouds(points=pts, normals=nrm, colors=col)
    out._set_counts(counts)
    return out


# --------------------------------------------------------------------------------------------- fused localisation
class _IcpWorkspace:
    _cache = {}

    def __init__(self, device, B, H, W, ds, capacity):
        n = _C.lib().gsx_icp_workspace_bytes(B, H, W, ds, capacity)
        self.buf = torch.zeros(n, dtype=torch.uint8, device=device)
        self.capacity = capacity
        self.epoch = 0

    @classmethod
    def get(cls, device, B, H, W, ds, capacity):
        key = (str(device), B, H, W, ds)
        ws = cls._cache.get(key)
        if ws is None or ws.capacity < capacity:
            ws = cls(device, B, H, W, ds, capacity)
            cls._cache[key] = ws
        return ws

    def next_epoch(self):
        self.epoch += 1
        if self.epoch >= (1 << 30) - 1:
            self.buf.zero_()
            self.epoch = 1
        return self.epoch


def localize_against_map(pointclouds, live_frame, prev_frame, dsratio, odomprov):
    """ICPSLAM._localize for odom in {icp, gradicp} (slam/icpslam.py:238-247) as ONE C call: gathers the source
    (live frame on the ds lattice at the previous pose) and target (lattice-active map points) clouds, runs the
    batched ICP loop and returns the new poses (B,1,4,4) = T_icp · prev pose.  No host synchronisation."""
    live = live_frame.to_channels_last()
    B, _, H, W = live.shape
    dev = pointclouds.device
    _C.require_cuda(live.depth_image, "depth_image")
    depth, d_bs = _frame_base(live.depth_image, H * W)
    K = live.intrinsics.contiguous()
    prev = prev_frame.poses.contiguous()
    _C.require_cuda(pointclouds._geo, "pointclouds (geometry rows)")
    geo = pointclouds._geo.contiguous()
    ws = _IcpWorkspace.get(dev, B, H, W, dsratio, pointclouds.capacity)
    # target capacity: lattice-active map points.  32 map points per lattice pixel on average is far beyond
    # anything a surfel map produces; if it is ever exceeded the kernel raises the map's overflow flag.
    ns_cap = ((H + dsratio - 1) // dsratio) * ((W + dsratio - 1) // dsratio)
    bound = max(1, min(pointclouds._bound, 32 * ns_cap))
    tgt = torch.empty(_C.lib().gsx_icp_tgt_scratch_bytes(B, bound), dtype=torch.uint8, device=dev)
    out = torch.empty((B, 1, 4, 4), dtype=torch.float32, device=dev)
    mode = 1 if hasattr(odomprov, "lambda_max") else 0
    dth = odomprov.dist_thresh
    with torch.cuda.device(dev):
        rc = _C.lib().gsx_icp_localize(
            _C.ptr(geo), _C.ptr(pointclouds._counts_dev[pointclouds._cur]),
            pointclouds.capacity, pointclouds._bound, _C.ptr(depth), d_bs, _C.ptr(K), 16, _C.ptr(prev), 16, B, H, W,
            int(dsratio), mode, int(odomprov.numiters), float(odomprov.damp), 0 if dth is None else 1,
            0.0 if dth is None else float(dth), float(getattr(odomprov, "lambda_max", 2.0)),
            float(getattr(odomprov, "B", 1.0)), float(getattr(odomprov, "B2", 1.0)),
            float(getattr(odomprov, "nu", 200.0)), _C.ptr(tgt), bound, _C.ptr(out), 16, _C.ptr(ws.buf),
            ws.capacity, ws.next_epoch(), _C.ptr(pointclouds._overflow_flag()), _C.stream_ptr(dev))
    _C.check(rc, "gsx_icp_localize")
    return out
