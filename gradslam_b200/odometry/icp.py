"""ICP odometry provider (mirror of gradslam/odometry/icp.py:11-97).  The reference loops over the batch in
Python calling point_to_plane_ICP per element; here the whole batch is one batched C call."""
from typing import Union

import torch

from ..structures.pointclouds import Pointclouds
from .base import OdometryProvider
from .icputils import _taped_icp, _wants_grad, icp_align

__all__ = ["ICPOdometryProvider"]


def _check_provide_args(maps_pointclouds, frames_pointclouds, who):
    if not isinstance(maps_pointclouds, Pointclouds):
        raise TypeError("Expected maps_pointclouds to be of type gradslam.Pointclouds. Got {0}.".format(
            type(maps_pointclouds)))
    if not isinstance(frames_pointclouds, Pointclouds):
        raise TypeError("Expected frames_pointclouds to be of type gradslam.Pointclouds. Got {0}.".format(
            type(frames_pointclouds)))
    if maps_pointclouds.normals_list is None:
        raise ValueError("maps_pointclouds missing normals. Map normals must be provided if using {}".format(who))
    if len(maps_pointclouds) != len(frames_pointclouds):
        raise ValueError("Batch size of maps_pointclouds and frames_pointclouds should be equal ({0} != {1})".format(
            len(maps_pointclouds), len(frames_pointclouds)))


def _provide(prov, maps_pc, frames_pc, mode):
    kw = dict(lambda_max=getattr(prov, "lambda_max", 2.0), B=getattr(prov, "B", 1.0), B2=getattr(prov, "B2", 1.0),
              nu=getattr(prov, "nu", 200.0))
    if _wants_grad(*frames_pc._grad_tensors(), *maps_pc._grad_tensors()):
        # differentiable mode: ONE chain of batched autograd ops for all elements (the reference's providers loop over
        # the batch in Python, odometry/icp.py:84-97)
        T, _ = _taped_icp(frames_pc.points_padded, frames_pc._counts_dev[frames_pc._cur], maps_pc.points_padded,
                          maps_pc.normals_padded, maps_pc._counts_dev[maps_pc._cur], None, mode, prov.numiters,
                          prov.damp, prov.dist_thresh, **kw)
        return T.unsqueeze(1)
    # (the padded views are strided slices of the packed rows; the ICP kernels take dense (B,N,3) clouds)
    src = frames_pc.points_padded.contiguous()
    tgt, tgt_n = maps_pc.points_padded.contiguous(), maps_pc.normals_padded.contiguous()
    src_c = frames_pc._counts_dev[frames_pc._cur]
    tgt_c = maps_pc._counts_dev[maps_pc._cur]
    T, _ = icp_align(src, src_c, tgt, tgt_n, tgt_c, None, mode, prov.numiters, prov.damp, prov.dist_thresh, **kw)
    return T.unsqueeze(1)


class ICPOdometryProvider(OdometryProvider):
    def __init__(self, numiters: int = 20, damp: float = 1e-8, dist_thresh: Union[float, int, None] = None):
        self.numiters = numiters
        self.damp = damp
        self.dist_thresh = dist_thresh

    def provide(self, maps_pointclouds: Pointclouds, frames_pointclouds: Pointclouds) -> torch.Tensor:
        """Transforms (B,1,4,4) aligning each frame cloud to its map cloud with point-to-plane ICP."""
        _check_provide_args(maps_pointclouds, frames_pointclouds, "ICPOdometryProvider")
        return _provide(self, maps_pointclouds, frames_pointclouds, 0)
