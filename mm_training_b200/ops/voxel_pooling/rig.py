"""Run plans straight from the camera rig: the (B, N, D, H, W, 3) geometry tensors are never made.

Reference being replaced (``layers/backbones/lss_fpn.py``): ``get_geometry`` :328-361 builds the float ego
coordinates of every frustum point with ~6 ATen passes, and :461-462 quantises them to int32 cell indices
(another 3 passes) that ``voxel_pooling`` then reads (12 B/point).  Here the plan builder derives the cell of
a point on the fly from what actually varies per sample -- ``combine = sensor2ego @ inverse(intrin)``, B*N
4x4 matrices left in torch -- and the frustum axes, op for op like the reference (float32 multiply, 4-term
dot product, IEEE subtract, true division, truncation toward zero).

Bit-exactness of the integer indices is the contract (SURVEY.md section 8a, rows a3/a4).  The one thing the
kernel cannot know a priori is the accumulation order of the reference's batched 4x4 @ 4x1 matmul (it is
whatever BLAS kernel torch dispatches to on the device in use), so ``rig_variant`` PROVES a variant on the
current device against ``mm_training_b200.geometry`` (= the reference's ops) over a randomised rig sweep
before it is used, and ``LiftSplatGeometry.plan`` falls back to the torch geometry + ``geom_xyz`` plan when
no variant reproduces torch exactly.
"""
from __future__ import annotations

import ctypes
import math
from typing import Dict, Optional, Sequence

import torch

from ... import _lib, geometry
from .voxel_pooling import PoolingPlan, RUN_CHANNELS  # noqa: F401

_VARIANT_CACHE: Dict[int, Optional[int]] = {}


def _f32x3(t: torch.Tensor):
    return (ctypes.c_float * 3)(*[float(v) for v in t.detach().cpu().tolist()])


def _random_rigs(batch: int, num_cams: int, gen: torch.Generator) -> (torch.Tensor, torch.Tensor):
    """sensor2ego / intrin pairs with arbitrary yaw, pitch, roll, lever arms and focal lengths."""
    def rot(axis, a):
        c, s = math.cos(a), math.sin(a)
        m = torch.eye(3)
        i, j = [(1, 2), (0, 2), (0, 1)][axis]
        m[i, i], m[i, j], m[j, i], m[j, j] = c, -s, s, c
        return m
    r0 = torch.tensor([[0, 0, 1.], [-1, 0, 0], [0, -1, 0]])
    s2e = torch.zeros(batch, num_cams, 4, 4)
    k = torch.zeros(batch, num_cams, 4, 4)
    for b in range(batch):
        for n in range(num_cams):
            u = torch.rand(8, generator=gen)
            yaw, pitch, roll = (u[0] * 2 - 1) * math.pi, (u[1] * 2 - 1) * 0.2, (u[2] * 2 - 1) * 0.1
            s2e[b, n, :3, :3] = rot(2, float(yaw)) @ rot(1, float(pitch)) @ rot(0, float(roll)) @ r0
            s2e[b, n, :3, 3] = torch.tensor([float(u[3] * 4 - 2), float(u[4] * 2 - 1), float(1 + u[5])])
            s2e[b, n, 3, 3] = 1.0
            f = float(400 + 900 * u[6])
            k[b, n] = torch.tensor([[f, 0, 352 + float(u[7] * 20), 0], [0, f * 1.01, 128, 0], [0, 0, 1, 0], [0, 0, 0, 1.]])
    return s2e, k


class LiftSplatGeometry:
    """The frustum / voxel buffers ``LSSFPN.__init__`` registers (``lss_fpn.py:278-291``) plus the two things
    the model does with them per step: ``geom_xyz`` (the reference's tensors, in torch) and ``plan`` (the run
    plan of the fused pooling op, built on the device without those tensors)."""

    def __init__(self, x_bound, y_bound, z_bound, d_bound, final_dim, downsample_factor, device='cuda'):
        self.device = torch.device(device)
        voxel_size, voxel_coord, voxel_num = geometry.voxel_buffers(x_bound, y_bound, z_bound)
        self.voxel_size, self.voxel_coord = voxel_size.to(self.device), voxel_coord.to(self.device)
        self.voxel_num = tuple(int(v) for v in voxel_num.tolist())
        self.frustum = geometry.create_frustum(final_dim, downsample_factor, d_bound).to(self.device)
        self.D, self.H, self.W, _ = self.frustum.shape
        # the axes the frustum was expanded from (lss_fpn.py:313-321): same float32 values, 1-D
        self.fx = self.frustum[0, 0, :, 0].contiguous()
        self.fy = self.frustum[0, :, 0, 1].contiguous()
        self.fd = self.frustum[:, 0, 0, 2].contiguous()
        # lss_fpn.py:461: (voxel_coord - voxel_size / 2.0), float32, computed by the same ATen ops
        self.lower = self.voxel_coord - self.voxel_size / 2.0
        self._lower_c, self._vs_c = _f32x3(self.lower), _f32x3(self.voxel_size)

    @classmethod
    def from_config(cls, cfg, device='cuda') -> 'LiftSplatGeometry':
        return cls(cfg.x_bound, cfg.y_bound, cfg.z_bound, cfg.d_bound, cfg.final_dim, cfg.downsample_factor, device)

    # ---- the reference's tensors (oracle for the integer indices) ------------------------------------
    def geom_xyz(self, sensor2ego_mat: torch.Tensor, intrin_mat: torch.Tensor) -> torch.Tensor:
        """int32 (B, N, D, H, W, 3) exactly as ``lss_fpn.py:455-462`` makes it (in float32: autocast is switched off here
        -- under bf16 autocast the matmuls of the reference's geometry would run in bf16 and move points by metres)."""
        with torch.autocast(device_type=self.device.type, enabled=False):
            pts = geometry.get_geometry(self.frustum, sensor2ego_mat.float(), intrin_mat.float())
            return geometry.quantise_geometry(pts, self.voxel_coord, self.voxel_size).contiguous()

    @staticmethod
    def combine(sensor2ego_mat: torch.Tensor, intrin_mat: torch.Tensor) -> torch.Tensor:
        """``sensor2ego @ inverse(intrin)`` (B, N, 4, 4) -- ``lss_fpn.py:354``, left in torch (B*N tiny matrices); always
        float32 (autocast off).  ``inv_ex(check_errors=False)`` runs the LU kernels of ``torch.inverse`` (same values)
        without its singularity check, which is a host synchronisation per call.  A singular intrinsic matrix (or a NaN / inf
        in ``sensor2ego_mat``) gives non-finite entries here, where the reference raises.  The plan kernels then give
        INT_MIN for every coordinate whose ``combine`` row is not finite, so every point of that image is dropped: it
        adds nothing to the pooled output, gets a zero depth gradient, and the other images' plan entries are those of
        a plan without it (``tests/test_gpu_quantise.py``)."""
        with torch.autocast(device_type=sensor2ego_mat.device.type, enabled=False):
            inv = torch.linalg.inv_ex(intrin_mat.float(), check_errors=False).inverse
            return sensor2ego_mat.float().matmul(inv).contiguous()

    # ---- device path ---------------------------------------------------------------------------------
    def rig_geom(self, combine: torch.Tensor, variant: int) -> torch.Tensor:
        """The kernel's indices as an int32 (B, N, D, H, W, 3) tensor (self-test / diagnostics)."""
        B, N = combine.shape[:2]
        out = torch.empty(B, N, self.D, self.H, self.W, 3, dtype=torch.int32, device=self.device)
        with torch.cuda.device(self.device):
            _lib.check(_lib.lib().bevpool_rig_geom(combine.data_ptr(), self.fx.data_ptr(), self.fy.data_ptr(),
                                                   self.fd.data_ptr(), self._lower_c, self._vs_c, variant, B, N,
                                                   self.D, self.H, self.W, out.data_ptr(),
                                                   _lib.stream_ptr(self.device)), 'bevpool_rig_geom')
        return out

    def plan(self, sensor2ego_mat: torch.Tensor, intrin_mat: torch.Tensor, max_runs: Optional[int] = None,
             variant: Optional[int] = None) -> PoolingPlan:
        """Run plan of the fused op for this rig.  Uses the on-device index path when a variant is proven on this
        device (``rig_variant``), else the reference's torch geometry + ``PoolingPlan(geom_xyz, ...)``."""
        B, N = sensor2ego_mat.shape[:2]
        if variant is None:
            variant = rig_variant(self.device)
        if variant is None:
            return PoolingPlan(self.geom_xyz(sensor2ego_mat, intrin_mat), self.voxel_num,
                               frustum=(N, self.D, self.H, self.W), max_runs=max_runs)
        return PoolingPlan.from_rig(self, self.combine(sensor2ego_mat, intrin_mat), variant, max_runs)


def rig_variant(device) -> Optional[int]:
    """Accumulation-order variant of the plan kernel that reproduces the reference's (torch's) indices bit for
    bit on ``device``, or None.  Proven once per device per process on ~10 M points chosen to discriminate
    between the orders (they only differ in the last bit of a coordinate, which flips a truncated index for about
    one point in 10^5): the shipped aiMotive frustum (depths to 206 m, 44 x 80 x 409) under randomised rigs
    (arbitrary yaw / pitch / roll, lever arms, focal lengths) on the 0.8 m grid and on a 0.2 m grid, plus the level
    4-camera rig.  A variant is accepted only with ZERO mismatching points; the order used by cuBLAS' batched
    4x4 @ 4x1 product on B200 (two k-slices) is tried first."""
    device = torch.device(device)
    key = device.index if device.index is not None else torch.cuda.current_device()
    if key in _VARIANT_CACHE:
        return _VARIANT_CACHE[key]
    from ...configs import CFG_2, CFG_AIM
    from ... import synthetic
    gen = torch.Generator().manual_seed(1234)
    cases = []
    g_aim = LiftSplatGeometry.from_config(CFG_AIM, device)
    s2e, k = _random_rigs(1, 2, gen)
    cases.append((g_aim, s2e.to(device), k.to(device)))
    g_fine = LiftSplatGeometry((-204.8, 204.8, 0.2), (-25.6, 25.6, 0.2), (-5.0, 3.0, 8.0), CFG_AIM.d_bound, CFG_AIM.final_dim,
                               CFG_AIM.downsample_factor, device)
    s2e, k = _random_rigs(1, 1, gen)
    cases.append((g_fine, s2e.to(device), k.to(device)))
    g2 = LiftSplatGeometry.from_config(CFG_2, device)
    s2e, k = _random_rigs(2, 4, gen)
    cases.append((g2, s2e.to(device), k.to(device)))
    kk = torch.eye(4)
    kk[0, 0] = kk[1, 1] = CFG_2.focal_px
    kk[0, 2], kk[1, 2] = CFG_2.final_dim[1] / 2, CFG_2.final_dim[0] / 2
    level = torch.stack([synthetic.cam2ego(y + 1.7) for y in CFG_2.cam_yaws_deg])[None]
    cases.append((g2, level.to(device), kk[None, None].repeat(1, 4, 1, 1).to(device)))
    refs = [(g, g.combine(a, b), g.geom_xyz(a, b)) for g, a, b in cases]
    found = None
    order = [2] + [v for v in range(_lib.lib().bevpool_rig_num_variants()) if v != 2]
    for v in order:
        if all(torch.equal(g.rig_geom(cmb, v), ref) for g, cmb, ref in refs):
            found = v
            break
    del refs
    _VARIANT_CACHE[key] = found
    return found


def voxel_pooling_rig(lsg: LiftSplatGeometry, sensor2ego_mat: torch.Tensor, intrin_mat: torch.Tensor,
                      depth: torch.Tensor, context: torch.Tensor, max_runs: Optional[int] = None) -> torch.Tensor:
    """``lss_fpn.py:455-464`` in one call: geometry, quantisation, outer product and pooling.  depth (B*N, D, H, W),
    context (B*N, C, H, W); returns (B, C, Y, X) like the reference op."""
    from .voxel_pooling import VoxelPoolingFused
    return VoxelPoolingFused.apply(None, depth, context, lsg.voxel_num, None,
                                   lambda: lsg.plan(sensor2ego_mat, intrin_mat, max_runs=max_runs), int(sensor2ego_mat.shape[0]))
