"""Operator surface: the Python functions the reference exposes in gsplat/cuda/_wrapper.py, with the
same names, argument meaning and error behaviour, implemented as torch.autograd.Function wrappers
around the C ABI of libgsplat_b200.so (include/gsplat_b200.h).

Reference wrappers mirrored here (file:line in /root/reference/gsplat/cuda/_wrapper.py):
  quat_scale_to_covar_preci :657   fully_fused_projection :819   spherical_harmonics :436
  isect_tiles :1196                isect_offset_encode :1328     rasterize_to_pixels :1497
and their autograd registrations (:559-716, :966-1191, :2010-2117).

PyTorch is plumbing here (device memory, streams, autograd graph); every number is produced by the
hand-written sm_100a kernels.
"""
from __future__ import annotations

import math
from typing import Optional, Tuple

import torch
from torch import Tensor

from . import _cabi
from ._cabi import check, f32c, lib, ptr, require_cuda, stream

# --------------------------------------------------------------------------------------------
# helpers


def _prod(shape) -> int:
    return int(math.prod(shape)) if len(shape) else 1


def _rows(t: Optional[Tensor], width: int, name: str) -> Tuple[Optional[Tensor], int]:
    """Return (tensor, row_stride_in_floats) for a gradient the kernels address as ptr[row * stride + k],
    row being the C-order flattened index over the leading dims.  ``width`` > 1: t is [..., width] with a
    unit inner stride; ``width`` == 1: t is [...] (no trailing dim).  Accepts any layout whose rows sit at
    one uniform stride (e.g. views into a packed per-gaussian record); copies otherwise."""
    if t is None:
        return None, 0
    if t.dtype != torch.float32:
        raise TypeError(f"{name}: expected a float32 gradient, got {t.dtype}")
    has_inner = width > 1
    lead_shape = t.shape[:-1] if has_inner else t.shape
    lead_strides = t.stride()[:-1] if has_inner else t.stride()
    ok = (not has_inner) or (t.shape[-1] == width and t.stride(-1) == 1)
    if ok:
        row, expect = None, None
        for size, st in zip(reversed(lead_shape), reversed(lead_strides)):
            if size == 1:
                continue
            if expect is None:
                row, expect = st, st * size
            elif st != expect:
                ok = False
                break
            else:
                expect *= size
        if row is None:
            row = width
        if ok and row >= width:
            return t, int(row)
    return t.contiguous(), width


class _Ctx:
    """device guard + stream fetch for one operator call"""

    __slots__ = ("dev", "_g")

    def __init__(self, dev: torch.device):
        self.dev = dev

    def __enter__(self):
        idx = self.dev.index
        if idx is None or torch._C._cuda_getDevice() != idx:  # not the current device: switch for the launches
            self._g = torch.cuda.device(self.dev)
            self._g.__enter__()
            return stream()
        self._g = None
        return stream(idx)

    def __exit__(self, *a):
        return self._g.__exit__(*a) if self._g is not None else None


def _camera_model_id(camera_model: str) -> int:
    table = {"pinhole": 0, "ortho": 1, "fisheye": 2, "ftheta": 3, "lidar": 4}
    if camera_model not in table:
        raise ValueError(f"unknown camera_model {camera_model!r}")
    if camera_model not in ("pinhole", "ortho", "fisheye"):
        raise NotImplementedError(
            f"camera_model={camera_model!r}: the EWA projection is built for pinhole / ortho / fisheye "
            "(reference: csrc/ProjectionEWA3DGSFused.cu:135-147); ftheta and lidar belong to the 3DGUT pipeline"
        )
    return table[camera_model]


# --------------------------------------------------------------------------------------------
# quat_scale_to_covar_preci


class _QuatScaleToCovarPreci(torch.autograd.Function):
    @staticmethod
    def forward(ctx, quats, scales, compute_covar: bool, compute_preci: bool, triu: bool):
        dev = require_cuda(quats, scales)
        q, s = f32c(quats, "quats"), f32c(scales, "scales")
        lead = q.shape[:-1]
        N = _prod(lead)
        shp = tuple(lead) + ((6,) if triu else (3, 3))
        covars = torch.empty(shp, device=dev, dtype=torch.float32) if compute_covar else None
        precis = torch.empty(shp, device=dev, dtype=torch.float32) if compute_preci else None
        with _Ctx(dev) as st:
            check(
                lib().gsb200_quat_scale_to_covar_preci_fwd(N, ptr(q), ptr(s), int(triu), ptr(covars), ptr(precis), st),
                "quat_scale_to_covar_preci",
            )
        ctx.save_for_backward(q, s)
        ctx.triu = triu
        return covars, precis

    @staticmethod
    def backward(ctx, v_covars, v_precis):
        q, s = ctx.saved_tensors
        N = _prod(q.shape[:-1])
        vc = None if v_covars is None else v_covars.contiguous()
        vp = None if v_precis is None else v_precis.contiguous()
        v_q, v_s = torch.empty_like(q), torch.empty_like(s)
        with _Ctx(q.device) as st:
            check(
                lib().gsb200_quat_scale_to_covar_preci_bwd(
                    N, ptr(q), ptr(s), int(ctx.triu), ptr(vc), ptr(vp), ptr(v_q), ptr(v_s), st
                ),
                "quat_scale_to_covar_preci_bwd",
            )
        return v_q, v_s, None, None, None


def quat_scale_to_covar_preci(
    quats: Tensor, scales: Tensor, compute_covar: bool = True, compute_preci: bool = True, triu: bool = False
) -> Tuple[Optional[Tensor], Optional[Tensor]]:
    """Quaternions (wxyz, need not be normalised) and scales -> covariance / precision matrices.
    Shapes: quats [..., 4], scales [..., 3] -> [..., 3, 3] or [..., 6] when ``triu``."""
    if quats.shape[-1] != 4 or scales.shape[-1] != 3 or quats.shape[:-1] != scales.shape[:-1]:
        raise ValueError(f"bad shapes quats {tuple(quats.shape)} scales {tuple(scales.shape)}")
    return _QuatScaleToCovarPreci.apply(quats, scales, compute_covar, compute_preci, triu)


# --------------------------------------------------------------------------------------------
# fully_fused_projection (dense)


class _FullyFusedProjection(torch.autograd.Function):
    @staticmethod
    def forward(
        ctx, means, covars, quats, scales, opacities, viewmats, Ks, width, height, eps2d, near_plane, far_plane,
        radius_clip, calc_compensations, camera_model_id,
    ):
        dev = require_cuda(means, viewmats, Ks)
        means, covars, quats, scales = f32c(means, "means"), f32c(covars, "covars"), f32c(quats, "quats"), f32c(scales, "scales")
        opacities, viewmats, Ks = f32c(opacities, "opacities"), f32c(viewmats, "viewmats"), f32c(Ks, "Ks")
        batch = tuple(means.shape[:-2])
        B, N, C = _prod(batch), means.shape[-2], viewmats.shape[-3]
        o = dict(device=dev, dtype=torch.float32)
        radii = torch.empty(batch + (C, N, 2), device=dev, dtype=torch.int32)
        means2d = torch.empty(batch + (C, N, 2), **o)
        depths = torch.empty(batch + (C, N), **o)
        conics = torch.empty(batch + (C, N, 3), **o)
        comps = torch.empty(batch + (C, N), **o) if calc_compensations else None
        with _Ctx(dev) as st:
            check(
                lib().gsb200_projection_fwd(
                    B, C, N, ptr(means), ptr(covars), ptr(quats), ptr(scales), ptr(opacities), ptr(viewmats), ptr(Ks),
                    width, height, eps2d, near_plane, far_plane, radius_clip, camera_model_id, ptr(radii), ptr(means2d),
                    ptr(depths), ptr(conics), ptr(comps), st,
                ),
                "projection_ewa_3dgs_fused",
            )
        ctx.save_for_backward(means, covars, quats, scales, viewmats, Ks, radii, conics, comps)
        ctx.meta = (width, height, eps2d, camera_model_id)
        ctx.mark_non_differentiable(radii)
        return radii, means2d, depths, conics, comps

    @staticmethod
    def backward(ctx, v_radii, v_means2d, v_depths, v_conics, v_comps):
        means, covars, quats, scales, viewmats, Ks, radii, conics, comps = ctx.saved_tensors
        width, height, eps2d, cam_id = ctx.meta
        batch = tuple(means.shape[:-2])
        B, N, C = _prod(batch), means.shape[-2], viewmats.shape[-3]
        dev = means.device
        z = lambda shape: torch.zeros(shape, device=dev, dtype=torch.float32)  # noqa: E731
        if v_means2d is None:
            v_means2d = z(batch + (C, N, 2))
        if v_depths is None:
            v_depths = z(batch + (C, N))
        if v_conics is None:
            v_conics = z(batch + (C, N, 3))
        v_means2d, s_m2 = _rows(v_means2d, 2, "v_means2d")
        v_depths, s_d = _rows(v_depths, 1, "v_depths")
        v_conics, s_c = _rows(v_conics, 3, "v_conics")
        v_comps = None if (v_comps is None or comps is None) else v_comps.contiguous()
        need_vm = ctx.needs_input_grad[5]
        v_means = torch.empty_like(means)
        v_covars = torch.empty_like(covars) if covars is not None else None
        v_quats = torch.empty_like(quats) if covars is None else None
        v_scales = torch.empty_like(scales) if covars is None else None
        v_viewmats = torch.empty_like(viewmats) if need_vm else None
        with _Ctx(dev) as st:
            check(
                lib().gsb200_projection_bwd(
                    B, C, N, ptr(means), ptr(covars), ptr(quats), ptr(scales), ptr(viewmats), ptr(Ks), width, height,
                    eps2d, cam_id, ptr(radii), ptr(conics), ptr(comps), ptr(v_means2d), s_m2, ptr(v_depths), s_d,
                    ptr(v_conics), s_c, ptr(v_comps), ptr(v_means), ptr(v_covars), ptr(v_quats), ptr(v_scales),
                    ptr(v_viewmats), st,
                ),
                "projection_ewa_3dgs_fused_bwd",
            )
        return (v_means, v_covars, v_quats, v_scales, None, v_viewmats) + (None,) * 9


class _FullyFusedProjectionPacked(torch.autograd.Function):
    """projection_ewa_3dgs_packed (/root/reference/gsplat/cuda/_wrapper.py:1065-1191): two-pass compacting
    projection; outputs are the nnz visible (batch, camera, gaussian) rows in ascending order."""

    @staticmethod
    def forward(
        ctx, means, covars, quats, scales, opacities, viewmats, Ks, width, height, eps2d, near_plane, far_plane,
        radius_clip, sparse_grad, calc_compensations, camera_model_id,
    ):
        dev = require_cuda(means, viewmats, Ks)
        means, covars, quats, scales = f32c(means, "means"), f32c(covars, "covars"), f32c(quats, "quats"), f32c(scales, "scales")
        opacities, viewmats, Ks = f32c(opacities, "opacities"), f32c(viewmats, "viewmats"), f32c(Ks, "Ks")
        batch = tuple(means.shape[:-2])
        if sparse_grad and len(batch) != 0:
            raise ValueError("sparse_grad does not support batch dimensions")
        B, N, C = _prod(batch), means.shape[-2], viewmats.shape[-3]
        if B * C > 65535:
            # same launch geometry limit as the reference's packed kernel (ProjectionEWA3DGSPacked.cu:325-333): B*C on grid.y
            raise RuntimeError(f"projection_ewa_3dgs_packed: B * C = {B * C} exceeds the CUDA grid.y limit of 65535")
        L = lib()
        o = dict(device=dev, dtype=torch.float32)
        nnz_dev = torch.empty(1, device=dev, dtype=torch.int32)
        args = (
            B, C, N, ptr(means), ptr(covars), ptr(quats), ptr(scales), ptr(opacities), ptr(viewmats), ptr(Ks), width, height,
            eps2d, near_plane, far_plane, radius_clip,
        )
        with _Ctx(dev) as st:
            ws = torch.empty(max(L.gsb200_projection_packed_workspace_bytes(B, C, N), 256), device=dev, dtype=torch.uint8)
            check(
                L.gsb200_projection_packed_count(*args, int(calc_compensations), camera_model_id, ptr(ws), ws.numel(), ptr(nnz_dev), st),
                "projection_ewa_3dgs_packed (count)",
            )
            nnz = int(nnz_dev.item())  # the host sync of the packed path (reference: Projection.cpp:924)
            ids = torch.empty((3, nnz), device=dev, dtype=torch.int64)
            indptr = torch.empty(B * C + 1, device=dev, dtype=torch.int32)
            radii = torch.empty((nnz, 2), device=dev, dtype=torch.int32)
            means2d, depths, conics = torch.empty((nnz, 2), **o), torch.empty((nnz,), **o), torch.empty((nnz, 3), **o)
            comps = torch.zeros((nnz,), **o) if calc_compensations else None
            check(
                L.gsb200_projection_packed_emit(
                    *args, camera_model_id, ptr(ws), ptr(indptr), ptr(ids[0]), ptr(ids[1]), ptr(ids[2]), ptr(radii), ptr(means2d),
                    ptr(depths), ptr(conics), ptr(comps), st,
                ),
                "projection_ewa_3dgs_packed (emit)",
            )
        batch_ids, camera_ids, gaussian_ids = ids[0], ids[1], ids[2]
        ctx.save_for_backward(means, covars, quats, scales, viewmats, Ks, batch_ids, camera_ids, gaussian_ids, conics, comps)
        ctx.meta = (width, height, eps2d, camera_model_id, bool(sparse_grad))
        ctx.mark_non_differentiable(batch_ids, camera_ids, gaussian_ids, indptr, radii)
        return batch_ids, camera_ids, gaussian_ids, indptr, radii, means2d, depths, conics, comps

    @staticmethod
    def backward(ctx, _vb, _vc, _vg, _vi, _vr, v_means2d, v_depths, v_conics, v_comps):
        means, covars, quats, scales, viewmats, Ks, batch_ids, camera_ids, gaussian_ids, conics, comps = ctx.saved_tensors
        width, height, eps2d, cam_id, sparse_grad = ctx.meta
        batch = tuple(means.shape[:-2])
        B, N, C = _prod(batch), means.shape[-2], viewmats.shape[-3]
        nnz = conics.shape[0]
        dev = means.device
        z = lambda shape: torch.zeros(shape, device=dev, dtype=torch.float32)  # noqa: E731
        v_means2d = z((nnz, 2)) if v_means2d is None else v_means2d
        v_depths = z((nnz,)) if v_depths is None else v_depths
        v_conics = z((nnz, 3)) if v_conics is None else v_conics
        v_means2d, s_m2 = _rows(v_means2d, 2, "v_means2d")
        v_depths, s_d = _rows(v_depths, 1, "v_depths")
        v_conics, s_c = _rows(v_conics, 3, "v_conics")
        v_comps = None if (v_comps is None or comps is None) else v_comps.contiguous()
        need_vm = ctx.needs_input_grad[5]
        lead = (nnz,) if sparse_grad else tuple(means.shape[:-1])
        e = lambda w: torch.empty(lead + (w,), device=dev, dtype=torch.float32)  # noqa: E731
        v_means = e(3)
        v_covars = e(6) if covars is not None else None
        v_quats = e(4) if covars is None else None
        v_scales = e(3) if covars is None else None
        v_viewmats = torch.empty_like(viewmats) if need_vm else None
        with _Ctx(dev) as st:
            check(
                lib().gsb200_projection_packed_bwd(
                    B, C, N, nnz, ptr(means), ptr(covars), ptr(quats), ptr(scales), ptr(viewmats), ptr(Ks), width, height, eps2d,
                    cam_id, ptr(batch_ids), ptr(camera_ids), ptr(gaussian_ids), ptr(conics), ptr(comps), ptr(v_means2d), s_m2,
                    ptr(v_depths), s_d, ptr(v_conics), s_c, ptr(v_comps), int(sparse_grad), ptr(v_means), ptr(v_covars),
                    ptr(v_quats), ptr(v_scales), ptr(v_viewmats), st,
                ),
                "projection_ewa_3dgs_packed_bwd",
            )
        if sparse_grad:
            # per-row gradients wrapped as COO over the gaussian index (reference Projection.cpp:1188-1206);
            # coalesced when there is a single camera (every gaussian id then appears at most once)
            idx = gaussian_ids[None]

            def coo(rows, like):
                return None if rows is None else torch.sparse_coo_tensor(idx, rows, size=like.shape, is_coalesced=(C == 1))

            v_means, v_covars = coo(v_means, means), coo(v_covars, covars)
            v_quats, v_scales = coo(v_quats, quats), coo(v_scales, scales)
        return (v_means, v_covars, v_quats, v_scales, None, v_viewmats) + (None,) * 10


def fully_fused_projection(
    means: Tensor,  # [..., N, 3]
    covars: Optional[Tensor],  # [..., N, 6] or None
    quats: Optional[Tensor],  # [..., N, 4] or None
    scales: Optional[Tensor],  # [..., N, 3] or None
    viewmats: Tensor,  # [..., C, 4, 4]
    Ks: Tensor,  # [..., C, 3, 3]
    width: int,
    height: int,
    eps2d: float = 0.3,
    near_plane: float = 0.01,
    far_plane: float = 1e10,
    radius_clip: float = 0.0,
    packed: bool = False,
    sparse_grad: bool = False,
    calc_compensations: bool = False,
    camera_model: str = "pinhole",
    opacities: Optional[Tensor] = None,  # [..., N] or None
):
    """Projects Gaussians to 2D (EWA).  Returns (radii int32 [..., C, N, 2], means2d [..., C, N, 2],
    depths [..., C, N], conics [..., C, N, 3], compensations [..., C, N] | None).  ``radii == 0`` marks
    culled entries; their float outputs are zero."""
    if sparse_grad and not packed:
        raise AssertionError("sparse_grad is only supported when packed is True")
    if covars is None and (quats is None or scales is None):
        raise ValueError("either covars or (quats, scales) must be given")
    if covars is not None:
        quats = scales = None
    cam = _camera_model_id(camera_model)
    if packed:
        # (batch_ids, camera_ids, gaussian_ids int64 [nnz], indptr int32 [B*C+1], radii [nnz,2], means2d [nnz,2],
        #  depths [nnz], conics [nnz,3], compensations [nnz] | None), rows in ascending (b, c, n) order
        return _FullyFusedProjectionPacked.apply(
            means, covars, quats, scales, opacities, viewmats, Ks, int(width), int(height), float(eps2d), float(near_plane),
            float(far_plane), float(radius_clip), bool(sparse_grad), bool(calc_compensations), cam,
        )
    return _FullyFusedProjection.apply(
        means, covars, quats, scales, opacities, viewmats, Ks, int(width), int(height), float(eps2d), float(near_plane),
        float(far_plane), float(radius_clip), bool(calc_compensations), cam,
    )


# --------------------------------------------------------------------------------------------
# spherical_harmonics (dense)


class _SphericalHarmonics(torch.autograd.Function):
    @staticmethod
    def forward(ctx, degrees_to_use, means, viewmats, coeffs, masks):
        dev = require_cuda(means, viewmats, coeffs)
        means, viewmats, coeffs = f32c(means, "means"), f32c(viewmats, "viewmats"), f32c(coeffs, "coeffs")
        batch = tuple(means.shape[:-2])
        B, N, C = _prod(batch), means.shape[-2], viewmats.shape[-3]
        K, D = coeffs.shape[-2:]
        m8 = None
        if masks is not None:
            m8 = masks.contiguous().view(torch.uint8) if masks.dtype == torch.bool else masks.to(torch.uint8).contiguous()
        colors = torch.empty(batch + (C, N, D), device=dev, dtype=torch.float32)
        with _Ctx(dev) as st:
            check(
                lib().gsb200_sh_fwd(B, C, N, K, D, degrees_to_use, ptr(means), ptr(viewmats), ptr(coeffs), ptr(m8), ptr(colors), st),
                "spherical_harmonics",
            )
        ctx.save_for_backward(means, viewmats, coeffs, m8)
        ctx.deg = degrees_to_use
        return colors

    @staticmethod
    def backward(ctx, v_colors):
        means, viewmats, coeffs, m8 = ctx.saved_tensors
        batch = tuple(means.shape[:-2])
        B, N, C = _prod(batch), means.shape[-2], viewmats.shape[-3]
        K, D = coeffs.shape[-2:]
        v_colors = v_colors.contiguous()
        v_coeffs = torch.empty_like(coeffs)
        v_means = torch.empty_like(means) if ctx.needs_input_grad[1] else None
        need_vm = ctx.needs_input_grad[2]
        v_dirsum = torch.empty(batch + (C, 3), device=means.device, dtype=torch.float32) if need_vm else None
        with _Ctx(means.device) as st:
            check(
                lib().gsb200_sh_bwd(
                    B, C, N, K, D, ctx.deg, ptr(means), ptr(viewmats), ptr(coeffs), ptr(m8), ptr(v_colors), ptr(v_coeffs),
                    ptr(v_means), ptr(v_dirsum), st,
                ),
                "spherical_harmonics_bwd",
            )
        v_viewmats = None
        if need_vm:
            # dir = mean + R^T t  =>  dL/dR[i][j] = t[i] S[j],  dL/dt[i] = sum_j R[i][j] S[j],  S = sum_n dL/ddir
            R, t = viewmats[..., :3, :3], viewmats[..., :3, 3]
            v_viewmats = torch.zeros_like(viewmats)
            v_viewmats[..., :3, :3] = t[..., :, None] * v_dirsum[..., None, :]
            v_viewmats[..., :3, 3] = torch.einsum("...ij,...j->...i", R, v_dirsum)
        return None, v_means, v_viewmats, v_coeffs, None


class _SphericalHarmonicsRows(torch.autograd.Function):
    """SH colours of packed rows (batch_ids, camera_ids, gaussian_ids) with the coefficient table [N, K, D] indexed
    inside the kernel -- what rasterization(packed=True) uses instead of gathering [nnz, K, D] rows first."""

    @staticmethod
    def forward(ctx, degrees_to_use, means, viewmats, coeffs, batch_ids, camera_ids, gaussian_ids):
        dev = require_cuda(means, viewmats, coeffs)
        means, viewmats, coeffs = f32c(means, "means"), f32c(viewmats, "viewmats"), f32c(coeffs, "coeffs")
        ids = [t.to(torch.int64).contiguous() for t in (batch_ids, camera_ids, gaussian_ids)]
        batch = tuple(means.shape[:-2])
        B, N, C = _prod(batch), means.shape[-2], viewmats.shape[-3]
        K, D = coeffs.shape[-2:]
        nnz = ids[0].shape[0]
        colors = torch.empty((nnz, D), device=dev, dtype=torch.float32)
        with _Ctx(dev) as st:
            check(
                lib().gsb200_sh_rows_fwd(
                    nnz, B, C, N, K, D, degrees_to_use, ptr(means), ptr(viewmats), ptr(coeffs), ptr(ids[0]), ptr(ids[1]),
                    ptr(ids[2]), ptr(colors), st,
                ),
                "spherical_harmonics (rows)",
            )
        ctx.save_for_backward(means, viewmats, coeffs, *ids)
        ctx.deg = degrees_to_use
        return colors

    @staticmethod
    def backward(ctx, v_colors):
        means, viewmats, coeffs, b_ids, c_ids, g_ids = ctx.saved_tensors
        batch = tuple(means.shape[:-2])
        B, N, C = _prod(batch), means.shape[-2], viewmats.shape[-3]
        K, D = coeffs.shape[-2:]
        v_colors = v_colors.contiguous()
        v_coeffs = torch.empty_like(coeffs)
        v_means = torch.empty_like(means) if ctx.needs_input_grad[1] else None
        need_vm = ctx.needs_input_grad[2]
        v_dirsum = torch.empty(batch + (C, 3), device=means.device, dtype=torch.float32) if need_vm else None
        with _Ctx(means.device) as st:
            check(
                lib().gsb200_sh_rows_bwd(
                    b_ids.shape[0], B, C, N, K, D, ctx.deg, ptr(means), ptr(viewmats), ptr(coeffs), ptr(b_ids), ptr(c_ids),
                    ptr(g_ids), ptr(v_colors), ptr(v_coeffs), ptr(v_means), ptr(v_dirsum), st,
                ),
                "spherical_harmonics_bwd (rows)",
            )
        v_viewmats = None
        if need_vm:  # dir = mean + R^T t  =>  dL/dR[i][j] = t[i] S[j],  dL/dt = R S,  S = sum of dL/ddir over the camera's rows
            R, t = viewmats[..., :3, :3], viewmats[..., :3, 3]
            v_viewmats = torch.zeros_like(viewmats)
            v_viewmats[..., :3, :3] = t[..., :, None] * v_dirsum[..., None, :]
            v_viewmats[..., :3, 3] = torch.einsum("...ij,...j->...i", R, v_dirsum)
        return None, v_means, v_viewmats, v_coeffs, None, None, None


def spherical_harmonics_rows(
    degrees_to_use: int, means: Tensor, viewmats: Tensor, coeffs: Tensor, batch_ids: Tensor, camera_ids: Tensor,
    gaussian_ids: Tensor,
) -> Tensor:
    """SH colours [nnz, D] of the packed rows (batch_ids, camera_ids, gaussian_ids); ``coeffs`` is the full
    [N, K, D] table (NOT pre-gathered).  Same values as ``spherical_harmonics(..., coeffs[gaussian_ids], ids)``."""
    if coeffs.dim() != 3 or coeffs.shape[0] != means.shape[-2]:
        raise ValueError(f"coeffs must be [N, K, D]; got {tuple(coeffs.shape)} for N={means.shape[-2]}")
    if not (0 <= degrees_to_use <= 4) or (degrees_to_use + 1) ** 2 > coeffs.shape[-2]:
        raise ValueError(f"degrees_to_use={degrees_to_use} needs K >= {(degrees_to_use + 1) ** 2}, got {coeffs.shape[-2]}")
    return _SphericalHarmonicsRows.apply(int(degrees_to_use), means, viewmats, coeffs, batch_ids, camera_ids, gaussian_ids)


def spherical_harmonics(
    degrees_to_use: int,
    means: Tensor,  # [..., N, 3]
    viewmats: Tensor,  # [..., C, 4, 4]
    coeffs: Tensor,  # [N, K, D]
    masks: Optional[Tensor] = None,  # [..., C, N]
    batch_ids: Optional[Tensor] = None,
    camera_ids: Optional[Tensor] = None,
    gaussian_ids: Optional[Tensor] = None,
    viewmats_rs: Optional[Tensor] = None,
) -> Tensor:
    """Evaluates SH colours for view directions ``mean - camera_position`` (camera position recovered as
    ``-R^T t``).  Returns [..., C, N, D]; masked-off rows are 0."""
    if viewmats_rs is not None:
        raise NotImplementedError("rolling-shutter view matrices are out of scope")
    # the reference rejects these with TORCH_CHECK (RuntimeError), csrc/SphericalHarmonics.cpp
    if not (0 <= degrees_to_use <= 4):
        raise RuntimeError(f"degrees_to_use must be between 0 and 4, got {degrees_to_use}")
    if coeffs.dim() == 3 and coeffs.shape[-1] == 0:
        raise RuntimeError("spherical_harmonics: coeffs must have at least one channel (D > 0)")
    if coeffs.dtype in (torch.float16, torch.bfloat16):
        # half-precision coefficient storage (the trainer's sh_fp16 option): evaluated in fp32 like the reference
        # kernel; the cast is differentiable, so v_coeffs comes back in the storage dtype
        coeffs = coeffs.float()
    if batch_ids is not None or camera_ids is not None or gaussian_ids is not None:
        # packed mode: coeffs [nnz, K, D] pre-gathered, one (batch, camera, gaussian) triple per row.  The view
        # direction mean + R^T t is formed per row (torch, differentiable) and evaluated by the dense kernel
        # with an identity view matrix, one "gaussian" per row.
        if batch_ids is None or camera_ids is None or gaussian_ids is None:
            raise ValueError("batch_ids, camera_ids and gaussian_ids must be given together")
        nb = means.dim() - 2
        N, C = means.shape[-2], viewmats.shape[-3]
        m = means.reshape(-1, N, 3)[batch_ids.long(), gaussian_ids.long()]  # [nnz, 3]
        vm = viewmats.reshape(-1, C, 4, 4)[batch_ids.long(), camera_ids.long()]  # [nnz, 4, 4]
        dirs = m + torch.einsum("nij,ni->nj", vm[:, :3, :3], vm[:, :3, 3])
        if coeffs.dim() != 3 or coeffs.shape[0] != dirs.shape[0]:
            raise ValueError(f"packed coeffs must be [nnz, K, D]; got {tuple(coeffs.shape)} for nnz={dirs.shape[0]}")
        if not (0 <= degrees_to_use <= 4) or (degrees_to_use + 1) ** 2 > coeffs.shape[-2]:
            raise ValueError(f"degrees_to_use={degrees_to_use} needs K >= {(degrees_to_use + 1) ** 2}")
        eye = torch.eye(4, device=dirs.device, dtype=dirs.dtype)[None]
        out = _SphericalHarmonics.apply(int(degrees_to_use), dirs, eye, coeffs, None if masks is None else masks[None])
        return out[0]
    if coeffs.dim() != 3 or coeffs.shape[0] != means.shape[-2]:
        raise ValueError(f"coeffs must be [N, K, D]; got {tuple(coeffs.shape)} for N={means.shape[-2]}")
    if not (0 <= degrees_to_use <= 4) or (degrees_to_use + 1) ** 2 > coeffs.shape[-2]:
        raise ValueError(f"degrees_to_use={degrees_to_use} needs K >= {(degrees_to_use + 1) ** 2}, got {coeffs.shape[-2]}")
    return _SphericalHarmonics.apply(int(degrees_to_use), means, viewmats, coeffs, masks)


# --------------------------------------------------------------------------------------------
# fused projection + conic + SH -> RGB (the rasterization() default path)


# Where the fused backward puts the parameter gradients.  The view-parallel trainer registers the segments of its
# symmetric (NVLS multicast) gradient buffer here, so that the backward kernel writes straight into the memory
# the all-reduce kernel works on (gsplat_b200.distributed.NvlsGradArena) -- no staging copy.
_grad_allocator = None


def set_gradient_allocator(fn) -> None:
    """fn(name, like) -> Tensor | None with name in {"means", "quats", "scales", "sh"}; None = default.
    The fused backward also asks for ``fn("seen_bits", None)``: an int32 [ceil(N / 32)] tensor that receives the
    row bitmap of the row-sparse all-reduce, or None."""
    global _grad_allocator
    _grad_allocator = fn


def _alloc_grad(name: str, like: Tensor) -> Tensor:
    if _grad_allocator is not None:
        t = _grad_allocator(name, like)
        if t is not None:
            if t.shape != like.shape or t.dtype != like.dtype or t.device != like.device or not t.is_contiguous():
                raise RuntimeError(f"gradient allocator returned a mismatching tensor for {name!r}")
            return t
    return torch.empty_like(like)


class _ProjectSH(torch.autograd.Function):
    @staticmethod
    def forward(
        ctx, means, quats, scales, opacities, sh_coeffs, viewmats, Ks, width, height, eps2d, near_plane, far_plane,
        radius_clip, sh_degree, calc_compensations, rows_out=None,
    ):
        dev = require_cuda(means, quats, scales, opacities, sh_coeffs, viewmats, Ks)
        means, quats, scales = f32c(means, "means"), f32c(quats, "quats"), f32c(scales, "scales")
        opacities, sh_coeffs = f32c(opacities, "opacities"), f32c(sh_coeffs, "colors")
        viewmats, Ks = f32c(viewmats, "viewmats"), f32c(Ks, "Ks")
        N, C, K = means.shape[0], viewmats.shape[0], sh_coeffs.shape[1]
        o = dict(device=dev, dtype=torch.float32)
        radii = torch.empty((C, N, 2), device=dev, dtype=torch.int32)
        means2d, depths, conics = torch.empty((C, N, 2), **o), torch.empty((C, N), **o), torch.empty((C, N, 3), **o)
        colors = torch.empty((C, N, 3), **o)
        comps = torch.empty((C, N), **o) if calc_compensations else None
        with _Ctx(dev) as st:
            if rows_out is not None and not calc_compensations:
                # + per-row tile counts / totals and the 64-byte compositing row records (see RowSideOutputs)
                rows_out.rows = torch.empty((C, N, 16), **o)
                rows_out.tiles_per_gauss = torch.empty((C, N), device=dev, dtype=torch.int32)
                rows_out.totals = torch.empty(3, device=dev, dtype=torch.int64)
                check(
                    lib().gsb200_project_sh_fwd_rows(
                        C, N, K, sh_degree, ptr(means), ptr(quats), ptr(scales), ptr(opacities), ptr(sh_coeffs),
                        ptr(viewmats), ptr(Ks), width, height, eps2d, near_plane, far_plane, radius_clip, rows_out.tile_size,
                        rows_out.tile_width, rows_out.tile_height, ptr(radii), ptr(means2d), ptr(depths), ptr(conics),
                        ptr(colors), ptr(rows_out.rows), ptr(rows_out.tiles_per_gauss), ptr(rows_out.totals), st,
                    ),
                    "project_sh_fwd_rows",
                )
            else:
                check(
                    lib().gsb200_project_sh_fwd(
                        C, N, K, sh_degree, ptr(means), ptr(quats), ptr(scales), ptr(opacities), ptr(sh_coeffs),
                        ptr(viewmats), ptr(Ks), width, height, eps2d, near_plane, far_plane, radius_clip,
                        int(calc_compensations), ptr(radii), ptr(means2d), ptr(depths), ptr(conics), ptr(comps), ptr(colors), st,
                    ),
                    "project_sh_fwd",
                )
        ctx.save_for_backward(means, quats, scales, sh_coeffs, viewmats, Ks, radii, conics, comps, colors)
        ctx.meta = (width, height, eps2d, sh_degree)
        ctx.mark_non_differentiable(radii)
        ctx.set_materialize_grads(False)  # no zero tensors for radii / depths / compensations nobody differentiated
        return radii, means2d, depths, conics, colors, comps

    @staticmethod
    def backward(ctx, v_radii, v_means2d, v_depths, v_conics, v_colors, v_comps):
        means, quats, scales, sh_coeffs, viewmats, Ks, radii, conics, comps, colors = ctx.saved_tensors
        width, height, eps2d, sh_degree = ctx.meta
        if ctx.needs_input_grad[5]:
            raise NotImplementedError("fused project+SH path does not produce viewmats gradients")
        N, C, K = means.shape[0], viewmats.shape[0], sh_coeffs.shape[1]
        dev = means.device
        z = lambda shape: torch.zeros(shape, device=dev, dtype=torch.float32)  # noqa: E731
        if v_means2d is None:
            v_means2d = z((C, N, 2))
        if v_conics is None:
            v_conics = z((C, N, 3))
        if v_colors is None:
            v_colors = z((C, N, 3))
        v_means2d, s_m2 = _rows(v_means2d, 2, "v_means2d")
        v_depths, s_d = _rows(v_depths, 1, "v_depths")
        v_conics, s_c = _rows(v_conics, 3, "v_conics")
        v_colors, s_col = _rows(v_colors, 3, "v_colors")
        v_comps = None if (v_comps is None or comps is None) else v_comps.contiguous()
        v_means, v_quats, v_scales = _alloc_grad("means", means), _alloc_grad("quats", quats), _alloc_grad("scales", scales)
        v_sh = _alloc_grad("sh", sh_coeffs)
        # optional row bitmap for the row-sparse gradient all-reduce (distributed.NvlsGradArena): int32 [ceil(N / 32)]
        seen_bits = _grad_allocator("seen_bits", None) if _grad_allocator is not None else None
        if seen_bits is not None and (seen_bits.dtype != torch.int32 or seen_bits.numel() < (N + 31) // 32 or not seen_bits.is_contiguous()):
            raise RuntimeError("gradient allocator returned a mismatching tensor for 'seen_bits'")
        with _Ctx(dev) as st:
            check(
                lib().gsb200_project_sh_bwd(
                    C, N, K, sh_degree, ptr(means), ptr(quats), ptr(scales), ptr(sh_coeffs), ptr(viewmats), ptr(Ks),
                    width, height, eps2d, ptr(radii), ptr(conics), ptr(comps), ptr(colors), ptr(v_means2d), s_m2,
                    ptr(v_depths), s_d, ptr(v_conics), s_c, ptr(v_colors), s_col, ptr(v_comps), ptr(v_means),
                    ptr(v_quats), ptr(v_scales), ptr(v_sh), ptr(seen_bits), st,
                ),
                "project_sh_bwd",
            )
        # opacities only steer culling / radius (non-differentiable there)
        return (v_means, v_quats, v_scales, None, v_sh, None, None) + (None,) * 9


class RowSideOutputs:
    """Side outputs of the fused projection for the two stages that follow it in rasterization(): per-row tile counts
    and their totals (what gsb200_isect_count_totals would compute) and the 64-byte compositing row records
    {cull | axis | geom | rgb0} that make the pack pass a pure gather.  Valid only while the compositing runs on exactly
    the projection's means2d / conics / colours and the INPUT opacities (no antialiasing compensation, 3 channels)."""

    __slots__ = ("tile_size", "tile_width", "tile_height", "rows", "tiles_per_gauss", "totals")

    def __init__(self, tile_size: int, tile_width: int, tile_height: int):
        self.tile_size, self.tile_width, self.tile_height = int(tile_size), int(tile_width), int(tile_height)
        self.rows = self.tiles_per_gauss = self.totals = None


def fused_project_sh(
    means, quats, scales, opacities, sh_coeffs, viewmats, Ks, width, height, sh_degree, eps2d=0.3, near_plane=0.01,
    far_plane=1e10, radius_clip=0.0, calc_compensations=False, rows_out: Optional[RowSideOutputs] = None,
):
    """One pass over the gaussians: world->camera, covariance->conic, SH->RGB (+0.5, clamped at 0).
    means [N,3] quats [N,4] scales [N,3] opacities [N] sh_coeffs [N,K,3] viewmats [C,4,4] Ks [C,3,3].
    Returns (radii, means2d, depths, conics, colors [C,N,3], compensations|None)."""
    if sh_coeffs.dim() != 3 or sh_coeffs.shape[-1] != 3:
        raise ValueError("fused_project_sh needs SH coefficients [N, K, 3]")
    if not (0 <= sh_degree <= 4) or (sh_degree + 1) ** 2 > sh_coeffs.shape[1]:
        raise ValueError(f"sh_degree={sh_degree} needs K >= {(sh_degree + 1) ** 2}")
    return _ProjectSH.apply(
        means, quats, scales, opacities, sh_coeffs, viewmats, Ks, int(width), int(height), float(eps2d),
        float(near_plane), float(far_plane), float(radius_clip), int(sh_degree), bool(calc_compensations), rows_out,
    )


# --------------------------------------------------------------------------------------------
# isect_tiles / isect_offset_encode

_scratch = {}


def _scratch_buffer(dev: torch.device, tag: str, nbytes: int) -> Tensor:
    """Grow-only per-device scratch (CUB temp storage).  Stream-ordered use only."""
    key = (dev, tag, stream(dev.index))
    buf = _scratch.get(key)
    if buf is None or buf.numel() < nbytes:
        buf = torch.empty(max(nbytes, 1 << 16), device=dev, dtype=torch.uint8)
        _scratch[key] = buf
    return buf


@torch.no_grad()
def isect_tiles(
    means2d: Tensor,  # [..., N, 2]
    radii: Tensor,  # [..., N, 2]
    depths: Tensor,  # [..., N]
    tile_size: int,
    tile_width: int,
    tile_height: int,
    sort: bool = True,
    segmented: bool = False,
    packed: bool = False,
    n_images: Optional[int] = None,
    image_ids: Optional[Tensor] = None,
    gaussian_ids: Optional[Tensor] = None,
    conics: Optional[Tensor] = None,
    opacities: Optional[Tensor] = None,
) -> Tuple[Tensor, Tensor, Tensor]:
    """Maps projected Gaussians to the tiles they touch.  With ``conics`` and ``opacities`` the
    conservative ellipse test (AccuTile / SNUGBOX) is used, otherwise the radius AABB.
    Returns (tiles_per_gauss int32 [..., N], isect_ids int64 [n_isects], flatten_ids int32 [n_isects])."""
    dev = require_cuda(means2d, radii, depths)
    means2d, depths = f32c(means2d, "means2d"), f32c(depths, "depths")
    conics, opacities = f32c(conics, "conics"), f32c(opacities, "opacities")
    if radii.dtype != torch.int32:
        raise TypeError("radii must be int32")
    radii = radii.contiguous()
    if packed:
        if n_images is None or image_ids is None:
            raise ValueError("n_images and image_ids are required when means2d is packed ([nnz, 2]).")
        if segmented:
            raise ValueError("segmented sort is not supported for packed inputs")
        if means2d.dim() != 2:
            raise ValueError(f"packed means2d must be [nnz, 2], got {tuple(means2d.shape)}")
        image_dims, I, N = (), int(n_images), means2d.shape[0]
        img_ids = image_ids.to(torch.int64).contiguous()
        I_count = 1  # pass 1 sees one flat list of nnz rows
    else:
        image_dims = tuple(means2d.shape[:-2])
        I, N = _prod(image_dims), means2d.shape[-2]
        img_ids, I_count = None, I
    L = lib()
    n_tiles = tile_width * tile_height
    image_bits, tile_bits = _cabi.bits_for_count(I), _cabi.bits_for_count(n_tiles)
    if image_bits + tile_bits > 32:
        raise RuntimeError(
            f"intersect_tile: (image, tile) id packing needs {image_bits + tile_bits} bits but only 32 are "
            f"available (I={I}, n_tiles={n_tiles})."
        )
    total = I_count * N
    tiles_per_gauss = torch.empty(image_dims + (N,), device=dev, dtype=torch.int32)
    if total == 0:
        return (tiles_per_gauss, torch.empty(0, device=dev, dtype=torch.int64), torch.empty(0, device=dev, dtype=torch.int32))
    accu = conics is not None and opacities is not None
    if sort and not packed:
        # dense, sorted (the rasterization() path): count first, read both totals with ONE host sync, then order and
        # scan only the rows that have tiles (a third of the rows at BASELINE configs[2]: the culled ones never enter
        # the four radix passes of the depth order)
        totals = torch.empty(3, device=dev, dtype=torch.int64)
        with _Ctx(dev) as st:
            check(
                L.gsb200_isect_count_totals(
                    I, N, ptr(means2d), ptr(radii), ptr(conics) if accu else None, ptr(opacities) if accu else None, tile_size,
                    tile_width, tile_height, ptr(tiles_per_gauss), ptr(totals), st,
                ),
                "intersect_tile (count)",
            )
            n_isects, n_vis, max_tiles = (int(v) for v in totals.tolist())  # the one host sync of the forward (reference: csrc/Intersect.cpp:259)
            isect_ids = torch.empty(n_isects, device=dev, dtype=torch.int64)
            flatten_ids = torch.empty(n_isects, device=dev, dtype=torch.int32)
            if n_isects == 0:
                return tiles_per_gauss, isect_ids, flatten_ids
            order = torch.empty(n_vis, device=dev, dtype=torch.int32)
            cum = torch.empty(n_vis, device=dev, dtype=torch.int64)
            ws = _scratch_buffer(dev, "vorder", L.gsb200_isect_order_visible_workspace_bytes(I, total, n_vis))
            check(
                L.gsb200_isect_order_visible(I, N, n_vis, ptr(tiles_per_gauss), ptr(depths), None, ptr(order), ptr(cum), ptr(ws), ws.numel(), st),
                "intersect_tile (order)",
            )
            check(
                L.gsb200_isect_emit_ordered(
                    I, N, n_vis, max_tiles, ptr(means2d), ptr(radii), ptr(depths), ptr(conics) if accu else None,
                    ptr(opacities) if accu else None, ptr(cum), None, ptr(order), tile_size, tile_width, tile_height,
                    ptr(isect_ids), ptr(flatten_ids), st,
                ),
                "intersect_tile (emit)",
            )
            begin_bit, end_bit = 32, 32 + tile_bits + image_bits
            keys_out, vals_out = torch.empty_like(isect_ids), torch.empty_like(flatten_ids)
            ws = _scratch_buffer(dev, "sort", L.gsb200_sort_workspace_bytes(n_isects, begin_bit, end_bit))
            check(
                L.gsb200_sort_pairs(
                    n_isects, begin_bit, end_bit, ptr(isect_ids), ptr(flatten_ids), ptr(keys_out), ptr(vals_out), ptr(ws), ws.numel(), st,
                ),
                "intersect_tile (sort)",
            )
        return tiles_per_gauss, keys_out, vals_out
    cum = torch.empty(total, device=dev, dtype=torch.int64)
    with _Ctx(dev) as st:
        order = None
        if sort:
            # pass 0: rows in (image, depth) order, so that the S-sized sort below only has the (image, tile) bits left
            order = torch.empty(total, device=dev, dtype=torch.int32)
            ws = _scratch_buffer(dev, "dorder", L.gsb200_isect_depth_order_workspace_bytes(I, total))
            check(
                L.gsb200_isect_depth_order(I, N, ptr(radii), ptr(depths), ptr(img_ids), ptr(order), ptr(ws), ws.numel(), st),
                "intersect_tile (depth order)",
            )
        ws = _scratch_buffer(dev, "scan", L.gsb200_isect_scan_workspace_bytes(total))
        check(
            L.gsb200_isect_count(
                I_count, N, ptr(means2d), ptr(radii), ptr(conics) if accu else None, ptr(opacities) if accu else None,
                ptr(order), tile_size, tile_width, tile_height, ptr(tiles_per_gauss), ptr(cum), ptr(ws), ws.numel(), st,
            ),
            "intersect_tile (count)",
        )
        n_isects = int(cum[-1].item())  # the one host sync of the forward (reference: csrc/Intersect.cpp:259)
        isect_ids = torch.empty(n_isects, device=dev, dtype=torch.int64)
        flatten_ids = torch.empty(n_isects, device=dev, dtype=torch.int32)
        if n_isects == 0:
            return tiles_per_gauss, isect_ids, flatten_ids
        check(
            L.gsb200_isect_emit(
                I, N, ptr(means2d), ptr(radii), ptr(depths), ptr(conics) if accu else None,
                ptr(opacities) if accu else None, ptr(cum), ptr(img_ids), ptr(order), tile_size, tile_width, tile_height,
                ptr(isect_ids), ptr(flatten_ids), st,
            ),
            "intersect_tile (emit)",
        )
        if sort:
            begin_bit, end_bit = 32, 32 + tile_bits + image_bits
            keys_out, vals_out = torch.empty_like(isect_ids), torch.empty_like(flatten_ids)
            ws = _scratch_buffer(dev, "sort", L.gsb200_sort_workspace_bytes(n_isects, begin_bit, end_bit))
            check(
                L.gsb200_sort_pairs(
                    n_isects, begin_bit, end_bit, ptr(isect_ids), ptr(flatten_ids), ptr(keys_out), ptr(vals_out), ptr(ws),
                    ws.numel(), st,
                ),
                "intersect_tile (sort)",
            )
            isect_ids, flatten_ids = keys_out, vals_out
    return tiles_per_gauss, isect_ids, flatten_ids


class _IsectPredictor:
    """Capacities for gsb200_isect_sorted from the totals of the last calls on the same (device, image count, tile grid),
    and the asynchronous host read of the current totals (a kernel stores them into pinned memory, the host polls)."""

    def __init__(self, dev: torch.device):
        self.hist = []  # (n_isects, n_vis, max_tiles) of the last 8 calls
        self.hits = self.misses = 0
        self.pinned = torch.zeros(4, dtype=torch.int64).pin_memory()  # totals[3] + sequence word, written by the GPU
        self.words = self.pinned.numpy()  # same memory: what the host polls
        self.seq = 0
        self.zero_copy, self.copied, self.copy_done = True, None, None
        self.dev = dev

    def capacities(self, total_rows: int):
        if not self.hist:
            return None
        n_isects = max(h[0] for h in self.hist)
        n_vis = max(h[1] for h in self.hist)
        if n_isects == 0 or n_vis == 0:
            return None
        cap_vis = min(total_rows, n_vis + n_vis // 32 + 512)
        cap_isects = min(0x7FFFFFFF, n_isects + n_isects // 32 + 2048)
        return cap_vis, cap_isects, max(h[2] for h in self.hist)

    def observe(self, n_isects: int, n_vis: int, max_tiles: int):
        self.hist.append((n_isects, n_vis, max_tiles))
        del self.hist[:-8]

    def stage(self, totals: Tensor, st: int):
        """Queues, right behind the kernel that produced them, a one-warp kernel that stores the totals and then a
        sequence number into pinned host memory (no copy engine, no event)."""
        self.seq += 1
        self.copied = None
        if self.zero_copy:
            rc = lib().gsb200_publish_totals(ptr(totals), self.pinned.data_ptr(), self.seq, st)
            if rc == 0:
                return
            self.zero_copy = False  # pinned memory not device-mapped on this system: plain asynchronous copy from now on
        self.copied = torch.empty(3, dtype=torch.int64).pin_memory()
        self.copied.copy_(totals, non_blocking=True)
        self.copy_done = torch.cuda.Event()
        self.copy_done.record(torch.cuda.current_stream(self.dev))

    def read(self):
        """Polls the sequence word; the stores before it are ordered by the kernel's system-scope fence."""
        if self.copied is not None:
            self.copy_done.synchronize()
            return tuple(int(v) for v in self.copied.tolist())
        words, seq = self.words, self.seq
        spins = 0
        while int(words[3]) != seq:
            spins += 1
            if spins % 4_000_000 == 0:  # seconds without progress: surface a device-side failure instead of hanging
                torch.cuda.synchronize(self.dev)
                if int(words[3]) != seq:
                    raise RuntimeError("intersect_tile: the totals never arrived from the device")
        return int(words[0]), int(words[1]), int(words[2])


_predictors = {}


def _isect_predictor(dev: torch.device, I: int, tile_width: int, tile_height: int) -> _IsectPredictor:
    key = (dev.index, I, tile_width, tile_height, stream(dev.index))
    p = _predictors.get(key)
    if p is None:
        p = _predictors[key] = _IsectPredictor(dev)
    return p


class SortedIntersections:
    """What the compositing needs from the tile intersection, from the narrow-key pipeline: ``tiles_per_gauss``,
    ``flatten_ids`` (sorted by (image, tile, depth)), ``isect_offsets`` [I, th, tw].  The reference's sorted int64
    ``isect_ids`` are rebuilt from the sorted tile ids and the depths only when asked for (``isect_ids()``)."""

    __slots__ = ("tiles_per_gauss", "flatten_ids", "isect_offsets", "_keys", "_key_bytes", "_depths", "_geom", "_ids")

    def __init__(self, tiles_per_gauss, flatten_ids, isect_offsets, keys, key_bytes, depths, geom):
        self.tiles_per_gauss, self.flatten_ids, self.isect_offsets = tiles_per_gauss, flatten_ids, isect_offsets
        self._keys, self._key_bytes, self._depths, self._geom, self._ids = keys, key_bytes, depths, geom, None

    def isect_ids(self) -> Tensor:
        if self._ids is None:
            I, tw, th = self._geom
            n = self.flatten_ids.shape[0]
            ids = torch.empty(n, device=self.flatten_ids.device, dtype=torch.int64)
            if n > 0:
                with _Ctx(ids.device) as st:
                    check(
                        lib().gsb200_isect_ids_from_tilekeys(
                            n, self._key_bytes, ptr(self._keys), ptr(self.flatten_ids), ptr(self._depths), I, tw, th, ptr(ids), st,
                        ),
                        "intersect_tile (ids)",
                    )
            self._ids = ids
        return self._ids


@torch.no_grad()
def isect_tiles_sorted(
    means2d: Tensor, radii: Tensor, depths: Tensor, tile_size: int, tile_width: int, tile_height: int,
    conics: Optional[Tensor] = None, opacities: Optional[Tensor] = None, precounted: Optional[RowSideOutputs] = None,
) -> SortedIntersections:
    """Dense-layout tile intersection + offsets for rasterization(): same intersections in the same order as
    ``isect_tiles(sort=True)`` + ``isect_offset_encode`` (reference: csrc/Intersect.cpp:203-326, 330-382), with the
    S-sized sort done on 2- or 4-byte dense tile ids instead of the 8-byte (image | tile | depth) ids."""
    dev = require_cuda(means2d, radii, depths)
    means2d, depths = f32c(means2d, "means2d"), f32c(depths, "depths")
    conics, opacities = f32c(conics, "conics"), f32c(opacities, "opacities")
    if radii.dtype != torch.int32:
        raise TypeError("radii must be int32")
    radii = radii.contiguous()
    image_dims = tuple(means2d.shape[:-2])
    I, N = _prod(image_dims), means2d.shape[-2]
    L = lib()
    n_tiles = tile_width * tile_height
    image_bits, tile_bits = _cabi.bits_for_count(I), _cabi.bits_for_count(n_tiles)
    if image_bits + tile_bits > 32:
        raise RuntimeError(
            f"intersect_tile: (image, tile) id packing needs {image_bits + tile_bits} bits but only 32 are "
            f"available (I={I}, n_tiles={n_tiles})."
        )
    key_bits = _cabi.bits_for_count(I * n_tiles)
    key_bytes = 2 if key_bits <= 16 else 4
    key_dtype = torch.int16 if key_bytes == 2 else torch.int32  # raw storage; the kernels read them unsigned
    total = I * N
    have_counts = (
        precounted is not None and precounted.totals is not None and total > 0
        and (precounted.tile_size, precounted.tile_width, precounted.tile_height) == (tile_size, tile_width, tile_height)
        and precounted.tiles_per_gauss.numel() == total and conics is not None and opacities is not None
    )
    if have_counts:  # counted by the fused projection (same device function, same inputs)
        tiles_per_gauss = precounted.tiles_per_gauss.view(image_dims + (N,))
    else:
        tiles_per_gauss = torch.empty(image_dims + (N,), device=dev, dtype=torch.int32)
    offsets = torch.empty((I, tile_height, tile_width), device=dev, dtype=torch.int32)
    geom = (I, tile_width, tile_height)
    accu = conics is not None and opacities is not None

    def empty():
        offsets.zero_()
        return SortedIntersections(
            tiles_per_gauss.zero_(), torch.empty(0, device=dev, dtype=torch.int32), offsets,
            torch.empty(0, device=dev, dtype=key_dtype), key_bytes, depths, geom,
        )

    if total == 0:
        return empty()
    totals = precounted.totals if have_counts else torch.empty(3, device=dev, dtype=torch.int64)
    pred = _isect_predictor(dev, I, tile_width, tile_height)
    with _Ctx(dev) as st:
        if not have_counts:
            check(
                L.gsb200_isect_count_totals(
                    I, N, ptr(means2d), ptr(radii), ptr(conics) if accu else None, ptr(opacities) if accu else None, tile_size,
                    tile_width, tile_height, ptr(tiles_per_gauss), ptr(totals), st,
                ),
                "intersect_tile (count)",
            )

        def run(cap_vis: int, cap_isects: int, max_tiles: int):
            # compaction, depth order, scan, emission, tile sort, offsets: one call, every launch sized by the capacities
            keys_out = torch.empty(cap_isects, device=dev, dtype=key_dtype)
            vals_out = torch.empty(cap_isects, device=dev, dtype=torch.int32)
            ws = _scratch_buffer(dev, "isect", L.gsb200_isect_sorted_workspace_bytes(I, N, cap_vis, cap_isects, key_bytes, tile_width, tile_height))
            check(
                L.gsb200_isect_sorted(
                    I, N, ptr(means2d), ptr(radii), ptr(depths), ptr(conics) if accu else None, ptr(opacities) if accu else None,
                    tile_size, tile_width, tile_height, ptr(tiles_per_gauss), ptr(totals), cap_vis, cap_isects, max_tiles, key_bytes,
                    ptr(keys_out), ptr(vals_out), ptr(offsets), ptr(ws), ws.numel(), st,
                ),
                "intersect_tile (sorted)",
            )
            return keys_out, vals_out

        caps = pred.capacities(total)
        if caps is not None:
            # Launch on PREDICTED capacities, then read the totals: the host read (the reference's one sync of the forward,
            # csrc/Intersect.cpp:259) overlaps the queued stage instead of idling the GPU.  A miss (a count above its
            # capacity) costs one exact re-run; nothing is ever written past a capacity.
            pred.stage(totals, st)
            keys_out, vals_out = run(*caps)
            n_isects, n_vis, max_tiles = pred.read()
            pred.observe(n_isects, n_vis, max_tiles)
            if n_isects == 0:
                return empty()
            if n_vis > caps[0] or n_isects > caps[1]:
                pred.misses += 1
                keys_out, vals_out = run(n_vis, n_isects, max_tiles)
            else:
                pred.hits += 1
                keys_out, vals_out = keys_out[:n_isects], vals_out[:n_isects]
        else:
            n_isects, n_vis, max_tiles = (int(v) for v in totals.tolist())  # first call of a shape: exact sizes
            pred.observe(n_isects, n_vis, max_tiles)
            if n_isects == 0:
                return empty()
            keys_out, vals_out = run(n_vis, n_isects, max_tiles)
    return SortedIntersections(tiles_per_gauss, vals_out, offsets, keys_out, key_bytes, depths, geom)


@torch.no_grad()
def isect_offset_encode(isect_ids: Tensor, n_images: int, tile_width: int, tile_height: int) -> Tensor:
    """Sorted intersection ids -> per-(image, tile) start offsets, int32 [n_images, tile_height, tile_width]."""
    dev = require_cuda(isect_ids)
    if isect_ids.dtype != torch.int64:
        raise TypeError("isect_ids must be int64")
    isect_ids = isect_ids.contiguous()
    offsets = torch.empty((n_images, tile_height, tile_width), device=dev, dtype=torch.int32)
    with _Ctx(dev) as st:
        check(
            lib().gsb200_isect_offsets(isect_ids.shape[0], ptr(isect_ids), n_images, tile_width, tile_height, ptr(offsets), st),
            "intersect_offset",
        )
    return offsets


# --------------------------------------------------------------------------------------------
# rasterize_to_pixels

_SUPPORTED_CHANNELS = (1, 2, 3, 4, 5, 8, 16, 32)


def _grad_record_width(D: int, absgrad: bool) -> int:
    return ((6 + D + (2 if absgrad else 0)) + 3) // 4 * 4


class _RasterizeToPixels(torch.autograd.Function):
    @staticmethod
    def forward(
        ctx, means2d, conics, colors, opacities, backgrounds, masks, width, height, tile_size, isect_offsets,
        flatten_ids, absgrad_holder, row_records=None,
    ):
        dev = require_cuda(means2d, conics, colors, opacities)
        means2d, conics, colors, opacities = f32c(means2d, "means2d"), f32c(conics, "conics"), f32c(colors, "colors"), f32c(opacities, "opacities")
        backgrounds = f32c(backgrounds, "backgrounds")
        # image dims come from the offsets; the gaussian rows may be dense [..., N, *] or packed [nnz, *]
        image_dims = tuple(isect_offsets.shape[:-2])
        row_dims = tuple(means2d.shape[:-1])
        I, R, D = _prod(image_dims), _prod(row_dims), colors.shape[-1]
        # N only feeds the C ABI's 32-bit offset guard (I * N * stride < 2^32).  Dense rows: R == I * N.  Packed rows
        # [nnz, *] are addressed flat: ceil(R / I) keeps I * N within I - 1 rows of the real row count R.
        N = (R + I - 1) // I if I > 0 else R
        th, tw = isect_offsets.shape[-2:]
        m8 = None
        if masks is not None:
            m8 = masks.contiguous().view(torch.uint8) if masks.dtype == torch.bool else masks.to(torch.uint8).contiguous()
        offsets = isect_offsets.contiguous()
        fl = flatten_ids.contiguous()
        if offsets.dtype != torch.int32 or fl.dtype != torch.int32:
            raise TypeError("isect_offsets and flatten_ids must be int32")
        S = fl.shape[0]
        L = lib()
        records = torch.empty(max(L.gsb200_raster_records_bytes(S, D, I * th * tw), 16), device=dev, dtype=torch.uint8)
        o = dict(device=dev, dtype=torch.float32)
        render_colors = torch.empty(image_dims + (height, width, D), **o)
        render_alphas = torch.empty(image_dims + (height, width, 1), **o)
        last_ids = torch.empty(image_dims + (height, width), device=dev, dtype=torch.int32)
        with _Ctx(dev) as st:
            if row_records is not None and D <= 4 and row_records.numel() == R * 16:
                check(
                    L.gsb200_raster_fwd_rows(
                        I, N, D, ptr(row_records), ptr(backgrounds), ptr(m8), width, height, tile_size, tw, th, ptr(offsets),
                        ptr(fl), S, ptr(records), ptr(render_colors), ptr(render_alphas), ptr(last_ids), st,
                    ),
                    "rasterize_to_pixels_3dgs (row records)",
                )
            else:
                check(
                    L.gsb200_raster_fwd(
                        I, N, D, ptr(means2d), ptr(conics), ptr(colors), ptr(opacities), ptr(backgrounds), ptr(m8), width,
                        height, tile_size, tw, th, ptr(offsets), ptr(fl), S, ptr(records), ptr(render_colors),
                        ptr(render_alphas), ptr(last_ids), st,
                    ),
                    "rasterize_to_pixels_3dgs",
                )
        ctx.save_for_backward(backgrounds, m8, offsets, fl, records, render_alphas, last_ids)
        ctx.set_materialize_grads(False)
        ctx.absgrad_holder = absgrad_holder  # filled in place by backward; deliberately not a saved tensor
        ctx.meta = (row_dims, I, N, R, D, width, height, tile_size, tw, th, S)
        return render_colors, render_alphas

    @staticmethod
    def backward(ctx, v_render_colors, v_render_alphas):
        backgrounds, m8, offsets, fl, records, render_alphas, last_ids = ctx.saved_tensors
        absgrad_holder = ctx.absgrad_holder
        row_dims, I, N, R, D, width, height, tile_size, tw, th, S = ctx.meta
        dev = render_alphas.device
        # set_materialize_grads(False): an output the loss does not use arrives as None instead of a zero-filled tensor
        # (render_alphas in a plain photometric loss: 8 MB of zeros per 1080p step); the kernel takes a null pointer for it
        if v_render_colors is None:
            v_render_colors = torch.zeros(render_alphas.shape[:-1] + (D,), device=dev, dtype=torch.float32)
        v_render_colors = v_render_colors.contiguous()
        v_render_alphas = v_render_alphas.contiguous() if v_render_alphas is not None else None
        absgrad = absgrad_holder is not None
        P = _grad_record_width(D, absgrad)
        # one packed gradient record per gaussian: [v_xy 2 | v_conic 3 | v_opacity 1 | v_rgb D | (abs 2) | pad]
        rec = torch.zeros((R, P), device=dev, dtype=torch.float32)
        base = rec.data_ptr()
        with _Ctx(dev) as st:
            check(
                lib().gsb200_raster_bwd(
                    I, N, D, ptr(backgrounds), ptr(m8), width, height, tile_size, tw, th, ptr(offsets), ptr(fl), S,
                    ptr(records), ptr(render_alphas), ptr(last_ids), ptr(v_render_colors), ptr(v_render_alphas),
                    base, P, base + 8, P, base + 24, P, base + 20, P, (base + 4 * (6 + D)) if absgrad else None, P, st,
                ),
                "rasterize_to_pixels_3dgs_bwd",
            )
        rec = rec.view(row_dims + (P,))
        v_means2d, v_conics, v_opacities, v_colors = rec[..., 0:2], rec[..., 2:5], rec[..., 5], rec[..., 6 : 6 + D]
        if absgrad:
            absgrad_holder.copy_(rec[..., 6 + D : 8 + D])
        v_backgrounds = None
        if backgrounds is not None and ctx.needs_input_grad[4]:
            v_backgrounds = (v_render_colors * (1.0 - render_alphas)).sum(dim=(-3, -2))
        return (v_means2d, v_conics, v_colors, v_opacities, v_backgrounds) + (None,) * 8


def rasterize_to_pixels(
    means2d: Tensor,  # [..., N, 2]
    conics: Tensor,  # [..., N, 3]
    colors: Tensor,  # [..., N, channels]
    opacities: Tensor,  # [..., N]
    image_width: int,
    image_height: int,
    tile_size: int,
    isect_offsets: Tensor,  # [..., tile_height, tile_width]
    flatten_ids: Tensor,  # [n_isects]
    backgrounds: Optional[Tensor] = None,  # [..., channels]
    masks: Optional[Tensor] = None,  # [..., tile_height, tile_width]
    packed: bool = False,
    absgrad: bool = False,
) -> Tuple[Tensor, Tensor]:
    """Front-to-back alpha compositing of depth-sorted Gaussians per 16x16 tile.
    Returns (render_colors [..., H, W, channels], render_alphas [..., H, W, 1]).  With ``absgrad`` the
    backward fills ``means2d.absgrad``."""
    return rasterize_to_pixels_rows(
        means2d, conics, colors, opacities, image_width, image_height, tile_size, isect_offsets, flatten_ids, backgrounds,
        masks, packed, absgrad, None,
    )


def rasterize_to_pixels_rows(
    means2d, conics, colors, opacities, image_width, image_height, tile_size, isect_offsets, flatten_ids, backgrounds=None,
    masks=None, packed=False, absgrad=False, _row_records: Optional[Tensor] = None,
) -> Tuple[Tensor, Tensor]:
    """rasterize_to_pixels with the optional ``RowSideOutputs.rows`` of the fused projection that produced the inputs
    (rasterization() passes them; the forward's pack pass then only gathers)."""
    if packed != (means2d.dim() == 2):
        raise ValueError(f"packed={packed} but means2d has shape {tuple(means2d.shape)}")
    if tile_size != 16:
        raise ValueError(f"Unsupported tile_size {tile_size}; gsplat_b200 is built for tile_size 16")
    D = colors.shape[-1]
    if D > 32:
        raise ValueError(
            f"Unsupported number of color channels: {D}. gsplat_b200 rasterizes up to 32 channels per pass "
            "(rasterization() chunks wider features with channel_chunk=32)."
        )
    pad = 0
    if D not in _SUPPORTED_CHANNELS:
        target = next(c for c in _SUPPORTED_CHANNELS if c >= D)
        pad = target - D
        colors = torch.nn.functional.pad(colors, (0, pad))
        if backgrounds is not None:
            backgrounds = torch.nn.functional.pad(backgrounds, (0, pad))
    holder = torch.zeros_like(means2d) if absgrad else None
    render_colors, render_alphas = _RasterizeToPixels.apply(
        means2d, conics, colors, opacities, backgrounds, masks, int(image_width), int(image_height), int(tile_size),
        isect_offsets, flatten_ids, holder, _row_records if pad == 0 else None,
    )
    if absgrad:
        means2d.absgrad = holder
    if pad:
        render_colors = render_colors[..., :D]
    return render_colors, render_alphas


# --------------------------------------------------------------------------------------------
# MCMC strategy ops ("next" row, SURVEY.md section 8f.3)


@torch.no_grad()
def compute_relocation(
    opacities: Tensor, scales: Tensor, ratios: Tensor, binoms: Tensor, min_opacity: float = 0.005
) -> Tuple[Tensor, Tensor]:
    """Eq. 9 of "3D Gaussian Splatting as Markov Chain Monte Carlo": opacities / scales of Gaussians that are
    split into ``ratios`` copies.  Mirrors gsplat.relocation.compute_relocation
    (/root/reference/gsplat/relocation.py:25-80): ``ratios`` is clamped to [1, n_max] in place."""
    dev = require_cuda(opacities, scales, ratios, binoms)
    N = opacities.shape[0]
    n_max = binoms.shape[0]
    assert scales.shape == (N, 3), scales.shape
    assert ratios.shape == (N,), ratios.shape
    opacities, scales, binoms = f32c(opacities, "opacities"), f32c(scales, "scales"), f32c(binoms, "binoms")
    ratios.clamp_(min=1, max=n_max)
    r32 = ratios.int().contiguous()
    new_opacities, new_scales = torch.empty_like(opacities), torch.empty_like(scales)
    with _Ctx(dev) as st:
        check(
            lib().gsb200_relocation(
                N, ptr(opacities), ptr(scales), ptr(r32), ptr(binoms), n_max, float(min_opacity), ptr(new_opacities),
                ptr(new_scales), st,
            ),
            "relocation",
        )
    return new_opacities, new_scales


@torch.no_grad()
def mcmc_perturb_positions(
    positions: Tensor, quats: Tensor, scales_log: Tensor, opacities_logit: Tensor, noise: Tensor, noise_scale: float,
    t: float = 0.005, k: float = 100.0,
) -> None:
    """In place: positions += Sigma(quats, exp(scales_log)) @ (noise * sigmoid(-k (sigmoid(opacities_logit) - t))
    * noise_scale)   (/root/reference/gsplat/cuda/csrc/MCMCPerturbCUDA.cu:28-60)."""
    dev = require_cuda(positions, quats, scales_log, opacities_logit, noise)
    if not positions.is_contiguous() or positions.dtype != torch.float32:
        raise ValueError("positions must be a contiguous float32 tensor (updated in place)")
    N = positions.shape[0]
    quats, scales_log = f32c(quats, "quats"), f32c(scales_log, "scales")
    opacities_logit, noise = f32c(opacities_logit, "opacities"), f32c(noise, "noise")
    with _Ctx(dev) as st:
        check(
            lib().gsb200_mcmc_perturb_positions(
                N, ptr(positions), ptr(quats), ptr(scales_log), ptr(opacities_logit), ptr(noise), float(noise_scale),
                float(t), float(k), st,
            ),
            "mcmc_perturb_positions",
        )


@torch.no_grad()
def adam(
    param: Tensor, param_grad: Tensor, exp_avg: Tensor, exp_avg_sq: Tensor, valid: Optional[Tensor], lr: float, b1: float,
    b2: float, eps: float,
) -> None:
    """Selective Adam step, in place on ``param`` / ``exp_avg`` / ``exp_avg_sq`` ([N, ...]); rows with
    ``valid[n] == False`` keep their value and their moments (/root/reference/gsplat/cuda/_wrapper.py:419-432,
    csrc/AdamCUDA.cu:34-70; no bias correction, like the reference)."""
    dev = require_cuda(param, param_grad, exp_avg, exp_avg_sq)
    for name, t in (("param", param), ("exp_avg", exp_avg), ("exp_avg_sq", exp_avg_sq)):
        if t.dtype != torch.float32 or not t.is_contiguous():
            raise ValueError(f"{name} must be a contiguous float32 tensor (updated in place)")
        if t.shape != param.shape:
            raise ValueError(f"{name} must have the shape of param")
    if param_grad.shape != param.shape:
        raise ValueError("param_grad must have the shape of param")
    param_grad = f32c(param_grad, "param_grad")
    N = param.shape[0] if param.dim() > 0 else 1
    D = param.numel() // max(N, 1)
    vmask = None
    if valid is not None:
        if valid.numel() != N:
            raise ValueError(f"valid must have {N} entries, got {valid.numel()}")
        vmask = valid.to(device=dev, dtype=torch.bool).contiguous()
    with _Ctx(dev) as st:
        check(
            lib().gsb200_adam(
                N, D, ptr(param), ptr(param_grad), ptr(exp_avg), ptr(exp_avg_sq), ptr(vmask), float(lr), float(b1), float(b2),
                float(eps), st,
            ),
            "adam",
        )
