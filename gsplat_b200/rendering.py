"""rasterization(): the public entry point, signature-compatible with the reference
(/root/reference/gsplat/rendering.py:234-690).  Orchestration (projection -> SH -> tile intersection ->
offsets -> compositing, channel chunking, depth channels, meta dict) stays in Python and follows the
reference's own Python restatement ``_rasterization`` (rendering.py:722-1106) and the C++ orchestrator it
mirrors (csrc/Rendering.cpp:745-1481); every kernel is ours (gsplat_b200.ops).

Scope: the 3DGS EWA path named by BASELINE.json (pinhole / orthographic / fisheye cameras, dense or
``packed=True`` rows with optional ``sparse_grad``, classic / antialiased, RGB / D / ED / RGB+D / RGB+ED,
backgrounds, masks, absgrad, SH or post-activation colours, ``distributed=True`` Gaussian sharding).
3DGUT (with_ut / with_eval3d), lidar, distortion, rolling shutter, extra signals and normals are out of scope
and raise NotImplementedError.
"""
from __future__ import annotations

import math
from typing import Dict, Optional, Tuple

import torch
from torch import Tensor

from .ops import (
    RowSideOutputs,
    fully_fused_projection,
    fused_project_sh,
    isect_offset_encode,
    isect_tiles,
    isect_tiles_sorted,
    rasterize_to_pixels,
    rasterize_to_pixels_rows,
    spherical_harmonics,
    spherical_harmonics_rows,
)


_COLOR_MODES = {"RGB", "RGB-d", "RGB-Ed", "RGB+D", "RGB+ED"}
_HIT_DISTANCE_MODES = {"d", "Ed", "RGB-d", "RGB-Ed"}
_DEPTH_MODES = {"D", "ED", "RGB+D", "RGB+ED"}
_EXPECTED_MODES = {"Ed", "ED", "RGB-Ed", "RGB+ED"}
_ALL_MODES = _COLOR_MODES | _HIT_DISTANCE_MODES | _DEPTH_MODES


class _Lazy:
    """A meta value that is only computed when somebody reads it."""

    __slots__ = ("fn",)

    def __init__(self, fn):
        self.fn = fn


class _Meta(dict):
    """The meta dict of rasterization(); ``_Lazy`` values are computed on first access and then stored.  Every read path
    resolves them (the Python-level ``__iter__`` also keeps ``dict(meta)`` / ``{**meta}`` off CPython's raw-entry fast path)."""

    def _resolve(self, key):
        v = dict.__getitem__(self, key)
        if isinstance(v, _Lazy):
            v = v.fn()
            dict.__setitem__(self, key, v)
        return v

    def _resolve_all(self):
        for k in list(dict.keys(self)):
            self._resolve(k)

    def __getitem__(self, key):
        return self._resolve(key)

    def get(self, key, default=None):
        return self._resolve(key) if dict.__contains__(self, key) else default

    def __iter__(self):
        return dict.__iter__(self)

    def items(self):
        self._resolve_all()
        return dict.items(self)

    def values(self):
        self._resolve_all()
        return dict.values(self)

    def copy(self):
        self._resolve_all()
        return dict(dict.items(self))

    def pop(self, key, *default):
        if dict.__contains__(self, key):
            self._resolve(key)
        return dict.pop(self, key, *default)


def _unsupported(name: str, why: str = "out of scope for the gsplat_b200 hot path (SURVEY.md section 8)"):
    raise NotImplementedError(f"rasterization({name}): {why}")


def _project_dense(
    means, covars, quats, scales, opacities, colors, viewmats, Ks, width, height, sh_degree, eps2d, near_plane, far_plane,
    radius_clip, antialiased, camera_model, has_color, nb, batch_dims, C, N, rows_out=None,
):
    """Dense [..., C, N] projection (+ SH): the fused single pass when it applies, else the per-op kernels."""
    fused = (
        has_color and sh_degree is not None and covars is None and nb == 0 and colors.shape[-1] == 3
        and not viewmats.requires_grad and camera_model == "pinhole"
    )
    if fused:
        radii, means2d, depths, conics, feat, compensations = fused_project_sh(
            means, quats, scales, opacities, colors, viewmats, Ks, width, height, sh_degree, eps2d, near_plane,
            far_plane, radius_clip, antialiased, rows_out=rows_out,
        )
    else:
        radii, means2d, depths, conics, compensations = fully_fused_projection(
            means, covars, quats, scales, viewmats, Ks, width, height, eps2d=eps2d, near_plane=near_plane,
            far_plane=far_plane, radius_clip=radius_clip, packed=False, calc_compensations=antialiased,
            camera_model=camera_model, opacities=opacities,
        )
        feat = None
        if has_color:
            if sh_degree is None:
                feat = colors
                if feat.dim() == nb + 2:
                    feat = torch.broadcast_to(feat[..., None, :, :], batch_dims + (C, N, feat.shape[-1]))
            else:
                valid = (radii > 0).all(dim=-1)
                feat = spherical_harmonics(sh_degree, means, viewmats, colors, masks=valid)
                feat = torch.clamp_min(feat + 0.5, 0.0)

    opac = torch.broadcast_to(opacities[..., None, :], batch_dims + (C, N))
    if compensations is not None:
        opac = opac * compensations
    return radii, means2d, depths, conics, feat, compensations, opac


def rasterization(
    means: Tensor,  # [..., N, 3]
    quats: Optional[Tensor],  # [..., N, 4]
    scales: Optional[Tensor],  # [..., N, 3]
    opacities: Tensor,  # [..., N]
    colors: Optional[Tensor],  # [..., (C,) N, D] or [N, K, 3] SH coefficients
    viewmats: Tensor,  # [..., C, 4, 4]
    Ks: Tensor,  # [..., C, 3, 3]
    width: int,
    height: int,
    near_plane: float = 0.01,
    far_plane: float = 1e10,
    radius_clip: float = 0.0,
    eps2d: float = 0.3,
    sh_degree: Optional[int] = None,
    packed: bool = True,
    tile_size: Optional[int] = None,
    backgrounds: Optional[Tensor] = None,
    render_mode: str = "RGB",
    sparse_grad: bool = False,
    absgrad: bool = False,
    rasterize_mode: str = "classic",
    channel_chunk: int = 32,
    distributed: bool = False,
    camera_model: str = "pinhole",
    segmented: bool = False,
    covars: Optional[Tensor] = None,
    with_ut: bool = False,
    with_eval3d: bool = False,
    return_normals: bool = False,
    global_z_order: bool = True,
    rays: Optional[Tensor] = None,
    radial_coeffs: Optional[Tensor] = None,
    tangential_coeffs: Optional[Tensor] = None,
    thin_prism_coeffs: Optional[Tensor] = None,
    ftheta_coeffs=None,
    lidar_coeffs=None,
    external_distortion_coeffs=None,
    rolling_shutter=None,
    viewmats_rs: Optional[Tensor] = None,
    ut_params=None,
    extra_signals: Optional[Tensor] = None,
    extra_signals_sh_degree: Optional[int] = None,
    renderer_config=None,
) -> Tuple[Tensor, Tensor, Dict]:
    """Rasterize N 3D Gaussians to C image planes.  Returns (render_colors [..., C, H, W, X],
    render_alphas [..., C, H, W, 1], meta) with the reference's meta keys."""
    # ---- features outside the path
    if with_ut or with_eval3d:
        _unsupported("with_ut/with_eval3d", "3DGUT is a different algorithm (SURVEY.md section 2.1 #16)")
    for name, val in (
        ("rays", rays), ("radial_coeffs", radial_coeffs), ("tangential_coeffs", tangential_coeffs),
        ("thin_prism_coeffs", thin_prism_coeffs), ("ftheta_coeffs", ftheta_coeffs), ("lidar_coeffs", lidar_coeffs),
        ("external_distortion_coeffs", external_distortion_coeffs), ("viewmats_rs", viewmats_rs),
        ("ut_params", ut_params), ("extra_signals", extra_signals),
    ):
        if val is not None:
            _unsupported(name)
    # renderer_config selects the implementation of the eval3d rasterizer (reference rendering.py:548-556); the classic
    # path only admits the default RendererConfig_MixedBatch, which changes nothing here
    if renderer_config is not None and type(renderer_config).__name__ != "RendererConfig_MixedBatch":
        _unsupported(f"renderer_config={type(renderer_config).__name__}", "eval3d renderer variants are out of scope")
    if return_normals:
        _unsupported("return_normals")
    if rolling_shutter is not None and getattr(rolling_shutter, "name", str(rolling_shutter)) not in ("GLOBAL", "RollingShutterType.GLOBAL"):
        _unsupported("rolling_shutter")
    if camera_model not in ("pinhole", "ortho", "fisheye"):
        _unsupported(f"camera_model={camera_model!r}", "the EWA projection is built for pinhole / ortho / fisheye")
    if render_mode not in _ALL_MODES:
        raise ValueError(f"unknown render_mode {render_mode!r}")
    if render_mode in _HIT_DISTANCE_MODES:
        _unsupported(f"render_mode={render_mode!r}", "hit-distance modes belong to the eval3d (3DGUT) renderer")
    if rasterize_mode not in ("classic", "antialiased"):
        raise ValueError(f"unknown rasterize_mode {rasterize_mode!r}")
    if sparse_grad and not packed:
        raise ValueError("sparse_grad requires packed=True")
    if sparse_grad and distributed:
        _unsupported("sparse_grad with distributed=True")
    world_size, world_rank = 1, 0
    if distributed:
        # reference: rendering.py:178-197 -- needs an initialised default group; NCCL in the reference (the CPU
        # tests of the host logic here run it over gloo)
        if not (torch.distributed.is_available() and torch.distributed.is_initialized()):
            raise ValueError("distributed=True requires an initialized default torch.distributed process group.")
        world_size, world_rank = torch.distributed.get_world_size(), torch.distributed.get_rank()
        # the reference's distributed-mode rejections (csrc/Rendering.cpp:187-232), same wording
        if len(tuple(means.shape[:-2])) != 0:
            raise ValueError("distributed=True does not support batch dimensions")
        if absgrad:
            raise ValueError("distributed=True does not support absgrad=True")
        if camera_model != "pinhole":
            raise ValueError("distributed=True only supports camera_model='pinhole'")
        if not global_z_order:
            raise ValueError("distributed=True does not support global_z_order=False")
        if colors is not None and sh_degree is None and colors.dim() == 3:
            raise ValueError("distributed=True only supports per-Gaussian colors")
    if tile_size is None:
        tile_size = 16
    if tile_size != 16:
        raise ValueError(f"Unsupported tile_size {tile_size}; gsplat_b200 is built for tile_size 16")

    has_color = render_mode in _COLOR_MODES
    has_depth = render_mode in _DEPTH_MODES
    batch_dims = tuple(means.shape[:-2])
    nb = len(batch_dims)
    B = math.prod(batch_dims) if batch_dims else 1
    N = means.shape[-2]
    C = viewmats.shape[-3]
    I = B * C

    # ---- shape validation (reference rendering.py:526-556 / Rendering.cpp:97-512)
    if means.shape[-1] != 3:
        raise ValueError(f"means must be [..., N, 3], got {tuple(means.shape)}")
    if covars is None:
        if quats is None or scales is None:
            raise ValueError("either covars or (quats, scales) is required")
        if tuple(quats.shape) != batch_dims + (N, 4) or tuple(scales.shape) != batch_dims + (N, 3):
            raise ValueError(f"quats/scales shape mismatch: {tuple(quats.shape)}, {tuple(scales.shape)}")
    else:
        if tuple(covars.shape) != batch_dims + (N, 3, 3):
            raise ValueError(f"covars must be [..., N, 3, 3], got {tuple(covars.shape)}")
        quats = scales = None
        tri = ([0, 0, 0, 1, 1, 2], [0, 1, 2, 1, 2, 2])
        covars = covars[..., tri[0], tri[1]]
    if tuple(opacities.shape) != batch_dims + (N,):
        raise ValueError(f"opacities must be [..., N], got {tuple(opacities.shape)}")
    if tuple(viewmats.shape) != batch_dims + (C, 4, 4) or tuple(Ks.shape) != batch_dims + (C, 3, 3):
        raise ValueError(f"viewmats/Ks shape mismatch: {tuple(viewmats.shape)}, {tuple(Ks.shape)}")
    if has_color:
        if colors is None:
            raise ValueError(f"render_mode={render_mode!r} needs colors")
        if sh_degree is None:
            ok = (colors.dim() == nb + 2 and tuple(colors.shape[:-1]) == batch_dims + (N,)) or (
                colors.dim() == nb + 3 and tuple(colors.shape[:-1]) == batch_dims + (C, N)
            )
            if not ok:
                raise ValueError(f"colors must be [..., N, D] or [..., C, N, D], got {tuple(colors.shape)}")
        else:
            if colors.dim() != 3 or colors.shape[0] != N:
                raise ValueError(f"SH colors must be [N, K, D], got {tuple(colors.shape)}")
            if (sh_degree + 1) ** 2 > colors.shape[-2]:
                raise ValueError(f"sh_degree={sh_degree} needs K >= {(sh_degree + 1) ** 2}, got {colors.shape[-2]}")

    antialiased = rasterize_mode == "antialiased"

    # ---- Seam A (distributed=True): every rank projects ITS gaussians onto ALL cameras
    C_world, N_world = [C], [N]
    if distributed and world_size > 1:
        from . import distributed as gdist

        N_world = gdist.all_gather_ints(N, means.device)
        C_world = gdist.all_gather_ints(C, means.device)
        viewmats, Ks = gdist.all_gather_rows([viewmats, Ks], C_world)
        C = sum(C_world)
        if backgrounds is not None and tuple(backgrounds.shape[:-1]) != (C_world[world_rank],):
            raise ValueError("backgrounds must be [C_local, D] under distributed=True")

    # ---- packed=True: native two-pass compacting projection; everything downstream works on the [nnz, ...] rows
    # (reference rendering.py:347-353, Rendering.cpp:936-973).  Under a multi-rank distributed=True the compacted
    # rows are what Seam B exchanges (only the visible (camera, gaussian) pairs travel).
    sharded = distributed and world_size > 1
    native_packed = packed
    camera_ids = gaussian_ids = batch_ids = None
    rows_out = None
    if native_packed:
        batch_ids, camera_ids, gaussian_ids, indptr, radii, means2d, depths, conics, compensations = fully_fused_projection(
            means, covars, quats, scales, viewmats, Ks, width, height, eps2d=eps2d, near_plane=near_plane,
            far_plane=far_plane, radius_clip=radius_clip, packed=True, sparse_grad=sparse_grad,
            calc_compensations=antialiased, camera_model=camera_model, opacities=opacities,
        )
        grow = batch_ids * N + gaussian_ids  # row of the gaussian in the flattened [B*N] parameter tensors
        # index_select: its backward is an atomic index_add (advanced indexing would sort the nnz indices)
        opac = torch.index_select(opacities.reshape(-1), 0, grow)
        if compensations is not None:
            opac = opac * compensations
        feat = None
        if has_color:
            if sh_degree is None:
                if colors.dim() == nb + 2:
                    feat = torch.index_select(colors.reshape(-1, colors.shape[-1]), 0, grow)
                else:
                    feat = torch.index_select(
                        colors.reshape(-1, colors.shape[-1]), 0, (batch_ids * C + camera_ids) * N + gaussian_ids
                    )
            else:
                feat = spherical_harmonics_rows(sh_degree, means, viewmats, colors, batch_ids, camera_ids, gaussian_ids)
                feat = torch.clamp_min(feat + 0.5, 0.0)
    else:
        # the fused projection can also count tiles and write the compositing row records, when what follows composites
        # exactly its outputs: plain RGB, input opacities (no antialiasing compensation), rows not exchanged between ranks
        if render_mode == "RGB" and not antialiased and not sharded:
            rows_out = RowSideOutputs(tile_size, math.ceil(width / float(tile_size)), math.ceil(height / float(tile_size)))
        radii, means2d, depths, conics, feat, compensations, opac = _project_dense(
            means, covars, quats, scales, opacities, colors, viewmats, Ks, width, height, sh_degree, eps2d, near_plane, far_plane,
            radius_clip, antialiased, camera_model, has_color, nb, batch_dims, C, N, rows_out=rows_out,
        )
        if rows_out is not None and rows_out.rows is None:
            rows_out = None  # the per-op projection ran: nothing precomputed

    # ---- Seam B (distributed=True): all-to-all so that each rank holds ALL gaussians projected onto ITS cameras
    if sharded and packed:
        # rows are sorted by (camera, gaussian): the rows of rank d's cameras are one contiguous range
        C_local = C_world[world_rank]
        cam0 = [sum(C_world[:d]) for d in range(world_size + 1)]
        ip = indptr.tolist()
        send = [ip[cam0[d + 1]] - ip[cam0[d]] for d in range(world_size)]
        recv = [row[world_rank] for row in gdist.all_gather_int_lists(send, means.device)]
        g0 = sum(N_world[:world_rank])  # global index of this rank's first gaussian
        ints = torch.stack([radii[:, 0], radii[:, 1], (gaussian_ids + g0).int(), camera_ids.int()], dim=-1)
        fields = [means2d, depths, conics, opac] + ([feat] if feat is not None else []) + [ints]
        got = gdist.all_to_all_rows(fields, send, recv)
        means2d, depths, conics, opac = got[0], got[1], got[2], got[3]
        if feat is not None:
            feat = got[4]
        ints = got[-1]
        radii = ints[:, :2].contiguous()
        gaussian_ids = ints[:, 2].long()
        camera_ids = ints[:, 3].long() - cam0[world_rank]
        batch_ids = torch.zeros_like(camera_ids)
        C, N = C_local, sum(N_world)
        I = C
    elif sharded:
        C_local = C_world[world_rank]
        send = [c * N for c in C_world]          # rows (camera-major) going to each camera owner
        recv = [C_local * n for n in N_world]    # rows arriving from each gaussian owner
        fields = [means2d.reshape(C * N, 2), depths.reshape(C * N), conics.reshape(C * N, 3), opac.reshape(C * N)]
        if feat is not None:
            if feat.dim() == 2:  # [N, D] shared by all cameras
                feat = torch.broadcast_to(feat[None], (C, N, feat.shape[-1]))
            fields.append(feat.reshape(C * N, feat.shape[-1]))
        fields.append(radii.reshape(C * N, 2))
        got = gdist.all_to_all_rows(fields, send, recv)
        loc = [gdist.camera_major_to_local(t, C_local, N_world) for t in got]
        means2d, depths, conics, opac = loc[0], loc[1], loc[2], loc[3]
        if feat is not None:
            feat = loc[4]
        radii = loc[-1].contiguous()
        C, N = C_local, sum(N_world)
        I = C

    # ---- tile intersection (AccuTile) + offsets
    tile_width = math.ceil(width / float(tile_size))
    tile_height = math.ceil(height / float(tile_size))
    # reference-shaped op sequence: (depth order,) count, emit, radix sort on the (image, tile) bits, offsets
    if native_packed:
        tiles_per_gauss, isect_ids, flatten_ids = isect_tiles(
            means2d, radii, depths, tile_size, tile_width, tile_height, sort=True, segmented=segmented, packed=True,
            n_images=I, image_ids=batch_ids * C + camera_ids, gaussian_ids=gaussian_ids, conics=conics, opacities=opac,
        )
        isect_offsets = isect_offset_encode(isect_ids, I, tile_width, tile_height)
    else:
        # dense rows: the S-sized sort runs on 2- / 4-byte tile ids; meta["isect_ids"] (the reference's 64-bit ids) is
        # rebuilt from them on first access
        hits = isect_tiles_sorted(
            means2d, radii, depths, tile_size, tile_width, tile_height, conics=conics, opacities=opac, precounted=rows_out,
        )
        tiles_per_gauss, flatten_ids, isect_offsets = hits.tiles_per_gauss, hits.flatten_ids, hits.isect_offsets
        isect_ids = _Lazy(hits.isect_ids)
    isect_offsets = isect_offsets.reshape(batch_dims + (C, tile_height, tile_width))

    # ---- assemble channels: [colour | depth]
    if has_color and has_depth:
        feat = torch.cat((feat, depths[..., None]), dim=-1)
        if backgrounds is not None:
            backgrounds = torch.cat([backgrounds, torch.zeros(batch_dims + (C, 1), device=backgrounds.device)], dim=-1)
    elif not has_color:
        feat = depths[..., None]
        if backgrounds is not None:
            backgrounds = torch.zeros(batch_dims + (C, 1), device=backgrounds.device)

    # ---- compositing (chunked over channels, reference Rendering.cpp:1353-1447)
    n_ch = feat.shape[-1]
    if n_ch > channel_chunk:
        outs, render_alphas = [], None
        for lo in range(0, n_ch, channel_chunk):
            bg = backgrounds[..., lo : lo + channel_chunk] if backgrounds is not None else None
            rc, ra = rasterize_to_pixels(
                means2d, conics, feat[..., lo : lo + channel_chunk], opac, width, height, tile_size, isect_offsets,
                flatten_ids, backgrounds=bg, packed=packed, absgrad=absgrad,
            )
            outs.append(rc)
            if render_alphas is None:
                render_alphas = ra
        render_colors = torch.cat(outs, dim=-1)
    else:
        render_colors, render_alphas = rasterize_to_pixels_rows(
            means2d, conics, feat, opac, width, height, tile_size, isect_offsets, flatten_ids, backgrounds=backgrounds,
            packed=packed, absgrad=absgrad, _row_records=rows_out.rows if (rows_out is not None and n_ch == 3) else None,
        )

    if render_mode in _EXPECTED_MODES:  # ED / RGB+ED: normalise accumulated depth
        depth = render_colors[..., -1:] / render_alphas.clamp(min=1e-10)
        render_colors = torch.cat([render_colors[..., :-1], depth], dim=-1)

    meta = _Meta({
        "batch_ids": batch_ids,
        "camera_ids": camera_ids,
        "gaussian_ids": gaussian_ids,
        "radii": radii,
        "means2d": means2d,
        "depths": depths,
        "conics": conics,
        "opacities": opac,
        "tile_width": tile_width,
        "tile_height": tile_height,
        "tiles_per_gauss": tiles_per_gauss,
        "isect_ids": isect_ids,
        "flatten_ids": flatten_ids,
        "isect_offsets": isect_offsets,
        "width": width,
        "height": height,
        "tile_size": tile_size,
        "n_batches": B,
        "n_cameras": C,
    })
    return render_colors, render_alphas, meta
