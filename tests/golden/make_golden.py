#!/usr/bin/env python
"""Generate the committed golden fixtures in tests/golden/ from the REFERENCE ITSELF.

Runs only in the build container (needs /root/reference).  The reference's pure-PyTorch
twins are imported unchanged and evaluated on the CPU in float64:

  * gsplat/cuda/_math.py:689        _quat_scale_to_covar_preci
  * gsplat/cuda/_torch_impl.py:262  _fully_fused_projection (+ _persp_proj :53, _world_to_cam :225)
  * gsplat/cuda/_torch_impl.py:1052 _spherical_harmonics (+ _eval_sh_bases_fast :968)
  * gsplat/cuda/_torch_impl.py:356  _isect_tiles, :455 _isect_offset_encode
  * gsplat/cuda/_torch_impl.py:713  accumulate  (alpha compositing; needs `nerfacc`)

`nerfacc` (setup.py:188 pins only ``nerfacc>=0.5.3``; not vendored, not installed) is replaced
by a 20-line shim restating its two published functions (render_weight_from_alpha =
alpha * exclusive cumprod(1 - alpha) per ray; accumulate_along_rays = segment sum of
weights * values) -- the reference's own alpha/sigma formula and autograd do the rest.

Also writes tests/golden/garden_{0,1}.npz: the cropped assets/test_garden.npz scene
(gsplat/_helper.py:51-102 load_test_data; crop [-2,2]^3 -> 111 785 points) so the GPU box,
which has no /root/reference, can rebuild BASELINE.json's configs.  quats / scales /
opacities are NOT stored: they are re-drawn with numpy's RandomState(42) by
tests/scene.py (the reference draws them on the device RNG, which is not portable).

Usage:  python tests/golden/make_golden.py        (from the repo root)
"""
import math
import os
import sys
import types

os.environ["CUDA_HOME"] = "/nonexistent"
os.environ["PATH"] = ":".join(p for p in os.environ["PATH"].split(":") if "cuda" not in p)
sys.path.insert(0, "/root/reference")
HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.abspath(os.path.join(HERE, "..", "..")))

import numpy as np
import torch

# ---- nerfacc shim (published algorithm, see module docstring) ----
nerfacc = types.ModuleType("nerfacc")


def render_weight_from_alpha(alphas, ray_indices=None, n_rays=None):
    # samples of one ray are contiguous and ordered front to back
    log1m = torch.log1p(-alphas)
    csum = torch.cumsum(log1m, 0)
    first = torch.ones_like(ray_indices, dtype=torch.bool)
    first[1:] = ray_indices[1:] != ray_indices[:-1]
    start_idx = torch.where(first)[0]
    seg = torch.cumsum(first.long(), 0) - 1
    base = (csum - log1m)[start_idx][seg]
    trans = torch.exp(csum - log1m - base)
    return alphas * trans, trans


def accumulate_along_rays(weights, values=None, ray_indices=None, n_rays=None):
    src = weights[:, None] if values is None else weights[:, None] * values
    out = torch.zeros((n_rays, src.shape[-1]), dtype=src.dtype)
    return out.index_add(0, ray_indices, src)


nerfacc.render_weight_from_alpha = render_weight_from_alpha
nerfacc.accumulate_along_rays = accumulate_along_rays
sys.modules["nerfacc"] = nerfacc

from gsplat.cuda._math import _quat_scale_to_covar_preci  # noqa: E402
from gsplat.cuda._torch_impl import (  # noqa: E402
    _fully_fused_projection,
    _isect_offset_encode,
    _isect_tiles,
    _spherical_harmonics,
    accumulate,
)

from oracle import gso  # noqa: E402  (used only to build the pair list for `accumulate`)

f64 = torch.float64


def save(name, **arrs):
    out = {}
    for k, v in arrs.items():
        if isinstance(v, torch.Tensor):
            v = v.detach().cpu().numpy()
        out[k] = v
    path = os.path.join(HERE, name)
    np.savez_compressed(path, **out)
    print(f"wrote {name}: {os.path.getsize(path) / 1e3:.1f} kB")


# ---------------------------------------------------------------- garden scene
def make_garden():
    d = np.load("/root/reference/assets/test_garden.npz")
    means = d["means3d"].astype(np.float32)
    sel = ((means >= -2.0) & (means <= 2.0)).all(-1)
    h = int(sel.sum()) // 2  # two halves: every stored file stays below 1 MB (tests/scene.py joins them)
    save(
        "garden_0.npz",
        means=means[sel][:h],
        colors=d["colors"][sel][:h],
        viewmats=d["viewmats"].astype(np.float32),
        Ks=d["Ks"].astype(np.float32),
        width=np.int64(d["width"]),
        height=np.int64(d["height"]),
    )
    save("garden_1.npz", means=means[sel][h:], colors=d["colors"][sel][h:])
    return means[sel], d["viewmats"].astype(np.float32), d["Ks"].astype(np.float32), int(d["width"]), int(d["height"])


# ---------------------------------------------------------------- quat/scale
def make_quat_scale(rng):
    N = 64
    quats = rng.standard_normal((N, 4)).astype(np.float32)
    scales = (rng.random((N, 3)) * 0.5 + 0.05).astype(np.float32)
    q = torch.tensor(quats, dtype=f64, requires_grad=True)
    s = torch.tensor(scales, dtype=f64, requires_grad=True)
    out = {}
    for triu in (False, True):
        cov, pre = _quat_scale_to_covar_preci(q, s, True, True, triu=triu)
        v_cov = torch.tensor(rng.standard_normal(tuple(cov.shape)))
        v_pre = torch.tensor(rng.standard_normal(tuple(pre.shape)))
        vq, vs = torch.autograd.grad((cov * v_cov).sum() + (pre * v_pre).sum(), (q, s))
        t = "_triu" if triu else ""
        out.update({f"covars{t}": cov, f"precis{t}": pre, f"v_covars{t}": v_cov, f"v_precis{t}": v_pre,
                    f"v_quats{t}": vq, f"v_scales{t}": vs})
    save("ref_quat_scale.npz", quats=quats, scales=scales, **out)


# ---------------------------------------------------------------- projection
def make_projection(rng, means_all, viewmats, Ks, W, H):
    N = 1500
    idx = rng.choice(len(means_all), N, replace=False)
    means = means_all[idx]
    quats = rng.standard_normal((N, 4)).astype(np.float32)
    quats /= np.linalg.norm(quats, axis=-1, keepdims=True)
    scales = (rng.random((N, 3)) * (0.02 - 1e-4) + 1e-4).astype(np.float32)
    scales[: N // 4] *= 20.0  # some big ones so the FOV clamp / large radii are exercised
    m = torch.tensor(means, dtype=f64, requires_grad=True)
    q = torch.tensor(quats, dtype=f64, requires_grad=True)
    s = torch.tensor(scales, dtype=f64, requires_grad=True)
    vm = torch.tensor(viewmats, dtype=f64, requires_grad=True)
    K = torch.tensor(Ks, dtype=f64)
    covars, _ = _quat_scale_to_covar_preci(q, s, True, False, triu=False)
    radii, means2d, depths, conics, comps = _fully_fused_projection(
        m, covars, vm, K, W, H, eps2d=0.3, near_plane=0.01, far_plane=1e10, calc_compensations=True
    )
    C = viewmats.shape[0]
    v_means2d = torch.tensor(rng.standard_normal((C, N, 2)))
    v_depths = torch.tensor(rng.standard_normal((C, N)))
    v_conics = torch.tensor(rng.standard_normal((C, N, 3)))
    v_comps = torch.tensor(rng.standard_normal((C, N)))
    valid = (radii > 0).all(-1)
    # cotangents only on the entries the CUDA path would also treat as valid
    loss = ((means2d * v_means2d).sum(-1) * valid).sum() + (depths * v_depths * valid).sum() \
        + ((conics * v_conics).sum(-1) * valid).sum() + (comps * v_comps * valid).sum()
    v_m, v_q, v_s, v_vm = torch.autograd.grad(loss, (m, q, s, vm), retain_graph=True)
    # same without the compensation cotangent (the CUDA rule's add_blur_vjp divides by comp + 1e-6,
    # include/Utils.cuh:486, so only this variant can agree to round-off)
    loss_nc = loss - (comps * v_comps * valid).sum()
    v_m_nc, v_q_nc, v_s_nc, v_vm_nc = torch.autograd.grad(loss_nc, (m, q, s, vm))
    save(
        "ref_projection.npz", means=means, quats=quats, scales=scales, viewmats=viewmats, Ks=Ks,
        width=np.int64(W), height=np.int64(H), radii=radii.int(), means2d=means2d, depths=depths, conics=conics,
        compensations=comps, v_means2d=v_means2d, v_depths=v_depths, v_conics=v_conics, v_compensations=v_comps,
        v_means=v_m, v_quats=v_q, v_scales=v_s, v_viewmats=v_vm,
        v_means_nc=v_m_nc, v_quats_nc=v_q_nc, v_scales_nc=v_s_nc, v_viewmats_nc=v_vm_nc,
    )


# ---------------------------------------------------------------- projection, ortho / fisheye cameras
def make_projection_cameras(means_all, viewmats, Ks, W, H):
    """_fully_fused_projection(camera_model=...) -> _ortho_proj (_torch_impl.py:180) / _fisheye_proj (:111),
    gradients by autograd (which differentiates the Jacobian as well, like the CUDA closed form)."""
    for model in ("ortho", "fisheye"):
        rng = np.random.RandomState({"ortho": 31, "fisheye": 32}[model])
        N = 600
        idx = rng.choice(len(means_all), N, replace=False)
        means = means_all[idx]
        quats = rng.standard_normal((N, 4)).astype(np.float32)
        quats /= np.linalg.norm(quats, axis=-1, keepdims=True)
        scales = (rng.random((N, 3)) * (0.02 - 1e-4) + 1e-4).astype(np.float32)
        scales[: N // 4] *= 20.0
        K_use = Ks.copy()
        if model == "ortho":  # pixels per world unit
            K_use[:, 0, 0] = 150.0
            K_use[:, 1, 1] = 140.0
        m = torch.tensor(means, dtype=f64, requires_grad=True)
        q = torch.tensor(quats, dtype=f64, requires_grad=True)
        s = torch.tensor(scales, dtype=f64, requires_grad=True)
        vm = torch.tensor(viewmats, dtype=f64, requires_grad=True)
        K = torch.tensor(K_use, dtype=f64)
        covars, _ = _quat_scale_to_covar_preci(q, s, True, False, triu=False)
        radii, means2d, depths, conics, comps = _fully_fused_projection(
            m, covars, vm, K, W, H, eps2d=0.3, near_plane=0.01, far_plane=1e10, calc_compensations=True, camera_model=model
        )
        C = viewmats.shape[0]
        v_means2d = torch.tensor(rng.standard_normal((C, N, 2)))
        v_depths = torch.tensor(rng.standard_normal((C, N)))
        v_conics = torch.tensor(rng.standard_normal((C, N, 3)))
        valid = (radii > 0).all(-1)
        loss = ((means2d * v_means2d).sum(-1) * valid).sum() + (depths * v_depths * valid).sum() \
            + ((conics * v_conics).sum(-1) * valid).sum()
        v_m, v_q, v_s, v_vm = torch.autograd.grad(loss, (m, q, s, vm))
        save(
            f"ref_projection_{model}.npz", means=means, quats=quats, scales=scales, viewmats=viewmats, Ks=K_use,
            width=np.int64(W), height=np.int64(H), radii=radii.int(), means2d=means2d, depths=depths, conics=conics,
            compensations=comps, v_means2d=v_means2d, v_depths=v_depths, v_conics=v_conics,
            v_means_nc=v_m, v_quats_nc=v_q, v_scales_nc=v_s, v_viewmats_nc=v_vm,
        )
        print(f"  {model}: {int(valid.sum())} of {valid.numel()} visible")


# ---------------------------------------------------------------- SH
def make_sh(rng, viewmats):
    N, D = 200, 3
    means = (rng.standard_normal((N, 3)) * 2).astype(np.float32)
    vm = torch.tensor(viewmats, dtype=f64)
    # camera position as the CUDA op recovers it: -R^T t (csrc/SphericalHarmonics.cuh:40-58), which
    # differs from inverse(viewmat) by ~1e-7 for the float32 (not exactly orthonormal) garden poses
    campos = -torch.einsum("cij,ci->cj", vm[:, :3, :3], vm[:, :3, 3])  # [C,3]
    out = {}
    for deg in range(5):
        K = (deg + 1) ** 2
        coeffs = rng.standard_normal((N, K, D)).astype(np.float32)
        m = torch.tensor(means, dtype=f64, requires_grad=True)
        cf = torch.tensor(coeffs, dtype=f64, requires_grad=True)
        dirs = m[None, :, :] - campos[:, None, :]
        colors = _spherical_harmonics(deg, dirs, cf)
        v_colors = torch.tensor(rng.standard_normal(tuple(colors.shape)))
        v_cf, v_m = torch.autograd.grad((colors * v_colors).sum(), (cf, m), allow_unused=True)
        if v_m is None:
            v_m = torch.zeros_like(m)
        out.update({f"coeffs{deg}": coeffs, f"colors{deg}": colors, f"v_colors{deg}": v_colors,
                    f"v_coeffs{deg}": v_cf, f"v_means{deg}": v_m})
    save("ref_sh.npz", means=means, viewmats=viewmats, **out)


# ---------------------------------------------------------------- isect (AABB mode), recipe of tests/test_basic.py:1288-1300
def make_isect(rng):
    C, N = 3, 1000
    width, height, tile_size = 40, 60, 16
    means2d = (rng.standard_normal((C, N, 2)) * width).astype(np.float32)
    radii = rng.randint(0, width, (C, N, 2)).astype(np.int32)
    depths = rng.random((C, N)).astype(np.float32)
    tw, th = math.ceil(width / tile_size), math.ceil(height / tile_size)
    tpg, ids, fl = _isect_tiles(torch.tensor(means2d), torch.tensor(radii), torch.tensor(depths), tile_size, tw, th)
    off = _isect_offset_encode(ids, C, tw, th)
    save("ref_isect.npz", means2d=means2d, radii=radii, depths=depths, tile_size=np.int64(tile_size),
         tile_width=np.int64(tw), tile_height=np.int64(th), tiles_per_gauss=tpg, isect_ids=ids, flatten_ids=fl,
         isect_offsets=off)


# ---------------------------------------------------------------- compositing through the reference's `accumulate`
def make_accumulate(rng):
    """Small synthetic scene (layout in the spirit of tests/test_basic.py:5421-5478): 160 gaussians on a
    48x40 image, 2 cameras, D=3 colours, with a background.  The (gaussian, pixel) pair list fed to the
    reference's accumulate() is the set of contributing pairs (sigma>=0, alpha>=1/255, not after the
    pixel's last contributor) -- what rasterize_to_indices (csrc/RasterizeToIndices3DGSSerialBatch.cu)
    would emit; it is built here from the oracle's forward (last_ids)."""
    C, N, D, W, H, ts = 2, 160, 3, 48, 40, 16
    means2d = np.stack([rng.random((C, N)) * W, rng.random((C, N)) * H], -1)
    sx, sy = rng.random((C, N)) * 6 + 0.8, rng.random((C, N)) * 6 + 0.8
    rho = rng.random((C, N)) * 1.6 - 0.8
    cov = np.stack([sx * sx, rho * sx * sy, sy * sy], -1)
    det = cov[..., 0] * cov[..., 2] - cov[..., 1] ** 2
    conics = np.stack([cov[..., 2] / det, -cov[..., 1] / det, cov[..., 0] / det], -1)
    opac = rng.random((C, N)) * 0.98 + 0.02
    opac[:, :20] = 1.0  # saturating ones -> exercises the 0.99 clamp and the transmittance stop
    colors = rng.random((C, N, D))
    depths = rng.random((C, N)) * 5 + 0.1
    radii = np.stack([np.ceil(3.33 * sx), np.ceil(3.33 * sy)], -1).astype(np.int32)
    bg = rng.random((C, D))
    f32 = lambda a: np.ascontiguousarray(a, np.float32)  # noqa: E731
    means2d, conics, opac, colors, depths, bg = map(f32, (means2d, conics, opac, colors, depths, bg))
    tw, th = math.ceil(W / ts), math.ceil(H / ts)
    d64 = lambda a: a.astype(np.float64)  # noqa: E731
    tpg, ids, fl = gso.isect_tiles(d64(means2d), radii, d64(depths), ts, tw, th, True, d64(conics), d64(opac))
    off = gso.isect_offset_encode(ids, C, tw, th)
    rc, ra, li, mg = gso.rasterize_to_pixels(d64(means2d), d64(conics), d64(colors), d64(opac), W, H, ts, off, fl,
                                             None, None, True)
    # pair list
    g_l, p_l, i_l = [], [], []
    offf = np.concatenate([off.reshape(-1), [len(fl)]])
    for img in range(C):
        for ty in range(th):
            for tx in range(tw):
                t = (img * th + ty) * tw + tx
                s0, s1 = int(offf[t]), int(offf[t + 1])
                for ly in range(ts):
                    for lx in range(ts):
                        i, j = ty * ts + ly, tx * ts + lx
                        if i >= H or j >= W:
                            continue
                        for s in range(s0, min(s1, li[img, i, j] + 1)):
                            g = fl[s] - img * N
                            dx, dy = (j + 0.5) - float(means2d[img, g, 0]), (i + 0.5) - float(means2d[img, g, 1])
                            a, b, c = map(float, conics[img, g])
                            sig = 0.5 * (a * dx * dx + c * dy * dy) + b * dx * dy
                            al = min(0.99, float(opac[img, g]) * math.exp(-sig))
                            if sig < 0 or al < 1.0 / 255.0:
                                continue
                            g_l.append(g), p_l.append(i * W + j), i_l.append(img)
    g_t, p_t, i_t = (torch.tensor(x, dtype=torch.long) for x in (g_l, p_l, i_l))
    # accumulate() wants pairs grouped per ray, front to back: sort by ray id, stable
    ray = i_t * H * W + p_t
    order = torch.sort(ray, stable=True)[1]
    g_t, p_t, i_t = g_t[order], p_t[order], i_t[order]
    m2 = torch.tensor(means2d, dtype=f64, requires_grad=True)
    cn = torch.tensor(conics, dtype=f64, requires_grad=True)
    op = torch.tensor(opac, dtype=f64, requires_grad=True)
    co = torch.tensor(colors, dtype=f64, requires_grad=True)
    bgt = torch.tensor(bg, dtype=f64, requires_grad=True)
    renders, alphas = accumulate(m2, cn, op, co, g_t, p_t, i_t, W, H)
    renders = renders + bgt[:, None, None, :] * (1.0 - alphas)  # _torch_impl.py:919-922
    v_rc = torch.tensor(rng.standard_normal((C, H, W, D)))
    v_ra = torch.tensor(rng.standard_normal((C, H, W, 1)))
    grads = torch.autograd.grad((renders * v_rc).sum() + (alphas * v_ra).sum(), (m2, cn, op, co, bgt))
    _d = np.abs(renders.detach().numpy() - (rc + bg[:, None, None, :] * (1 - ra)))
    print("accumulate-vs-oracle fwd max diff", _d.max(), "alpha diff", np.abs(alphas.detach().numpy() - ra).max(), "pairs", len(g_l))
    assert _d.max() < 1e-7, "oracle fwd != reference accumulate"  # 0.99f vs 0.99 clamp constant
    save(
        "ref_accumulate.npz", means2d=means2d, conics=conics, opacities=opac, colors=colors, depths=depths,
        radii=radii, backgrounds=bg, width=np.int64(W), height=np.int64(H), tile_size=np.int64(ts),
        isect_offsets=off, flatten_ids=fl, n_pairs=np.int64(len(g_l)),
        render_colors=renders, render_alphas=alphas, v_render_colors=v_rc, v_render_alphas=v_ra,
        v_means2d=grads[0], v_conics=grads[1], v_opacities=grads[2], v_colors=grads[3], v_backgrounds=grads[4],
        min_margin=np.float64(mg.min()),
    )


# ---------------------------------------------------------------- MCMC strategy ops ("next" row)
def make_mcmc(rng):
    """relocation: the reference's own Python restatement in its test-suite
    (/root/reference/tests/test_relocation.py:42-76 _reference_relocation, loaded by path);
    perturbation: the reference's PyTorch fallback (gsplat/strategy/ops.py:494-512) with an explicit noise."""
    import importlib.util

    spec = importlib.util.spec_from_file_location("ref_test_relocation", "/root/reference/tests/test_relocation.py")
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    N, n_max = 257, 51
    op = (rng.random(N) * 0.98 + 0.01).astype(np.float32)
    op[:8] = [1e-4, 0.9999, 0.5, 0.003, 0.999999, 0.25, 0.75, 0.01]
    sc = (rng.random((N, 3)) * 0.5 + 0.01).astype(np.float32)
    ratios = rng.randint(1, n_max + 1, N).astype(np.int32)
    ratios[:4] = [1, n_max, 2, 3]
    binoms = mod._binomial_table(n_max, torch.device("cpu"))
    out = {}
    for tag, mo in (("", 0.005), ("_mo0", 0.0)):
        no, ns = mod._reference_relocation(
            torch.tensor(op, dtype=f64), torch.tensor(sc, dtype=f64), torch.tensor(ratios), binoms.to(f64), mo
        )
        out["new_opacities" + tag], out["new_scales" + tag] = no, ns
    # perturbation
    M = 300
    pos = rng.standard_normal((M, 3)).astype(np.float32)
    quats = rng.standard_normal((M, 4)).astype(np.float32)
    slog = (rng.standard_normal((M, 3)) * 0.5 - 3).astype(np.float32)
    ologit = (rng.standard_normal(M) * 3).astype(np.float32)
    noise = rng.standard_normal((M, 3)).astype(np.float32)
    noise_scale, t, k = 5e5 * 1.6e-4, 0.005, 100.0
    covars, _ = _quat_scale_to_covar_preci(torch.tensor(quats, dtype=f64), torch.exp(torch.tensor(slog, dtype=f64)), True, False, triu=False)
    opac = torch.sigmoid(torch.tensor(ologit, dtype=f64))
    nz = torch.tensor(noise, dtype=f64) * torch.sigmoid(-k * (opac - t)).unsqueeze(-1) * noise_scale
    new_pos = torch.tensor(pos, dtype=f64) + torch.einsum("bij,bj->bi", covars, nz)
    save("ref_mcmc.npz", opacities=op, scales=sc, ratios=ratios, binoms=binoms, n_max=np.int64(n_max), positions=pos,
         quats=quats, scales_log=slog, opacities_logit=ologit, noise=noise, noise_scale=np.float64(noise_scale),
         t=np.float64(t), k=np.float64(k), new_positions=new_pos, **out)


if __name__ == "__main__":
    if "--cameras-only" in sys.argv:  # adds the ortho / fisheye fixtures without rewriting the others
        sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))
        from tests import scene

        d = scene.load_garden()
        make_projection_cameras(d["means"], d["viewmats"], d["Ks"], int(d["width"]), int(d["height"]))
        sys.exit(0)
    rng = np.random.RandomState(20260922)
    means_all, viewmats, Ks, W, H = make_garden()
    make_quat_scale(rng)
    make_projection(rng, means_all, viewmats, Ks, W, H)
    make_projection_cameras(means_all, viewmats, Ks, W, H)
    make_sh(rng, viewmats)
    make_isect(rng)
    make_accumulate(rng)
    make_mcmc(np.random.RandomState(7))
