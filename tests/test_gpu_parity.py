"""GPU parity tests: every CUDA kernel, called through the C ABI / operator surface, against the CPU
oracle (oracle/) on the same seeded inputs, and against the committed golden vectors produced by the
reference's own Python twins (tests/golden/).  Run on the B200 box:  pytest -m gpu

Tolerances (written here as the contract):
  * integer / index outputs (radii, tiles_per_gauss, isect_ids, flatten_ids, offsets): bit-exact
    given identical float inputs;
  * per-gaussian float outputs (projection, SH): the kernels are compiled without FMA contraction and
    mirror the oracle's operation order, so they are expected to be BIT-EXACT against the float32
    oracle; the assertion is exactness on >= 99.9 % of entries and rtol 1e-5 / atol 1e-6 on all;
  * rendered colours / alphas: rtol 1e-4, atol 1e-5 (BASELINE.json north_star) against the float64
    oracle on every pixel whose discrete decisions are not within 1e-4 (relative) of flipping
    (alpha >= 1/255, T <= 1e-4, alpha clamp) -- `margins` from the oracle; flagged pixels (a handful)
    only have to agree to 2e-2;
  * compositing gradients: |cuda - oracle64| <= 1e-4 * mag + 1e-5 on >= 99.9 % of the entries and
    <= 1e-3 * mag + 1e-4 on all, where mag is the sum of the absolute values of the terms that make up
    that gradient (a float32 sum cannot do better than eps * sum|terms|); gaussians touching a flagged
    pixel are excluded.  Against the real reference CUDA kernels the bound is relative L2
    (tests/test_gpu_vs_reference_cuda.py).
"""
import math
import os

import numpy as np
import pytest
import torch

from oracle import gso
from tests import scene

pytestmark = pytest.mark.gpu

DEV = "cuda:0"


def _t(a, requires_grad=False):
    t = torch.from_numpy(np.ascontiguousarray(a)).to(DEV)
    if requires_grad:
        t.requires_grad_(True)
    return t


def _n(t):
    return t.detach().cpu().numpy()


def _close(a, b, rtol, atol, what=""):
    a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
    err = np.abs(a - b) - (atol + rtol * np.abs(b))
    assert err.max() <= 0, f"{what}: max violation {err.max():.3e} (max abs diff {np.abs(a - b).max():.3e})"


def _exactish(a, b, what, frac=0.999, rtol=1e-5, atol=1e-6):
    a, b = np.asarray(a), np.asarray(b)
    eq = (a == b).mean()
    _close(a, b, rtol, atol, what)
    assert eq >= frac, f"{what}: only {eq * 100:.3f}% bit-exact"
    return eq


@pytest.fixture(scope="module")
def gs():
    import gsplat_b200

    assert torch.cuda.is_available(), "needs a GPU"
    return gsplat_b200


def _load(name):
    d = np.load(os.path.join(os.path.dirname(__file__), "golden", name))
    return {k: d[k] for k in d.files}


# ------------------------------------------------------------------------------------------
def test_quat_scale(gs):
    g = _load("ref_quat_scale.npz")
    for triu in (False, True):
        t = "_triu" if triu else ""
        q, s = _t(g["quats"], True), _t(g["scales"], True)
        cov, pre = gs.quat_scale_to_covar_preci(q, s, True, True, triu)
        ocov, opre = gso.quat_scale_to_covar_preci(g["quats"], g["scales"], True, True, triu)
        _exactish(_n(cov), ocov, "covars")
        _exactish(_n(pre), opre, "precis")
        _close(_n(cov), g["covars" + t], 1e-5, 1e-6, "covars vs reference golden")
        v_cov, v_pre = _t(g["v_covars" + t].astype(np.float32)), _t(g["v_precis" + t].astype(np.float32))
        vq, vs = torch.autograd.grad((cov * v_cov).sum() + (pre * v_pre).sum(), (q, s))
        scale = np.abs(g["v_scales" + t]).max()
        _close(_n(vq), g["v_quats" + t], 2e-3, 1e-4 * np.abs(g["v_quats" + t]).max(), "v_quats vs golden")
        _close(_n(vs), g["v_scales" + t], 2e-3, 1e-4 * scale, "v_scales vs golden")
        # only one output requested
        c2, p2 = gs.quat_scale_to_covar_preci(q, s, True, False, triu)
        assert p2 is None and torch.equal(c2, cov)


def test_projection_vs_oracle_and_golden(gs):
    g = _load("ref_projection.npz")
    W, H = int(g["width"]), int(g["height"])
    means, quats, scales = _t(g["means"], True), _t(g["quats"], True), _t(g["scales"], True)
    vm, Ks = _t(g["viewmats"], True), _t(g["Ks"])
    radii, m2, dep, con, comp = gs.fully_fused_projection(
        means, None, quats, scales, vm, Ks, W, H, calc_compensations=True
    )
    o = gso.fully_fused_projection(g["means"], None, g["quats"], g["scales"], g["viewmats"], g["Ks"], W, H, 0.3, 0.01, 1e10, 0.0, True)
    assert np.array_equal(_n(radii), o[0]), "radii differ from the float32 oracle"
    for a, b, name in ((m2, o[1], "means2d"), (dep, o[2], "depths"), (con, o[3], "conics"), (comp, o[4], "compensations")):
        _exactish(_n(a), b, name)
    both = (o[0] > 0).all(-1) & (g["radii"] > 0).all(-1)
    _close(_n(m2)[both], g["means2d"][both], 1e-4, 1e-3, "means2d vs reference golden")
    _close(_n(con)[both], g["conics"][both], 2e-3, 1e-5, "conics vs reference golden")
    # backward with the golden cotangents (no compensation term -> same formulas as torch autograd)
    valid = _t((g["radii"] > 0).all(-1))
    v_m2, v_d, v_c = (_t(g[k].astype(np.float32)) for k in ("v_means2d", "v_depths", "v_conics"))
    loss = ((m2 * v_m2).sum(-1) * valid).sum() + (dep * v_d * valid).sum() + ((con * v_c).sum(-1) * valid).sum()
    gm, gq, gsc, gvm = torch.autograd.grad(loss, (means, quats, scales, vm))
    ov = gso.fully_fused_projection_bwd(
        g["means"], None, g["quats"], g["scales"], g["viewmats"], g["Ks"], W, H, 0.3, o[0], o[3], None,
        (g["v_means2d"] * (g["radii"] > 0).all(-1)[..., None]).astype(np.float32),
        (g["v_depths"] * (g["radii"] > 0).all(-1)).astype(np.float32),
        (g["v_conics"] * (g["radii"] > 0).all(-1)[..., None]).astype(np.float32), None, True,
    )
    for a, b, name in ((gm, ov[0], "v_means"), (gq, ov[2], "v_quats"), (gsc, ov[3], "v_scales")):
        _close(_n(a), b, 1e-4, 1e-5 * np.abs(b).max(), name + " vs f32 oracle")
    _close(_n(gvm), ov[4], 1e-3, 1e-4 * np.abs(ov[4]).max(), "v_viewmats vs f32 oracle")
    # vs the float64 reference autograd: float32 conditioning (tiny scales -> 1/s^2) limits agreement
    sel = (g["radii"] > 0).all(-1).any(0)
    for a, name, rt in ((gm, "v_means", 2e-2), (gq, "v_quats", 2e-2), (gsc, "v_scales", 2e-2)):
        ref = g[name + "_nc"]
        rel = np.linalg.norm(_n(a)[sel] - ref[sel]) / np.linalg.norm(ref[sel])
        assert rel < rt, f"{name}: relative L2 error vs reference golden {rel:.3e}"


@pytest.mark.parametrize("model", ["ortho", "fisheye"])
def test_projection_camera_models(gs, model):
    """Orthographic / fisheye EWA projection (reference Utils.cuh:498-565, 692-846) vs the float32 oracle (bit-exact
    for ortho; fisheye goes through atan2f, and its Jacobian derivative is computed with dual numbers on the GPU
    and with the reference's closed form in the oracle -> tolerance) and vs the reference's torch twin goldens."""
    g = _load(f"ref_projection_{model}.npz")
    W, H = int(g["width"]), int(g["height"])
    means, quats, scales = _t(g["means"], True), _t(g["quats"], True), _t(g["scales"], True)
    vm, Ks = _t(g["viewmats"], True), _t(g["Ks"])
    radii, m2, dep, con, comp = gs.fully_fused_projection(
        means, None, quats, scales, vm, Ks, W, H, calc_compensations=True, camera_model=model
    )
    o = gso.fully_fused_projection(
        g["means"], None, g["quats"], g["scales"], g["viewmats"], g["Ks"], W, H, 0.3, 0.01, 1e10, 0.0, True, camera_model=model
    )
    if model == "ortho":
        assert np.array_equal(_n(radii), o[0]), "radii differ from the float32 oracle"
        for a, b, name in ((m2, o[1], "means2d"), (dep, o[2], "depths"), (con, o[3], "conics"), (comp, o[4], "compensations")):
            _exactish(_n(a), b, name)
    else:
        assert (np.abs(_n(radii) - o[0]) <= 1).all() and (_n(radii) != o[0]).mean() < 2e-3
        vis = (o[0] > 0).all(-1) & (_n(radii) > 0).all(-1)
        _close(_n(m2)[vis], o[1][vis], 1e-5, 1e-3, "means2d")
        _close(_n(con)[vis], o[3][vis], 2e-3, 1e-5, "conics")
    both = (_n(radii) > 0).all(-1) & (g["radii"] > 0).all(-1)
    assert both.sum() > 1000
    _close(_n(m2)[both], g["means2d"][both], 1e-4, 2e-3, "means2d vs reference golden")
    _close(_n(con)[both], g["conics"][both], 5e-3, 1e-5, "conics vs reference golden")
    valid_np = (g["radii"] > 0).all(-1) & (_n(radii) > 0).all(-1)
    valid = _t(valid_np)
    v_m2, v_d, v_c = (_t(g[k].astype(np.float32)) for k in ("v_means2d", "v_depths", "v_conics"))
    loss = ((m2 * v_m2).sum(-1) * valid).sum() + (dep * v_d * valid).sum() + ((con * v_c).sum(-1) * valid).sum()
    gm, gq, gsc, gvm = torch.autograd.grad(loss, (means, quats, scales, vm))
    radii_v = (o[0] * valid_np[..., None]).astype(np.int32)
    ov = gso.fully_fused_projection_bwd(
        g["means"], None, g["quats"], g["scales"], g["viewmats"], g["Ks"], W, H, 0.3, radii_v, o[3], None,
        g["v_means2d"].astype(np.float32), g["v_depths"].astype(np.float32), g["v_conics"].astype(np.float32), None, True,
        camera_model=model,
    )
    for a, b, name in ((gm, ov[0], "v_means"), (gq, ov[2], "v_quats"), (gsc, ov[3], "v_scales")):
        rel = np.linalg.norm(_n(a) - b) / np.linalg.norm(b)
        assert rel < (1e-5 if model == "ortho" else 2e-4), f"{name}: rel L2 error vs f32 oracle {rel:.3e}"
    rel = np.linalg.norm(_n(gvm) - ov[4]) / np.linalg.norm(ov[4])
    assert rel < 1e-3, f"v_viewmats: rel L2 error vs f32 oracle {rel:.3e}"
    sel = valid_np.any(0)
    for a, name in ((gm, "v_means"), (gq, "v_quats"), (gsc, "v_scales")):
        ref = g[name + "_nc"]
        # the golden masks with the twin's own visibility; restrict to gaussians visible in the same cameras
        same = (valid_np == (g["radii"] > 0).all(-1)).all(0) & sel
        rel = np.linalg.norm(_n(a)[same] - ref[same]) / np.linalg.norm(ref[same])
        assert rel < 2e-2, f"{name}: relative L2 error vs reference golden {rel:.3e}"


@pytest.mark.parametrize("model", ["ortho", "fisheye"])
def test_rasterization_camera_models(gs, model):
    """End to end with a non-pinhole camera: matches the float64 oracle chain projection -> SH -> isect -> raster."""
    sc = scene.make_scene(n_max=30000, sh_degree=1)
    W, H = 320, 200
    Ks = scene.rescale_K(sc["Ks"], sc["width"], sc["height"], W, H)[:1].copy()
    if model == "ortho":
        Ks[:, 0, 0], Ks[:, 1, 1] = 60.0, 60.0
    vm = sc["viewmats"][:1]
    sh = np.ascontiguousarray(sc["sh"][:, :4])
    P = [_t(sc[k], True) for k in ("means", "quats", "scales", "opacities")]
    tsh = _t(sh, True)
    rc, ra, meta = gs.rasterization(*P, tsh, _t(vm), _t(Ks), W, H, sh_degree=1, camera_model=model)
    d = lambda a: a.astype(np.float64)  # noqa: E731
    o = gso.fully_fused_projection(d(sc["means"]), None, d(sc["quats"]), d(sc["scales"]), d(vm), d(Ks), W, H, 0.3, 0.01, 1e10,
                                   0.0, False, model, d(sc["opacities"]))
    vis = (o[0] > 0).all(-1)
    assert vis.sum() > 2000
    col = np.maximum(gso.spherical_harmonics(1, d(sc["means"]), d(vm), d(sh), vis) + 0.5, 0.0)
    op = np.broadcast_to(d(sc["opacities"])[None], vis.shape)
    tw, th = math.ceil(W / 16), math.ceil(H / 16)
    _, ids, fl = gso.isect_tiles(o[1], o[0], o[2], 16, tw, th, True, o[3], op)
    off = gso.isect_offset_encode(ids, 1, tw, th)
    orc, ora, _, omg = gso.rasterize_to_pixels(o[1], o[3], col, op, W, H, 16, off, fl, None, None, True)
    ok = omg > 1e-4
    assert ok.mean() > 0.99
    _close(_n(rc)[ok], orc[ok], 2e-4, 2e-5, "render_colors")
    _close(_n(ra)[ok], ora[ok], 2e-4, 2e-5, "render_alphas")
    (rc.sum() + ra.sum()).backward()
    assert all(torch.isfinite(p.grad).all() and p.grad.abs().sum() > 0 for p in P) and torch.isfinite(tsh.grad).all()


def test_projection_opacity_aware_and_covars(gs):
    sc = scene.make_scene(n_max=20000, sh_degree=0)
    W, H = sc["width"], sc["height"]
    args = (sc["means"], None, sc["quats"], sc["scales"], sc["viewmats"], sc["Ks"], W, H)
    o = gso.fully_fused_projection(*args, 0.3, 0.01, 1e10, 2.0, False, "pinhole", sc["opacities"])
    r = gs.fully_fused_projection(
        _t(sc["means"]), None, _t(sc["quats"]), _t(sc["scales"]), _t(sc["viewmats"]), _t(sc["Ks"]), W, H,
        radius_clip=2.0, opacities=_t(sc["opacities"]),
    )
    assert np.array_equal(_n(r[0]), o[0])
    assert (o[0] > 0).all(-1).sum() > 1000
    _exactish(_n(r[1]), o[1], "means2d")
    _exactish(_n(r[3]), o[3], "conics")
    assert r[4] is None
    # covars input path == quats/scales path
    cov6, _ = gso.quat_scale_to_covar_preci(sc["quats"], sc["scales"], True, False, True)
    r2 = gs.fully_fused_projection(
        _t(sc["means"]), _t(cov6), None, None, _t(sc["viewmats"]), _t(sc["Ks"]), W, H, radius_clip=2.0,
        opacities=_t(sc["opacities"]),
    )
    assert torch.equal(r2[0], r[0]) and torch.equal(r2[1], r[1]) and torch.equal(r2[3], r[3])


@pytest.mark.parametrize("deg", [0, 1, 2, 3, 4])
def test_sh(gs, deg):
    g = _load("ref_sh.npz")
    means, vm, cf = _t(g["means"], True), _t(g["viewmats"]), _t(g[f"coeffs{deg}"], True)
    colors = gs.spherical_harmonics(deg, means, vm, cf)
    oc = gso.spherical_harmonics(deg, g["means"], g["viewmats"], g[f"coeffs{deg}"])
    _exactish(_n(colors), oc, "colors")
    _close(_n(colors), g[f"colors{deg}"], 1e-4, 1e-5, "colors vs reference golden")
    v_col = _t(g[f"v_colors{deg}"].astype(np.float32))
    v_cf, v_m = torch.autograd.grad((colors * v_col).sum(), (cf, means), allow_unused=True)
    _close(_n(v_cf), g[f"v_coeffs{deg}"], 1e-4, 1e-5, "v_coeffs vs reference golden")
    if deg > 0:
        _close(_n(v_m), g[f"v_means{deg}"], 1e-3, 1e-4 * np.abs(g[f"v_means{deg}"]).max(), "v_means vs reference golden")
    if deg > 0:
        # pose gradient through the view direction (dir = mean + R^T t): one camera at a time,
        # dL/dR = t S^T, dL/dt = R S with S = sum_n dL/ddir_n = sum_n v_means_n
        for c in range(vm.shape[0]):
            vmc = vm[c : c + 1].clone().requires_grad_(True)
            m1 = means.detach().clone().requires_grad_(True)
            col_c = gs.spherical_harmonics(deg, m1, vmc, cf.detach())
            g_vm, g_m = torch.autograd.grad((col_c * v_col[c : c + 1]).sum(), (vmc, m1))
            S = g_m.sum(0)
            R, t = vmc.detach()[0, :3, :3], vmc.detach()[0, :3, 3]
            expect = torch.zeros(4, 4, device=DEV)
            expect[:3, :3] = t[:, None] * S[None, :]
            expect[:3, 3] = R @ S
            torch.testing.assert_close(g_vm[0], expect, rtol=2e-3, atol=2e-4 * float(expect.abs().max()))
    # masks: masked rows are zero and get zero gradient
    mask = np.zeros(oc.shape[:-1], bool)
    mask[:, ::3] = True
    cm = gs.spherical_harmonics(deg, means, vm, cf, masks=_t(mask))
    assert torch.equal(cm[_t(mask)], colors[_t(mask)]) and (cm[~_t(mask)] == 0).all()


def test_isect_exact(gs):
    g = _load("ref_isect.npz")
    ts, tw, th = int(g["tile_size"]), int(g["tile_width"]), int(g["tile_height"])
    tpg, ids, fl = gs.isect_tiles(_t(g["means2d"]), _t(g["radii"]), _t(g["depths"]), ts, tw, th)
    assert np.array_equal(_n(tpg), g["tiles_per_gauss"])
    assert np.array_equal(_n(ids), g["isect_ids"])
    assert np.array_equal(_n(fl), g["flatten_ids"])
    off = gs.isect_offset_encode(ids, g["means2d"].shape[0], tw, th)
    assert np.array_equal(_n(off), g["isect_offsets"])
    # unsorted emit order == oracle emit order
    tpg2, ids2, fl2 = gs.isect_tiles(_t(g["means2d"]), _t(g["radii"]), _t(g["depths"]), ts, tw, th, sort=False)
    o = gso.isect_tiles(g["means2d"], g["radii"], g["depths"], ts, tw, th, sort=False)
    assert np.array_equal(_n(ids2), o[1]) and np.array_equal(_n(fl2), o[2])
    # empty input
    e = gs.isect_tiles(_t(np.zeros((1, 4, 2), np.float32)), _t(np.zeros((1, 4, 2), np.int32)), _t(np.ones((1, 4), np.float32)), 16, 3, 2)
    assert e[1].numel() == 0 and (gs.isect_offset_encode(e[1], 1, 3, 2) == 0).all()


def _project_scene(sc, W, H, Ks, C=1, sh_degree=None):
    vm = sc["viewmats"][:C]
    o = gso.fully_fused_projection(sc["means"], None, sc["quats"], sc["scales"], vm, Ks[:C], W, H, 0.3, 0.01, 1e10, 0.0, False, "pinhole", sc["opacities"])
    return o


def test_isect_accutile_exact_on_scene(gs):
    sc = scene.make_scene(n_max=60000)
    W, H = 640, 360
    Ks = scene.rescale_K(sc["Ks"], sc["width"], sc["height"], W, H)
    radii, m2, dep, con, _ = _project_scene(sc, W, H, Ks, C=2)
    op = np.ascontiguousarray(np.broadcast_to(sc["opacities"][None], dep.shape))
    tw, th = math.ceil(W / 16), math.ceil(H / 16)
    o = gso.isect_tiles(m2, radii, dep, 16, tw, th, True, con, op)
    r = gs.isect_tiles(_t(m2), _t(radii), _t(dep), 16, tw, th, conics=_t(con), opacities=_t(op))
    assert o[1].shape[0] > 50000
    assert np.array_equal(_n(r[0]), o[0]), "tiles_per_gauss"
    assert np.array_equal(_n(r[1]), o[1]), "isect_ids"
    assert np.array_equal(_n(r[2]), o[2]), "flatten_ids"
    off = gs.isect_offset_encode(r[1], 2, tw, th)
    assert np.array_equal(_n(off), gso.isect_offset_encode(o[1], 2, tw, th))
    # properties at this size: sorted keys, offsets partition the list
    ids = _n(r[1])
    assert (np.diff(ids) >= 0).all()
    offn = _n(off).reshape(-1)
    assert offn[0] == 0 and (np.diff(offn) >= 0).all() and offn[-1] <= len(ids)


@pytest.mark.parametrize("accu", [True, False])
def test_isect_large_gaussians_cooperative_emit(gs, accu):
    """Gaussians that cover many tiles take the warp-cooperative emit path (row intervals in closed form, rows
    placed by a warp scan): counts, unsorted emission order and the sorted lists must stay EXACTLY the oracle's."""
    sc = scene.make_scene(n_max=20000)
    sc["scales"] = sc["scales"] * 6.0
    W, H = 640, 360
    Ks = scene.rescale_K(sc["Ks"], sc["width"], sc["height"], W, H)
    radii, m2, dep, con, _ = _project_scene(sc, W, H, Ks, C=2)
    op = np.ascontiguousarray(np.broadcast_to(sc["opacities"][None], dep.shape))
    tw, th = math.ceil(W / 16), math.ceil(H / 16)
    kw_o = (con, op) if accu else (None, None)
    kw = dict(conics=_t(con), opacities=_t(op)) if accu else {}
    for sort in (False, True):
        o = gso.isect_tiles(m2, radii, dep, 16, tw, th, sort, *kw_o)
        r = gs.isect_tiles(_t(m2), _t(radii), _t(dep), 16, tw, th, sort=sort, **kw)
        assert o[1].shape[0] > 200000 and _n(r[0]).max() > 100, "the case must contain many-tile gaussians"
        assert np.array_equal(_n(r[0]), o[0]), "tiles_per_gauss"
        assert np.array_equal(_n(r[1]), o[1]), f"isect_ids (sort={sort})"
        assert np.array_equal(_n(r[2]), o[2]), f"flatten_ids (sort={sort})"


@pytest.mark.parametrize("big_gaussians", [False, True])
def test_isect_narrow_keys_match_wide_pipeline(gs, big_gaussians):
    """rasterization()'s narrow-key pipeline (2- / 4-byte dense tile ids through the S-sized sort, int64 ids rebuilt on
    demand) must give bit for bit what isect_tiles(sort=True) + isect_offset_encode -- and the oracle -- give."""
    from gsplat_b200.ops import isect_tiles_sorted

    sc = scene.make_scene(n_max=30000)
    if big_gaussians:
        sc["scales"] = sc["scales"] * 6.0
    W, H = 640, 360
    Ks = scene.rescale_K(sc["Ks"], sc["width"], sc["height"], W, H)
    radii, m2, dep, con, _ = _project_scene(sc, W, H, Ks, C=3)
    op = np.ascontiguousarray(np.broadcast_to(sc["opacities"][None], dep.shape))
    tw, th = math.ceil(W / 16), math.ceil(H / 16)
    o = gso.isect_tiles(m2, radii, dep, 16, tw, th, True, con, op)
    hits = isect_tiles_sorted(_t(m2), _t(radii), _t(dep), 16, tw, th, conics=_t(con), opacities=_t(op))
    assert hits._key_bytes == 2 and o[1].shape[0] > 20000
    assert np.array_equal(_n(hits.tiles_per_gauss), o[0])
    assert np.array_equal(_n(hits.flatten_ids), o[2])
    assert np.array_equal(_n(hits.isect_ids()), o[1])
    assert np.array_equal(_n(hits.isect_offsets), gso.isect_offset_encode(o[1], 3, tw, th))
    # 4-byte keys: more than 65536 (image, tile) cells -- checked against the wide pipeline of this library
    tw4, th4 = 300, 120  # a 4800 x 1920 canvas, 36000 tiles x 3 images
    m2b = m2 * np.float32(7.5)
    r = gs.isect_tiles(_t(m2b), _t(radii), _t(dep), 16, tw4, th4, conics=_t(con), opacities=_t(op))
    hits = isect_tiles_sorted(_t(m2b), _t(radii), _t(dep), 16, tw4, th4, conics=_t(con), opacities=_t(op))
    assert hits._key_bytes == 4 and r[1].numel() > 20000
    assert torch.equal(hits.tiles_per_gauss, r[0]) and torch.equal(hits.isect_ids(), r[1]) and torch.equal(hits.flatten_ids, r[2])
    assert torch.equal(hits.isect_offsets, gs.isect_offset_encode(r[1], 3, tw4, th4))
    # nothing visible
    z = isect_tiles_sorted(_t(np.zeros((1, 4, 2), np.float32)), _t(np.zeros((1, 4, 2), np.int32)), _t(np.ones((1, 4), np.float32)), 16, 3, 2)
    assert z.flatten_ids.numel() == 0 and z.isect_ids().numel() == 0 and (z.isect_offsets == 0).all() and (z.tiles_per_gauss == 0).all()


def test_isect_speculative_capacities(gs):
    """rasterization() sizes the intersection stage by capacities predicted from earlier calls and reads the real totals
    afterwards: a hit (counts fit: padded slots must not leak into the result), a miss (counts grew: exact re-run) and a
    large over-estimate (counts shrank) must all give exactly the lists of the exact pipeline."""
    from gsplat_b200 import ops

    sc = scene.make_scene(n_max=30000)
    W, H = 800, 448  # a tile grid no other test uses: this test owns its predictor
    tw, th = math.ceil(W / 16), math.ceil(H / 16)
    Ks = scene.rescale_K(sc["Ks"], sc["width"], sc["height"], W, H)
    pred = ops._isect_predictor(torch.device(DEV), 2, tw, th)
    pred.hist.clear()
    pred.hits = pred.misses = 0
    seen = []
    for scale in (1.0, 1.0, 3.0, 0.4, 0.4, 1.0):
        sc2 = dict(sc, scales=sc["scales"] * np.float32(scale))
        radii, m2, dep, con, _ = _project_scene(sc2, W, H, Ks, C=2)
        op = np.ascontiguousarray(np.broadcast_to(sc["opacities"][None], dep.shape))
        a = (_t(m2), _t(radii), _t(dep))
        kw = dict(conics=_t(con), opacities=_t(op))
        ref = gs.isect_tiles(*a, 16, tw, th, **kw)
        hits = ops.isect_tiles_sorted(*a, 16, tw, th, **kw)
        assert torch.equal(hits.tiles_per_gauss, ref[0]) and torch.equal(hits.flatten_ids, ref[2])
        assert torch.equal(hits.isect_ids(), ref[1])
        assert torch.equal(hits.isect_offsets, gs.isect_offset_encode(ref[1], 2, tw, th))
        seen.append((ref[1].numel(), pred.hits, pred.misses))
    # call 1 exact, call 2 hit, call 3 (3x scales) miss, call 4 (0.4x) hit with a large over-estimate, ...
    assert [s[1:] for s in seen] == [(0, 0), (1, 0), (1, 1), (2, 1), (3, 1), (4, 1)], seen
    assert seen[2][0] > 1.5 * seen[0][0] and seen[0][0] > seen[3][0] > 0, seen


def test_fused_projection_row_side_outputs(gs):
    """The fused projection's side outputs (per-row tile counts + totals, 64-byte compositing row records) must reproduce
    what the stand-alone stages compute: counts / totals bit for bit, and a forward that is BIT-identical to the one that
    packs its records from means2d / conics / colours / opacities (the extents only steer a conservative culling)."""
    from gsplat_b200.ops import RowSideOutputs, fused_project_sh, isect_tiles_sorted, rasterize_to_pixels_rows

    sc = scene.make_scene(n_max=40000, sh_degree=3)
    W, H, C = 640, 360, 2
    tw, th = math.ceil(W / 16), math.ceil(H / 16)
    Ks = scene.rescale_K(sc["Ks"], sc["width"], sc["height"], W, H)[:C]
    P = {k: _t(sc[k]) for k in ("means", "quats", "scales", "opacities", "sh")}
    vm, K = _t(sc["viewmats"][:C]), _t(Ks)
    plain = fused_project_sh(P["means"], P["quats"], P["scales"], P["opacities"], P["sh"], vm, K, W, H, 3)
    side = RowSideOutputs(16, tw, th)
    rows = fused_project_sh(P["means"], P["quats"], P["scales"], P["opacities"], P["sh"], vm, K, W, H, 3, rows_out=side)
    for a, b in zip(plain[:5], rows[:5]):
        assert torch.equal(a, b)
    radii, m2, dep, con, col = rows[:5]
    op = torch.broadcast_to(P["opacities"][None], dep.shape).contiguous()
    ref = gs.isect_tiles(m2, radii, dep, 16, tw, th, conics=con, opacities=op)
    assert torch.equal(side.tiles_per_gauss, ref[0])
    tot = side.totals.tolist()
    assert tot == [ref[1].numel(), int((ref[0] > 0).sum()), int(ref[0].max())] and tot[0] > 30000
    hits = isect_tiles_sorted(m2, radii, dep, 16, tw, th, conics=con, opacities=op, precounted=side)
    assert torch.equal(hits.flatten_ids, ref[2]) and torch.equal(hits.isect_ids(), ref[1])
    bg = torch.rand(C, 3, device=DEV)
    outs = []
    for rr in (None, side.rows):
        m2g, cong, colg, opg = (x.clone().requires_grad_(True) for x in (m2, con, col, op))
        rc, ra = rasterize_to_pixels_rows(m2g, cong, colg, opg, W, H, 16, hits.isect_offsets.view(C, th, tw), hits.flatten_ids, backgrounds=bg, _row_records=rr)
        w = torch.linspace(0.5, 1.5, rc.numel(), device=DEV).view_as(rc)
        ((rc * w).sum() + ra.sum()).backward()
        outs.append((rc.detach(), ra.detach(), m2g.grad, cong.grad, colg.grad, opg.grad))
    assert torch.equal(outs[0][0], outs[1][0]) and torch.equal(outs[0][1], outs[1][1])
    for a, b, name in zip(outs[0][2:], outs[1][2:], ("v_means2d", "v_conics", "v_colors", "v_opacities")):
        rel = float((a - b).norm() / a.norm())
        assert rel < 1e-5, (name, rel)  # same pairs, same arithmetic; only the order of the atomic adds differs


def test_isect_sorted_equals_stable_sort_of_unsorted(gs):
    """The two-level sort (rows by depth, then intersections by (image, tile) bits only) must give exactly what
    one stable sort of the reference's unsorted emission gives (csrc/Intersect.cpp:283-326)."""

    def check(m2, radii, dep, tw, th, **kw):
        a = gs.isect_tiles(_t(m2), _t(radii), _t(dep), 16, tw, th, **kw)
        u = gs.isect_tiles(_t(m2), _t(radii), _t(dep), 16, tw, th, sort=False, **kw)
        ids, perm = torch.sort(u[1], stable=True)
        assert torch.equal(a[0], u[0]) and torch.equal(a[1], ids) and torch.equal(a[2], u[2][perm])
        return a

    sc = scene.make_scene(n_max=80000)
    W, H = 800, 450
    Ks = scene.rescale_K(sc["Ks"], sc["width"], sc["height"], W, H)
    radii, m2, dep, con, _ = _project_scene(sc, W, H, Ks, C=3)
    op = np.ascontiguousarray(np.broadcast_to(sc["opacities"][None], dep.shape))
    tw, th = math.ceil(W / 16), math.ceil(H / 16)
    for accu in (True, False):
        kw = dict(conics=_t(con), opacities=_t(op)) if accu else {}
        assert check(m2, radii, dep, tw, th, **kw)[1].numel() > 10000
    # ties in depth inside a tile keep emit (gaussian index) order
    m2t = np.tile(np.array([[20.0, 20.0]], np.float32), (1, 64, 1))
    a = check(m2t, np.full((1, 64, 2), 10, np.int32), np.full((1, 64), 1.5, np.float32), 4, 4)
    assert (np.diff(_n(a[2]).reshape(-1, 64), axis=1) > 0).all()
    # crowded tiles with heavy depth ties (depths quantised to 1/64), two images, some culled rows
    rng = np.random.RandomState(3)
    for n in (7000, 40000):
        m2c = (rng.rand(2, n, 2) * 64).astype(np.float32)
        rc = rng.randint(0, 80, size=(2, n, 2)).astype(np.int32)
        rc[:, ::7] = 0
        dc = (np.round(rng.rand(2, n) * 64) / 64 + 0.5).astype(np.float32)
        check(m2c, rc, dc, 4, 4)
    # packed rows with image ids
    nnz = 5000
    img = np.sort(rng.randint(0, 3, size=nnz)).astype(np.int64)
    m2p = (rng.rand(nnz, 2) * 64).astype(np.float32)
    rp = rng.randint(0, 30, size=(nnz, 2)).astype(np.int32)
    dp = (np.round(rng.rand(nnz) * 16) / 16 + 0.5).astype(np.float32)
    check(m2p, rp, dp, 4, 4, packed=True, n_images=3, image_ids=_t(img), gaussian_ids=_t(np.arange(nnz, dtype=np.int64)))
    # empty
    e = gs.isect_tiles(_t(np.zeros((1, 4, 2), np.float32)), _t(np.zeros((1, 4, 2), np.int32)), _t(np.ones((1, 4), np.float32)), 16, 3, 2)
    assert e[1].numel() == 0


def _raster_case(gs, m2, con, col, op, W, H, off, fl, bg=None, absgrad=False, seed=0, strict_frac=0.995):
    """Runs fwd+bwd on the GPU and in the oracle (f64) and applies the module's tolerance contract."""
    D = col.shape[-1]
    tm2, tcon, tcol, top = _t(m2, True), _t(con, True), _t(col, True), _t(op, True)
    tbg = _t(bg, True) if bg is not None else None
    rc, ra = gs.rasterize_to_pixels(tm2, tcon, tcol, top, W, H, 16, _t(off), _t(fl), backgrounds=tbg, absgrad=absgrad)
    d = lambda a: None if a is None else a.astype(np.float64)  # noqa: E731
    orc, ora, oli, omg = gso.rasterize_to_pixels(d(m2), d(con), d(col), d(op), W, H, 16, off, fl, d(bg), None, True)
    ok = omg > 1e-4
    assert ok.mean() > strict_frac, f"too many marginal pixels: {1 - ok.mean():.4f}"
    _close(_n(rc)[ok], orc[ok], 1e-4, 1e-5, "render_colors")
    _close(_n(ra)[ok], ora[ok], 1e-4, 1e-5, "render_alphas")
    _close(_n(rc)[~ok], orc[~ok], 0, 2e-2, "render_colors (marginal pixels)")
    rng = np.random.RandomState(seed)
    v_rc = rng.standard_normal(orc.shape).astype(np.float32)
    v_ra = rng.standard_normal(ora.shape).astype(np.float32)
    ins = [tm2, tcon, tcol, top] + ([tbg] if tbg is not None else [])
    grads = torch.autograd.grad((rc * _t(v_rc)).sum() + (ra * _t(v_ra)).sum(), ins)
    og = gso.rasterize_to_pixels_bwd(d(m2), d(con), d(col), d(op), W, H, 16, off, fl, ora, oli, d(v_rc), d(v_ra), d(bg), None, absgrad)
    # gaussians that touch a marginal pixel are excluded from the strict check
    th, tw = off.shape[-2:]
    I = int(np.prod(off.shape[:-2]))
    bad_tiles = np.zeros(I * th * tw, bool)
    bad_pix = np.argwhere(~ok.reshape(I, H, W))
    for im, y, x in bad_pix:
        bad_tiles[(im * th + y // 16) * tw + x // 16] = True
    offf = np.concatenate([off.reshape(-1), [len(fl)]])
    tainted = np.zeros(int(np.prod(m2.shape[:-1])), bool)
    for t in np.nonzero(bad_tiles)[0]:
        tainted[fl[offf[t] : offf[t + 1]]] = True
    good = ~tainted.reshape(m2.shape[:-1])
    mag = og["mag"]
    for a, key, mi in ((grads[0], "v_means2d", 0), (grads[1], "v_conics", 1), (grads[3], "v_opacities", 2), (grads[2], "v_colors", 3)):
        ref = og[key]
        m = mag[..., mi]
        m = m[..., None] if ref.ndim > m.ndim else m
        diff = np.abs(_n(a).astype(np.float64) - ref)
        g3 = np.broadcast_to(good[..., None] if ref.ndim > good.ndim else good, diff.shape)
        strict = (diff <= 1e-4 * m + 1e-5) | ~g3
        # float32 evaluates sigma = 0.5(a dx^2 + c dy^2) + b dx dy with cancellation between large terms
        # (elongated gaussians far from the pixel), so a few entries see a relative alpha error near 1e-4
        # that no summation-order argument covers: >= 99.9 % must meet the strict bound, all the loose one
        assert strict.mean() >= 0.999, f"{key}: only {strict.mean() * 100:.3f}% within 1e-4*mag + 1e-5"
        loose = (diff <= 1e-3 * m + 1e-4) | ~g3
        assert loose.all(), f"{key}: max violation of the loose bound {(diff - (1e-3 * m + 1e-4))[g3].max():.3e}"
        # and nothing anywhere is wildly off
        rel = np.linalg.norm(_n(a) - ref) / max(np.linalg.norm(ref), 1e-30)
        assert rel < 1e-3, f"{key}: relative L2 error {rel:.3e}"
    if tbg is not None:
        _close(_n(grads[4]), og["v_backgrounds"], 1e-3, 1e-2, "v_backgrounds")
    if absgrad:
        ref = og["v_means2d_abs"]
        rel = np.linalg.norm(_n(tm2.absgrad) - ref) / np.linalg.norm(ref)
        assert rel < 1e-4, f"absgrad: relative L2 error {rel:.3e}"
    return rc, ra


def test_raster_golden_accumulate(gs):
    """The reference's own accumulate() (+autograd) fixture, straight against the CUDA kernels."""
    g = _load("ref_accumulate.npz")
    W, H = int(g["width"]), int(g["height"])
    m2, con, col, op, bg = (_t(g[k], True) for k in ("means2d", "conics", "colors", "opacities", "backgrounds"))
    rc, ra = gs.rasterize_to_pixels(m2, con, col, op, W, H, 16, _t(g["isect_offsets"]), _t(g["flatten_ids"]), backgrounds=bg)
    _close(_n(rc), g["render_colors"], 1e-4, 1e-5, "render_colors vs reference accumulate")
    _close(_n(ra), g["render_alphas"], 1e-4, 1e-5, "render_alphas vs reference accumulate")
    v_rc, v_ra = _t(g["v_render_colors"].astype(np.float32)), _t(g["v_render_alphas"].astype(np.float32))
    grads = torch.autograd.grad((rc * v_rc).sum() + (ra * v_ra).sum(), (m2, con, op, col, bg))
    for a, k in zip(grads, ("v_means2d", "v_conics", "v_opacities", "v_colors", "v_backgrounds")):
        ref = g[k]
        rel = np.linalg.norm(_n(a) - ref) / np.linalg.norm(ref)
        assert rel < 1e-4, f"{k}: relative L2 error vs reference autograd {rel:.3e}"  # fp32 sums vs float64 autograd
        _close(_n(a), ref, 1e-3, 1e-4 * np.abs(ref).max(), k)


@pytest.mark.parametrize("D,bg,absgrad", [(3, False, False), (3, True, True), (1, False, False), (4, True, False), (8, False, False), (32, False, False), (7, True, False)])
def test_raster_vs_oracle(gs, D, bg, absgrad):
    sc = scene.make_scene(n_max=30000)
    W, H = 320, 200  # partial tiles on the bottom edge (200 = 12.5 tiles)
    Ks = scene.rescale_K(sc["Ks"], sc["width"], sc["height"], W, H)
    C = 2
    radii, m2, dep, con, _ = _project_scene(sc, W, H, Ks, C=C)
    op = np.ascontiguousarray(np.broadcast_to(sc["opacities"][None], dep.shape)).copy()
    op[:, ::50] = 1.0  # saturating gaussians exercise the 0.99 clamp
    tw, th = math.ceil(W / 16), math.ceil(H / 16)
    _, ids, fl = gso.isect_tiles(m2, radii, dep, 16, tw, th, True, con, op)
    off = gso.isect_offset_encode(ids, C, tw, th)
    rng = np.random.RandomState(D)
    col = rng.random_sample(m2.shape[:-1] + (D,)).astype(np.float32)
    bgv = rng.random_sample((C, D)).astype(np.float32) if bg else None
    _raster_case(gs, m2, con, col, op, W, H, off, fl, bgv, absgrad, seed=D)


def test_raster_dense_overdraw_and_termination(gs):
    """Large opaque gaussians: every pixel saturates (T <= 1e-4 stop), lists longer than one batch."""
    rng = np.random.RandomState(3)
    C, N, W, H = 1, 3000, 64, 48
    m2 = np.stack([rng.random_sample((C, N)) * W, rng.random_sample((C, N)) * H], -1).astype(np.float32)
    s = (rng.random_sample((C, N)) * 12 + 4).astype(np.float32)
    con = np.stack([1 / s**2, np.zeros_like(s), 1 / s**2], -1).astype(np.float32)
    op = (rng.random_sample((C, N)) * 0.6 + 0.39).astype(np.float32)
    dep = (rng.random_sample((C, N)) + 0.1).astype(np.float32)
    radii = np.stack([np.ceil(3.33 * s), np.ceil(3.33 * s)], -1).astype(np.int32)
    tw, th = 4, 3
    _, ids, fl = gso.isect_tiles(m2, radii, dep, 16, tw, th, True, con, op)
    off = gso.isect_offset_encode(ids, C, tw, th)
    assert (np.diff(np.concatenate([off.reshape(-1), [len(fl)]])) > 300).all()
    col = rng.random_sample((C, N, 3)).astype(np.float32)
    rc, ra = _raster_case(gs, m2, con, col, op, W, H, off, fl, None, False, seed=1, strict_frac=0.97)
    assert (_n(ra) > 0.999).mean() > 0.9


def test_raster_masks_and_empty(gs):
    rng = np.random.RandomState(5)
    C, N, W, H = 1, 50, 40, 40
    m2 = (rng.random_sample((C, N, 2)) * 40).astype(np.float32)
    con = np.tile(np.array([0.05, 0.0, 0.05], np.float32), (C, N, 1))
    op = np.full((C, N), 0.5, np.float32)
    dep = rng.random_sample((C, N)).astype(np.float32)
    radii = np.full((C, N, 2), 15, np.int32)
    _, ids, fl = gso.isect_tiles(m2, radii, dep, 16, 3, 3, True, con, op)
    off = gso.isect_offset_encode(ids, C, 3, 3)
    col = rng.random_sample((C, N, 3)).astype(np.float32)
    bg = rng.random_sample((C, 3)).astype(np.float32)
    masks = np.ones((C, 3, 3), bool)
    masks[0, 1, 1] = False
    rc, ra = gs.rasterize_to_pixels(_t(m2), _t(con), _t(col), _t(op), W, H, 16, _t(off), _t(fl), backgrounds=_t(bg), masks=_t(masks))
    orc, ora = gso.rasterize_to_pixels(m2, con, col, op, W, H, 16, off, fl, bg, masks)
    _close(_n(rc), orc, 1e-4, 1e-5, "masked render")
    assert (_n(ra)[0, 16:32, 16:32] == 0).all()
    # no intersections at all
    e_off = np.zeros((C, 3, 3), np.int32)
    rc, ra = gs.rasterize_to_pixels(_t(m2, True), _t(con), _t(col), _t(op), W, H, 16, _t(e_off), _t(np.zeros(0, np.int32)), backgrounds=_t(bg))
    assert (_n(ra) == 0).all() and np.allclose(_n(rc), bg[:, None, None, :])
    rc.sum().backward()  # backward with n_isects == 0 must be a clean no-op


def _pipeline_case(gs, sc, W, H, Ks, C, sh_degree, packed=False, **kw):
    c32 = lambda k: sc[k].astype(np.float32)  # noqa: E731
    vm = sc["viewmats"][:C]
    K = (sh_degree + 1) ** 2
    sh = np.ascontiguousarray(sc["sh"][:, :K])
    rng = np.random.RandomState(11)
    v_rc = rng.standard_normal((C, H, W, 3)).astype(np.float32)
    v_ra = rng.standard_normal((C, H, W, 1)).astype(np.float32)
    f64 = lambda a: a.astype(np.float64)  # noqa: E731
    fwd, grads = gso.rasterization_fwd_bwd(
        f64(c32("means")), f64(c32("quats")), f64(c32("scales")), f64(c32("opacities")), f64(sh), f64(vm), f64(Ks[:C]),
        W, H, sh_degree, f64(v_rc), f64(v_ra), **kw,
    )
    tens = {k: _t(c32(k), True) for k in ("means", "quats", "scales", "opacities")}
    tsh = _t(sh, True)
    rc, ra, meta = gs.rasterization(
        tens["means"], tens["quats"], tens["scales"], tens["opacities"], tsh, _t(vm), _t(Ks[:C]), W, H,
        sh_degree=sh_degree, packed=packed, **kw,
    )
    ok = fwd["margins"] > 1e-4
    # the float32 projection can move a gaussian across a tile / cull boundary relative to float64; such
    # (rare) pixels show up as mismatches and are bounded, not excused: <= 0.05 % of pixels
    err = np.abs(_n(rc).astype(np.float64) - fwd["render_colors"]) - (1e-4 * np.abs(fwd["render_colors"]) + 1e-5)
    bad = (err.max(-1) > 0) & ok
    assert bad.mean() < 5e-4, f"{bad.mean() * 100:.4f}% of non-marginal pixels exceed rtol 1e-4 / atol 1e-5"
    assert np.abs(_n(rc) - fwd["render_colors"]).max() < 5e-2
    loss = (rc * _t(v_rc)).sum() + (ra * _t(v_ra)).sum()
    meta["means2d"].retain_grad()
    loss.backward()
    for k, ok_rel in (("means", 2e-3), ("quats", 2e-3), ("scales", 2e-3), ("opacities", 1e-3)):
        a, ref = _n(tens[k].grad), grads["v_" + k]
        rel = np.linalg.norm(a - ref) / np.linalg.norm(ref)
        assert rel < ok_rel, f"v_{k}: relative L2 error vs float64 oracle {rel:.3e}"
    # SH colours pass through max(x + 0.5, 0): gaussians whose pre-activation value sits on the kink
    # (|x + 0.5| < 1e-5 in any view / channel -- e.g. pure black points at SH degree 0) legitimately get
    # either sub-gradient depending on float32 rounding and are excluded, like marginal pixels
    kink = (np.abs(fwd["sh_raw"] + 0.5) < 1e-5).any(axis=(0, 2))
    a, ref = _n(tsh.grad)[~kink], grads["v_sh"][~kink]
    rel = np.linalg.norm(a - ref) / np.linalg.norm(ref)
    assert kink.mean() < 0.2 and rel < 1e-3, f"v_sh: relative L2 error {rel:.3e} (kink fraction {kink.mean():.3f})"
    assert meta["means2d"].grad is not None and meta["means2d"].grad.abs().sum() > 0
    return rc, ra, meta, fwd


def test_rasterization_cfg1_garden_256(gs):
    """BASELINE.json configs[0]: test_garden, 1 camera, 256x256, SH degree 0, fwd + bwd."""
    sc = scene.make_scene(sh_degree=0)
    W = H = 256
    rc, ra, meta, fwd = _pipeline_case(gs, sc, W, H, sc["Ks"], 1, 0)
    assert tuple(rc.shape) == (1, H, W, 3) and tuple(ra.shape) == (1, H, W, 1)
    assert meta["radii"].dtype == torch.int32 and tuple(meta["radii"].shape) == (1, sc["means"].shape[0], 2)
    assert meta["gaussian_ids"] is None and meta["tile_width"] == 16 and meta["n_cameras"] == 1
    # integer outputs vs the float32 oracle run on the float32 projection
    o32, _ = gso.rasterization_fwd_bwd(
        sc["means"], sc["quats"], sc["scales"], sc["opacities"], np.ascontiguousarray(sc["sh"][:, :1]), sc["viewmats"][:1],
        sc["Ks"][:1], W, H, 0, None, None,
    )
    assert np.array_equal(_n(meta["radii"]), o32["radii"])
    assert np.array_equal(_n(meta["isect_ids"]), o32["isect_ids"])
    assert np.array_equal(_n(meta["flatten_ids"]), o32["flatten_ids"])
    assert np.array_equal(_n(meta["isect_offsets"]), o32["isect_offsets"])
    _exactish(_n(meta["means2d"]), o32["means2d"], "means2d")
    _exactish(_n(meta["conics"]), o32["conics"], "conics")


def test_rasterization_sh3_two_cameras_packed_and_dense(gs):
    sc = scene.make_scene(n_max=50000, sh_degree=3)
    W, H = 400, 240
    Ks = scene.rescale_K(sc["Ks"], sc["width"], sc["height"], W, H)
    rc_d, ra_d, meta_d, _ = _pipeline_case(gs, sc, W, H, Ks, 2, 3, packed=False)
    rc_p, ra_p, meta_p, _ = _pipeline_case(gs, sc, W, H, Ks, 2, 3, packed=True)
    # packed mode evaluates SH on gathered rows (view direction formed per row), the dense mode in the fused kernel
    torch.testing.assert_close(rc_p, rc_d, rtol=1e-5, atol=2e-6)
    assert torch.equal(ra_d, ra_p)
    nnz = int((meta_d["radii"] > 0).all(-1).sum())
    assert meta_p["means2d"].shape == (nnz, 2) and meta_p["gaussian_ids"].shape == (nnz,)
    assert meta_p["camera_ids"].max() == 1 and meta_p["gaussian_ids"].dtype == torch.int64
    # gradients of packed == dense; sparse_grad=True returns the geometry gradients as COO tensors with the same values
    P = {k: _t(sc[k], True) for k in ("means", "quats", "scales", "opacities")}
    sh = _t(sc["sh"], True)
    cam = (_t(sc["viewmats"][:1]), _t(Ks[:1]), W, H)
    outs = {}
    for mode in ("dense", "packed", "sparse"):
        for t in list(P.values()) + [sh]:
            t.grad = None
        rc, ra, _ = gs.rasterization(
            P["means"], P["quats"], P["scales"], P["opacities"], sh, *cam, sh_degree=3, packed=mode != "dense",
            sparse_grad=mode == "sparse",
        )
        (rc.square().sum() + ra.sum()).backward()
        outs[mode] = {k: v.grad for k, v in P.items()} | {"sh": sh.grad}
    for k in ("means", "quats", "scales"):
        g = outs["sparse"][k]
        if k != "means":  # means also receives a dense gradient through the SH view direction (as in the reference)
            assert g.is_sparse
        g = g.to_dense() if g.is_sparse else g
        assert float((g - outs["packed"][k]).norm() / outs["packed"][k].norm()) < 1e-5
    for k in outs["dense"]:
        assert float((outs["packed"][k] - outs["dense"][k]).norm() / outs["dense"][k].norm()) < 2e-5, k


def test_rasterization_modes(gs):
    sc = scene.make_scene(n_max=20000, sh_degree=1)
    W, H = 160, 96
    Ks = scene.rescale_K(sc["Ks"], sc["width"], sc["height"], W, H)
    t = lambda k: _t(sc[k])  # noqa: E731
    sh = _t(np.ascontiguousarray(sc["sh"][:, :4]))
    base = (t("means"), t("quats"), t("scales"), t("opacities"))
    cam = (_t(sc["viewmats"][:1]), _t(Ks[:1]), W, H)
    rgb, a, _ = gs.rasterization(*base, sh, *cam, sh_degree=1, packed=False)
    rgbd, a2, _ = gs.rasterization(*base, sh, *cam, sh_degree=1, packed=False, render_mode="RGB+D")
    rgbed, _, _ = gs.rasterization(*base, sh, *cam, sh_degree=1, packed=False, render_mode="RGB+ED")
    d, _, _ = gs.rasterization(*base, None, *cam, packed=False, render_mode="D")
    assert rgbd.shape[-1] == 4 and d.shape[-1] == 1
    assert torch.allclose(rgbd[..., :3], rgb, atol=1e-6) and torch.allclose(a, a2)
    assert torch.allclose(rgbd[..., 3:], d, atol=1e-5)
    assert torch.allclose(rgbed[..., 3:], d / a.clamp(min=1e-10), rtol=1e-5, atol=1e-6)
    # post-activation colours [N, D] and antialiased mode run and differ from classic
    col = _t(sc["colors"])
    c1, _, _ = gs.rasterization(*base, col, *cam, packed=False)
    c2, _, m2 = gs.rasterization(*base, col, *cam, packed=False, rasterize_mode="antialiased")
    assert (c1 - c2).abs().max() > 1e-4 and (m2["opacities"] <= t("opacities")[None] + 1e-6).all()
    # 40 feature channels -> chunked compositing == two direct passes
    feat = torch.rand((sc["means"].shape[0], 40), device=DEV)
    f, _, _ = gs.rasterization(*base, feat, *cam, packed=False)
    f0, _, _ = gs.rasterization(*base, feat[:, :32].contiguous(), *cam, packed=False)
    assert f.shape[-1] == 40 and torch.equal(f[..., :32], f0)
    for bad in (dict(with_ut=True), dict(camera_model="ftheta"), dict(render_mode="RGB-d"), dict(tile_size=8)):
        with pytest.raises((NotImplementedError, ValueError)):
            gs.rasterization(*base, col, *cam, packed=False, **bad)


def test_full_size_properties_1080p(gs):
    """BASELINE.json configs[1] scale (111 785 gaussians, 1080p, SH3): size-independent properties."""
    sc = scene.make_scene(sh_degree=3)
    W, H = 1920, 1080
    Ks = scene.rescale_K(sc["Ks"], sc["width"], sc["height"], W, H)
    t = {k: _t(sc[k], True) for k in ("means", "quats", "scales", "opacities", "sh")}
    args = (t["means"], t["quats"], t["scales"], t["opacities"], t["sh"], _t(sc["viewmats"][:1]), _t(Ks[:1]), W, H)
    rc, ra, meta = gs.rasterization(*args, sh_degree=3, packed=False)
    ids = meta["isect_ids"]
    assert (ids[1:] >= ids[:-1]).all(), "sorted keys"
    assert int(meta["tiles_per_gauss"].sum()) == ids.numel() == meta["flatten_ids"].numel()
    off = meta["isect_offsets"].reshape(-1)
    assert off[0] == 0 and (off[1:] >= off[:-1]).all()
    assert (ra >= 0).all() and (ra <= 1).all() and torch.isfinite(rc).all()
    # determinism of the forward, linearity of the backward in the cotangent
    rc2, ra2, _ = gs.rasterization(*args, sh_degree=3, packed=False)
    assert torch.equal(rc, rc2) and torch.equal(ra, ra2)
    v = torch.randn_like(rc)
    g1 = torch.autograd.grad((rc * v).sum(), t["sh"], retain_graph=True)[0]
    g2 = torch.autograd.grad((rc * (2 * v)).sum(), t["sh"], retain_graph=True)[0]
    assert torch.allclose(g2, 2 * g1, rtol=1e-3, atol=1e-6)
    # background only changes pixels by T * bg
    bg = torch.tensor([[0.2, 0.4, 0.6]], device=DEV)
    rc_bg, _, _ = gs.rasterization(*args, sh_degree=3, packed=False, backgrounds=bg)
    assert torch.allclose(rc_bg, rc + (1 - ra) * bg, atol=1e-5)


def test_mcmc_ops(gs):
    g = _load("ref_mcmc.npz")
    binoms = _t(g["binoms"].astype(np.float32))
    for tag, mo in (("", 0.005), ("_mo0", 0.0)):
        ratios = _t(g["ratios"].astype(np.int64))
        no, ns = gs.compute_relocation(_t(g["opacities"]), _t(g["scales"]), ratios, binoms, mo)
        _close(_n(no), g["new_opacities" + tag], 2e-5, 1e-6, "new_opacities vs reference restatement")
        # 1 - (1-o)^(1/n) loses relative precision for tiny o in float32 and the scale inherits it
        sel = g["opacities"] > 1e-3
        _close(_n(ns)[sel], g["new_scales" + tag][sel], 2e-3, 1e-6, "new_scales vs reference restatement")
    # ratios beyond n_max are clamped in place, like the reference wrapper does
    r = torch.full((4,), 999, device=DEV, dtype=torch.int64)
    gs.compute_relocation(_t(g["opacities"][:4]), _t(g["scales"][:4]), r, binoms)
    assert (r == int(g["n_max"])).all()
    pos = _t(g["positions"])
    gs.mcmc_perturb_positions(pos, _t(g["quats"]), _t(g["scales_log"]), _t(g["opacities_logit"]), _t(g["noise"]),
                              float(g["noise_scale"]), float(g["t"]), float(g["k"]))
    _close(_n(pos), g["new_positions"], 1e-4, 1e-5, "perturbed positions")


def test_packed_operator_variants(gs):
    """packed=True forms of the per-op surface (COO rows) against the dense ops."""
    from gsplat_b200 import ops
    sc = scene.make_scene(n_max=30000, sh_degree=2)
    W, H, C = 320, 180, 2
    Ks = scene.rescale_K(sc["Ks"], sc["width"], sc["height"], W, H)[:C]
    means, quats, scales, opac = (_t(sc[k], True) for k in ("means", "quats", "scales", "opacities"))
    vm, K = _t(sc["viewmats"][:C]), _t(Ks)
    radii, m2, dep, con, _ = gs.fully_fused_projection(means, None, quats, scales, vm, K, W, H, opacities=opac)
    b_ids, c_ids, g_ids, indptr, p_radii, p_m2, p_dep, p_con, p_comp = gs.fully_fused_projection(
        means, None, quats, scales, vm, K, W, H, opacities=opac, packed=True
    )
    sel = (radii > 0).all(-1)
    nnz = int(sel.sum())
    assert p_m2.shape == (nnz, 2) and p_comp is None and indptr.tolist() == [0, int(sel[0].sum()), nnz]
    assert torch.equal(p_m2, m2[sel]) and torch.equal(p_con, con[sel]) and torch.equal(p_radii, radii[sel])
    assert torch.equal(g_ids.long(), torch.nonzero(sel)[:, 1]) and torch.equal(c_ids.long(), torch.nonzero(sel)[:, 0])
    assert b_ids.dtype == torch.int64 and indptr.dtype == torch.int32 and int(b_ids.max()) == 0
    g1 = torch.autograd.grad(p_m2.sum() + p_con.sum() + p_dep.sum(), (means, quats, scales), retain_graph=True)
    g2 = torch.autograd.grad(m2[sel].sum() + con[sel].sum() + dep[sel].sum(), (means, quats, scales))
    for a, b in zip(g1, g2):  # the dense kernel sums over cameras before the quat/scale VJP, the packed one after
        assert float((a - b).norm() / b.norm()) < 1e-5
    # sparse_grad: COO gradients over the gaussian index (single camera -> coalesced)
    sp = gs.fully_fused_projection(means, None, quats, scales, vm[:1], K[:1], W, H, opacities=opac, packed=True, sparse_grad=True)
    gsp = torch.autograd.grad(sp[5].sum() + sp[7].sum(), (means, quats, scales))
    dn = gs.fully_fused_projection(means, None, quats, scales, vm[:1], K[:1], W, H, opacities=opac, packed=True)
    gdn = torch.autograd.grad(dn[5].sum() + dn[7].sum(), (means, quats, scales))
    for a, b in zip(gsp, gdn):
        assert a.is_sparse and a.is_coalesced() and a.shape == b.shape and a._nnz() == sp[5].shape[0]
        assert torch.equal(a.to_dense(), b)
    # covars input, compensations, batch dimension: packed rows == dense rows
    cov6 = _t(gso.quat_scale_to_covar_preci(sc["quats"], sc["scales"], True, False, True)[0])
    mb = torch.stack([means.detach(), means.detach() + 0.05])
    cb, ob = torch.stack([cov6, cov6]), torch.stack([opac.detach(), opac.detach()])
    vmb, Kb = torch.stack([vm, vm]), torch.stack([K, K])
    d = gs.fully_fused_projection(mb, cb, None, None, vmb, Kb, W, H, opacities=ob, calc_compensations=True)
    pk = gs.fully_fused_projection(mb, cb, None, None, vmb, Kb, W, H, opacities=ob, calc_compensations=True, packed=True)
    selb = (d[0] > 0).all(-1)
    assert pk[3].tolist() == [0] + torch.cumsum(selb.reshape(-1, selb.shape[-1]).sum(-1), 0).tolist()
    nzb = torch.nonzero(selb)
    assert torch.equal(pk[0], nzb[:, 0]) and torch.equal(pk[1], nzb[:, 1]) and torch.equal(pk[2], nzb[:, 2])
    assert torch.equal(pk[5], d[1][selb]) and torch.equal(pk[7], d[3][selb]) and torch.equal(pk[8], d[4][selb])
    # isect on packed rows == isect on the dense layout (same keys; flatten ids index the packed rows)
    tw, th = math.ceil(W / 16), math.ceil(H / 16)
    op_cn = opac.detach()[None].expand(C, -1).contiguous()
    d_tpg, d_ids, d_fl = gs.isect_tiles(m2, radii, dep, 16, tw, th, conics=con, opacities=op_cn)
    image_ids = c_ids.long()
    p_tpg, p_ids, p_fl = gs.isect_tiles(
        p_m2.detach(), p_radii, p_dep.detach(), 16, tw, th, packed=True, n_images=C, image_ids=image_ids, gaussian_ids=g_ids,
        conics=p_con.detach(), opacities=op_cn[sel],
    )
    assert torch.equal(p_ids, d_ids)
    rows = torch.nonzero(sel.reshape(-1)).squeeze(-1)
    assert torch.equal(rows[p_fl.long()], d_fl.long())
    assert torch.equal(p_tpg, d_tpg[sel])
    # packed SH == dense SH on the visible rows
    sh = _t(np.ascontiguousarray(sc["sh"][:, :9]), True)
    dense = gs.spherical_harmonics(2, means, vm, sh, masks=sel)
    packed = gs.spherical_harmonics(2, means, vm, sh[g_ids.long()], batch_ids=b_ids, camera_ids=c_ids, gaussian_ids=g_ids)
    torch.testing.assert_close(packed, dense[sel], rtol=1e-5, atol=1e-6)
    # rows variant (coefficient table indexed in the kernel) == dense kernel on the visible rows, bit for bit; grads close
    rows_col = ops.spherical_harmonics_rows(2, means, vm, sh, b_ids, c_ids, g_ids)
    assert torch.equal(rows_col, dense[sel])
    v = torch.randn_like(rows_col)
    ga = torch.autograd.grad((rows_col * v).sum(), (sh, means), retain_graph=True)
    gb = torch.autograd.grad((dense[sel] * v).sum(), (sh, means), retain_graph=True)
    for a, b in zip(ga, gb):
        assert float((a - b).norm() / b.norm()) < 1e-5
    # and the packed rows render the same image through rasterize_to_pixels(packed=True)
    off = gs.isect_offset_encode(p_ids, C, tw, th)
    col = torch.clamp_min(packed + 0.5, 0.0)
    rc_p, ra_p = gs.rasterize_to_pixels(p_m2, p_con, col, op_cn[sel], W, H, 16, off, p_fl, packed=True)
    dcol = torch.clamp_min(dense + 0.5, 0.0) * sel[..., None]
    rc_d, ra_d = gs.rasterize_to_pixels(m2, con, dcol, op_cn, W, H, 16, gs.isect_offset_encode(d_ids, C, tw, th), d_fl)
    torch.testing.assert_close(rc_p, rc_d, rtol=1e-5, atol=1e-6)
    assert torch.equal(ra_p, ra_d)


def test_distributed_single_rank_is_identity(gs):
    """distributed=True on a 1-rank group == local render (reference: tests/test_rasterization.py:816-870)."""
    import torch.distributed as dist

    if not dist.is_initialized():
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        os.environ.setdefault("MASTER_PORT", "29577")
        dist.init_process_group("nccl", rank=0, world_size=1)
    sc = scene.make_scene(n_max=20000, sh_degree=1)
    W, H = 160, 96
    Ks = scene.rescale_K(sc["Ks"], sc["width"], sc["height"], W, H)
    P = [_t(sc[k], True) for k in ("means", "quats", "scales", "opacities")]
    sh = _t(np.ascontiguousarray(sc["sh"][:, :4]), True)
    cam = (_t(sc["viewmats"][:2]), _t(Ks[:2]), W, H)
    a, aa, _ = gs.rasterization(*P, sh, *cam, sh_degree=1, packed=False)
    b, ba, _ = gs.rasterization(*P, sh, *cam, sh_degree=1, packed=False, distributed=True)
    assert torch.equal(a, b) and torch.equal(aa, ba)


def _torchrun2(script, port):
    import subprocess
    import sys as _sys

    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    root = os.path.abspath(os.path.join(os.path.dirname(__file__), ".."))
    r = subprocess.run(
        [_sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr", "127.0.0.1",
         "--master-port", str(port), os.path.join(root, "tests", script)],
        capture_output=True, text=True, timeout=600,
    )
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-3000:]
    return r.stdout


def test_distributed_two_ranks_sharded():
    """Launches tests/dist_sharded_check.py on 2 GPUs (skipped on a 1-GPU box)."""
    assert _torchrun2("dist_sharded_check.py", 29588).count("sharded check ok") == 4


def test_nvls_allreduce_two_ranks():
    """Own all-reduce kernels (multimem + peer-to-peer) vs NCCL, bit-exact at 2 ranks (skipped on a 1-GPU box)."""
    out = _torchrun2("dist_nvls_check.py", 29590)
    # dense multicast / peer kernels at two grid sizes, the two row-sparse variants, the end-to-end fused backward
    assert "AssertionError" not in out and out.count("nvls check ok") >= 9, out[-2000:]
    assert "rows-p2p moved" in out and "rows-nvls moved" in out and "end-to-end gradients in the arena" in out


def test_selective_adam(gs):
    """adam op + SelectiveAdam vs the float32 oracle (bit-exact: same operations in the same order) and, for the
    visible rows, vs a hand-rolled torch Adam without bias correction."""
    rng = np.random.RandomState(5)
    N = 5000
    for shape in ((N, 3), (N, 16, 3), (N,)):
        p0 = rng.standard_normal(shape).astype(np.float32)
        g = (rng.standard_normal(shape) * 0.1).astype(np.float32)
        m0 = (rng.standard_normal(shape) * 0.01).astype(np.float32)
        v0 = (rng.random_sample(shape) * 1e-3).astype(np.float32)
        vis = rng.random_sample(N) < 0.4
        p, m, v = _t(p0), _t(m0), _t(v0)
        gs.adam(p, _t(g), m, v, _t(vis), 1e-2, 0.9, 0.999, 1e-8)
        op, om, ov = gso.adam(p0, g, m0, v0, vis, 1e-2, 0.9, 0.999, 1e-8)
        assert np.array_equal(_n(m), om) and np.array_equal(_n(v), ov)
        _exactish(_n(p), op, "param")
        assert np.array_equal(_n(p)[~vis], p0[~vis]) and np.array_equal(_n(m)[~vis], m0[~vis])
        gs.adam(p, _t(g), m, v, None, 1e-2, 0.9, 0.999, 1e-8)  # valid=None: every row
        assert not np.array_equal(_n(p)[~vis], p0[~vis])
    # the optimizer front-end (reference API: one tensor per group, step(visibility))
    w = torch.nn.Parameter(_t(rng.standard_normal((N, 3)).astype(np.float32)))
    opt = gs.SelectiveAdam([{"params": [w], "lr": 1e-2}], eps=1e-8, betas=(0.9, 0.999))
    w0 = w.detach().clone()
    (w**2).sum().backward()
    vis_t = _t(rng.random_sample(N) < 0.5)
    opt.step(vis_t)
    gref = 2 * w0
    expect = w0 - 1e-2 * (0.1 * gref) / ((0.001 * gref * gref).sqrt() + 1e-8)
    torch.testing.assert_close(w.detach()[vis_t], expect[vis_t], rtol=1e-5, atol=1e-6)
    assert torch.equal(w.detach()[~vis_t], w0[~vis_t])


def test_fused_l1_loss(gs):
    """l1_loss == (a - b).abs().mean() and its autograd gradient; deterministic; odd sizes; scaled upstream gradient."""
    g = torch.Generator(device=DEV).manual_seed(9)
    for shape in ((1, 1080, 1920, 3), (3, 37, 53, 3), (5,)):
        a = torch.rand(shape, device=DEV, generator=g).requires_grad_(True)
        b = torch.rand(shape, device=DEV, generator=g)
        b.view(-1)[::7] = a.detach().view(-1)[::7]  # exact zeros of a - b: subgradient 0 like torch
        ours = gs.l1_loss(a, b)
        ref = (a - b).abs().mean()
        np.testing.assert_allclose(float(ours), float((a.double() - b.double()).abs().mean()), rtol=2e-6)
        np.testing.assert_allclose(float(ours), float(ref), rtol=1e-5)
        (g1,) = torch.autograd.grad(ours * 3.0, a)
        (g2,) = torch.autograd.grad(ref * 3.0, a)
        torch.testing.assert_close(g1, g2, rtol=1e-6, atol=0)
        assert float(gs.l1_loss(a, b)) == float(ours)


def _torch_ssim_loss_f64(img1, img2):
    """float64 restatement of the reference's torch path (gsplat/losses.py:82-151, 190-201): 11-tap Gaussian
    window sigma 1.5, zero padding, per channel, 1 - mean."""
    import torch.nn.functional as F

    x = torch.arange(11, dtype=torch.float32)
    g = torch.exp(-((x - 5) ** 2) / (2 * 1.5**2))
    g = (g / g.sum()).double()
    C = img1.shape[1]
    w = (g[:, None] @ g[None, :])[None, None].expand(C, 1, 11, 11).contiguous().to(img1.device)
    conv = lambda t: F.conv2d(t, w, padding=5, groups=C)  # noqa: E731
    mu1, mu2 = conv(img1), conv(img2)
    s11, s22, s12 = conv(img1 * img1) - mu1 * mu1, conv(img2 * img2) - mu2 * mu2, conv(img1 * img2) - mu1 * mu2
    m = ((2 * mu1 * mu2 + 0.01**2) * (2 * s12 + 0.03**2)) / ((mu1 * mu1 + mu2 * mu2 + 0.01**2) * (s11 + s22 + 0.03**2))
    return 1.0 - m.mean()


@pytest.mark.parametrize("layout", ["nchw", "nhwc_view"])
@pytest.mark.parametrize("shape", [(2, 3, 70, 95), (1, 3, 16, 16), (1, 1, 5, 37)])
def test_fused_ssim_loss(gs, layout, shape):
    torch.manual_seed(3)
    B, C, H, W = shape
    if layout == "nchw":
        a = torch.rand(shape, device=DEV)
        b = torch.rand(shape, device=DEV)
    else:  # what the trainer passes: render[B,H,W,C].permute(0,3,1,2)
        a = torch.rand((B, H, W, C), device=DEV).permute(0, 3, 1, 2)
        b = torch.rand((B, H, W, C), device=DEV).permute(0, 3, 1, 2)
    b = (0.7 * a + 0.3 * b).detach()  # correlated images: SSIM away from 0
    a.requires_grad_(True)
    loss = gs.ssim_loss(a, b)
    (loss * 1.7).backward()
    a64 = a.detach().double().contiguous().requires_grad_(True)
    ref = _torch_ssim_loss_f64(a64, b.double().contiguous())
    (ref * 1.7).backward()
    assert abs(loss.item() - ref.item()) <= 1e-5 * abs(ref.item()) + 1e-6, (loss.item(), ref.item())
    g, gr = a.grad.double(), a64.grad
    assert g.shape == gr.shape
    err = (g - gr).abs().max().item()
    assert err <= 1e-4 * gr.abs().max().item() + 1e-9, f"ssim grad max err {err:.3e} vs max {gr.abs().max().item():.3e}"
    # forward-only call allocates no derivative maps and agrees
    with torch.no_grad():
        assert abs(gs.ssim_loss(a.detach(), b).item() - loss.item()) < 1e-7
