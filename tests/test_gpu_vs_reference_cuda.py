"""GPU parity against the REAL reference CUDA operators (nerfstudio-project/gsplat v1.6.0, built for sm_100a with
its release flags by oracle/build_ref.py and called through torch.ops.gsplat.*).  What the reference computed is
stored under tests/golden/ref_cuda/ (tests/golden/make_ref_cuda_golden.py, run once on a B200): a fixed, seeded
sample of its outputs (Gaussians / rows / pixels), full-size visibility masks, and statistics of its full outputs
such as its run-to-run spread.  The inputs are regenerated here from the same seeds.

The reference is built with -use_fast_math (its default) and accumulates gradients with float atomics,
so it is itself only reproducible to ~1e-6 relative; its own tests compare at rtol 1e-5..2.5e-4 /
atol 1e-3..2e-3 for gradients (tests/test_basic.py:2664-2692).  Here: north_star's rtol 1e-4 / atol 1e-5
on rendered colours / alphas (with a bounded count of threshold-flip pixels), relative-L2 bounds on
gradients, exact equality on sort keys when fed identical projections.
"""
import math
import os

import numpy as np
import pytest
import torch

from tests import scene

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "ref_cuda")


@pytest.fixture(scope="module")
def gs():
    import gsplat_b200

    return gsplat_b200


def _gold(name):
    d = np.load(os.path.join(GOLDEN, name))
    return {k: d[k] for k in d.files}


def _t(a, rg=False):
    t = torch.from_numpy(np.ascontiguousarray(a)).to(DEV)
    return t.requires_grad_(True) if rg else t


def _bits(packed, shape):
    """Boolean mask stored with np.packbits."""
    return _t(np.unpackbits(packed)[: math.prod(shape)].reshape(shape).astype(bool))


def _rel(a, b):
    a, b = a.double(), b.double()
    return float((a - b).norm() / b.norm().clamp_min(1e-30))


def _scene(n_max, W, H, C, sh_degree=3, grid=1):
    sc = scene.make_scene(scene_grid=grid, n_max=n_max, sh_degree=sh_degree)
    Ks = scene.rescale_K(sc["Ks"], sc["width"], sc["height"], W, H)[:C]
    return sc, _t(sc["viewmats"][:C]), _t(Ks)


def test_projection_and_sh_vs_reference(gs):
    W, H, C = 960, 540, 2
    sc, vm, Ks = _scene(80000, W, H, C)
    ref = _gold("projection_sh.npz")
    means, quats, scales, opac, sh = (_t(sc[k]) for k in ("means", "quats", "scales", "opacities", "sh"))
    N = len(means)
    radii, m2, dep, con, col, _ = gs.fused_project_sh(means, quats, scales, opac, sh, vm, Ks, W, H, 3)
    rv, ov = _bits(ref["vis"], (C, N)), (radii > 0).all(-1)
    assert (rv != ov).float().mean() < 1e-4, "visibility sets differ"
    assert (rv & ov).sum() > 10000
    # per-element comparisons on the stored sample of Gaussians
    i = _t(ref["idx"])
    sub = lambda x: x[:, i].contiguous()  # noqa: E731
    both = sub(rv & ov)
    r_radii, r_m2, r_dep, r_con, r_col = (_t(ref[k]) for k in ("radii", "means2d", "depths", "conics", "colors"))
    radii, m2, dep, con, col = (sub(x) for x in (radii, m2, dep, con, col))
    assert ((r_radii[both] - radii[both]).abs() <= 1).all() and (r_radii[both] != radii[both]).float().mean() < 1e-3
    torch.testing.assert_close(m2[both], r_m2[both], rtol=1e-4, atol=1e-3)
    torch.testing.assert_close(dep[both], r_dep[both], rtol=1e-5, atol=1e-6)
    assert _rel(con[both], r_con[both]) < 1e-4
    torch.testing.assert_close(con[both], r_con[both], rtol=5e-3, atol=1e-5)  # fast-math conic of tiny gaussians
    torch.testing.assert_close(col[both], r_col[both], rtol=1e-4, atol=1e-5)
    # backward of both ops with common cotangents, on the sampled Gaussians and the reference's radii / conics
    g = torch.Generator(device=DEV).manual_seed(0)
    v_m2, v_dep, v_con = (torch.randn(s, device=DEV, generator=g) for s in ((C, N, 2), (C, N), (C, N, 3)))
    v_col = torch.randn((C, N, 3), device=DEV, generator=g)
    v_m2, v_dep, v_con, v_col = (sub(x) for x in (v_m2, v_dep, v_con, v_col))
    means, quats, scales, sh = (x[i].contiguous() for x in (means, quats, scales, sh))
    L = gs._cabi.lib()
    from gsplat_b200._cabi import ptr, stream

    v_means, v_quats, v_scales, v_sh = (torch.empty_like(x) for x in (means, quats, scales, sh))
    rc = L.gsb200_project_sh_bwd(
        C, len(means), 16, 3, ptr(means), ptr(quats), ptr(scales), ptr(sh), ptr(vm), ptr(Ks), W, H, 0.3, ptr(r_radii),
        ptr(r_con), None, ptr(r_col), ptr(v_m2), 2, ptr(v_dep), 1, ptr(v_con), 3, ptr(v_col), 3, None,
        ptr(v_means), ptr(v_quats), ptr(v_scales), ptr(v_sh), None, stream(),
    )
    assert rc == 0
    assert _rel(v_means, _t(ref["v_means"])) < 1e-4
    assert _rel(v_quats, _t(ref["v_quats"])) < 1e-3 and _rel(v_scales, _t(ref["v_scales"])) < 1e-3
    assert _rel(v_sh, _t(ref["v_sh"])) < 1e-5


@pytest.mark.parametrize("model,cam_id", [("ortho", 1), ("fisheye", 2)])
def test_projection_camera_models_vs_reference(gs, model, cam_id):
    """Ortho / fisheye projection fwd + bwd against the reference CUDA kernels (CameraModelType 1 / 2)."""
    W, H, C = 960, 540, 2
    sc, vm, Ks = _scene(60000, W, H, C)
    if model == "ortho":
        Ks = Ks.clone()
        Ks[:, 0, 0], Ks[:, 1, 1] = 180.0, 170.0
    ref = _gold(f"projection_{model}.npz")
    means, quats, scales, opac = (_t(sc[k]) for k in ("means", "quats", "scales", "opacities"))
    N = len(means)
    o = gs.fully_fused_projection(means, None, quats, scales, vm, Ks, W, H, opacities=opac, camera_model=model)
    rv, ov = _bits(ref["vis"], (C, N)), (o[0] > 0).all(-1)
    assert (rv != ov).float().mean() < 1e-4
    assert (rv & ov).sum() > 5000
    i = _t(ref["idx"])
    sub = lambda x: x[:, i].contiguous()  # noqa: E731
    both = sub(rv & ov)
    r = [_t(ref[k]) for k in ("radii", "means2d", "depths", "conics")]
    o = [sub(x) for x in o[:4]]
    assert ((r[0][both] - o[0][both]).abs() <= 1).all()
    torch.testing.assert_close(o[1][both], r[1][both], rtol=1e-4, atol=2e-3)
    torch.testing.assert_close(o[2][both], r[2][both], rtol=1e-5, atol=1e-6)
    assert _rel(o[3][both], r[3][both]) < 1e-4
    g = torch.Generator(device=DEV).manual_seed(1)
    v_m2, v_dep, v_con = (sub(torch.randn(s, device=DEV, generator=g)) for s in ((C, N, 2), (C, N), (C, N, 3)))
    means, quats, scales = (x[i].contiguous() for x in (means, quats, scales))
    S = len(means)
    L = gs._cabi.lib()
    from gsplat_b200._cabi import ptr, stream

    v_means, v_quats, v_scales, v_vm = (torch.empty_like(x) for x in (means, quats, scales, vm))
    rc = L.gsb200_projection_bwd(
        1, C, S, ptr(means), None, ptr(quats), ptr(scales), ptr(vm), ptr(Ks), W, H, 0.3, cam_id, ptr(r[0]), ptr(r[3]), None,
        ptr(v_m2), 2, ptr(v_dep), 1, ptr(v_con), 3, None, ptr(v_means), None, ptr(v_quats), ptr(v_scales), ptr(v_vm), stream(),
    )
    assert rc == 0
    assert _rel(v_means, _t(ref["v_means"])) < 2e-4 and _rel(v_quats, _t(ref["v_quats"])) < 2e-4
    assert _rel(v_scales, _t(ref["v_scales"])) < 2e-4
    assert _rel(v_vm, _t(ref["v_viewmats"])) < 2e-3


def test_isect_vs_reference_on_identical_projection(gs):
    W, H, C = 1280, 720, 2
    sc, vm, Ks = _scene(100000, W, H, C)
    ref = _gold("isect.npz")
    means, quats, scales, opac = (_t(sc[k]) for k in ("means", "quats", "scales", "opacities"))
    radii, m2, dep, con, _ = gs.fully_fused_projection(means, None, quats, scales, vm, Ks, W, H, opacities=opac)
    op = opac[None].expand(C, -1).contiguous()
    tw, th = math.ceil(W / 16), math.ceil(H / 16)
    tpg, ids, fl = gs.isect_tiles(m2, radii, dep, 16, tw, th, conics=con, opacities=op)
    # the reference evaluates the ellipse bounds with fast-math (approximate div / sqrt / log): a gaussian
    # whose bound falls within an ulp of a tile edge may gain or lose a tile.  Such tiles hold no pixel with
    # alpha >= 1/255, so images are unaffected; here the symmetric difference must stay below 1e-4.
    diff = (tpg != _t(ref["tiles_per_gauss"]).to(tpg.dtype)).float().mean()
    assert diff < 1e-4, f"tiles_per_gauss differs on {diff * 100:.4f}% of gaussians"
    n_ref = int(ref["n_isects"])
    if ids.numel() == n_ref:
        same = (ids[_t(ref["pos"])] == _t(ref["isect_ids"])).float().mean()
        assert same > 0.999
    assert abs(ids.numel() - n_ref) <= 1e-4 * ids.numel() + 2


@pytest.mark.parametrize("D,with_bg", [(3, False), (3, True), (4, False), (1, False)])
def test_raster_vs_reference(gs, D, with_bg):
    W, H, C = 1280, 720, 1
    sc, vm, Ks = _scene(150000, W, H, C)
    ref = _gold(f"raster_D{D}_bg{int(with_bg)}.npz")
    means, quats, scales, opac = (_t(sc[k]) for k in ("means", "quats", "scales", "opacities"))
    radii, m2, dep, con, _ = gs.fully_fused_projection(means, None, quats, scales, vm, Ks, W, H, opacities=opac)
    op = opac[None].expand(C, -1).contiguous()
    tw, th = math.ceil(W / 16), math.ceil(H / 16)
    # the reference rendered from its own intersection lists, which equal ours on the same projection
    # (test_isect_vs_reference_on_identical_projection)
    _, ids, fl = gs.isect_tiles(m2, radii, dep, 16, tw, th, conics=con, opacities=op)
    off = gs.isect_offset_encode(ids, C, tw, th)
    g = torch.Generator(device=DEV).manual_seed(D)
    col = torch.rand((C, len(means), D), device=DEV, generator=g)
    bg = torch.rand((C, D), device=DEV, generator=g) if with_bg else None
    ins = [x.detach().clone().requires_grad_(True) for x in (m2, con, col, op)]
    rc, ra = gs.rasterize_to_pixels(*ins, W, H, 16, off, fl, backgrounds=bg)
    p = _t(ref["pix"])
    r_rc, r_ra = _t(ref["render_colors"]), _t(ref["render_alphas"])
    s_rc, s_ra = rc.detach().reshape(-1, D)[p], ra.detach().reshape(-1)[p]
    err = (s_rc - r_rc).abs() - (1e-4 * r_rc.abs() + 1e-5)
    bad = (err.amax(-1) > 0).float().mean()
    # __expf and the alpha >= 1/255 / T <= 1e-4 decisions can flip on a few pixels between two correct
    # implementations; a flip changes a pixel by at most ~0.4 % of a colour
    assert bad < 2e-4, f"{bad * 100:.4f}% of pixels exceed rtol 1e-4 / atol 1e-5"
    assert (s_rc - r_rc).abs().max() < 2e-2 and (s_ra - r_ra).abs().max() < 2e-2
    v_rc = torch.randn(rc.shape, device=DEV, generator=g)
    v_ra = torch.randn(ra.shape, device=DEV, generator=g)
    grads = torch.autograd.grad((rc * v_rc).sum() + (ra * v_ra).sum(), ins)
    i = _t(ref["idx"])
    # two runs of the reference itself differ by its atomic order; that spread was measured on its full outputs,
    # ours must be within a small multiple of it (and within absolute bounds)
    for name, a, lim in (
        ("v_means2d", grads[0], 2e-4), ("v_conics", grads[1], 2e-4), ("v_colors", grads[2], 5e-5), ("v_opacities", grads[3], 2e-4),
    ):
        spread = float(ref["spread_" + name])
        rel = _rel(a[:, i], _t(ref[name]))
        assert rel < max(lim, 20 * spread), f"{name}: rel L2 {rel:.3e} (reference run-to-run {spread:.3e})"


def test_full_path_vs_reference_1080p(gs):
    """BASELINE configs[1]: ~100k gaussians, 1 camera 1080p, SH3, fwd + bwd vs the reference CUDA ops chained
    exactly as its orchestrator does (csrc/Rendering.cpp:976-1447)."""
    W, H, C = 1920, 1080, 1
    sc, vm, Ks = _scene(None, W, H, C)
    ref = _gold("full_1080p.npz")
    P = {k: _t(sc[k], True) for k in ("means", "quats", "scales", "opacities", "sh")}
    rc, ra, meta = gs.rasterization(P["means"], P["quats"], P["scales"], P["opacities"], P["sh"], vm, Ks, W, H, sh_degree=3, packed=False)
    s_rc, r_rc = rc.detach().reshape(-1, 3)[_t(ref["pix"])], _t(ref["render_colors"])
    err = (s_rc - r_rc).abs() - (1e-4 * r_rc.abs() + 1e-5)
    bad = (err.amax(-1) > 0).float().mean()
    assert bad < 1e-3, f"{bad * 100:.4f}% of pixels exceed rtol 1e-4 / atol 1e-5 vs the reference CUDA rasterizer"
    assert (s_rc - r_rc).abs().max() < 5e-2
    g = torch.Generator(device=DEV).manual_seed(3)
    v_rc, v_ra = torch.randn(rc.shape, device=DEV, generator=g), torch.randn(ra.shape, device=DEV, generator=g)
    ((rc * v_rc).sum() + (ra * v_ra).sum()).backward()
    i = _t(ref["idx"])
    grad = lambda k: P[k].grad[i]  # noqa: E731
    assert _rel(grad("sh"), _t(ref["v_sh"])) < 1e-3
    assert _rel(grad("opacities"), _t(ref["v_opacities"])) < 1e-3
    assert _rel(grad("means"), _t(ref["v_means"])) < 2e-3
    assert _rel(grad("quats"), _t(ref["v_quats"])) < 5e-3 and _rel(grad("scales"), _t(ref["v_scales"])) < 5e-3


def test_adam_and_relocation_vs_reference(gs):
    """Trainer-side ops against the reference kernels (csrc/AdamCUDA.cu, RelocationCUDA.cu, MCMCPerturbCUDA.cu)."""
    ref = _gold("adam_relocation.npz")
    g = torch.Generator(device=DEV).manual_seed(3)
    N = 20000
    for tag, shape in (("a", (N, 3)), ("b", (N, 16, 3))):
        p = torch.randn(shape, device=DEV, generator=g)
        grad = torch.randn(shape, device=DEV, generator=g) * 0.1
        m = torch.randn(shape, device=DEV, generator=g) * 0.01
        v = torch.rand(shape, device=DEV, generator=g) * 1e-3
        vis = torch.rand(N, device=DEV, generator=g) < 0.3
        b = [x.clone() for x in (p, m, v)]
        gs.adam(b[0], grad, b[1], b[2], vis, 1e-2, 0.9, 0.999, 1e-8)
        i = _t(ref[f"adam_{tag}_idx"])
        for x, name in zip(b, ("param", "exp_avg", "exp_avg_sq")):
            # the reference is built with fast-math (FMA: cancellation in m)
            torch.testing.assert_close(x[i], _t(ref[f"adam_{tag}_{name}"]), rtol=1e-5, atol=1e-7)
        assert torch.equal(b[0][~vis], p[~vis])
    # relocation
    n_max = 51
    binoms = torch.zeros((n_max, n_max), device=DEV)
    for n in range(n_max):
        for k in range(n + 1):
            binoms[n, k] = math.comb(n, k)
    opac = torch.rand(N, device=DEV, generator=g) * 0.98 + 0.01
    scales = torch.rand((N, 3), device=DEV, generator=g) * 0.1 + 1e-3
    ratios = torch.randint(1, 12, (N,), device=DEV, generator=g)
    o, s = gs.compute_relocation(opac, scales, ratios.clone(), binoms, 0.005)
    i = _t(ref["reloc_idx"])
    torch.testing.assert_close(o[i], _t(ref["reloc_opacities"]), rtol=1e-5, atol=1e-7)
    torch.testing.assert_close(s[i], _t(ref["reloc_scales"]), rtol=1e-4, atol=1e-8)


def test_packed_projection_vs_reference(gs):
    """Two-pass compacting projection fwd + bwd against the reference's projection_ewa_3dgs_packed kernels."""
    W, H, C = 960, 540, 3
    sc, vm, Ks = _scene(70000, W, H, C)
    ref = _gold("packed_projection.npz")
    means, quats, scales, opac = (_t(sc[k]) for k in ("means", "quats", "scales", "opacities"))
    o = gs.fully_fused_projection(means, None, quats, scales, vm, Ks, W, H, opacities=opac, packed=True, calc_compensations=True)
    # the reference's rows are the visible (camera, gaussian) pairs in ascending order: key = camera * N + gaussian
    N = len(means)
    rk = np.flatnonzero(np.unpackbits(ref["vis"])[: C * N])
    ok = (o[1] * N + o[2]).cpu().numpy()
    # visibility differs on a handful of borderline rows (fast-math radius): compare on the common (camera, gaussian) keys
    assert abs(len(rk) - len(ok)) <= max(2, int(1e-4 * len(rk)))
    common = np.intersect1d(rk, ok)
    assert len(common) > 0.999 * len(rk)
    assert (np.diff(ok) > 0).all(), "rows must be in ascending (camera, gaussian) order"
    sel = ref["sel"]
    keys = rk[sel]
    oi = np.searchsorted(ok, keys).clip(max=len(ok) - 1)
    found = ok[oi] == keys
    oi, fi = _t(oi[found]), _t(found)
    torch.testing.assert_close(o[5][oi], _t(ref["means2d"])[fi], rtol=1e-4, atol=1e-3)
    torch.testing.assert_close(o[6][oi], _t(ref["depths"])[fi], rtol=1e-5, atol=1e-6)
    assert _rel(o[7][oi], _t(ref["conics"])[fi]) < 1e-4 and _rel(o[8][oi], _t(ref["compensations"])[fi]) < 1e-5
    if len(rk) == len(ok):
        assert torch.equal(o[3], _t(ref["indptr"]).to(o[3].dtype))
    # backward on the reference's own rows / conics (the sampled rows; dense accumulation)
    g = torch.Generator(device=DEV).manual_seed(2)
    nnz = len(rk)
    s = _t(sel)
    v_m2, v_dep, v_con = (torch.randn(sh, device=DEV, generator=g)[s].contiguous() for sh in ((nnz, 2), (nnz,), (nnz, 3)))
    ids = o[1].dtype
    rc_, rg = _t(keys // N).to(ids), _t(keys % N).to(ids)
    rb = torch.zeros_like(rc_)
    rcon = _t(ref["conics"])
    L = gs._cabi.lib()
    from gsplat_b200._cabi import ptr, stream

    v_means, v_quats, v_scales, v_vm = (torch.zeros_like(x) for x in (means, quats, scales, vm))
    rc = L.gsb200_projection_packed_bwd(
        1, C, N, len(sel), ptr(means), None, ptr(quats), ptr(scales), ptr(vm), ptr(Ks), W, H, 0.3, 0, ptr(rb), ptr(rc_), ptr(rg),
        ptr(rcon), None, ptr(v_m2), 2, ptr(v_dep), 1, ptr(v_con), 3, None, 0, ptr(v_means), None, ptr(v_quats), ptr(v_scales),
        ptr(v_vm), stream(),
    )
    assert rc == 0
    t = _t(ref["touched"])
    assert _rel(v_means[t], _t(ref["v_means"])) < 1e-4 and _rel(v_quats[t], _t(ref["v_quats"])) < 1e-4
    assert _rel(v_scales[t], _t(ref["v_scales"])) < 1e-4
    assert _rel(v_vm, _t(ref["v_viewmats"])) < 1e-3


def _stock_step(G, P, vm, Ks, W, H, deg, v_rc, v_ra):
    """fwd + bwd through a rasterization() callable G; returns render, alpha and the parameter gradients."""
    ins = {k: v.detach().clone().requires_grad_(True) for k, v in P.items()}
    rc, ra, _ = G(ins["means"], ins["quats"], ins["scales"], ins["opacities"], ins["sh"], vm, Ks, W, H, sh_degree=deg, packed=False)
    ((rc * v_rc).sum() + (ra * v_ra).sum()).backward()
    return rc.detach(), ra.detach(), {k: ins[k].grad.detach() for k in ins}


@pytest.mark.parametrize("cfg", ["cfg1_garden_256_sh0", "cfg2_100k_1080p_sh3"])
def test_stock_rasterization_with_gradient_spread(gs, cfg):
    """BASELINE configs[0] / configs[1] against the reference's STOCK path -- the unmodified gsplat package:
    gsplat.rasterization() -> rasterization_3dgs orchestrator + its registered autograd.

    What is measured and printed, per gradient tensor:
      * the reference's own run-to-run spread (two runs, same inputs; stored);
      * ours vs the reference: relative L2, max |diff| / max |g|, and the fraction of elements outside
        rtol 1e-4 + atol 1e-5 * max|g| (north_star's per-element tolerance, the absolute part scaled to the tensor),
        on the stored sample of Gaussians;
      * cfg1 only: BOTH implementations against the float64 CPU oracle (the ground truth of the reference's formulas).
    Measured on B200 (round 2): the reference's run-to-run spread is 3e-8 ... 1e-5 in relative L2, i.e. its float
    atomics are NOT what separates two correct implementations; ours and the reference differ by 2e-5 ... 4e-4 in
    relative L2 because the reference is a -use_fast_math build (approximate division / rsqrt / log in the projection
    and conic inversion) while the b200 per-gaussian kernels are bit-exact against the float32 oracle, and because
    discrete decisions (alpha >= 1/255, T <= 1e-4, radius / tile cuts) flip on a few (pixel, gaussian) pairs.
    Contract asserted here: render / alpha rtol 1e-4, atol 1e-5 on all but < 0.1 % decision-flip pixels; every
    gradient tensor within 1e-3 relative L2 of the reference and >= 99 % of its elements within
    rtol 1e-4 + atol 1e-5 * max|g|; on cfg1 ours must be at least as close to the float64 oracle as the reference is
    (factor 1.5 + 2e-5)."""
    import json

    from oracle import gso

    ref = _gold(f"stock_{cfg}.npz")
    if cfg.startswith("cfg1"):
        sc = scene.make_scene(sh_degree=0)
        W = H = 256
        vm, Ks, deg = _t(sc["viewmats"][:1]), _t(sc["Ks"][:1]), 0
    else:
        W, H, deg = 1920, 1080, 3
        sc, vm, Ks = _scene(100000, W, H, 1)
    P = {k: _t(sc[k]) for k in ("means", "quats", "scales", "opacities", "sh")}
    g = torch.Generator(device=DEV).manual_seed(11)
    v_rc, v_ra = torch.randn((1, H, W, 3), device=DEV, generator=g), torch.randn((1, H, W, 1), device=DEV, generator=g)
    o1 = _stock_step(gs.rasterization, P, vm, Ks, W, H, deg, v_rc, v_ra)
    oracle = None
    if cfg.startswith("cfg1"):
        f8 = lambda a: np.ascontiguousarray(a, np.float64)  # noqa: E731
        _, og = gso.rasterization_fwd_bwd(
            f8(sc["means"]), f8(sc["quats"]), f8(sc["scales"]), f8(sc["opacities"]), f8(sc["sh"]), f8(sc["viewmats"][:1]),
            f8(sc["Ks"][:1]), W, H, 0, f8(v_rc.cpu().numpy()), f8(v_ra.cpu().numpy()),
        )
        oracle = {k: torch.from_numpy(np.asarray(og["v_" + k])).to(DEV) for k in ("means", "quats", "scales", "opacities", "sh")}
    p = _t(ref["pix"])
    rc, ra = o1[0].reshape(-1, 3)[p], o1[1].reshape(-1)[p]
    r_rc, r_ra = _t(ref["render_colors"]), _t(ref["render_alphas"])
    err = (rc - r_rc).abs() - (1e-4 * r_rc.abs() + 1e-5)
    bad = float((err.amax(-1) > 0).float().mean())
    bad_a = float((((ra - r_ra).abs() - (1e-4 * r_ra.abs() + 1e-5)) > 0).float().mean())
    report = {"cfg": cfg, "n_gaussians": int(P["means"].shape[0]), "render_pixels_out_of_1e-4_1e-5": bad, "alpha_pixels_out": bad_a, "grads": {}}
    fails = []
    i = _t(ref["idx"])
    for k in ("means", "quats", "scales", "opacities", "sh"):
        ref_g, our_g = _t(ref["v_" + k]), o1[2][k][i]
        scale = float(ref["scale_" + k])
        tol = 1e-4 * ref_g.abs() + 1e-5 * scale
        row = {
            "ref_run_to_run_rel_l2": float(ref["run_to_run_rel_l2_" + k]), "ours_vs_ref_rel_l2": _rel(our_g, ref_g),
            "ref_run_to_run_max_over_scale": float(ref["run_to_run_max_over_scale_" + k]),
            "ours_vs_ref_max_over_scale": float((our_g - ref_g).abs().max()) / scale,
            "ours_vs_ref_frac_outside_rtol1e-4_atol1e-5scale": float(((our_g - ref_g).abs() > tol).float().mean()),
        }
        if oracle is not None:
            og64 = oracle[k].reshape(o1[2][k].shape)
            row["ours_vs_oracle64_rel_l2"] = float((o1[2][k].double() - og64).norm() / og64.norm())
            row["ref_vs_oracle64_rel_l2"] = float(ref["vs_oracle64_rel_l2_" + k])
            # (sh is reported but not asserted against the oracle: the garden colours contain exact zeros, whose SH
            # value sits exactly on the relu edge of clamp_min(sh + 0.5, 0) -- float32 and float64 evaluations fall on
            # different sides of it, for the reference and for us alike: both read 0.177 against the float64 oracle)
            if k != "sh" and not row["ours_vs_oracle64_rel_l2"] <= 1.5 * row["ref_vs_oracle64_rel_l2"] + 2e-5:
                fails.append(f"{k}: ours vs float64 oracle {row['ours_vs_oracle64_rel_l2']:.3e}, reference vs oracle {row['ref_vs_oracle64_rel_l2']:.3e}")
        report["grads"][k] = row
        if not row["ours_vs_ref_rel_l2"] <= 1e-3:
            fails.append(f"{k}: rel L2 {row['ours_vs_ref_rel_l2']:.3e} vs the reference")
        if not row["ours_vs_ref_frac_outside_rtol1e-4_atol1e-5scale"] <= 1e-2:
            fails.append(f"{k}: {row['ours_vs_ref_frac_outside_rtol1e-4_atol1e-5scale'] * 100:.3f} % of the elements outside rtol 1e-4 + atol 1e-5 max|g|")
    print(json.dumps(report))
    assert bad < 1e-3 and bad_a < 1e-3, report
    assert (rc - r_rc).abs().max() < 5e-2
    assert not fails, (fails, report)
