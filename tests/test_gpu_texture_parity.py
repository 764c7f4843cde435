"""GPU parity of the texture fetch (DESIGN.md 3.6), bit for bit against the oracle: the fused attribute map of
render() (render_attr=True: the shading kernel samples the texture in groups of four channels) on every channel
count, non-square and non-power-of-two textures, UVs far outside [0, 1) and on texel edges, per-channel
backgrounds and texture_override; the dr.texture operator (wr_texture) with per-view textures and edge coordinates
in all six filter x boundary modes; and the maps SmartPainter renders (one-channel nearest texture + bake view map,
render.py's generic shading instantiation with out_geo) with the view scores taken from them."""
import numpy as np
import pytest
import torch

import cases
import worldrenderer_b200 as wr
from oracle import render_oracle, shim
from oracle.render_oracle import DepthSpec
from test_gpu_render_parity import make_mesh
from test_gpu_stitched_mesh import stitched_mesh
from worldrenderer_b200 import _native, smart_paint
from worldrenderer_b200.render import render_geometry_raw

pytestmark = pytest.mark.gpu

f32 = np.float32


def _np(t):
    return t.detach().cpu().numpy()


def _uv_mesh(form, device, TH, TW, seed):
    """icosphere(8) with one atlas cell per face pair, plain (tri_nrm = NULL) or in the seams form of load_mesh (with
    the texture vertices listed in another order, so that t_tex_idx != t_pos_idx there too).  Every face is shifted
    as a whole by one of 0, +-1, +2, -2, 0.37, -0.61, -1.25 (UVs in about [-2, 3]); a few faces sit with all corners
    on one edge value -- 0, 1, -1e-9, k / TW, (k + 1/2) / TW -- and a few single corners on such values."""
    if form == "plain":
        mesh = make_mesh(*cases.icosphere_mesh(8), device, with_uv=True)
    else:
        mesh = stitched_mesh("seams", device)
    rng = np.random.default_rng(seed)
    vt = _np(mesh.v_tex).reshape(-1, 3, 2).astype(f32)
    nf = vt.shape[0]
    shifts = np.array([0.0, 1.0, -1.0, 2.0, -2.0, 0.37, -0.61, -1.25], f32)
    vt = vt + shifts[rng.integers(0, len(shifts), nf)][:, None, None]
    k = int(rng.integers(1, max(TW, 2)))   # a 1-texel axis has only the edges 0 and 1
    j = int(rng.integers(1, max(TH, 2)))
    edges = np.array([[0.0, 0.0], [1.0, 1.0], [-1e-9, -1e-9], [0.0, 1.0], [1.0, -1e-9],
                      [k / TW, j / TH], [(k + 0.5) / TW, (j + 0.5) / TH], [1.0 / TW, 0.5], [-1e-9, (TH - 1.0) / TH]], f32)
    faces = rng.choice(nf, 2 * len(edges), replace=False)
    for n, e in enumerate(edges):
        vt[faces[n]] = e                                        # a whole face on the edge value
        vt[faces[len(edges) + n], n % 3] = e                    # one corner of another face
    vt = vt.reshape(-1, 2)
    ft = np.arange(vt.shape[0], dtype=np.int64).reshape(-1, 3)
    if form != "plain":
        p = rng.permutation(vt.shape[0])
        inv = np.argsort(p)
        vt, ft = vt[p], inv[ft]
        assert not np.array_equal(ft, _np(mesh.t_pos_idx))
    mesh.v_tex = torch.from_numpy(np.ascontiguousarray(vt)).to(device)
    mesh.t_tex_idx = torch.from_numpy(ft).to(device)
    return mesh


@pytest.mark.parametrize("TC", [1, 2, 3, 4, 5, 8])
@pytest.mark.parametrize("TH,TW", [(37, 53), (1, 7), (2048, 1024)])
def test_fused_attr_matches_oracle(wr_ctx, TH, TW, TC):
    """render(render_attr=True) against render_oracle.render(texture=...): nearest and linear, a scalar and a
    per-channel background, the mesh's texture and texture_override, on the plain and the seams mesh."""
    dev = wr_ctx.device
    rng = np.random.default_rng(1000 * TH + TW + TC)
    tex = rng.uniform(-1.0, 1.0, (TH, TW, TC)).astype(f32)
    cam = cases.canonical_cameras(device=dev)
    H, W = 72, 88
    for form in ("plain", "seams"):
        mesh = _uv_mesh(form, dev, TH, TW, seed=TC)
        for filt in ("nearest", "linear"):
            override = (form == "seams") != (filt == "linear")
            if override:   # the mesh's own texture must not be read
                mesh.texture = torch.full((3, 5, TC), 7.0, device=dev)
                kw = dict(texture_override=torch.from_numpy(tex).to(dev))
            else:
                mesh.texture = torch.from_numpy(tex).to(dev)
                kw = {}
            per_channel = (form == "plain") == (filt == "linear")
            bg = rng.uniform(-2, 2, TC).astype(f32) if per_channel else np.full(TC, 0.25, f32)
            out = wr.render(wr_ctx, mesh, cam, H, W, render_attr=True, texture_filter_mode=filt,
                            attr_background=torch.from_numpy(bg) if per_channel else 0.25, **kw)
            ref = render_oracle.render(_np(mesh.v_pos), _np(mesh.t_pos_idx).astype(np.int32), _np(cam.mvp_mtx),
                                       _np(cam.w2c), H, W, v_nrm=_np(mesh.v_nrm),
                                       tri_nrm=_np(mesh.stitched_t_pos_idx).astype(np.int32),
                                       depth=DepthSpec("controlnet"), v_tex=_np(mesh.v_tex),
                                       tri_tex=_np(mesh.t_tex_idx).astype(np.int32), texture=tex,
                                       texture_filter_mode=filt, attr_background=0.0)
            want = np.where(ref["mask"][..., None], ref["attr"], bg).astype(f32)
            assert out.attr.shape == (6, H, W, TC)
            msg = f"{form} {filt} override={override} per_channel_bg={per_channel}"
            np.testing.assert_array_equal(_np(out.mask), ref["mask"], err_msg=msg)
            np.testing.assert_array_equal(_np(out.attr), want, err_msg=msg)
            for k in ("pos", "normal", "depth"):
                np.testing.assert_array_equal(_np(getattr(out, k)), ref[k], err_msg=f"{msg} {k}")
            assert ref["mask"].sum() > 0.3 * 6 * H * W


def _edge_coords(rng, B, H, W, TH, TW):
    """uv [B,H,W,2]: uniform in [-2, 3], and at the front of every view a grid of edge values on each axis --
    0, 1, -0.0, +-1e-9, texel edges k / n and centres (k + 1/2) / n (k in -1, 0, 1, n / 2, n - 1, n, n + 1),
    +-1e9 (beyond the int range once scaled by the texture size), +-inf and NaN."""
    def specials(n):
        ks = sorted({-1, 0, 1, n // 2, n - 1, n, n + 1})
        c = [0.0, 1.0, -0.0, -1e-9, 1e-9, 1.0 - 1e-7, 1e9, -1e9, np.inf, -np.inf, np.nan]
        c += [k / n for k in ks] + [(k + 0.5) / n for k in ks]
        return np.array(c, f32)
    su, sv = specials(TW), specials(TH)
    grid = np.stack(np.meshgrid(su, sv, indexing="ij"), -1).reshape(-1, 2)
    assert len(grid) <= H * W
    uv = rng.uniform(-2.0, 3.0, (B, H, W, 2)).astype(f32)
    flat = uv.reshape(B, -1, 2)
    for b in range(B):
        flat[b, :len(grid)] = grid[rng.permutation(len(grid))]
    return uv


@pytest.mark.parametrize("C", [1, 2, 4, 5, 8])
@pytest.mark.parametrize("per_view", [False, True], ids=["tex_B=1", "tex_B=B"])
def test_texture_operator_matches_oracle(wr_ctx, per_view, C):
    """ctx.texture (dr.texture, k_texture) against shim.texture in all six filter x boundary modes, bit for bit.  A
    non-finite coordinate takes no tap (0); under 'zero', |u| = 1e9 scales past the int range and takes none either."""
    rng = np.random.default_rng(10 * C + per_view)
    B, H, W, TH, TW = 3, 24, 40, 37, 53
    tex = rng.standard_normal((B if per_view else 1, TH, TW, C)).astype(f32)
    uv = _edge_coords(rng, B, H, W, TH, TW)
    dev = wr_ctx.device
    t, q = torch.from_numpy(tex).to(dev), torch.from_numpy(uv).to(dev)
    for filt in ("nearest", "linear"):
        for bnd in ("wrap", "clamp", "zero"):
            got = _np(wr_ctx.texture(t, q, filter_mode=filt, boundary_mode=bnd))
            want = shim.texture(tex, uv, filt, bnd)
            assert got.shape == (B, H, W, C)
            np.testing.assert_array_equal(got, want, err_msg=f"{filt}/{bnd}")
            assert np.isfinite(got).all() and (got != 0).mean() > (0.05 if bnd == "zero" else 0.5)
    # -1e-9 wraps to exactly 1.0: x = TW, which the nearest tap must wrap to texel 0
    one = np.zeros((B, 1, 1, 2), f32)
    one[..., 0] = -1e-9
    got = _np(wr_ctx.texture(t, torch.from_numpy(one).to(dev), filter_mode="nearest", boundary_mode="wrap"))
    np.testing.assert_array_equal(got[:, 0, 0], np.broadcast_to(tex[:, 0, 0], (B, C)))


def _score_map(rng, Hu, Wu):
    """0 (unpainted), 1 (painted) and partial scores, as the painter's score map holds after a few rounds."""
    r = rng.random((Hu, Wu))
    return np.where(r < 0.35, 0.0, np.where(r < 0.6, 1.0, rng.uniform(0.0, 1.0, (Hu, Wu)))).astype(f32)


def _painter_oracle(mesh, cam, size, score, depth):
    """attr (score texture, nearest, background 1) and the bake view map (pos, aoi_cos) of the oracle."""
    args = (_np(mesh.v_pos), _np(mesh.t_pos_idx).astype(np.int32), _np(mesh.v_nrm),
            _np(mesh.stitched_t_pos_idx).astype(np.int32), _np(cam.mvp_mtx), _np(cam.w2c), size, size)
    geo = render_oracle.uv_render_geometry(*args, {"uv_pos": np.zeros((1, 1, 3), f32)}, False)
    ref = render_oracle.render(args[0], args[1], args[4], args[5], size, size, v_nrm=args[2], tri_nrm=args[3],
                               depth=depth, v_tex=_np(mesh.v_tex), tri_tex=_np(mesh.t_tex_idx).astype(np.int32),
                               texture=score[..., None], texture_filter_mode="nearest", attr_background=1.0)
    np.testing.assert_array_equal(geo["view_mask"], ref["mask"])
    return ref, geo


@pytest.mark.parametrize("form", ["plain", "seams"])
def test_smart_painter_maps_and_view_scores(wr_ctx, form):
    """SmartPainter's two renders (smart_paint.py score_views and _best_view_inputs): no position or normal map, a
    one-channel nearest score texture and the bake view map, without and with controlnet depth.  attr, geo, mask and
    depth bit-exact against the oracle; then wr_view_scores on the 108 candidate maps: the counts exact, the sums
    within 2e-6 of their float64 value, and score_views returns the same scores."""
    dev = wr_ctx.device
    mesh = make_mesh(*cases.icosphere_mesh(8), dev, with_uv=True) if form == "plain" else stitched_mesh("seams", dev)
    score = _score_map(np.random.default_rng(5), 96, 96)
    tex = torch.from_numpy(score[..., None]).to(dev)
    cams = smart_paint.candidate_cameras(str(dev))
    B, S = cams.mvp_mtx.shape[0], smart_paint._SCORE_RES
    raw = render_geometry_raw(wr_ctx, mesh, cams, S, S, want_pos=False, want_depth=False, want_normal=False,
                              want_attr=True, want_geo=True, attr_background=1.0, texture_override=tex,
                              texture_filter_mode="nearest")
    assert set(raw) == {"mask", "attr", "geo"}
    ref, geo = _painter_oracle(mesh, cams, S, score, None)
    np.testing.assert_array_equal(_np(raw["mask"]), ref["mask"])
    np.testing.assert_array_equal(_np(raw["attr"]), ref["attr"])
    np.testing.assert_array_equal(_np(raw["geo"][..., :3]), geo["view_position"])
    np.testing.assert_array_equal(_np(raw["geo"][..., 3]), geo["view_aoi_cos"])

    count = torch.empty((B,), dtype=torch.int32, device=dev)
    fsum = torch.empty((B,), dtype=torch.float32, device=dev)
    c = wr_ctx.ctx
    c.check(_native.lib().wr_view_scores(c.handle, _native.ptr(raw["attr"]), 1, _native.ptr(raw["geo"]), B, S, S,
                                         smart_paint._ATTR_EPS, smart_paint._AOI_MIN, smart_paint._MARGIN,
                                         _native.ptr(count), _native.ptr(fsum), c.stream()), "wr_view_scores")
    s, aoi = ref["attr"][..., 0], geo["view_aoi_cos"]
    lo, amin, margin = f32(smart_paint._ATTR_EPS), f32(smart_paint._AOI_MIN), f32(smart_paint._MARGIN)
    want_count = ((s < lo) & (aoi > amin)).sum((1, 2))
    term = np.maximum((aoi - s) - margin, f32(0))
    want_sum = np.where((s > lo) & (aoi > amin), term, 0).astype(np.float64).sum((1, 2))
    assert want_count.min() > 0 and (want_sum > 0).mean() > 0.9
    np.testing.assert_array_equal(_np(count), want_count)
    np.testing.assert_allclose(_np(fsum), want_sum, rtol=2e-6)
    scores = smart_paint.score_views(wr_ctx, mesh, cams, torch.from_numpy(score).to(dev))
    np.testing.assert_array_equal(scores, (_np(count).astype(np.float64) + _np(fsum).astype(np.float64)) / (S * S))

    # the inpaint render of the best view: 1024^2, with render()'s default controlnet depth
    best = int(np.argmax(scores))
    cam = cams[best:best + 1]
    R = smart_paint._INPAINT_RES
    raw = render_geometry_raw(wr_ctx, mesh, cam, R, R, want_pos=False, want_depth=True, want_normal=False,
                              want_attr=True, want_geo=True, attr_background=1.0, texture_override=tex,
                              texture_filter_mode="nearest", depth_normalization_strategy=wr.DepthControlNetNormalization())
    ref, geo = _painter_oracle(mesh, cam, R, score, DepthSpec("controlnet"))
    assert ref["mask"].sum() > 0.1 * R * R
    np.testing.assert_array_equal(_np(raw["mask"]), ref["mask"])
    np.testing.assert_array_equal(_np(raw["attr"]), ref["attr"])
    np.testing.assert_array_equal(_np(raw["depth"]), ref["depth"])
    np.testing.assert_array_equal(_np(raw["geo"][..., :3]), geo["view_position"])
    np.testing.assert_array_equal(_np(raw["geo"][..., 3]), geo["view_aoi_cos"])
