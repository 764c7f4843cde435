"""render(output_dtype=torch.float16 / torch.bfloat16): every float map equals the float32 render cast by torch, bit
for bit (NaN by position), on every kernel path -- packed and unpacked vertex records, the specialised and the generic
shading instantiations, the 16-byte background rows and the per-pixel stores, every depth normaliser (the two-pass ones
finalise from a float32 copy of the view depth), the torch post-processing of user strategies and tensor backgrounds,
RenderGraph replays -- and the refusals of other dtypes."""
import ctypes

import numpy as np
import pytest
import torch

import cases
import worldrenderer_b200 as wr
from worldrenderer_b200 import _native, synth
from worldrenderer_b200.render import render_geometry_raw

pytestmark = pytest.mark.gpu

HALF = [torch.float16, torch.bfloat16]
MAPS = ("pos", "depth", "normal", "tangent", "attr")


def _mesh(v, f, dev, channels=None, tex_size=32, seed=0):
    m = wr.TexturedMesh(v_pos=torch.tensor(v, dtype=torch.float32), t_pos_idx=torch.tensor(f, dtype=torch.int64))
    m.set_stitched_mesh(m.v_pos, m.t_pos_idx)
    if channels is not None:
        vt, ft = synth.cell_atlas_uv(f.shape[0])
        m.v_tex = torch.tensor(vt, dtype=torch.float32)
        m.t_tex_idx = torch.tensor(ft, dtype=torch.int64)
        rng = np.random.default_rng(seed)
        m.texture = torch.tensor(rng.uniform(0, 1, (tex_size, tex_size, channels)), dtype=torch.float32)
    m.to(dev)
    return m


def _assert_cast_equal(got, want, dt):
    """got: a map rendered in dt; want: the float32 map.  Same bits as want.to(dt); NaN only where want.to(dt) has it."""
    assert got.dtype == dt and got.is_contiguous() and got.shape == want.shape
    ref = want.to(dt)
    nan = torch.isnan(ref)
    assert torch.equal(torch.isnan(got), nan)
    assert torch.equal(got.view(torch.int16)[~nan], ref.view(torch.int16)[~nan])


def _assert_outputs(got, want, dt):
    assert got.mask.dtype == torch.bool and torch.equal(got.mask, want.mask)
    for name in MAPS:
        a, b = getattr(got, name), getattr(want, name)
        assert (a is None) == (b is None), name
        if b is not None:
            assert b.dtype == torch.float32
            _assert_cast_equal(a, b, dt)


def _check(ctx, mesh, cam, H, W, dt, **kw):
    want = wr.render(ctx, mesh, cam, H, W, **kw)
    got = wr.render(ctx, mesh, cam, H, W, output_dtype=dt, **kw)
    _assert_outputs(got, want, dt)
    return want


class Halve(wr.DepthNormalizationStrategy):
    def __init__(self):
        pass

    def __call__(self, depth, mask):
        return depth * 0.5 + 0.125


STRATEGIES = {
    "controlnet": wr.DepthControlNetNormalization(),
    "controlnet_custom": wr.DepthControlNetNormalization(far_clip=0.1, near_clip=0.9, bg_value=0.3),
    "zero123pp": wr.Zero123PlusPlusNormalization(),
    "simple_clamp": wr.SimpleNormalization(),
    "simple_raw": wr.SimpleNormalization(scale=1.0, offset=0.0, clamp=False, bg_value=1e2),
    "none": None,
    "user": Halve(),
}


@pytest.mark.parametrize("dt", HALF)
@pytest.mark.parametrize("strategy", list(STRATEGIES))
@pytest.mark.parametrize("shape", ["icosphere_packed", "terrain_unpacked"])
def test_every_depth_strategy_on_both_vertex_paths(wr_ctx, shape, strategy, dt):
    """Icosphere on the canonical rig: few vertices, many pixels -- 16-byte vertex records; terrain: the per-float
    gathers.  160 x 160: W % 8 == 0, the 16-bit background rows go out as 16-byte stores."""
    dev = wr_ctx.device
    mesh = _mesh(*cases.icosphere_mesh(8), dev) if shape == "icosphere_packed" else _mesh(*cases.terrain_mesh(96, 64), dev)
    cam = cases.canonical_cameras(device=dev)
    want = _check(wr_ctx, mesh, cam, 160, 160, dt, render_attr=False,
                  depth_normalization_strategy=STRATEGIES[strategy])
    assert 0 < int(want.mask.sum()) < want.mask.numel()


@pytest.mark.parametrize("dt", HALF)
@pytest.mark.parametrize("rig", ["perspective", "inside", "low_terrain"])
def test_perspective_and_near_plane_rigs(wr_ctx, rig, dt):
    dev = wr_ctx.device
    if rig == "low_terrain":
        mesh, cam = _mesh(*cases.terrain_mesh(64, 32), dev), cases.low_terrain_cameras(96, 128, device=dev)
    else:
        mesh = _mesh(*cases.icosphere_mesh(8), dev)
        cam = cases.perspective_cameras(4, device=dev) if rig == "perspective" else cases.inside_cameras(device=dev)
    for strategy in ("controlnet", "zero123pp", "simple_raw"):
        _check(wr_ctx, mesh, cam, 96, 128, dt, render_attr=False, depth_normalization_strategy=STRATEGIES[strategy])


@pytest.mark.parametrize("dt", HALF)
@pytest.mark.parametrize("H,W", [(30, 34), (33, 31), (7, 5), (64, 36), (1, 16), (50, 52), (64, 64)])
def test_viewport_shapes(wr_ctx, H, W, dt):
    """W % 4 != 0, H % 4 != 0, W % 8 == 4 (float32 takes the 16-byte background rows, 16-bit maps do not), H*W % 4 !=
    0 (the scalar form of the second depth pass)."""
    dev = wr_ctx.device
    mesh = _mesh(*cases.icosphere_mesh(6), dev)
    cam = cases.canonical_cameras(device=dev)
    for strategy in ("controlnet", "zero123pp", "none", "simple_clamp"):
        _check(wr_ctx, mesh, cam, H, W, dt, render_attr=False, depth_normalization_strategy=STRATEGIES[strategy])


@pytest.mark.parametrize("dt", HALF)
def test_one_view_and_40_views(wr_ctx, dt):
    dev = wr_ctx.device
    mesh = _mesh(*cases.icosphere_mesh(6), dev)
    _check(wr_ctx, mesh, cases.canonical_cameras(device=dev)[2:3], 64, 64, dt, render_attr=False)
    _check(wr_ctx, mesh, cases.mixed_40_view_cameras(48, 64, device=dev), 48, 64, dt, render_attr=False)


@pytest.mark.parametrize("dt", HALF)
def test_render_normal_off(wr_ctx, dt):
    dev = wr_ctx.device
    mesh = _mesh(*cases.icosphere_mesh(8), dev)
    cam = cases.canonical_cameras(device=dev)
    for strategy in ("controlnet", "simple_clamp"):
        want = _check(wr_ctx, mesh, cam, 96, 96, dt, render_attr=False, render_normal=False,
                      depth_normalization_strategy=STRATEGIES[strategy])
        assert want.normal is None


@pytest.mark.parametrize("dt", HALF)
@pytest.mark.parametrize("channels", [1, 3, 4])
@pytest.mark.parametrize("filt", ["linear", "nearest"])
def test_render_attr(wr_ctx, filt, channels, dt):
    dev = wr_ctx.device
    mesh = _mesh(*cases.icosphere_mesh(6), dev, channels=channels, seed=channels)
    cam = cases.canonical_cameras(device=dev)
    _check(wr_ctx, mesh, cam, 96, 100, dt, render_attr=True, texture_filter_mode=filt, attr_background=0.3)


@pytest.mark.parametrize("dt", HALF)
def test_render_tangent(wr_ctx, dt):
    dev = wr_ctx.device
    mesh = _mesh(*cases.icosphere_mesh(6), dev, channels=3)
    cam = cases.canonical_cameras(device=dev)
    _check(wr_ctx, mesh, cam, 96, 96, dt, render_attr=True, render_tangent=True, tangent_background=0.25)
    _check(wr_ctx, mesh, cam, 96, 96, dt, render_attr=False, render_tangent=True,
           tangent_background=torch.tensor([0.1, 0.2, 0.3], device=dev))


@pytest.mark.parametrize("dt", HALF)
def test_tensor_backgrounds_and_user_strategy_are_cast_once(wr_ctx, dt):
    """The maps torch post-processes are kept in float32 through the post-processing: per-pixel normal / tangent
    backgrounds, a per-channel attribute background, a user-defined depth strategy."""
    dev = wr_ctx.device
    mesh = _mesh(*cases.icosphere_mesh(6), dev, channels=3)
    cam = cases.canonical_cameras(device=dev)
    H, W = 64, 72
    n_bg = int((~wr.render(wr_ctx, mesh, cam, H, W, render_attr=False).mask).sum())
    g = torch.Generator(device="cpu").manual_seed(0)
    nbg = (torch.rand((n_bg, 3), generator=g) * 3.0 - 1.0).to(dev)
    tbg = (torch.rand((n_bg, 3), generator=g) * 1e-3).to(dev)
    abg = torch.tensor([0.1, 0.7, 1.0 / 3.0], device=dev)
    _check(wr_ctx, mesh, cam, H, W, dt, render_attr=True, render_tangent=True, normal_background=nbg,
           tangent_background=tbg, attr_background=abg, depth_normalization_strategy=Halve())
    _check(wr_ctx, mesh, cam, H, W, dt, render_attr=True, attr_background=abg)
    _check(wr_ctx, mesh, cam, H, W, dt, render_attr=False, normal_background=nbg)


@pytest.mark.parametrize("dt", HALF)
def test_bake_view_set_with_half_depth(wr_ctx, dt):
    """The bake's output set (geo map + simple depth) with a 16-bit depth map: geo stays float32 and unchanged."""
    dev = wr_ctx.device
    mesh = _mesh(*cases.icosphere_mesh(8), dev)
    cam = cases.canonical_cameras(device=dev)
    kw = dict(want_pos=False, want_depth=True, want_normal=False, want_geo=True,
              depth_normalization_strategy=wr.SimpleNormalization(scale=1.0, offset=0.0, clamp=False, bg_value=1e2))
    want = render_geometry_raw(wr_ctx, mesh, cam, 128, 128, **kw)
    got = render_geometry_raw(wr_ctx, mesh, cam, 128, 128, output_dtype=dt, **kw)
    assert got["geo"].dtype == torch.float32 and torch.equal(got["geo"].view(torch.int32), want["geo"].view(torch.int32))
    assert torch.equal(got["mask"], want["mask"])
    _assert_cast_equal(got["depth"], want["depth"], dt)


@pytest.mark.parametrize("dt", HALF)
def test_config_b_full_size(wr_ctx, dt):
    """1M-face terrain, canonical 6-view rig, 768^2, render()'s defaults without the texture."""
    v, f = synth.terrain(1000, 500, 0)
    v = v / np.abs(v).max() * 0.5
    v = np.stack([v[:, 0], -v[:, 2], v[:, 1]], -1).astype(np.float32)
    mesh = _mesh(v, f.astype(np.int32), wr_ctx.device)
    cam = cases.canonical_cameras(device=wr_ctx.device)
    want = _check(wr_ctx, mesh, cam, 768, 768, dt, render_attr=False)
    assert int(want.mask.sum()) > 700_000


@pytest.mark.parametrize("dt", HALF)
def test_render_graph_replays_equal_eager(wr_ctx, dt):
    dev = wr_ctx.device
    cam = cases.canonical_cameras(device=dev)
    meshes = [_mesh(*cases.terrain_mesh(96, 64, seed=1), dev), _mesh(*cases.icosphere_mesh(8), dev)]
    for kw in (dict(lanes=2), dict(view_lanes=2, stagger=True)):
        g = wr.RenderGraph(wr_ctx, [(m, cam) for m in meshes], 64, 64, render_attr=False, output_dtype=dt, **kw)
        for _ in range(2):
            outs = g.replay()
        torch.cuda.synchronize()
        for m, o in zip(meshes, outs):
            want = wr.render(wr_ctx, m, cam, 64, 64, render_attr=False, output_dtype=dt)
            assert torch.equal(o.mask, want.mask)
            for name in ("pos", "depth", "normal"):
                a, b = getattr(o, name), getattr(want, name)
                assert a.dtype == dt and torch.equal(a.view(torch.int16), b.view(torch.int16)), (kw, name)
    # a user strategy renders float32 and casts: the graph copies the result into its 16-bit outputs
    g = wr.RenderGraph(wr_ctx, [(meshes[0], cam)], 64, 64, view_lanes=2, render_attr=False, output_dtype=dt,
                       depth_normalization_strategy=Halve())
    o = g.replay()[0]
    torch.cuda.synchronize()
    _assert_outputs(o, wr.render(wr_ctx, meshes[0], cam, 64, 64, render_attr=False,
                                 depth_normalization_strategy=Halve()), dt)


def test_default_is_float32_and_other_dtypes_are_refused(wr_ctx):
    dev = wr_ctx.device
    mesh = _mesh(*cases.icosphere_mesh(4), dev)
    cam = cases.canonical_cameras(device=dev)
    out = wr.render(wr_ctx, mesh, cam, 32, 32, render_attr=False)
    assert all(getattr(out, n).dtype == torch.float32 for n in ("pos", "depth", "normal"))
    for bad in (torch.float64, torch.int32, torch.uint8, "float16"):
        with pytest.raises(ValueError):
            wr.render(wr_ctx, mesh, cam, 32, 32, render_attr=False, output_dtype=bad)


def test_c_abi_refuses_out_of_range_out_dtype(wr_ctx):
    dev = wr_ctx.device
    cam = cases.canonical_cameras(device=dev)
    mvp = cam.mvp_mtx[:1].contiguous()
    mask = torch.empty((1, 8, 8), dtype=torch.uint8, device=dev)
    depth = torch.empty((1, 8, 8), dtype=torch.float16, device=dev)
    c = wr_ctx.ctx

    def call(out_dtype):
        a = _native.RenderArgs()
        a.mvp, a.w2c, a.B, a.H, a.W = _native.ptr(mvp), _native.ptr(cam.w2c), 1, 8, 8
        a.depth_mode = _native.DEPTH_CONTROLNET
        a.out_mask, a.out_depth = _native.ptr(mask), _native.ptr(depth)
        a.out_dtype = out_dtype
        return _native.lib().wr_render(c.handle, ctypes.byref(a), c.stream())

    assert call(_native.DTYPE_F16) == 0   # an empty mesh: background only
    torch.cuda.synchronize()
    assert not bool(mask.any())
    for bad in (-1, 3, 1 << 20):
        assert call(bad) == -1   # WR_ERR_INVALID_ARGUMENT
