"""A context returns the same results whatever ran on it before.

Every entry point of a wr_ctx works in one grow-only scratch block that carries state from call to call (DESIGN.md
section 2): the packed visibility buffer at offset 0 is self-cleaning (k_resolve_rast and every k_shade instantiation
write WR_EMPTY_PIXEL back over the entries they read), `clean_bytes` lets the next raster call skip its clear when its
buffer fits in the prefix the last consumer left, the blend / view-score scratch sits behind that prefix, and the
vertex normal / tangent kernels and scratch growth reset it.  A slip in any of these shows only in a LATER call of
equal or smaller size, which skips the clear and finds stale entries.

The probe reads that prefix: a full-screen quad (ids 0 and 1) at z/w = 0.999, behind everything drawn here, padded
with degenerate off-screen faces to PROBE_F faces, at exactly the (B, H, W) of the call that consumed the buffer
before it.  It skips the clear, so a stale entry wins the depth test against the quad and shows up as an id other than
0 / 1 -- a valid id, PROBE_F being at least the face count of every mesh drawn here.  Every consuming call below is
followed by the probe, and a test stops at the first probe that finds a stale entry: a later call with fewer faces
never gets to read a stale id beyond its face buffer.  Empty meshes (F = 0, a NULL face buffer) are only rendered right
after a clean probe.

Every other output is compared, bit for bit, with the same call on a fresh context."""
import random

import numpy as np
import pytest
import torch

import cases
import worldrenderer_b200 as wr
from oracle import shim
from test_gpu_render_parity import make_mesh
from worldrenderer_b200 import _native, synth
from worldrenderer_b200.render import render_geometry_raw

pytestmark = pytest.mark.gpu

PROBE_F = 50_000        # >= the face count of every mesh of this file (checked where the meshes are built)
PROBE_Z = 0.999
INSTANTIATIONS = ("default", "simple", "bake", "generic")
DTYPES = (torch.float32, torch.float16, torch.bfloat16)
CONFIG_C = dict(uv_size=1024, poisson_blending=False, uv_padding=False, depth_grad_dilation=5, uv_exp_blend_alpha=3,
                aoi_cos_valid_threshold=0.2, depth_grad_threshold=0.1, iou_rejection_threshold=None, return_dict=True)


# ---- contexts, cameras, meshes -----------------------------------------------------------------------------------

def fresh(dev):
    return wr.NVDiffRastContextWrapper(str(dev), "cuda")


def identity_cameras(B, dev, stretch=0.0):
    """B views of a clip-space mesh: mvp = diag(1 + stretch b, 1, 1, 1), w2c = identity."""
    eye = torch.eye(4, device=dev).repeat(B, 1, 1)
    mvp = eye.clone()
    mvp[:, 0, 0] = 1.0 + stretch * torch.arange(B, device=dev, dtype=torch.float32)
    return wr.Camera(c2w=eye.clone(), w2c=eye.clone(), proj_mtx=mvp.clone(), mvp_mtx=mvp.contiguous(),
                     cam_pos=torch.zeros(B, 3, device=dev))


def perspective_rig(B, H, W, dev):
    return wr.get_camera(elevation_deg=np.linspace(-50.0, 60.0, B).tolist(), distance=[1.8] * B, fovy_deg=[40.0] * B,
                         azimuth_deg=((np.arange(B) * 137.5) % 360.0).tolist(), aspect_wh=W / H, device=dev)


def cameras_for(name, B, H, W, dev):
    return identity_cameras(B, dev, 1 / 64) if name == "huge" else perspective_rig(B, H, W, dev)


def raster_path(mesh, B, H, W):
    """(raster path, vertex-record form) wr_render takes (raster.cu use_mv, render.cu use_pack), as in
    test_gpu_stitched_mesh.py."""
    F, V, Vn = mesh.t_pos_idx.shape[0], mesh.v_pos.shape[0], mesh.v_nrm.shape[0]
    return ("multi-view" if 4 * F > H * W else "per-view",
            "packed" if B * H * W >= 32 * (V + Vn) else "unpacked")


@pytest.fixture(scope="module")
def meshes(cuda_device):
    """coarse: packed vertex records, per-view set-up; fine: the multi-view path (4 F > H W); huge: the tile pass
    (cases.huge_triangle_scene as a clip-space mesh); config_c: the bake mesh of bench.py; empty: F = V = 0."""
    out = {}
    v, f = cases.icosphere_mesh(8)
    out["coarse"] = make_mesh(v, f, cuda_device, with_uv=True)
    v, f = cases.icosphere_mesh(40)
    out["fine"] = make_mesh(v, f, cuda_device, with_uv=True)
    pos, tri = cases.huge_triangle_scene(B=1)
    out["huge"] = make_mesh(pos[0, :, :3], tri, cuda_device, with_uv=True)
    v, f = synth.icosphere(50, 0.5)
    out["config_c"] = make_mesh(v.astype(np.float32), f.astype(np.int32), cuda_device, with_uv=True, tex_size=1024)
    for m in out.values():
        assert m.t_pos_idx.shape[0] <= PROBE_F
        m.v_nrm, m.v_tang   # computed once, on the package's shared context
    empty = wr.TexturedMesh(v_pos=torch.zeros((0, 3)), t_pos_idx=torch.zeros((0, 3), dtype=torch.int64))
    empty.to(cuda_device)
    out["empty"] = empty
    return out


# ---- the probe ---------------------------------------------------------------------------------------------------

_PROBE = {}
_PROBE_WANT = {}


def _probe_geometry(dev):
    if dev not in _PROBE:
        z = PROBE_Z
        pos = torch.tensor([[-1, -1, z, 1], [1, -1, z, 1], [1, 1, z, 1], [-1, 1, z, 1], [3, 3, 0, 1]],
                           dtype=torch.float32)
        tri = torch.full((PROBE_F, 3), 4, dtype=torch.int32)   # padding: one off-screen point, culled
        tri[0] = torch.tensor([0, 1, 2])
        tri[1] = torch.tensor([0, 2, 3])
        mesh = wr.TexturedMesh(v_pos=pos[:, :3].clone(), t_pos_idx=tri.long())
        mesh.to(dev)
        _PROBE[dev] = (pos.to(dev), tri.to(dev), mesh)
    return _PROBE[dev]


def _run_probe(ctx, B, H, W):
    pos, tri, mesh = _probe_geometry(ctx.device)
    rast, ids = ctx.rasterize_with_ids(pos[None].expand(B, -1, -1), tri, (H, W))
    raw = render_geometry_raw(ctx, mesh, identity_cameras(B, ctx.device), H, W, want_pos=False, want_depth=False,
                              want_normal=False, want_tri_id=True)
    return rast, ids, raw["tri_id"]


def _stale_report(ids, what):
    bad = (ids != 0) & (ids != 1)
    if not bool(bad.any()):
        return None
    where = bad.nonzero()
    kind = "uncovered pixels (the probe no longer covers the viewport)" if bool((ids[bad] == -1).all()) \
        else "stale entries left by an earlier call"
    return (f"{what}: {int(bad.sum())} {kind}, in views "
            f"{sorted(set(where[:, 0].tolist()))[:8]}, columns {sorted(set(where[:, 2].tolist()))[:8]}, "
            f"rows {sorted(set(where[:, 1].tolist()))[:8]}; ids found {ids[bad].unique()[:8].tolist()}")


def probe(ctx, B, H, W):
    """Rasterises the probe at (B, H, W) through wr_rasterize (k_resolve_rast) and wr_render (generic k_shade), both
    skipping the clear when the context believes that prefix clean.  Every id must be 0 or 1, and the result that of
    the same probe on a fresh context."""
    held = ctx.ctx.scratch_bytes()
    rast, ids, tri_id = _run_probe(ctx, B, H, W)
    for name, t in (("rasterize_with_ids", ids), ("render", tri_id)):
        msg = _stale_report(t, f"probe {name} at B={B} H={H} W={W}")
        assert msg is None, msg
    # a probe that grew the scratch cleared the buffer and checked nothing: warm() reserves enough up front
    assert ctx.ctx.scratch_bytes() == held, "the probe grew the scratch: warm the context for this shape first"
    key = (str(ctx.device), B, H, W)
    if key not in _PROBE_WANT:
        if len(_PROBE_WANT) > 8:
            _PROBE_WANT.clear()
        _PROBE_WANT[key] = _run_probe(fresh(ctx.device), B, H, W)
    want = _PROBE_WANT[key]
    assert same(rast, want[0]) and same(ids, want[1]) and same(tri_id, want[2]), \
        f"probe at B={B} H={H} W={W} differs from the same probe on a fresh context"


def warm(ctx, shapes):
    """Grows the scratch once for the probes at `shapes` ((B, H, W) tuples), so that no later probe grows it."""
    B = max(s[0] for s in shapes)
    pix = max(s[0] * s[1] * s[2] for s in shapes)
    H = min(8192, max(s[1] for s in shapes))
    W = min(8192, -(-pix // (B * H)) + 1)
    _run_probe(ctx, B, H, W)
    _run_probe(ctx, B, H, W)


# ---- comparisons -------------------------------------------------------------------------------------------------

def same(a, b):
    """Bit-equal tensors; NaNs (tangents of vertices without a face) compared by position."""
    if a is None or b is None:
        return a is None and b is None
    if a.dtype != b.dtype or a.shape != b.shape:
        return False
    if a.is_floating_point():
        na, nb = torch.isnan(a), torch.isnan(b)
        if not torch.equal(na, nb):
            return False
        return torch.equal(a[~na], b[~nb])
    return torch.equal(a, b)


def assert_same(got, want, what):
    assert set(got) == set(want), (what, sorted(got), sorted(want))
    for k in want:
        assert same(got[k], want[k]), f"{what}: {k} differs from the same call on a fresh context"


# ---- calls -------------------------------------------------------------------------------------------------------

def render_case(ctx, mesh, cam, H, W, inst, dtype):
    """One shading instantiation: the default controlnet set, SimpleNormalization, the bake view set (want_geo, as
    CameraProjection issues it) or the generic one (attr, triangle ids, rast, tangent)."""
    if inst == "default":
        o = wr.render(ctx, mesh, cam, H, W, render_attr=False, output_dtype=dtype)
        return {k: getattr(o, k) for k in ("mask", "pos", "depth", "normal")}
    if inst == "simple":
        o = wr.render(ctx, mesh, cam, H, W, render_attr=False, depth_normalization_strategy=wr.SimpleNormalization(),
                      normal_background=0.5, output_dtype=dtype)
        return {k: getattr(o, k) for k in ("mask", "pos", "depth", "normal")}
    if inst == "bake":
        return render_geometry_raw(ctx, mesh, cam, H, W, want_pos=False, want_depth=True, want_normal=False,
                                   want_geo=True, output_dtype=dtype,
                                   depth_normalization_strategy=wr.SimpleNormalization(1.0, 0.0, False, 1e2))
    return render_geometry_raw(ctx, mesh, cam, H, W, want_attr=True, want_tri_id=True, want_rast=True, want_tangent=True,
                               tangent_background=0.25, output_dtype=dtype,
                               depth_normalization_strategy=wr.DepthControlNetNormalization())


def soup(seed, B, n_tri, dev):
    pos, tri = cases.random_soup(seed, n_tri, B=B)
    return torch.from_numpy(pos).to(dev), torch.from_numpy(tri).to(dev)


def raster_null_outputs(ctx, pos, tri, H, W):
    """wr_rasterize with neither rast nor tri_id: nothing consumes the buffer, the next call must clear it."""
    c = ctx.ctx
    c.check(_native.lib().wr_rasterize(c.handle, pos.data_ptr(), pos.shape[0], pos.shape[1], 1, tri.data_ptr(),
                                       tri.shape[0], None, H, W, None, None, c.stream()), "wr_rasterize")


def _images(shape, seed, dev):
    g = torch.Generator().manual_seed(seed)
    return torch.rand(shape, generator=g).to(dev)


def _region(H, W, seed, dev, density=0.5):
    g = torch.Generator().manual_seed(seed + 1)
    m = torch.rand((H, W), generator=g) < density
    m[: H // 3, : W // 2] = True
    return m.to(dev)


def scratch_user(c, kind, size, seed):
    """One call of a scratch user on NativeContext `c` with inputs drawn from `seed`.  size = (H, W) or, for the view
    scores, (B, H, W).  Returns {name: output}."""
    dev = c.device
    L = _native.lib()
    if kind == "view_scores":
        B, H, W = size
        attr = _images((B, H, W, 3), seed, dev)
        attr[..., 0] = torch.where(attr[..., 0] < 0.2, torch.zeros_like(attr[..., 0]), attr[..., 0])
        geo = _images((B, H, W, 4), seed + 7, dev)
        count = torch.empty(B, dtype=torch.int32, device=dev)
        fsum = torch.empty(B, dtype=torch.float32, device=dev)
        c.check(L.wr_view_scores(c.handle, attr.data_ptr(), 3, geo.data_ptr(), B, H, W, 1e-3, 0.1, 0.3,
                                 count.data_ptr(), fsum.data_ptr(), c.stream()), "wr_view_scores")
        return {"count": count, "fsum": fsum, "_attr": attr, "_geo": geo}
    H, W = size
    if kind == "poisson":
        src, tgt = _images((H, W, 3), seed, dev), _images((H, W, 3), seed + 3, dev)
        mask = _region(H, W, seed, dev)
        out = torch.empty_like(tgt)
        c.check(L.wr_poisson_blend(c.handle, src.data_ptr(), mask.view(torch.uint8).data_ptr(), tgt.data_ptr(), H, W,
                                   3, 24, 0, out.data_ptr(), c.stream()), "wr_poisson_blend")
        return {"out": out, "_src": src, "_tgt": tgt, "_mask": mask}
    if kind == "uv_padding":
        attr, inside = _images((H, W, 3), seed, dev) * 1.2 - 0.1, _region(H, W, seed, dev)
        out = torch.empty_like(attr)
        c.check(L.wr_uv_padding(c.handle, attr.data_ptr(), inside.view(torch.uint8).data_ptr(), H, W, 3, 3,
                                out.data_ptr(), c.stream()), "wr_uv_padding")
        return {"out": out, "_attr": attr, "_mask": inside}
    if kind == "uv_padding_sets":
        attrs = [_images((H, W, 3), seed + k, dev) for k in range(3)]
        inside = _region(H, W, seed, dev)
        outs = [torch.empty_like(a) for a in attrs]
        c.check(L.wr_uv_padding_sets(c.handle, _native.ptr_array(attrs), inside.view(torch.uint8).data_ptr(), H, W, 3,
                                     3, _native.ptr_array(outs), c.stream()), "wr_uv_padding_sets")
        return {**{f"out{k}": o for k, o in enumerate(outs)}, **{f"_attr{k}": a for k, a in enumerate(attrs)},
                "_mask": inside}
    if kind == "inpaint":
        img = (_images((H, W, 4), seed, dev) * 255).to(torch.uint8)
        mask = ~_region(H, W, seed, dev)
        out = torch.empty_like(img)
        c.check(L.wr_inpaint_u8(c.handle, img.data_ptr(), mask.view(torch.uint8).data_ptr(), H, W, 4, 5,
                                out.data_ptr(), c.stream()), "wr_inpaint_u8")
        return {"out": out, "_img": img, "_mask": mask}
    raise ValueError(kind)


USERS = ("view_scores", "poisson", "uv_padding", "uv_padding_sets", "inpaint")


def user_bytes(kind, size):
    """Scratch bytes a user asks for behind the clean prefix (csrc/blend.cu blend_scratch, csrc/score.cu)."""
    a = lambda x: (x + 255) // 256 * 256
    if kind == "view_scores":
        return 2 * a(size[0] * 64 * 4)
    H, W = size
    if kind == "poisson":
        Hp, Wp = -(-H // 48) * 48 + 16, -(-W // 112) * 112 + 16
        return 3 * a(Hp * Wp * 4 * 3) + a(Hp * Wp)
    return 2 * a(H * W * 4)


def check_user_oracle(kind, out):
    """The oracle where one exists (oracle/shim.py); the view scores against a float64 sum."""
    n = lambda t: t.cpu().numpy()
    if kind == "poisson":
        np.testing.assert_array_equal(n(out["out"]), shim.poisson_blend(n(out["_src"]), n(out["_mask"]), n(out["_tgt"]), 24))
    elif kind == "uv_padding":
        np.testing.assert_array_equal(n(out["out"]), shim.uv_padding(n(out["_attr"]), n(out["_mask"]), 3))
    elif kind == "uv_padding_sets":
        for k in range(3):
            np.testing.assert_array_equal(n(out[f"out{k}"]), shim.uv_padding(n(out[f"_attr{k}"]), n(out["_mask"]), 3))
    elif kind == "inpaint":
        np.testing.assert_array_equal(n(out["out"]), shim.inpaint_u8(n(out["_img"]), n(out["_mask"]), 5))
    elif kind == "view_scores":
        a, aoi = out["_attr"][..., 0].double(), out["_geo"][..., 3].double()
        lo, aoi_min, margin = (float(np.float32(x)) for x in (1e-3, 0.1, 0.3))   # the kernel's float arguments
        ok = aoi > aoi_min
        cnt = ((a < lo) & ok).flatten(1).sum(1)
        fs = torch.where((a > lo) & ok, (aoi - a - margin).clamp(min=0), torch.zeros_like(a)).flatten(1).sum(1)
        assert torch.equal(out["count"].long(), cnt)
        torch.testing.assert_close(out["fsum"].double(), fs, rtol=1e-5, atol=1e-3)


def outputs(d):
    return {k: v for k, v in d.items() if not k.startswith("_")}


def split_mesh(mesh):
    """Every face with its own three vertices: each vertex sums one face, so the tangents do not depend on the order
    of the float atomics and compare bit for bit."""
    f = mesh.t_pos_idx.long()
    v = mesh.v_pos[f.reshape(-1)].contiguous()
    corners = torch.arange(v.shape[0], device=v.device, dtype=torch.int32).reshape(-1, 3)
    vt, ft = synth.cell_atlas_uv(f.shape[0])
    return v, corners, torch.from_numpy(vt.astype(np.float32)).to(v.device), \
        torch.from_numpy(ft.astype(np.int32)).to(v.device)


def normals_and_tangents(c, v, tri, vt, ft):
    """wr_vertex_normals then wr_vertex_tangents on NativeContext `c`, as examples/c_abi_render.cpp calls them."""
    L = _native.lib()
    V, F = v.shape[0], tri.shape[0]
    nrm = torch.empty_like(v)
    c.check(L.wr_vertex_normals(c.handle, v.data_ptr(), V, tri.data_ptr(), F, nrm.data_ptr(), c.stream()),
            "wr_vertex_normals")
    tang = torch.empty_like(v)
    c.check(L.wr_vertex_tangents(c.handle, v.data_ptr(), V, tri.data_ptr(), vt.data_ptr(), vt.shape[0], ft.data_ptr(),
                                 F, nrm.data_ptr(), tang.data_ptr(), c.stream()), "wr_vertex_tangents")
    return {"normal": nrm, "tangent": tang}


# ---- 2. every consumer, then the probe ---------------------------------------------------------------------------

def test_raster_operators_leave_the_buffer_clean(cuda_device):
    """rasterize_with_ids, rasterize, wr_rasterize without outputs and range mode (with an empty view), at viewports
    that are not multiples of the kernels' block shapes."""
    dev = cuda_device
    ctx = fresh(dev)
    shapes = [(3, 97, 131), (5, 61, 250), (1, 7, 9), (4, 96, 96)]
    warm(ctx, shapes)
    for B, H, W in shapes:
        pos, tri = soup(B * H + W, B, 600, dev)
        for want_ids in (True, False):
            got = ctx.rasterize_with_ids(pos, tri, (H, W), want_ids=want_ids)
            want = fresh(dev).rasterize_with_ids(pos, tri, (H, W), want_ids=want_ids)
            assert bool((got[0][..., 3] > 0).any())
            assert same(got[0], want[0]) and same(got[1], want[1]), (B, H, W, want_ids)
            probe(ctx, B, H, W)
            probe(ctx, B, max(1, H // 2), max(1, W - 5))
        raster_null_outputs(ctx, pos, tri, H, W)
        probe(ctx, B, H, W)
    # range mode: one [V,4] vertex table, one face range per view, the last one empty
    pos, tri = soup(21, 1, 600, dev)
    ranges = torch.tensor([[0, 250], [250, 300], [100, 100], [0, 0]], dtype=torch.int32)
    for H, W in ((96, 96), (101, 130)):
        got = ctx.rasterize_with_ids(pos[0], tri, (H, W), ranges=ranges)
        want = fresh(dev).rasterize_with_ids(pos[0], tri, (H, W), ranges=ranges)
        assert same(got[0], want[0]) and same(got[1], want[1])
        assert bool((got[1][2] >= 100).any()) and bool((got[1][3] == -1).all())
        probe(ctx, 4, H, W)
        probe(ctx, 2, H - 3, W)


# (mesh, B, H, W, expected raster path): W % 128 != 0 and H % 4 != 0 (kShadeThreads, kShadeRows) everywhere
RENDER_CASES = [
    ("coarse", 6, 101, 130, ("per-view", "packed")),
    ("fine", 6, 131, 250, ("multi-view", "unpacked")),
    ("huge", 2, 333, 517, ("per-view", "unpacked")),   # and the tile pass (cases.huge_triangle_scene)
]


@pytest.mark.parametrize("name,B,H,W,path", RENDER_CASES, ids=[c[0] for c in RENDER_CASES])
def test_render_leaves_the_buffer_clean(meshes, cuda_device, name, B, H, W, path):
    """Each shading instantiation in float32, float16 and bfloat16, then the probe at the same and a smaller shape;
    last an empty mesh, right after a clean probe."""
    dev = cuda_device
    mesh = meshes[name]
    cam = cameras_for(name, B, H, W, dev)
    assert raster_path(mesh, B, H, W) == path
    ctx = fresh(dev)
    warm(ctx, [(B, H, W)])
    small = (B, H // 2 + 1, W // 3 + 1)
    for inst in INSTANTIATIONS:
        for dtype in DTYPES:
            got = render_case(ctx, mesh, cam, H, W, inst, dtype)
            want = render_case(fresh(dev), mesh, cam, H, W, inst, dtype)
            assert bool(got["mask"].any())
            assert_same(got, want, f"{name} {inst} {dtype}")
            probe(ctx, B, H, W)
            probe(ctx, *small)
    probe(ctx, B, H, W)
    got = render_geometry_raw(ctx, meshes["empty"], cam, H, W, want_normal=False, want_tri_id=True, want_rast=True,
                              depth_normalization_strategy=None)
    assert not bool(got["mask"].any()) and bool((got["tri_id"] == -1).all())
    probe(ctx, B, H, W)


# ---- 3. scratch users behind the prefix, and the ones that reset it -----------------------------------------------

def test_scratch_users_and_resets(meshes, cuda_device):
    """After a render has left a clean prefix: each scratch user once at a size that fits behind the prefix and once at
    a size that grows the scratch, bit-equal to a fresh context and to the oracle; the probe after each must be
    clean.  Then the vertex normals and tangents on the same context, and a render after them."""
    dev = cuda_device
    S = (4, 61, 90)
    mesh = meshes["coarse"]
    cam = cameras_for("coarse", S[0], S[1], S[2], dev)
    ctx = fresh(dev)
    c = ctx.ctx
    warm(ctx, [S])
    base = render_case(fresh(dev), mesh, cam, S[1], S[2], "default", torch.float32)
    prefix = S[0] * S[1] * S[2] * 8
    for seed, kind in enumerate(USERS):
        for grow in (False, True):
            assert_same(render_case(ctx, mesh, cam, S[1], S[2], "default", torch.float32), base, "render")
            held = c.scratch_bytes()
            if kind == "view_scores":
                size = (max(2, (held // 512) + 64), 1, 3) if grow else (5, 33, 47)
                assert size[0] <= 65535
            else:
                size = (40, 56)
                while grow and user_bytes(kind, size) + prefix <= held:
                    size = (size[0] * 2, size[1] * 2)
            assert (user_bytes(kind, size) + prefix + 256 > held) == grow, (kind, size, held)
            got = scratch_user(c, kind, size, seed)
            assert (c.scratch_bytes() > held) == grow, (kind, size, held, c.scratch_bytes())
            want = scratch_user(_native.NativeContext(dev), kind, size, seed)
            assert_same(outputs(got), outputs(want), f"{kind} {size}")
            check_user_oracle(kind, got)
            probe(ctx, *S)
    # mesh-level kernels on the render context overwrite the head of the scratch
    assert_same(render_case(ctx, mesh, cam, S[1], S[2], "default", torch.float32), base, "render")
    args = split_mesh(mesh)
    got = normals_and_tangents(c, *args)
    want = normals_and_tangents(_native.NativeContext(dev), *args)
    assert_same(got, want, "normals / tangents")
    v, f = cases.icosphere_mesh(8)
    v_d, f_d = torch.from_numpy(v).to(dev), torch.from_numpy(f).to(dev)
    nrm = torch.empty_like(v_d)
    c.check(_native.lib().wr_vertex_normals(c.handle, v_d.data_ptr(), v_d.shape[0], f_d.data_ptr(), f_d.shape[0],
                                            nrm.data_ptr(), c.stream()), "wr_vertex_normals")
    np.testing.assert_allclose(nrm.cpu().numpy(), cases.exact_vertex_normals(v, f), rtol=0, atol=1.2e-7)
    probe(ctx, *S)
    assert_same(render_case(ctx, mesh, cam, S[1], S[2], "default", torch.float32), base, "render after the normals")
    probe(ctx, *S)


# ---- 4. seeded sequences -----------------------------------------------------------------------------------------

MAX_PIX = 1 << 22


def _shape(rng):
    H = int(round(np.exp(rng.uniform(np.log(7), np.log(2048)))))
    W = int(round(np.exp(rng.uniform(np.log(7), np.log(2048)))))
    B = rng.randint(1, 40)
    while B > 1 and B * H * W > MAX_PIX:
        B = max(1, B // 2)
    return B, H, W


def draw_calls(seed, n=30):
    """About n calls of every kind: raster operators, renders (instantiation x dtype x mesh), scratch users, normals
    and tangents, one 4096^2 uv_precompute and one config C bake, in a seeded order."""
    rng = random.Random(seed)
    calls = []
    for i in range(n - 2):
        kind = rng.choice(["ids", "rast", "null", "ranges", "render", "render", "render", "render", "user", "mesh"])
        B, H, W = _shape(rng)
        call = dict(kind=kind, B=B, H=H, W=W, seed=seed * 1000 + i)
        if kind == "render":
            call.update(mesh=rng.choice(["coarse", "fine", "huge"]), inst=rng.choice(INSTANTIATIONS),
                        dtype=rng.choice(DTYPES))
        elif kind == "user":
            call.update(user=rng.choice(USERS), H=min(H, 1024), W=min(W, 1024))
        calls.append(call)
    calls.insert(rng.randint(0, len(calls)), dict(kind="uv_precompute", B=1, H=4096, W=4096))
    calls.insert(rng.randint(0, len(calls)), dict(kind="bake", B=6, H=768, W=768))
    return calls


def run_call(ctx, call, meshes, dev):
    """Runs one call on `ctx`; returns (outputs, (B, H, W) of the buffer it consumed last, or None)."""
    kind, B, H, W = call["kind"], call["B"], call["H"], call["W"]
    shape = (B, H, W)
    if kind in ("ids", "rast"):
        pos, tri = soup(call["seed"], B, 600, dev)
        rast, ids = ctx.rasterize_with_ids(pos, tri, (H, W), want_ids=kind == "ids")
        return {"rast": rast, "ids": ids}, shape
    if kind == "null":
        pos, tri = soup(call["seed"], B, 600, dev)
        raster_null_outputs(ctx, pos, tri, H, W)
        return {}, shape
    if kind == "ranges":
        pos, tri = soup(call["seed"], 1, 600, dev)
        starts = torch.randint(0, 600, (B,), generator=torch.Generator().manual_seed(call["seed"]))
        ranges = torch.stack([starts, (600 - starts) // 2], 1).to(torch.int32)
        ranges[-1] = torch.tensor([0, 0])
        rast, ids = ctx.rasterize_with_ids(pos[0], tri, (H, W), ranges=ranges)
        return {"rast": rast, "ids": ids}, shape
    if kind == "render":
        cam = cameras_for(call["mesh"], B, H, W, dev)
        return render_case(ctx, meshes[call["mesh"]], cam, H, W, call["inst"], call["dtype"]), shape
    if kind == "user":
        size = (B, H, W) if call["user"] == "view_scores" else (H, W)
        return outputs(scratch_user(ctx.ctx, call["user"], size, call["seed"])), None
    if kind == "mesh":
        return normals_and_tangents(ctx.ctx, *split_mesh(meshes["coarse"])), None
    if kind == "uv_precompute":
        pre = wr.uv_precompute(ctx, meshes["config_c"], H, W)
        return {"uv_mask": pre.uv_mask, "uv_pos": pre.uv_pos}, shape
    if kind == "bake":
        mesh = meshes["config_c"]
        cam = cases.canonical_cameras(device=dev)
        images = torch.from_numpy(synth.view_images(B, H, W, seed=1)).to(dev)
        proj = wr.CameraProjection(None, None, str(dev), "cuda")
        proj.ctx = ctx
        out = proj(images, mesh, cam, uv_exp_blend_view_weight=torch.ones(B), **CONFIG_C)
        return {k: getattr(out, k) for k in ("uv_proj", "uv_proj_mask", "uv_depth_grad", "uv_aoi_cos")}, shape
    raise ValueError(kind)


def run_sequence(ctx, calls, meshes, dev, seed):
    """Every call against a fresh context, then the probe at the shape the call consumed, or at the last consumed
    shape after a call that only uses the scratch behind the prefix.  Stops at the first difference."""
    shapes = [(c["B"], c["H"], c["W"]) for c in calls if c["kind"] not in ("user", "mesh")]
    warm(ctx, shapes)
    results = []
    last = None
    for i, call in enumerate(calls):
        try:
            got, consumed = run_call(ctx, call, meshes, dev)
            want, _ = run_call(fresh(dev), call, meshes, dev)
            assert_same(got, want, call["kind"])
            last = consumed or last
            if last is not None:
                probe(ctx, *last)
        except AssertionError as e:
            listing = "\n".join(f"  {j:2d} {c}" for j, c in enumerate(calls[: i + 1]))
            raise AssertionError(f"seed {seed}, call {i} ({call}): {e}\ncalls so far:\n{listing}") from e
        results.append(got)
    return results


@pytest.mark.parametrize("seed", [0, 1, 2])
def test_seeded_sequence(meshes, cuda_device, seed):
    calls = draw_calls(seed)
    run_sequence(fresh(cuda_device), calls, meshes, cuda_device, seed)


# ---- 5. error paths and profiling mode ---------------------------------------------------------------------------

def test_range_error_after_earlier_views_leaves_the_context_usable(meshes, cuda_device):
    """A range-mode call whose third view has an out-of-range face range: views 0 and 1 are rasterised before the host
    check returns an error.  The call raises; the probe after it is clean and the next render equals a fresh one."""
    dev = cuda_device
    ctx = fresh(dev)
    B, H, W = 3, 97, 131
    warm(ctx, [(B, H, W), (6, 101, 130)])
    pos, tri = soup(5, 1, 600, dev)
    ranges = torch.tensor([[0, 300], [300, 300], [500, 200]], dtype=torch.int32)
    with pytest.raises(RuntimeError, match="wr_rasterize"):
        ctx.rasterize_with_ids(pos[0], tri, (H, W), ranges=ranges)
    probe(ctx, B, H, W)
    with pytest.raises(RuntimeError, match="wr_rasterize"):
        ctx.rasterize_with_ids(pos[0], tri, (H, W), ranges=ranges)
    mesh = meshes["coarse"]
    cam = cameras_for("coarse", 6, 101, 130, dev)
    got = render_case(ctx, mesh, cam, 101, 130, "generic", torch.float32)
    assert_same(got, render_case(fresh(dev), mesh, cam, 101, 130, "generic", torch.float32), "render after the error")
    probe(ctx, 6, 101, 130)


def test_profiling_mode_matches_plain_launches(meshes, cuda_device):
    """ctx.profile(True) launches without programmatic dependent launch and records stage events: the same sequence
    returns the same bits."""
    dev = cuda_device
    calls = [c for c in draw_calls(3, n=14) if c["kind"] != "bake"]
    plain = run_sequence(fresh(dev), calls, meshes, dev, seed=3)
    ctx = fresh(dev)
    ctx.ctx.profile(True)
    profiled = run_sequence(ctx, calls, meshes, dev, seed=3)
    assert ctx.ctx.profile_read()   # the stages of the last call were recorded
    for call, a, b in zip(calls, profiled, plain):
        assert_same(a, b, f"profiled {call}")
