"""Coarse meshes (few large triangles): set-up / queue-pass times of render() and uv_precompute at large atlases."""
import os, sys
import numpy as np, torch
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__))); sys.path.insert(0, ROOT)
import worldrenderer_b200 as wr
from worldrenderer_b200 import synth
dev = torch.device("cuda", 0)
cam = wr.get_orthogonal_camera(device="cuda:0", **synth.CANONICAL_RIG)
ctx = wr.NVDiffRastContextWrapper("cuda:0", "cuda")
def mk(v, f, uv=False):
    m = wr.TexturedMesh(v_pos=torch.tensor(v, dtype=torch.float32, device=dev), t_pos_idx=torch.tensor(f, device=dev))
    if uv:
        vt, ft = synth.cell_atlas_uv(f.shape[0])
        m.v_tex, m.t_tex_idx = torch.tensor(vt, dtype=torch.float32, device=dev), torch.tensor(ft, device=dev)
    m.set_stitched_mesh(m.v_pos, m.t_pos_idx); m.v_nrm; return m
def stages(fn, keys=("k_setup_triangles", "k_raster_queues")):
    ctx.ctx.profile(True); acc = {}
    for k in range(10):
        fn()
        for n, ms in ctx.ctx.profile_read(): acc.setdefault(n, []).append(ms * 1e3)
    ctx.ctx.profile(False)
    return {n: round(float(np.mean(x[2:])), 1) for n, x in acc.items() if n in keys}
def wall(fn, reps=10):
    for _ in range(3): fn()
    torch.cuda.synchronize()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(reps)]
    for a, b in ev:
        a.record(); fn(); b.record()
    torch.cuda.synchronize()
    return round(float(np.mean([a.elapsed_time(b) for a, b in ev])) * 1e3, 1)
box_v = np.array([[x, y, z] for x in (-.4, .4) for y in (-.4, .4) for z in (-.4, .4)], np.float32)
box_f = np.array([[0,1,3],[0,3,2],[4,6,7],[4,7,5],[0,4,5],[0,5,1],[2,3,7],[2,7,6],[0,2,6],[0,6,4],[1,5,7],[1,7,3]], np.int64)
box = mk(box_v, box_f)
for res in (768, 2048, 4096):
    print(f"box (12 faces) 6 views {res}^2:", stages(lambda: wr.render(ctx, box, cam, res, res, render_attr=False)),
          "render() total us", wall(lambda: wr.render(ctx, box, cam, res, res, render_attr=False)))
for freq in (1, 2, 4, 8, 16):
    m = mk(*synth.icosphere(freq, 0.5))
    print(f"icosphere f={freq:2d} faces={20*freq*freq:5d}", "6v 768:", stages(lambda: wr.render(ctx, m, cam, 768, 768, render_attr=False)),
          "6v 2048:", stages(lambda: wr.render(ctx, m, cam, 2048, 2048, render_attr=False)))
for freq, uvs in ((50, 1024), (50, 3072), (50, 4096), (16, 4096), (4, 4096)):
    m = mk(*synth.icosphere(freq, 0.5), uv=True)
    print(f"uv_precompute {20*freq*freq} faces -> {uvs}^2 atlas:", stages(lambda: wr.uv_precompute(ctx, m, uvs, uvs), ("k_setup_triangles", "k_raster_queues", "k_resolve_rast")),
          "total us", wall(lambda: wr.uv_precompute(ctx, m, uvs, uvs)))
