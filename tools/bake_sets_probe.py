"""K image sets baked in one CameraProjection.project_sets call against K separate __call__s, on one GPU.

Two shapes: config C (50k-face icosphere, 6 x 768^2 views, 1024^2 atlas) and the single-GPU config-E shape (5M-face
terrain, 32 x 2048^2 views, 4096^2 atlas).  The texture pipeline's colour keywords (aoi_cos_valid_threshold -1,
no depth-gradient test, alpha 3, unit view weights, no Poisson blend), seam padding off and on, K = 1..4.  Each time is
the median and min-max of --reps device-event timings, with a 256 MB buffer overwritten before each run so that no
input stays in L2 from the run before.  Every project_sets result (atlas and mask) is compared with torch.equal to the
separate call on its set.

--compare-tree DIR times the one-set __call__ of another checkout (e.g. the parent commit, its library built) against
this tree's __call__ and project_sets([images]), alternating between the two trees in child processes.

    python tools/bake_sets_probe.py [--reps 9] [--out FILE.json] [--compare-tree DIR] [--rounds 3]
"""
from __future__ import annotations

import argparse
import contextlib
import io
import json
import os
import subprocess
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
COLOUR_KW = dict(aoi_cos_valid_threshold=-1.0, depth_grad_threshold=None, uv_exp_blend_alpha=3,
                 iou_rejection_threshold=None, poisson_blending=False, return_uv_projection_mask=True)


def scene(shape, dev, n_sets):
    """(mesh, cam, [image sets], uv size, description) of config C or the single-GPU config-E shape."""
    import torch

    import worldrenderer_b200 as wr
    from worldrenderer_b200 import synth
    if shape == "C":
        v, f = synth.icosphere(50, 0.5)
        vt, ft = synth.cell_atlas_uv(f.shape[0])
        NV, RES, UV = 6, 768, 1024
        mesh = wr.TexturedMesh(v_pos=torch.tensor(v, dtype=torch.float32), t_pos_idx=torch.tensor(f, dtype=torch.int64),
                               v_tex=torch.tensor(vt, dtype=torch.float32), t_tex_idx=torch.tensor(ft, dtype=torch.int64),
                               texture=torch.zeros((UV, UV, 3), dtype=torch.float32))
        mesh.set_stitched_mesh(mesh.v_pos, mesh.t_pos_idx)
        mesh.to(dev)
        cam = wr.get_orthogonal_camera(device=str(dev), **synth.CANONICAL_RIG)
        sets = [torch.from_numpy(synth.view_images(NV, RES, RES, seed=1 + k)).to(dev) for k in range(n_sets)]
    else:
        NX, NY, NV, RES, UV = 2500, 1000, 32, 2048, 4096
        v, f = synth.terrain(NX, NY, 0)
        v = v / np.abs(v).max() * 0.5
        v = np.ascontiguousarray(np.stack([v[:, 0], -v[:, 2], v[:, 1]], -1), np.float32)
        f = np.ascontiguousarray(f, np.int64)
        vt = synth.terrain_uv(NX, NY).astype(np.float32)
        mesh = wr.TexturedMesh(v_pos=torch.from_numpy(v).to(dev), t_pos_idx=torch.from_numpy(f).to(dev),
                               v_tex=torch.from_numpy(vt).to(dev), t_tex_idx=torch.from_numpy(f).to(dev),
                               texture=torch.zeros((UV, UV, 3), device=dev))
        mesh.set_stitched_mesh(mesh.v_pos, mesh.t_pos_idx)
        cam = wr.get_orthogonal_camera(elevation_deg=[20.0] * NV, distance=[1.0] * NV, left=-0.55, right=0.55,
                                       bottom=-0.55, top=0.55, azimuth_deg=list(np.linspace(0, 360, NV + 1)[:-1]),
                                       device=str(dev))
        y, x = torch.meshgrid(torch.arange(RES, device=dev, dtype=torch.float32),
                              torch.arange(RES, device=dev, dtype=torch.float32), indexing="ij")
        sets = []
        for k in range(n_sets):   # img[v, y, x, c] = .5 + .5 sin(w_c . (x, y) + phi_vc), one seed per set
            g = torch.Generator(device="cpu").manual_seed(1 + k)
            omega = torch.empty(3, 2).uniform_(0.01, 0.06, generator=g).to(dev)
            phi = torch.empty(NV, 3).uniform_(0.0, 6.2831853, generator=g).to(dev)
            arg = omega[None, :, 0, None, None] * x + omega[None, :, 1, None, None] * y + phi[:, :, None, None]
            sets.append((0.5 + 0.5 * torch.sin(arg)).permute(0, 2, 3, 1).contiguous())
    mesh.v_nrm
    desc = f"{f.shape[0]} faces, {NV} x {RES}^2 views, {UV}^2 atlas"
    return mesh, cam, sets, UV, desc


def timer(dev):
    import torch
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)

    def timed(fn, reps):
        for _ in range(2):
            fn()
        ms = []
        for k in range(reps):
            flush.fill_(k & 0xFF)
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            fn()
            b.record()
            torch.cuda.synchronize()
            ms.append(a.elapsed_time(b))
        return {"median_ms": float(np.median(ms)), "min_ms": float(min(ms)), "max_ms": float(max(ms)), "runs": reps}
    return timed


def worker(root, label, reps):
    """One-set timings of the package at `root` (printed as one JSON line)."""
    sys.path.insert(0, root)
    import torch

    import worldrenderer_b200 as wr
    dev = torch.device("cuda:0")
    timed = timer(dev)
    res = {"tree": label}
    with contextlib.redirect_stdout(io.StringIO()):
        for shape in ("C", "E"):
            mesh, cam, sets, uv, _ = scene(shape, dev, 1)
            proj = wr.CameraProjection(None, None, str(dev), "cuda")
            for pad in (False, True):
                kw = dict(COLOUR_KW, uv_size=uv, uv_padding=pad,
                          uv_exp_blend_view_weight=torch.ones(cam.mvp_mtx.shape[0]))
                res[f"{shape} pad={pad} __call__"] = timed(lambda: proj(sets[0], mesh, cam, **kw), reps)
                if hasattr(proj, "project_sets"):
                    res[f"{shape} pad={pad} project_sets K=1"] = timed(
                        lambda: proj.project_sets(sets[:1], mesh, cam, **kw), reps)
            del mesh, cam, sets, proj
            torch.cuda.empty_cache()
    print("WORKER " + json.dumps(res), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=9)
    ap.add_argument("--out", default=None, help="write the results as JSON here")
    ap.add_argument("--compare-tree", default=None)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--worker", nargs=2, default=None, help=argparse.SUPPRESS)
    args = ap.parse_args()
    if args.worker:
        worker(args.worker[0], args.worker[1], args.reps)
        return
    sys.path.insert(0, ROOT)
    import torch

    import worldrenderer_b200 as wr
    dev = torch.device("cuda:0")
    smi = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip()
    result = {"device": torch.cuda.get_device_name(dev), "nvidia_smi_name_power_limit_max_sm_clock": smi,
              "keywords": {k: v for k, v in COLOUR_KW.items()}, "shapes": {}}
    print(f"device: {result['device']} | nvidia-smi name, power limit, max SM clock: {smi}")
    timed = timer(dev)
    for shape in ("C", "E"):
        mesh, cam, sets, uv, desc = scene(shape, dev, 4)
        proj = wr.CameraProjection(None, None, str(dev), "cuda")
        rows = []
        for pad in (False, True):
            kw = dict(COLOUR_KW, uv_size=uv, uv_padding=pad, uv_exp_blend_view_weight=torch.ones(cam.mvp_mtx.shape[0]))
            with contextlib.redirect_stdout(io.StringIO()):
                got = proj.project_sets(sets, mesh, cam, **kw)
                want = [proj(s, mesh, cam, **kw) for s in sets]
            equal = all(torch.equal(g[0], w[0]) and torch.equal(g[1], w[1]) for g, w in zip(got, want))
            del got, want
            for K in range(1, 5):
                with contextlib.redirect_stdout(io.StringIO()):
                    sep = timed(lambda: [proj(s, mesh, cam, **kw) for s in sets[:K]], args.reps)
                    one = timed(lambda: proj.project_sets(sets[:K], mesh, cam, **kw), args.reps)
                rows.append({"uv_padding": pad, "K": K, "separate_calls": sep, "project_sets": one,
                             "ratio": one["median_ms"] / sep["median_ms"], "bit_equal_K4": equal})
                print(f"{shape} pad={pad!s:5} K={K}: {K} calls {sep['median_ms']:8.3f} ms "
                      f"[{sep['min_ms']:.3f}-{sep['max_ms']:.3f}]  project_sets {one['median_ms']:8.3f} ms "
                      f"[{one['min_ms']:.3f}-{one['max_ms']:.3f}]  ratio {rows[-1]['ratio']:.3f}  "
                      f"equal(K=4) {equal}", flush=True)
        result["shapes"][shape] = {"workload": desc, "rows": rows}
        del mesh, cam, sets, proj
        torch.cuda.empty_cache()
    if args.compare_tree:
        runs = []
        for r in range(args.rounds):
            for tree, label in ((os.path.abspath(args.compare_tree), "compare"), (ROOT, "this")):
                p = subprocess.run([sys.executable, os.path.abspath(__file__), "--worker", tree, label,
                                    "--reps", str(args.reps)], capture_output=True, text=True, cwd=tree)
                line = [x for x in p.stdout.splitlines() if x.startswith("WORKER ")]
                if p.returncode != 0 or not line:
                    raise RuntimeError(f"worker for {tree} failed:\n{p.stdout[-2000:]}\n{p.stderr[-4000:]}")
                runs.append(json.loads(line[0][7:]))
                print(f"round {r} {label}: " + ", ".join(f"{k} {v['median_ms']:.3f}" for k, v in runs[-1].items()
                                                       if isinstance(v, dict)), flush=True)
        result["one_set_trees_alternating"] = runs
    if args.out:
        with open(args.out, "w") as fh:
            json.dump(result, fh, indent=1)


if __name__ == "__main__":
    main()
