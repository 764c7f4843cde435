"""render(output_dtype=...) on config B: float32 against float16 and bfloat16 maps, alternating in one run, on one GPU.

Config B is bench.py's workload: 1M-face terrain, canonical 6-view orthographic rig, 768^2, mask + position + depth
(ControlNet) + normal.  For each output dtype, in --rounds rounds that alternate float32 / float16 / bfloat16:

- step: median (and min / max) of --steps RenderGraph replays, each between two CUDA events, with a 512 MiB device
  write before every step (outside the events) so that nothing of the step before stays in L2 -- as bench.py times it;
- stages: k_shade and k_depth_finalize of the eager call (wr_ctx_profile events), mean over --stage-reps calls;
- e2e: views/s of eager render() calls whose four maps are copied to pinned host buffers on a second stream, double
  buffered as in bench.py's e2e loop (the mesh stays on the device), wall clock over --e2e-steps steps; next to it the
  copies alone (the same maps device -> pinned host, nothing else running): the ceiling of that loop.

Before timing, the 16-bit maps are checked against the float32 maps cast by torch (bit-identical).  The card name, its
power limit and its maximum SM clock are read in the same run.

    python tools/render_dtype_probe.py [--steps 200] [--rounds 3] [--out FILE.json]
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import time

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
sys.path.insert(0, ROOT)

H = W = 768
N_VIEWS = 6
SHAPES = {"mask": (N_VIEWS, H, W), "pos": (N_VIEWS, H, W, 3), "depth": (N_VIEWS, H, W), "normal": (N_VIEWS, H, W, 3)}


def card():
    q = "name,power.limit,clocks.max.sm,driver_version"
    try:
        line = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader", "-i", "0"],
                              capture_output=True, text=True, timeout=60).stdout.strip()
        return dict(zip(q.split(","), [x.strip() for x in line.split(",")]))
    except Exception as exc:   # the timing does not depend on it; the record says it is missing
        return {"error": repr(exc)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--stage-reps", type=int, default=20)
    ap.add_argument("--e2e-steps", type=int, default=100)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()

    import torch

    import worldrenderer_b200 as wr
    from worldrenderer_b200 import synth
    if not torch.cuda.is_available():
        raise RuntimeError("render_dtype_probe needs a CUDA device")
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)

    v, f = synth.terrain(1000, 500, 0)
    v = v / np.abs(v).max() * 0.5
    v = np.stack([v[:, 0], -v[:, 2], v[:, 1]], -1).astype(np.float32)
    mesh = wr.TexturedMesh(v_pos=torch.from_numpy(v).to(dev), t_pos_idx=torch.from_numpy(f.astype(np.int64)).to(dev))
    mesh.set_stitched_mesh(mesh.v_pos, mesh.t_pos_idx)
    mesh.v_nrm
    cam = wr.get_orthogonal_camera(device=str(dev), **synth.CANONICAL_RIG)
    ctx = wr.NVDiffRastContextWrapper(str(dev), "cuda")
    kw = dict(render_attr=False, render_depth=True, render_normal=True)
    dtypes = {"float32": torch.float32, "float16": torch.float16, "bfloat16": torch.bfloat16}

    # ---- same numbers as the float32 render, cast -------------------------------------------------------------
    ref = wr.render(ctx, mesh, cam, H, W, **kw)
    exact = {}
    for name, dt in dtypes.items():
        got = wr.render(ctx, mesh, cam, H, W, output_dtype=dt, **kw)
        ok = torch.equal(got.mask, ref.mask)
        for m in ("pos", "depth", "normal"):
            a, b = getattr(got, m), getattr(ref, m).to(dt)
            bits = torch.int32 if dt == torch.float32 else torch.int16
            ok = ok and a.dtype == dt and torch.equal(a.view(bits), b.view(bits))
        exact[name] = bool(ok)
    bytes_per_step = {name: sum(int(np.prod(shape)) * (1 if m == "mask" else dt.itemsize) for m, shape in SHAPES.items())
                      for name, dt in dtypes.items()}
    del ref, got

    flush = torch.empty(512 << 20, dtype=torch.uint8, device=dev)
    graphs = {name: wr.RenderGraph(ctx, [(mesh, cam)], H, W, output_dtype=dt, **kw) for name, dt in dtypes.items()}

    def time_steps(g, n):
        ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(n)]
        for k in range(n):
            flush.fill_(k & 0xFF)
            ev[k][0].record()
            g.replay()
            ev[k][1].record()
        torch.cuda.synchronize()
        return [a.elapsed_time(b) for a, b in ev]

    def stages(dt):
        ctx.ctx.profile(True)
        acc = {}
        for k in range(args.stage_reps):
            flush.fill_(k & 0xFF)
            wr.render(ctx, mesh, cam, H, W, output_dtype=dt, **kw)
            for n, ms in ctx.ctx.profile_read():
                acc.setdefault(n, []).append(ms)
        ctx.ctx.profile(False)
        return {n: float(np.mean(ms)) for n, ms in acc.items()}

    main_s = torch.cuda.current_stream(dev)
    s_d2h = torch.cuda.Stream(dev)

    def e2e(dt, n):
        host = [{m: torch.empty(shape, dtype=(torch.bool if m == "mask" else dt)).pin_memory()
                 for m, shape in SHAPES.items()} for _ in range(2)]
        done = [torch.cuda.Event(), torch.cuda.Event()]
        pending = [None, None]

        def run(steps):
            for k in range(steps):
                if pending[k % 2] is not None:
                    main_s.wait_event(done[k % 2])   # the copy of step k - 2 is finished before its maps are freed
                    pending[k % 2] = None
                o = wr.render(ctx, mesh, cam, H, W, output_dtype=dt, **kw)
                ready = torch.cuda.Event()
                ready.record(main_s)
                with torch.cuda.stream(s_d2h):
                    s_d2h.wait_event(ready)
                    for m, dst in host[k % 2].items():
                        dst.copy_(getattr(o, m), non_blocking=True)
                    done[k % 2].record(s_d2h)
                pending[k % 2] = o
            torch.cuda.synchronize()
            pending[0] = pending[1] = None

        run(6)
        t0 = time.perf_counter()
        run(n)
        dt_s = time.perf_counter() - t0
        # the copies alone: the same maps, device -> the same pinned buffers, back to back on one stream
        src = {m: torch.empty(t.shape, dtype=t.dtype, device=dev) for m, t in host[0].items()}
        for _ in range(3):
            for m in SHAPES:
                host[0][m].copy_(src[m], non_blocking=True)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for _ in range(n):
            for m in SHAPES:
                host[0][m].copy_(src[m], non_blocking=True)
        torch.cuda.synchronize()
        c_s = time.perf_counter() - t0
        return {"views_per_s": N_VIEWS * n / dt_s, "copies_only_steps_per_s": n / c_s,
                "copy_ceiling_views_per_s": N_VIEWS * n / c_s, "frac_of_copy_ceiling": (n / dt_s) / (n / c_s)}

    for g in graphs.values():   # warm-up of every shape the timed window uses
        time_steps(g, 10)
    steps = {name: [] for name in dtypes}
    stage = {name: [] for name in dtypes}
    e2e_r = {name: [] for name in dtypes}
    for r in range(args.rounds):
        order = list(dtypes) if r % 2 == 0 else list(reversed(dtypes))
        for name in order:
            steps[name].append(time_steps(graphs[name], args.steps))
        for name in order:
            stage[name].append(stages(dtypes[name]))
        for name in order:
            e2e_r[name].append(e2e(dtypes[name], args.e2e_steps))

    result = {"card": card(), "torch_device_name": torch.cuda.get_device_name(dev),
              "workload": "config B: 1M-face terrain, canonical 6-view orthographic rig, 768x768, "
                          "mask + pos + depth(controlnet) + normal",
              "timing": "step: RenderGraph replay between CUDA events, 512 MiB device write before every step outside "
                        "the events (L2 flushed); stages: wr_ctx_profile events of the eager call; e2e: wall clock of "
                        "eager calls with the maps copied to pinned host memory on a second stream, double-buffered",
              "rounds": args.rounds, "steps_per_round": args.steps, "bit_identical_to_float32_cast": exact,
              "map_bytes_per_step": bytes_per_step, "by_dtype": {}}
    for name in dtypes:
        all_ms = [x for rnd in steps[name] for x in rnd]
        st = {n: float(np.mean([s[n] for s in stage[name]])) for n in stage[name][0]}
        result["by_dtype"][name] = {
            "step_ms_median": statistics.median(all_ms),
            "step_ms_min": min(all_ms), "step_ms_max": max(all_ms),
            "step_ms_median_per_round": [statistics.median(rnd) for rnd in steps[name]],
            "views_per_s_from_median": N_VIEWS / (statistics.median(all_ms) * 1e-3),
            "stage_ms": st,
            "k_shade_ms": st.get("k_shade"), "k_depth_finalize_ms": st.get("k_depth_finalize"),
            "e2e_views_per_s_per_round": [e["views_per_s"] for e in e2e_r[name]],
            "e2e_views_per_s_median": statistics.median(e["views_per_s"] for e in e2e_r[name]),
            "copy_ceiling_views_per_s_median": statistics.median(e["copy_ceiling_views_per_s"] for e in e2e_r[name]),
            "e2e_frac_of_copy_ceiling_median": statistics.median(e["frac_of_copy_ceiling"] for e in e2e_r[name]),
        }
    text = json.dumps(result, indent=1)
    print(text)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as fh:
            fh.write(text + "\n")


if __name__ == "__main__":
    main()
