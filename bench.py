#!/usr/bin/env python
"""bench.py -- headline measurement of the geometry path (BASELINE.json metric).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]

Workload (config B of SURVEY.md section 8d, `configs[1]` of BASELINE.json): one synthetic 1M-face
terrain mesh per GPU, the canonical 6-view orthographic rig, 768x768, outputs mask + position +
view depth (DepthControlNetNormalization) + normal.  One STEP = one render() call = 6 views.
With N GPUs every rank renders its own mesh (seed = rank) -- the by-mesh sharding of config D, no
data-path collective -- so scaling is weak and `value` = N * 6 * K / (max over ranks of the timed time).

JSON keys beyond the base contract:
  roofline      dominant kernel: algorithmic bytes / CUDA-event duration vs MEASURED_PEAKS.json
  pipeline      whole render step against the same peak (SURVEY 8d: 12F + 24V + 33HW bytes per view)
  stages        per-kernel ms (CUDA events recorded by the library on its launch stream; recording them
                turns the dependent launches off, so the stages sum to more than ms_per_step)
  cpu_baseline  the oracle port of the reference's render path timed on this box's host cores
  e2e           same metric through the public API with host buffers (H2D of the mesh, D2H of the maps)
  bake          ms per UV bake, config C (6 x 768^2 images -> 1024^2 atlas), device resident: the
                CameraProjection call of SURVEY 8d, the unprojection kernel alone, uv_precompute alone (1024^2 and
                4096^2), and the same call with the reference's default tail (seam padding; padding + 1000 sweeps)
  timing        how the timed region ran (launch path, L2 policy); kept out of `config`, which names the workload
                only and is identical in both arms
  config_a      config A (50k-face icosphere, same rig): ms per step and views/s on this GPU
  config_d      config D (BASELINE.json configs[3]): 8 meshes x 6 views per GPU per step, one CUDA-graph replay per
                step (RenderGraph), whole-job views/s and the ratio to N x the config-B value
  bake_sharded  config E (BASELINE.json configs[4]): 32 views of 2048^2 of a 5M-face mesh baked into a 4096^2
                atlas, views sharded over the ranks, accumulators exchanged ("auto" = fused peer-memory /
                NVSwitch-multicast kernel, "nccl" = all_reduce + finalize); ms per bake, the exchange step alone,
                equality with a 1-rank bake, and strong-scaling efficiency against the 1-rank time measured on
                rank 0 in the same run

`--impl reference` times the reference's render path on the host cores.  The reference has no CPU
implementation of its own (its rasterizer is the GPU-only nvdiffrast), so this arm is the oracle
port: the reference's Python restated in NumPy over the C/OpenMP restatement of the operators.

`--dump-outputs DIR` writes the four maps of the last timed step (rank 0's mesh) as DIR/{mask,pos,depth,normal}.npy,
float32, at a fixed sample of pixels (see dump_outputs); the inputs are seeded, so two builds, or the two arms, can be
compared file by file.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

H = W = 768
N_VIEWS = 6
TERRAIN = (1000, 500)  # quads -> 1 000 000 faces, 501 501 vertices
METRIC = "views_per_sec_768sq_pos_normal_1M_face_mesh"
UNIT = "views/s"
MAPS = ("mask", "pos", "depth", "normal")   # what render() returns to the caller of the timed step
DUMP_PIXELS = 1 << 20                       # 32 MiB of float32 for the four maps (a step has 3.5 M pixels, 113 MB)


def dump_outputs(dump_dir: str, maps: dict) -> None:
    """Writes each map (torch tensor or NumPy array, leading dims views x H x W) as DIR/<name>.npy in float32, the mask
    as 0 / 1, at the same DUMP_PIXELS (view, y, x) positions: drawn with seed 0 without replacement, in increasing
    flat order.  pos and normal keep their channel axis: (DUMP_PIXELS, 3)."""
    os.makedirs(dump_dir, exist_ok=True)
    n_pix = N_VIEWS * H * W
    idx = np.sort(np.random.default_rng(0).choice(n_pix, DUMP_PIXELS, replace=False))
    for name, m in maps.items():
        a = m.cpu().numpy() if hasattr(m, "cpu") else np.asarray(m)
        a = a.reshape(n_pix, -1)[idx].reshape((DUMP_PIXELS,) + a.shape[3:])
        np.save(os.path.join(dump_dir, f"{name}.npy"), a.astype(np.float32))


def terrain_arrays(seed: int):
    from worldrenderer_b200 import synth
    v, f = synth.terrain(TERRAIN[0], TERRAIN[1], seed)
    v = v / np.abs(v).max() * 0.5                       # load_mesh(rescale=True, scale=0.5)
    v = np.stack([v[:, 0], -v[:, 2], v[:, 1]], -1)      # load_mesh axis remap (up=+y, front=+x)
    return np.ascontiguousarray(v, np.float32), np.ascontiguousarray(f, np.int64)


def algorithmic_bytes_per_view(F: int, V: int) -> dict:
    """SURVEY.md 8(d): compulsory HBM traffic of one rendered view, split by the kernel that owns it."""
    return {
        "k_snap_vertices": 12 * V,                 # f32 positions read once
        "k_setup_triangles": 12 * F,               # i32 indices read once
        "k_shade4": 12 * V + 33 * H * W,           # f32 normals + per pixel 4 id + 4 depth + 12 pos + 12 normal + 1 mask
        "k_shade": 12 * V + 33 * H * W,
        "total": 12 * F + 24 * V + 33 * H * W,
    }


def peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as fh:
            return float(json.load(fh)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """Samples SM clock and throttle reasons through NVML while the timed region runs."""

    def __init__(self, index: int):
        self.samples, self.reasons, self.max_mhz = [], set(), None
        self._stop = threading.Event()
        self._thread = None
        try:
            import pynvml
            pynvml.nvmlInit()
            self._nv = pynvml
            self._h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = int(pynvml.nvmlDeviceGetMaxClockInfo(self._h, pynvml.NVML_CLOCK_SM))
        except Exception:
            self._nv = None

    def _run(self):
        nv = self._nv
        names = {
            getattr(nv, "nvmlClocksEventReasonHwSlowdown", 0x8): "hw_slowdown",
            getattr(nv, "nvmlClocksEventReasonHwThermalSlowdown", 0x40): "hw_thermal_slowdown",
            getattr(nv, "nvmlClocksEventReasonSwThermalSlowdown", 0x20): "sw_thermal_slowdown",
            getattr(nv, "nvmlClocksEventReasonSwPowerCap", 0x4): "sw_power_cap",
        }
        while not self._stop.is_set():
            try:
                self.samples.append(int(nv.nvmlDeviceGetClockInfo(self._h, nv.NVML_CLOCK_SM)))
                try:
                    mask = nv.nvmlDeviceGetCurrentClocksEventReasons(self._h)
                except Exception:
                    mask = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self._h)
                for bit, name in names.items():
                    if mask & bit:
                        self.reasons.add(name)
            except Exception:
                pass
            time.sleep(0.002)

    def __enter__(self):
        if self._nv is not None:
            self._thread = threading.Thread(target=self._run, daemon=True)
            self._thread.start()
        return self

    def __exit__(self, *exc):
        self._stop.set()
        if self._thread is not None:
            self._thread.join()

    def summary(self):
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": [], "note": "NVML unavailable"}
        return {"sm_mhz": int(statistics.median(self.samples)), "sm_max_mhz": self.max_mhz,
                "reasons": sorted(self.reasons), "samples": len(self.samples)}


# ------------------------------------------------------------------------------------------------
# reference arm / cpu baseline: the oracle port on the host cores
# ------------------------------------------------------------------------------------------------

def cpu_render_setup(seed: int = 0):
    import worldrenderer_b200 as wr
    from oracle import render_oracle
    from worldrenderer_b200 import synth
    v, f = terrain_arrays(seed)
    f32 = f.astype(np.int32)
    cam = wr.get_orthogonal_camera(**synth.CANONICAL_RIG)
    v_nrm = render_oracle.vertex_normals(v, f32)  # once per mesh, outside the timed steps (as on the GPU arm's value)
    return v, f32, v_nrm, cam.mvp_mtx.numpy(), cam.w2c.numpy()


def cpu_threads() -> int:
    """Host threads the CPU arm uses: every core this process may run on (torchrun exports OMP_NUM_THREADS=1,
    so the count is passed to the oracle explicitly instead of being left to the OpenMP default)."""
    try:
        return max(1, len(os.sched_getaffinity(0)))
    except AttributeError:
        return max(1, os.cpu_count() or 1)


def cpu_render_step(state, views: int = N_VIEWS, nthreads: int = 0):
    from oracle import render_oracle
    v, f32, v_nrm, mvp, w2c = state
    return render_oracle.render(v, f32, mvp[:views], w2c[:views], H, W, v_nrm=v_nrm,
                                nthreads=nthreads or cpu_threads(), elementwise="by_view")


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    state = cpu_render_setup(0)
    for _ in range(max(1, min(args.warmup, 2))):
        cpu_render_step(state)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        out = cpu_render_step(state)
    dt = time.perf_counter() - t0
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {name: out[name] for name in MAPS})
    value = N_VIEWS * args.steps / dt
    cores = cpu_threads()
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * dt / args.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": workload_config(args.gpus),
        "timing": {"l2": "n/a (host run)", "launch_path": "n/a (host run)"},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": "port",
                         "sample": f"{args.steps} full steps (6 views 768^2 of the 1M-face mesh each), "
                                   f"oracle/render_oracle.py over oracle/wr_oracle.c (-O3 -march=native) with {cores} "
                                   "OpenMP threads, element-wise tail of each view on its own thread; "
                                   "the reference itself has no CPU path (nvdiffrast is GPU-only)"},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


def workload_config(n_gpus: int):
    """Names the workload only -- identical in both arms (how a run was timed goes into `timing`)."""
    return {"workload": "config B: 1M-face procedural terrain (501501 vertices), canonical 6-view orthographic rig, "
                        "768x768, outputs mask+position+depth(controlnet)+normal; one mesh per GPU (seed = rank)",
            "faces": 2 * TERRAIN[0] * TERRAIN[1], "views_per_step": N_VIEWS, "resolution": [H, W],
            "parallelism": f"by-mesh x{n_gpus}, no collective"}


# ------------------------------------------------------------------------------------------------
# our arm
# ------------------------------------------------------------------------------------------------

def run_ours(args):
    import torch
    import torch.distributed as dist

    import worldrenderer_b200 as wr
    from worldrenderer_b200 import synth

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise RuntimeError("bench.py needs a CUDA device: worldrenderer_b200 has no CPU path")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    K, Wm = args.steps, max(args.warmup, 3)
    v_np, f_np = terrain_arrays(rank)
    V, F = v_np.shape[0], f_np.shape[0]
    ctx = wr.NVDiffRastContextWrapper(str(dev), "cuda")
    cam = wr.get_orthogonal_camera(device=str(dev), **synth.CANONICAL_RIG)

    def make_mesh(v_t, f_t):
        m = wr.TexturedMesh(v_pos=v_t, t_pos_idx=f_t)
        m.set_stitched_mesh(m.v_pos, m.t_pos_idx)
        return m

    mesh = make_mesh(torch.from_numpy(v_np).to(dev), torch.from_numpy(f_np).to(dev))
    mesh.v_nrm  # vertex normals: once per mesh, like the reference's lazy property

    def step_eager():
        return wr.render(ctx, mesh, cam, H, W, render_attr=False, render_depth=True, render_normal=True)

    # The step of the timed region: the same render() captured once into a CUDA graph (wr.RenderGraph) and replayed
    # -- one host call per step, so eight ranks sharing one host cannot fall behind their GPUs (--eager times the
    # plain call instead; `eager_ms_per_step` is reported either way).
    graph = None if args.eager else wr.RenderGraph(ctx, [(mesh, cam)], H, W, render_attr=False, render_depth=True,
                                                   render_normal=True)

    def step():
        return graph.replay()[0] if graph is not None else step_eager()

    flush_buf = torch.empty(512 << 20, dtype=torch.uint8, device=dev)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(Wm):
        out = step()
    barrier()

    # ---- timed region: K steps, per-step CUDA events, L2 flushed between steps -------------------
    starts = [torch.cuda.Event(enable_timing=True) for _ in range(K)]
    stops = [torch.cuda.Event(enable_timing=True) for _ in range(K)]
    sampler = ClockSampler(local)
    barrier()
    with sampler:
        t_wall0 = time.perf_counter()
        for k in range(K):
            flush_buf.fill_(k & 0xFF)
            starts[k].record()
            out = step()
            stops[k].record()
        barrier()
        t_wall = time.perf_counter() - t_wall0
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, {name: getattr(out, name) for name in MAPS})
    step_ms = [starts[k].elapsed_time(stops[k]) for k in range(K)]
    total_ms = float(sum(step_ms))
    tot = torch.tensor([total_ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(tot, op=dist.ReduceOp.MAX)
    total_ms_max = float(tot.item())
    value = world * N_VIEWS * K / (total_ms_max * 1e-3)

    # ---- the same step issued eagerly (ctypes call per step) ---------------------------------------
    Ke_ = min(K, 30)
    keep_ = None
    for _ in range(5):   # un-timed: capturing the graph emptied torch's allocator cache, the first eager calls re-fill it
        keep_ = step_eager()
    torch.cuda.synchronize()
    del keep_
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(Ke_)]
    for k in range(Ke_):
        flush_buf.fill_(k & 0xFF)
        ev[k][0].record()
        step_eager()
        ev[k][1].record()
    torch.cuda.synchronize()
    eager_ms = float(np.mean([a.elapsed_time(b) for a, b in ev]))

    # ---- per-kernel stage timing (same steps, library-side events), rank 0 ------------------------
    stages, launches_per_step = {}, 0
    if rank == 0:
        ctx.ctx.profile(True)
        reps = min(K, 20)
        for k in range(reps):
            flush_buf.fill_(k & 0xFF)
            step_eager()
            for name, ms in ctx.ctx.profile_read():
                stages.setdefault(name, []).append(ms)
        ctx.ctx.profile(False)
        launches_per_step = sum(1 for n in stages if n.startswith("k_"))
        stages = {n: float(np.mean(ms)) for n, ms in stages.items()}
    torch.cuda.synchronize()

    # ---- end to end through the public API with host buffers ---------------------------------------
    v_host = torch.from_numpy(v_np).pin_memory()
    f_host = torch.from_numpy(f_np).pin_memory()
    mvp_host, w2c_host = cam.mvp_mtx.cpu().pin_memory(), cam.w2c.cpu().pin_memory()
    host_out = {
        "mask": torch.empty((N_VIEWS, H, W), dtype=torch.bool).pin_memory(),
        "pos": torch.empty((N_VIEWS, H, W, 3), dtype=torch.float32).pin_memory(),
        "depth": torch.empty((N_VIEWS, H, W), dtype=torch.float32).pin_memory(),
        "normal": torch.empty((N_VIEWS, H, W, 3), dtype=torch.float32).pin_memory(),
    }
    h2d = v_host.numel() * 4 + f_host.numel() * 8 + 2 * mvp_host.numel() * 4
    d2h = sum(t.numel() * t.element_size() for t in host_out.values())

    # Software pipeline over steps, as a serving loop would run it: while step k renders on the main stream,
    # the mesh of step k+1 is uploaded on a copy stream and the maps of step k-1 are read back on another.
    # Every step's inputs still come from pinned host memory and every step's four maps still land in pinned
    # host memory inside the timed region.
    main = torch.cuda.current_stream(dev)
    s_h2d, s_d2h = torch.cuda.Stream(dev), torch.cuda.Stream(dev)
    dev_in = [{"v": torch.empty_like(v_host, device=dev), "f": torch.empty_like(f_host, device=dev),
               "mvp": torch.empty_like(mvp_host, device=dev), "w2c": torch.empty_like(w2c_host, device=dev),
               "ready": torch.cuda.Event(), "free": torch.cuda.Event()} for _ in range(2)]
    host_outs = [host_out, {k: torch.empty_like(t).pin_memory() for k, t in host_out.items()}]
    d2h_done = [torch.cuda.Event(), torch.cuda.Event()]

    def upload(k):
        slot = dev_in[k % 2]
        with torch.cuda.stream(s_h2d):
            s_h2d.wait_event(slot["free"])  # the render that last read this slot has finished
            slot["v"].copy_(v_host, non_blocking=True)
            slot["f"].copy_(f_host, non_blocking=True)
            slot["mvp"].copy_(mvp_host, non_blocking=True)
            slot["w2c"].copy_(w2c_host, non_blocking=True)
            slot["ready"].record(s_h2d)

    pending = [None, None]  # render outputs of the step that last used each host buffer set

    def render_and_read_back(k):
        slot = dev_in[k % 2]
        # The maps of step k-2 are released here.  Their copy must be complete before the main stream may reuse
        # that memory, so the wait is put on the main stream BEFORE the references are dropped (no
        # record_stream: the caching allocator then recycles the blocks at once and never has to grow).
        if pending[k % 2] is not None:
            main.wait_event(d2h_done[k % 2])
            pending[k % 2] = None
        main.wait_event(slot["ready"])
        m = make_mesh(slot["v"], slot["f"])
        c = wr.Camera(c2w=None, w2c=slot["w2c"], proj_mtx=cam.proj_mtx, mvp_mtx=slot["mvp"], cam_pos=None)
        o = wr.render(ctx, m, c, H, W, render_attr=False, render_depth=True, render_normal=True)
        slot["free"].record(main)
        done = torch.cuda.Event()
        done.record(main)
        with torch.cuda.stream(s_d2h):
            s_d2h.wait_event(done)
            for name, dst in host_outs[k % 2].items():
                dst.copy_(getattr(o, name), non_blocking=True)
            d2h_done[k % 2].record(s_d2h)
        pending[k % 2] = (o, m)

    def e2e_run(n):
        for slot in dev_in:
            slot["free"].record(main)
        upload(0)
        for k in range(n):
            if k + 1 < n:
                upload(k + 1)
            render_and_read_back(k)
        torch.cuda.synchronize()
        pending[0] = pending[1] = None

    e2e_run(6)
    barrier()
    Ke = min(K, 100)
    t0 = time.perf_counter()
    e2e_run(Ke)
    barrier()
    e2e_dt = torch.tensor([time.perf_counter() - t0], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(e2e_dt, op=dist.ReduceOp.MAX)
    e2e_value = world * N_VIEWS * Ke / float(e2e_dt.item())

    # ---- what the box's PCIe path gives all ranks at once: the same pinned buffers, copies only -------
    # (the e2e loop above is bound by its read-back; this is the ceiling it is compared with: every rank moves the
    # step's 102.6 MB of maps to the host and the 30 MB mesh to the device, concurrently, nothing else running)
    pcie = None
    try:
        src = {k: torch.empty(t.shape, dtype=t.dtype, device=dev) for k, t in host_out.items()}

        def copies(n):
            for _ in range(n):
                with torch.cuda.stream(s_d2h):
                    for name, dst in host_out.items():
                        dst.copy_(src[name], non_blocking=True)
                with torch.cuda.stream(s_h2d):
                    dev_in[0]["v"].copy_(v_host, non_blocking=True)
                    dev_in[0]["f"].copy_(f_host, non_blocking=True)
            torch.cuda.synchronize()

        copies(3)
        barrier()
        reps_c = 30
        t0 = time.perf_counter()
        copies(reps_c)
        barrier()
        c_dt = torch.tensor([time.perf_counter() - t0], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(c_dt, op=dist.ReduceOp.MAX)
        c_dt = float(c_dt.item())
        pcie = {"d2h_gbs_all_ranks": world * reps_c * d2h / c_dt / 1e9,
                "h2d_gbs_all_ranks": world * reps_c * (h2d - 2 * mvp_host.numel() * 4) / c_dt / 1e9,
                "steps_per_s_all_ranks_copies_only": world * reps_c / c_dt,
                "e2e_d2h_gbs_all_ranks": e2e_value / N_VIEWS * d2h / 1e9,
                "e2e_frac_of_copy_ceiling": (e2e_value / N_VIEWS) / (world * reps_c / c_dt),
                "what": f"{world} rank(s) at once, {reps_c} x (the step's four maps device -> pinned host on one "
                        "stream + the step's mesh pinned host -> device on another), wall clock, max over ranks"}
        del src
    except Exception as exc:  # a measurement aid: never let it take the bench line down
        pcie = {"error": repr(exc)}

    # ---- bake (config C) and config A, rank 0 ------------------------------------------------------
    bake, config_a = None, None
    if rank == 0 and not args.no_bake:
        bake = bench_bake(ctx, dev, flush_buf)
        config_a = bench_config_a(ctx, dev, flush_buf, cam)
    # ---- config D (8 meshes per GPU per step) and config E (view-sharded bake), all ranks ----------
    config_d = None if args.no_extra else bench_config_d(dev, rank, world, flush_buf, cam, min(K, 20), value)
    bake_sharded = None if args.no_extra else bench_bake_sharded(ctx, dev, rank, world, flush_buf, full=not args.small_e)

    if rank == 0:
        peak, peak_src = peaks()
        ab = algorithmic_bytes_per_view(F, V)
        kernel_stages = {n: ms for n, ms in stages.items() if n.startswith("k_") and n in ab}
        dom = max(kernel_stages, key=kernel_stages.get) if kernel_stages else None
        roofline = None
        if dom is not None:
            achieved = ab[dom] * N_VIEWS / (kernel_stages[dom] * 1e-3) / 1e9
            traffic = None
            tpath = os.path.join(ROOT, "profiles", "ncu_traffic_r02.json")
            if not os.path.exists(tpath):
                tpath = os.path.join(ROOT, "profiles", "ncu_traffic_r01.json")
            if os.path.exists(tpath):
                with open(tpath) as fh:
                    traffic = json.load(fh).get(dom)  # DRAM bytes per launch of this kernel from the committed ncu capture
            roofline = {"bound": "hbm", "kernel": dom, "achieved": achieved, "peak": peak, "unit": "GB/s",
                        "frac": achieved / peak, "frac_of_nominal_8000": achieved / 8000.0, "traffic": traffic,
                        "peak_source": peak_src,
                        "algorithmic_bytes_per_launch": ab[dom] * N_VIEWS, "kernel_ms": kernel_stages[dom],
                        "share_of_step": kernel_stages[dom] / max(sum(stages.values()), 1e-9)}
        ms_per_step = total_ms_max / K
        pipe_achieved = ab["total"] * N_VIEWS / (ms_per_step * 1e-3) / 1e9
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": K, "warmup": Wm,
            "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic", "config": workload_config(world),
            "timing": {"l2": "flushed between timed steps by a 512 MiB device write outside the per-step events",
                       "launch_path": "eager ctypes call per step" if graph is None else
                       "one CUDA-graph replay per step (wr.RenderGraph capture of the same render() call)",
                       "eager_ms_per_step": eager_ms},
            "roofline": roofline,
            "pipeline": {"bound": "hbm", "achieved": pipe_achieved, "peak": peak, "unit": "GB/s",
                         "frac": pipe_achieved / peak, "frac_of_nominal_8000": pipe_achieved / 8000.0,
                         "algorithmic_bytes_per_step": ab["total"] * N_VIEWS},
            "stages_ms": stages,
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                    "steps": Ke, "what": "render() per step on a mesh uploaded from pinned host memory (positions f32 + "
                                         "faces i64 + cameras), vertex normals, 6 views, all four maps copied back to "
                                         "pinned host memory; steps are software-pipelined over three streams "
                                         "(upload k+1 | render k | read back k-1)",
                    "pcie_ceiling": pcie},
            "gpu_launches": launches_per_step * K,
            "gpu_launches_per_step": launches_per_step,
            "clocks": sampler.summary(),
            "wall_s_timed_region": t_wall,
            "bake": bake,
            "config_a": config_a,
            "config_d": config_d,
            "bake_sharded": bake_sharded,
        }
        if not args.no_cpu and world == 1:
            line["cpu_baseline"] = bench_cpu_baseline()
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def _timed(torch, flush_buf, fn, reps=20, warm=3):
    for _ in range(warm):
        fn()
    ms = []
    for k in range(reps):
        flush_buf.fill_(k & 0xFF)
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        torch.cuda.synchronize()
        ms.append(a.elapsed_time(b))
    return ms


def bench_config_a(ctx, dev, flush_buf, cam):
    """Config A (BASELINE.json configs[0]): 50k-face icosphere, the canonical rig, 768^2."""
    import torch

    import worldrenderer_b200 as wr
    from worldrenderer_b200 import synth
    v, f = synth.icosphere(50, 0.5)
    mesh = wr.TexturedMesh(v_pos=torch.tensor(v, dtype=torch.float32, device=dev), t_pos_idx=torch.tensor(f, dtype=torch.int64, device=dev))
    mesh.set_stitched_mesh(mesh.v_pos, mesh.t_pos_idx)
    mesh.v_nrm
    ms = float(np.median(_timed(torch, flush_buf, lambda: wr.render(ctx, mesh, cam, H, W, render_attr=False))))
    bytes_step = N_VIEWS * (12 * f.shape[0] + 24 * v.shape[0] + 33 * H * W)
    peak, _ = peaks()
    return {"workload": "config A: 50k-face icosphere, canonical 6-view rig, 768^2, same outputs as config B",
            "ms_per_step": ms, "views_per_s": N_VIEWS / (ms * 1e-3), "algorithmic_bytes_per_step": bytes_step,
            "frac_of_hbm_peak": bytes_step / (ms * 1e-3) / 1e9 / peak}


def bench_config_d(dev, rank, world, flush_buf, cam, K, config_b_value):
    """Config D (BASELINE.json configs[3]): a batch of 8 x world meshes x 6 views at 768^2 sharded by mesh, 8 meshes
    per GPU and step, no communication.  One step = one RenderGraph replay (8 render() calls)."""
    import torch
    import torch.distributed as dist

    import worldrenderer_b200 as wr
    per_gpu = 8
    meshes = []
    for j in range(per_gpu):
        v_np, f_np = terrain_arrays(rank * per_gpu + j)
        m = wr.TexturedMesh(v_pos=torch.from_numpy(v_np).to(dev), t_pos_idx=torch.from_numpy(f_np).to(dev))
        m.set_stitched_mesh(m.v_pos, m.t_pos_idx)
        m.v_nrm
        meshes.append(m)
    ctx = wr.NVDiffRastContextWrapper(str(dev), "cuda")
    g = wr.RenderGraph(ctx, [(m, cam) for m in meshes], H, W, lanes=2, render_attr=False)
    for _ in range(3):
        g.replay()
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(K)]
    for k in range(K):
        flush_buf.fill_(k & 0xFF)
        ev[k][0].record()
        g.replay()
        ev[k][1].record()
    torch.cuda.synchronize()
    tot = torch.tensor([sum(a.elapsed_time(b) for a, b in ev)], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(tot, op=dist.ReduceOp.MAX)
    ms = float(tot.item()) / K
    value = world * per_gpu * N_VIEWS / (ms * 1e-3)
    del g, meshes
    torch.cuda.empty_cache()
    return {"workload": f"config D: {per_gpu * world} terrain meshes (1M faces each, seeds 0..{per_gpu * world - 1}) x 6 views "
                        f"at 768^2, {per_gpu} meshes per GPU and step, sharded by mesh, no collective",
            "meshes_per_gpu": per_gpu, "ms_per_step": ms, "views_per_s": value,
            "ratio_to_config_b_value": value / config_b_value,
            "launch_path": "one CUDA-graph replay per step (8 render() calls captured by wr.RenderGraph on two concurrent "
                           "lanes: the shading pass of one mesh runs under the raster set-up of the next)"}


def bench_bake_sharded(ctx, dev, rank, world, flush_buf, full=True):
    """Config E (BASELINE.json configs[4]): 32 views at 2048^2 of a 5M-face terrain baked into a 4096^2 atlas, the
    views sharded over the ranks and the weighted accumulators exchanged (the one collective of the path).
    full=False: the scaled shape (1M faces, 32 x 1024^2 views, 2048^2 atlas)."""
    import contextlib
    import io

    import torch
    import torch.distributed as dist

    import worldrenderer_b200 as wr
    from worldrenderer_b200 import parallel, synth
    from worldrenderer_b200.uv import uv_finalize

    NV, RES, UV = (32, 2048, 4096) if full else (32, 1024, 2048)
    NX, NY = (2500, 1000) if full else TERRAIN
    v, f = synth.terrain(NX, NY, 0)
    v = v / np.abs(v).max() * 0.5
    v = np.ascontiguousarray(np.stack([v[:, 0], -v[:, 2], v[:, 1]], -1), np.float32)
    f = np.ascontiguousarray(f, np.int64)
    vt = synth.terrain_uv(NX, NY).astype(np.float32)
    mesh = wr.TexturedMesh(v_pos=torch.from_numpy(v).to(dev), t_pos_idx=torch.from_numpy(f).to(dev),
                           v_tex=torch.from_numpy(vt).to(dev), t_tex_idx=torch.from_numpy(f).to(dev),
                           texture=torch.zeros((UV, UV, 3), device=dev))
    mesh.set_stitched_mesh(mesh.v_pos, mesh.t_pos_idx)
    mesh.v_nrm
    cam = wr.get_orthogonal_camera(elevation_deg=[20.0] * NV, distance=[1.0] * NV, left=-0.55, right=0.55,
                                   bottom=-0.55, top=0.55, azimuth_deg=list(np.linspace(0, 360, NV + 1)[:-1]),
                                   device=str(dev))

    def images_for(lo, hi):
        # img[v, y, x, c] = .5 + .5 sin(w_c . (x, y) + phi_vc), generated on the device (seeded per global view)
        g = torch.Generator(device="cpu").manual_seed(1)
        omega = torch.empty(3, 2).uniform_(0.01, 0.06, generator=g).to(dev)
        phi = torch.empty(NV, 3).uniform_(0.0, 6.2831853, generator=g)[lo:hi].to(dev)
        y, x = torch.meshgrid(torch.arange(RES, device=dev, dtype=torch.float32),
                              torch.arange(RES, device=dev, dtype=torch.float32), indexing="ij")
        arg = omega[None, :, 0, None, None] * x + omega[None, :, 1, None, None] * y + phi[:, :, None, None]
        return (0.5 + 0.5 * torch.sin(arg)).permute(0, 2, 3, 1).contiguous()

    # interleaved view shards (rank, rank + world, ...): neighbouring ring views cost alike, so contiguous blocks
    # leave the ranks unevenly loaded (tools/bake_balance_probe.py)
    mine = parallel.shard_slice(NV, rank, world, interleave=True)
    images = images_for(0, NV)[mine].contiguous() if world > 1 else images_for(0, NV)
    kw = dict(aoi_cos_valid_threshold=0.2, depth_grad_threshold=0.1, uv_exp_blend_alpha=3.0)

    def sync():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()

    solo = dist.new_group([0]) if world > 1 else None   # rank 0 alone: the 1-rank bake of this run

    def time_bake(mode, cam_l, img_l, group_sync=True, reps=8, group=None):
        kw_ = dict(kw, group=group)
        for _ in range(2):
            parallel.sharded_bake(ctx, mesh, cam_l, img_l, UV, exchange=mode, **kw_)
        if group_sync:
            sync()
        else:
            torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(reps):
            out = parallel.sharded_bake(ctx, mesh, cam_l, img_l, UV, exchange=mode, **kw_)
        e1.record()
        torch.cuda.synchronize()
        t = torch.tensor([e0.elapsed_time(e1) / reps], dtype=torch.float64, device=dev)
        if group_sync and world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item()), out

    res = {"workload": f"config E{'' if full else ' (scaled)'}: {f.shape[0]} faces, {NV} views of {RES}^2 on a ring, "
                       f"{UV}^2 atlas, views sharded over {world} rank(s), accumulators exchanged and finalised on every rank",
           "views": NV, "view_resolution": RES, "atlas": UV, "faces": int(f.shape[0])}
    with contextlib.redirect_stdout(io.StringIO()):
        if world == 1:
            ms, (atlas, any_) = time_bake("auto", cam, images)
            res.update({"ms_per_bake": ms, "ms_per_bake_1_rank": ms, "covered_texels": int(any_.sum())})
            bytes_bake = 32 * NV * RES * RES + 38 * UV * UV + NV * (12 * f.shape[0] + 24 * v.shape[0] + 33 * RES * RES)
            peak, _ = peaks()
            res["algorithmic_bytes_per_bake"] = bytes_bake
            res["frac_of_hbm_peak"] = bytes_bake / (ms * 1e-3) / 1e9 / peak
            return res
        ms_auto, (atlas, any_) = time_bake("auto", cam[mine], images)
        atlas, any_ = atlas.clone(), any_.clone()
        ms_nccl, (atlas_n, any_n) = time_bake("nccl", cam[mine], images)
        # the exchange step alone, on this bake's accumulators
        ws = parallel._p2p_workspace(UV, UV, dev, None)
        exch = {}
        if ws is not None:
            old = mesh.texture

            def run_fused():
                return ws.reduce_finalize(ctx, old)

            def run_nccl():
                t = ws.accum.clone()
                parallel.all_reduce_accumulators(t)
                return uv_finalize(ctx, t, old)

            for name, fn in (("fused", run_fused), ("nccl_all_reduce_plus_finalize", run_nccl)):
                for _ in range(2):
                    fn()
                sync()
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                for _ in range(8):
                    fn()
                e1.record()
                torch.cuda.synchronize()
                t = torch.tensor([e0.elapsed_time(e1) / 8], dtype=torch.float64, device=dev)
                dist.all_reduce(t, op=dist.ReduceOp.MAX)
                exch[name] = float(t.item())
            exch["kernel"] = "k_uv_reduce_finalize_mc (multimem.ld_reduce / multimem.st)" if (ws.mc_ptr and world >= 4) \
                else "k_uv_reduce_finalize_p2p (peer loads / stores)"
        # batched baking: a stream of bakes through parallel.BakePipeline (the exchange of bake k on its own stream,
        # under the view passes of bake k + 1)
        pipe = parallel.BakePipeline(ctx, UV, depth=2)
        NB = 8
        for _ in range(2):
            tickets = [pipe.submit(mesh, cam[mine], images, **kw) for _ in range(3)]
            atlas_p, any_p = tickets[-1].result()
        sync()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        tickets = [pipe.submit(mesh, cam[mine], images, **kw) for _ in range(NB)]
        for tk in tickets:
            atlas_p, any_p = tk.result()
        e1.record()
        torch.cuda.synchronize()
        tp = torch.tensor([e0.elapsed_time(e1) / NB], dtype=torch.float64, device=dev)
        dist.all_reduce(tp, op=dist.ReduceOp.MAX)
        ms_pipe = float(tp.item())
        pipe_same = bool(torch.equal(atlas_p, atlas) and torch.equal(any_p, any_))
        sync()
        # rank 0 bakes all views alone: the 1-rank time of THIS run and the result to compare with
        same_mask, max_err, ms_one = True, 0.0, None
        if rank == 0:
            img_all = images_for(0, NV)
            ms_one, (atlas1, any1) = time_bake("nccl", cam, img_all, group_sync=False, reps=4, group=solo)
            same_mask = bool(torch.equal(any1, any_))
            max_err = float((atlas1 - atlas).abs().max())
            dd = (atlas1 - atlas).abs().max(-1).values
            iy, ix = divmod(int(dd.argmax()), UV)
            print(f"[diag] texels > 1e-5: {int((dd > 1e-5).sum())}, > 1e-3: {int((dd > 1e-3).sum())}, max at {(iy, ix)}: "
                  f"1-rank {atlas1[iy, ix].tolist()} N-rank {atlas[iy, ix].tolist()} nccl-path {atlas_n[iy, ix].tolist()} "
                  f"any {bool(any1[iy, ix])}", file=sys.stderr, flush=True)
            del img_all
        sync()
        gathered = [torch.empty_like(atlas) for _ in range(world)]
        dist.all_gather(gathered, atlas)
        identical = all(torch.equal(g, gathered[0]) for g in gathered)
        res.update({"ms_per_bake": ms_auto, "ms_per_bake_nccl": ms_nccl, "exchange_step_ms": exch,
                    "ms_per_bake_1_rank": ms_one, "mask_equal_to_1_rank": same_mask, "max_abs_err_vs_1_rank": max_err,
                    "ranks_identical": identical,
                    "strong_scaling_efficiency": None if ms_one is None else ms_one / (world * ms_auto),
                    "batched": {"what": f"{NB} bakes back to back through parallel.BakePipeline (depth 2): the exchange "
                                        "of bake k runs on its own stream under the view passes of bake k + 1",
                                "ms_per_bake": ms_pipe, "same_result_as_single_bake": pipe_same,
                                "scaling_efficiency": None if ms_one is None else ms_one / (world * ms_pipe)},
                    "nvlink_bytes_per_texel": {"fused_multicast": "20 B out (in-switch sum) + 13 B in", "nccl": "2 x 20 B"}})
    return res


def bench_cpu_baseline():
    state = cpu_render_setup(0)
    cpu_render_step(state)
    reps, t0 = 0, time.perf_counter()
    while reps < 3 or (time.perf_counter() - t0 < 10.0 and reps < 30):
        cpu_render_step(state)
        reps += 1
    dt = time.perf_counter() - t0
    cores = cpu_threads()
    t1 = time.perf_counter()
    cpu_render_step(state, nthreads=1)      # single-core figure (BASELINE.md 4.3): one full step on one thread
    dt1 = time.perf_counter() - t1
    return {"value": N_VIEWS * reps / dt, "unit": UNIT, "cores": cores, "kind": "port",
            "sample": f"{reps} full steps (6 views 768^2, same 1M-face mesh), oracle port of render.py:220-286 "
                      f"(C operators -O3 -march=native, {cores} OpenMP threads; NumPy tail of each view on its own "
                      "thread); vertex normals excluded on both sides",
            "ms_per_step": 1e3 * dt / reps,
            "single_core": {"value": N_VIEWS / dt1, "unit": UNIT, "cores": 1, "ms_per_step": 1e3 * dt1}}


def bench_bake(ctx, dev, flush_buf):
    """Config C: icosphere 50k faces with a cell atlas, 6 synthetic 768^2 images -> 1024^2 atlas."""
    import torch

    import worldrenderer_b200 as wr
    from worldrenderer_b200 import synth
    from worldrenderer_b200.uv import fused_unproject, fused_view_maps

    v, f = synth.icosphere(50, 0.5)
    vt, ft = synth.cell_atlas_uv(f.shape[0])
    uv = 1024
    mesh = wr.TexturedMesh(v_pos=torch.tensor(v, dtype=torch.float32), t_pos_idx=torch.tensor(f, dtype=torch.int64),
                           v_tex=torch.tensor(vt, dtype=torch.float32), t_tex_idx=torch.tensor(ft, dtype=torch.int64),
                           texture=torch.zeros((uv, uv, 3), dtype=torch.float32))
    mesh.set_stitched_mesh(mesh.v_pos, mesh.t_pos_idx)
    mesh.to(dev)
    mesh.v_nrm
    cam = wr.get_orthogonal_camera(device=str(dev), **synth.CANONICAL_RIG)
    images = torch.from_numpy(synth.view_images(N_VIEWS, H, W, seed=1)).to(dev)
    proj = wr.CameraProjection(None, None, str(dev), "cuda")
    proj.ctx = ctx
    kw = dict(uv_size=uv, poisson_blending=False, uv_padding=False, depth_grad_dilation=5, uv_exp_blend_alpha=3,
              uv_exp_blend_view_weight=torch.ones(N_VIEWS), aoi_cos_valid_threshold=0.2, depth_grad_threshold=0.1,
              iou_rejection_threshold=None, return_dict=True)

    def timed(fn, reps=20):
        for _ in range(3):
            fn()
        ms = []
        for k in range(reps):
            flush_buf.fill_(k & 0xFF)
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            fn()
            b.record()
            torch.cuda.synchronize()
            ms.append(a.elapsed_time(b))
        return float(np.median(ms))

    import contextlib
    import io
    with contextlib.redirect_stdout(io.StringIO()):  # the call prints the reference's "No view mask" notice
        e2e_ms = timed(lambda: proj(images, mesh, cam, **kw))
        pre = wr.uv_precompute(ctx, mesh, uv, uv)
        _, geo, att = fused_view_maps(ctx, mesh, cam, images, H, W, 5)
        unproj_ms = timed(lambda: fused_unproject(ctx, pre, cam, H, W, geo, att, aoi_cos_thresh=0.2,
                                                  depth_grad_thresh=0.1, alpha=3.0,
                                                  view_weight=torch.ones(N_VIEWS, device=dev)))
        # uv_precompute (uv.py:24-53) on its own: UV-space raster of the 50k faces + position interpolation.
        # CameraProjection caches it per (mesh, size), so it is outside ms_per_uv_bake_end_to_end after the first call.
        pre_ms = {str(s_): timed(lambda: wr.uv_precompute(ctx, mesh, s_, s_), reps=10) for s_ in (1024, 4096)}
        # the same CameraProjection call replayed from a CUDA graph (wr.BakeGraph): no launch gaps
        graph_ms = None
        try:
            bg = wr.BakeGraph(proj, images, mesh, cam, **kw)
            graph_ms = timed(bg.replay)
            del bg
        except Exception as exc:
            graph_ms = repr(exc)
        # the reference's default tail (uv.py:426-461): seam padding, and Poisson blending with 1000 sweeps
        proj_pb = wr.CameraProjection("torch-cuda", None, str(dev), "cuda")
        proj_pb.ctx = ctx
        kw_pad = dict(kw, uv_padding=True)
        kw_pb = dict(kw, uv_padding=True, poisson_blending=True, pb_num_iters=1000)
        pad_ms = timed(lambda: proj_pb(images, mesh, cam, **kw_pad), reps=10)
        pb_ms = timed(lambda: proj_pb(images, mesh, cam, **kw_pb), reps=5)
    peak, _ = peaks()
    bytes_unproj = 32 * N_VIEWS * H * W + 38 * uv * uv
    return {"workload": "config C: 50k-face icosphere, 6 x 768^2 images -> 1024^2 atlas, validity + cosine^3 weights",
            "ms_per_uv_bake_end_to_end": e2e_ms, "ms_per_uv_bake_graph_replay": graph_ms,
            "ms_unprojection_only": unproj_ms, "ms_uv_precompute": pre_ms,
            "ms_per_uv_bake_with_seam_padding": pad_ms,
            "ms_per_uv_bake_with_padding_and_poisson_1000_sweeps": pb_ms,
            "unprojection_algorithmic_bytes": bytes_unproj,
            "unprojection_frac_of_hbm_peak": bytes_unproj / (unproj_ms * 1e-3) / 1e9 / peak}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--no-bake", action="store_true", help="skip the config C bake timing")
    ap.add_argument("--no-extra", action="store_true", help="skip config D and the config E sharded bake")
    ap.add_argument("--small-e", action="store_true", help="config E at the scaled shape (1M faces, 32 x 1024^2, 2048^2 atlas)")
    ap.add_argument("--eager", action="store_true", help="time the eager render() call instead of its CUDA-graph replay")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the maps of the last timed step to DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
