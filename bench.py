#!/usr/bin/env python
"""bench.py — physics steps/s of the avian3d substep hot path on B200 (BASELINE.json metric).

A "step" is ONE pass of the hot path over one frozen snapshot of the headline scene (100 000-cube coupled stack, f32, 8 substeps):
sweep-and-prune broad phase over the 100 001 collider AABBs + the whole solver stage (prepare, 8 x [integrate velocities, warm start,
biased solve, integrate positions, relax], restitution, writeback, store impulses) over the snapshot's bodies and contact manifolds.
The narrow phase is NOT in the step (outside the hot path, SURVEY.md 8f #1); its manifolds are part of the snapshot, identical for every arm.

  e2e          THE HEADLINE: steps/s from pinned HOST body / AABB columns to HOST results through the public C-ABI calls of the device-resident
               pipeline (SURVEY 8f #1 + #3): avn_broadphase_upload/run/download_order -> avn_contacts_step (the new pairs are taken in device
               memory; contact rows, geometry + match_contacts, touching state machine, ContactGraph, ConstraintGraph colouring and the
               colour-major list all live on the device) -> avn_solver_upload_resident + run + download; every step uploads the body, collider
               and AABB columns and reads back the persistent order, ~40 counters and the bodies (wall clock around K steps of a LIVE world,
               barrier + synchronize on both sides).  It does MORE than the CPU arm's step (narrow phase and graph maintenance are inside).
               `e2e.host_manifolds` is round 1's arm: the manifolds computed by a host narrow phase outside the step and uploaded as columns
               through avn_solver_step (80 MB up / 24 MB down).
  value        steps/s with the snapshot resident in HBM: K x (avn_broadphase_run + avn_solver_run) back to back, timed as ONE span by two
               CUDA events on the library's stream (host launch gaps included, no copies), max over ranks; N > 1 = N independent piles
               (island sharding of independent scenes, no collective), value = N * K / T.
  breakdown_ms per-call device times of the two stages (CUDA events inside the library), for the roofline.
  roofline     the dominant kernel (the persistent step megakernel): algorithmic bytes per launch (SURVEY 8d formulas with the measured
               B, M, P) / its CUDA-event duration, vs MEASURED_PEAKS.json hbm_gbs; `solver_pass` = the same for ONE solver-iteration pass
               (biased solve over all colours), the kernel BASELINE.json's 40 % bar names.
  parity       the GPU step vs the CPU oracle step from the same full-size snapshot, element-wise (bar 1e-5; pairs bit-exact).  Missing the
               bar fails the run.
  partition    ONE scene over the N GPUs (strong scaling, SURVEY 8e): `spheres1m_slab` = the 1M-sphere f64 scene cut into x-slabs, one NCCL
               all-gather of boundary state per substep INSIDE the library (avn_comm_init + avn_solver_step_partitioned);
               `ragdolls5k_island` = the 5 000-ragdoll field dealt out by island (no collective in the data path).  Printed at every N
               (N = 1 is the baseline of the curve).
  cpu_baseline the CPU oracle (C++ restatement of the reference path, colour-parallel, all host cores) on the same snapshot.
  --impl reference   times only that CPU arm (the reference itself is Rust and cannot be built in this image).
  --dump-outputs DIR the arrays the last timed step returned (`value`'s arm, or the CPU arm with --impl reference): bodies, impulses, joint
                     forces, the count of new pairs (and their columns when there are any), persistent order, as DIR/<name>.npy, so that
                     two builds can be compared output for output.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))

SCENES = {
    # name: (builder, substeps, default settle steps)
    "stack100k": (lambda sc: sc.cube_stack(51, 40, 50, brick=True), 8, 2),   # BASELINE configs[2] (headline): exactly 100 000 cubes
    "stack10k": (lambda sc: sc.cube_stack(23, 20, 22, brick=True), 8, 2),    # BASELINE configs[1]-sized: ~10 000 cubes
    "stack1k": (lambda sc: sc.cube_stack(11, 10, 10, brick=True), 8, 2),
    "ragdolls5k": (lambda sc: sc.ragdoll_field(5000, pitch=3.0, drop_height=0.2), 8, 30),  # BASELINE configs[3]: 85 000 bodies, 80 000 joints
    "ragdolls500": (lambda sc: sc.ragdoll_field(500, pitch=3.0, drop_height=0.2), 8, 30),
    # BASELINE configs[4]: 1M spheres r=0.5, f64, uniform in a 200x50x200 box (seed 42); broad-phase heavy
    "spheres1m": (lambda sc: sc.falling_spheres(1_000_000, seed=42, scalar=np.float64), 8, 2),
    "spheres100k": (lambda sc: sc.falling_spheres(100_000, seed=42, box=(93.0, 50.0, 93.0), scalar=np.float64), 8, 2),
}
LABEL = {"stack100k": "100k-cube stack", "stack10k": "10k-cube stack", "stack1k": "1k-cube stack", "ragdolls5k": "5k-ragdoll field",
         "ragdolls500": "500-ragdoll field", "spheres1m": "1M falling spheres (f64)", "spheres100k": "100k falling spheres (f64)"}
MODES = {0: "phases", 1: "megakernel, grid barriers", 2: "megakernel, wavefront records", 3: "megakernel, one warp per island"}


def metric_name(scene: str) -> str:
    return f"physics steps/sec on {LABEL[scene]} (broad phase + solver stage per step)"


def workload_config(sc, prm, B, M, P, J, settle, scalar_name, iters) -> dict:
    """The part of `config` both arms print identically (the driver compares the two lines)."""
    return {"workload": f"{sc.name}: {B - 1} dynamic bodies on a ground slab, {scalar_name}, {int(prm.substeps)} substeps, reference solver semantics "
                        f"(1 warm start + {iters} biased + 1 relax pass per substep), one step = broad phase + solver stage of a frozen snapshot",
            "bodies": B, "manifolds": M, "contact_points": P, "joints": J, "solver_iterations": iters, "settle_steps": settle}


def algorithmic_bytes(B: int, M: int, P: int, substeps: int, scalar_bytes: int = 4) -> dict:
    """SURVEY.md 8(d), f32 figures scaled by the scalar size; P = total contact points (P/M = mean points/manifold)."""
    k = scalar_bytes / 4.0
    pbar = P / max(M, 1)
    solve_pass = (52 + 76 * pbar) * M + 216 * B
    warm = (28 + 36 * pbar) * M + 136 * B
    a_sub = 84 * B + 80 * B + warm + 2 * solve_pass
    prepare = (100 + 80 * pbar) * M + 170 * B
    step = substeps * a_sub + prepare + 152 * B + 16 * pbar * M
    return {"solve_pass": solve_pass * k, "substep": a_sub * k, "step": step * k}


class ClockSampler(threading.Thread):
    """nvidia-smi clocks/throttle reasons sampled DURING the timed region (B200_PROFILING.md recipe); rank 0 only."""
    Q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
        "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index: int, enabled: bool = True):
        super().__init__(daemon=True)
        self.index, self.rows, self.stop_flag, self.enabled = index, [], threading.Event(), enabled

    def run(self):
        while self.enabled and not self.stop_flag.is_set():
            try:
                out = subprocess.run(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits"],
                                     capture_output=True, text=True, timeout=5).stdout.strip()
                if out:
                    self.rows.append([x.strip() for x in out.split(",")])
            except Exception:
                pass
            self.stop_flag.wait(0.2)

    def summary(self) -> dict:
        self.stop_flag.set()
        if not self.rows:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["unavailable"]}
        sm = sorted(float(r[0]) for r in self.rows if r[0].replace(".", "").isdigit())
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(len(r) > 3 + i and r[3 + i].lower().startswith("active") for r in self.rows)]
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": float(self.rows[0][1]) if self.rows[0][1].replace(".", "").isdigit() else None,
                "reasons": reasons, "samples": len(self.rows)}


def build_snapshot(scene_name: str, settle: int, ctx=None):
    """Scene -> (scene, params, bodies, manifolds, aabbs, joints) frozen after `settle` full pipeline steps.  With ctx (GPU arm) the
    pipeline's hot path runs on the GPU; without it on the CPU oracle, so that the CPU arm never needs the GPU.  Both give the same
    snapshot (the two paths are bit-identical on contact scenes, tests/test_gpu_parity_at_size.py)."""
    from avian_b200 import plugins, scenes
    builder, substeps, _ = SCENES[scene_name]
    sc = builder(scenes)
    if ctx is not None:
        w = plugins.World(sc, plugins.PhysicsPlugins(ctx), substeps=substeps)
    else:
        sys.path.insert(0, str(ROOT / "tests"))
        import oracle_lib
        w = plugins.World(sc, oracle_lib.oracle_plugins(threads=os.cpu_count() or 1), substeps=substeps)
    for _ in range(settle):
        w.step()
    w.broad_phase()
    man = w.narrow_phase()
    # the steady-state broad-phase input: every current pair is already in the contact graph
    aabbs = w.pipeline.intervals(w.bodies, w.aabb_min, w.aabb_max, with_existing=True)
    aabbs.joint_disabled_body_pairs = sc.joint_disabled_body_pairs
    return sc, w.params, w.bodies, man, aabbs, w.joints


DUMP_BUDGET = 60 << 20     # bytes of array data per --dump-outputs directory: under 64 MB with the .npy headers


def step_outputs(bodies, man, joints, pairs, aabbs) -> dict:
    """What a caller of one step receives: the bodies' new state, the contact impulses, the joint forces, the number of new pairs the
    broad phase found and, when there are any, their columns, and its persistent order (the retained intervals only: the rest of
    order_out is not written).  A steady-state snapshot has every current pair in its contact graph, so its count of new pairs is 0."""
    out = {k: getattr(bodies, k) for k in ("position", "rotation", "linear_velocity", "angular_velocity")}
    out.update({k: getattr(man, k) for k in ("warm_start_normal_impulse", "warm_start_tangent_impulse", "normal_impulse")})
    for t, j in ({} if joints is None else joints.types).items():
        for k in ("force", "torque"):
            if getattr(j, k) is not None:
                out[f"joint{int(t)}_{k}"] = getattr(j, k)
    out["pair_count"] = np.array([pairs.count])
    if pairs.count:
        out.update({f"pairs_{k}": getattr(pairs, k)[:pairs.count] for k in ("collider1", "collider2", "body1", "body2", "flags")})
    if aabbs.order_out is not None:
        out["order"] = aabbs.order_out[:aabbs.retained_count]
    return out


def dump_outputs(out_dir: str, arrays: dict) -> None:
    """<out_dir>/<name>.npy for every array: float columns in their own type, integer columns as float64 (exact below 2**53).  When the
    arrays exceed DUMP_BUDGET, each keeps the same seeded sample of its rows (the same rows for arrays of the same length, at least one
    row), so that the dumps of two builds still compare element for element.  An array without elements is not written."""
    out = {k: np.array(v, dtype=v.dtype if v.dtype in (np.float32, np.float64) else np.float64) for k, v in arrays.items() if v.size}
    total = sum(v.nbytes for v in out.values())
    if total > DUMP_BUDGET:
        share = DUMP_BUDGET / total
        for k, v in out.items():
            rows = np.random.default_rng(0).choice(v.shape[0], max(1, int(v.shape[0] * share)), replace=False)
            out[k] = v[np.sort(rows)]
    path = Path(out_dir)
    path.mkdir(parents=True, exist_ok=True)
    for k, v in out.items():
        np.save(path / f"{k}.npy", v)


def pin_columns(ctx, obj):
    """Move every numpy column of a Bodies/Manifolds/Aabbs dataclass into pinned host memory."""
    for k, v in list(obj.__dict__.items()):
        if isinstance(v, np.ndarray):
            setattr(obj, k, ctx.pin_like(v))
    return obj


class StreamTimer:
    """Two CUDA events on the LIBRARY's stream (torch.cuda.Event only sees torch's current stream: make the library's stream current)."""

    def __init__(self, ctx):
        import torch
        self.torch = torch
        self.stream = torch.cuda.ExternalStream(ctx.stream(), device=torch.device("cuda", ctx.device))
        self.e0, self.e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)

    def start(self):
        with self.torch.cuda.stream(self.stream):
            self.e0.record()

    def stop_ms(self) -> float:
        with self.torch.cuda.stream(self.stream):
            self.e1.record()
        self.e1.synchronize()
        return self.e0.elapsed_time(self.e1)


def run_gpu(args, info):
    import torch
    from avian_b200 import api, parallel
    rank, world, local_rank = info.rank, info.world, info.local_rank
    torch.cuda.set_device(local_rank)
    scalar = np.float64 if args.scene.startswith("spheres") else np.float32
    ctx = api.Context(device=local_rank, scalar=scalar)
    sc, prm, bodies, man, aabbs, joints = build_snapshot(args.scene, args.settle, ctx)
    prm.solver_iterations = args.solver_iterations
    B, M, P = bodies.count, man.count, int(man.penetration.shape[0])
    J = 0 if joints is None else joints.count
    pin_columns(ctx, bodies); pin_columns(ctx, man); pin_columns(ctx, aabbs)
    pairs_out = api.PairList.empty(1 << 20)
    b0, m0 = bodies.copy(), man.copy()     # the frozen snapshot (the step writes results into bodies/man in place)
    K = args.steps

    def barrier():
        parallel.barrier(info)
        torch.cuda.synchronize()

    def restore():
        for name in ("position", "rotation", "linear_velocity", "angular_velocity"):
            getattr(bodies, name)[...] = getattr(b0, name)
        for name in ("warm_start_normal_impulse", "warm_start_tangent_impulse", "normal_impulse"):
            getattr(man, name)[...] = getattr(m0, name)

    sampler = ClockSampler(local_rank, enabled=(rank == 0)); sampler.start()
    # ---- resident arm: upload once, K x (broad phase + solver stage) back to back, ONE event span on the library's stream ---------------
    ctx.solver_upload(prm, bodies, man, joints)
    ctx.broadphase_upload(aabbs)
    for _ in range(args.warmup):
        ctx.broadphase_run(); ctx.solver_run()
    timer = StreamTimer(ctx)
    barrier()
    t0 = time.perf_counter()
    timer.start()
    for _ in range(K):
        ctx.broadphase_run()
        ctx.solver_run()
    span_ms = timer.stop_ms()
    barrier()
    wall_resident = time.perf_counter() - t0
    if args.dump_outputs and rank == 0:     # every run restarts from the uploaded snapshot: this is what the last timed step computed
        ctx.broadphase_download(pairs_out)
        ctx.solver_download()
        dump_outputs(args.dump_outputs, step_outputs(bodies, man, joints, pairs_out, aabbs))
    # ---- the same loop with the per-call device times read back (stage breakdown, launch count); results are downloaded here
    mega_ms, bp_ms, launches, mode = 0.0, 0.0, 0, None
    n_break = min(K, 10)
    for _ in range(n_break):
        ctx.broadphase_run()
        ctx.broadphase_download(pairs_out)
        tb = ctx.timings()
        ctx.solver_run()
        ctx.solver_download()
        ts = ctx.timings()
        bp_ms += tb["broad_phase_ms"]; mega_ms += ts["total_ms"]
        launches += tb["kernel_launches"] + ts["kernel_launches"]
        mode = ts["launch_mode"]
    bp_ms, mega_ms = bp_ms / n_break, mega_ms / n_break
    launches_per_step = launches / n_break
    new_pairs = int(pairs_out.count)
    restore()

    # ---- one solver-iteration pass on its own (the kernel BASELINE.json's 40 % bar names)
    solver_pass = measure_solver_pass(args, prm, bodies, man, joints, scalar, local_rank) if (rank == 0 and not args.no_pass) else None
    restore()

    # ---- end-to-end arm: host buffers in, host buffers out, every step ----------------------------------------------------------------
    for _ in range(max(1, args.warmup // 2)):
        ctx.broadphase(aabbs); ctx.solver_step(prm, bodies, man, joints); restore()
    barrier()
    t0 = time.perf_counter()
    for _ in range(K):
        ctx.broadphase_upload(aabbs); ctx.broadphase_run(); ctx.broadphase_download(pairs_out)
        ctx.solver_step(prm, bodies, man, joints)
    barrier()
    wall_e2e = time.perf_counter() - t0
    te = ctx.timings()     # of the last end-to-end solver call: where its time went
    e2e_break = {"solver_h2d": te["h2d_ms"], "solver_kernels": te["total_ms"], "solver_d2h": te["d2h_ms"]}
    # keep the GPU under the same load until the sampler has a few readings (nvidia-smi takes ~100 ms per call)
    t_hold = time.perf_counter()
    while rank == 0 and len(sampler.rows) < 3 and time.perf_counter() - t_hold < 3.0:
        ctx.broadphase_run(); ctx.solver_run(); ctx.solver_download()
    clocks = sampler.summary()
    sb = bodies.position.dtype.itemsize
    h2d = sum(v.nbytes for k, v in bodies.__dict__.items() if isinstance(v, np.ndarray)) + \
        sum(v.nbytes for k, v in man.__dict__.items() if isinstance(v, np.ndarray) and k != "normal_impulse") + \
        sum(v.nbytes for k, v in aabbs.__dict__.items() if isinstance(v, np.ndarray) and k != "order_out")
    d2h = B * (3 + 4 + 3 + 3) * sb + P * 4 * sb + B * 4 + new_pairs * 17
    restore()
    # one more end-to-end step from the frozen snapshot whose outputs are kept: the parity block compares them with the CPU arm's
    gpu_pairs = ctx.broadphase(aabbs)
    ctx.solver_step(prm, bodies, man, joints)
    gpu_out = (bodies.copy(), man.copy(), gpu_pairs, None if aabbs.order_out is None else aabbs.order_out.copy())
    restore()

    # ---- end-to-end arm of the device-resident pipeline: its own context and world (the contact rows must have lived through the settle steps)
    resident = e2e_resident(args, info, barrier) if not args.no_resident else None

    # max over ranks
    span_ms, wall_res_ms, wall_e2e_ms, mega_ms, bp_ms = parallel.reduce_max([span_ms, wall_resident * 1e3, wall_e2e * 1e3, mega_ms, bp_ms], info, device="cuda")
    # the pinned columns die with the context: what the CPU arm still needs moves to ordinary memory first
    aabbs = api.Aabbs(**{k: (v.copy() if isinstance(v, np.ndarray) else v) for k, v in aabbs.__dict__.items()})
    n_colliders = int(aabbs.collider.shape[0])
    n_existing = 0 if aabbs.existing_pairs is None else int(aabbs.existing_pairs.shape[0])
    del bodies, man
    ctx.close()

    # ---- ONE scene over the N GPUs (every rank takes part; rank 0 reports)
    partition = None
    if not args.no_partition:
        partition = {}
        for name, fn in (("spheres1m_slab", partition_slab), ("ragdolls5k_island", partition_islands)):
            t_part = time.perf_counter()
            try:
                partition[name] = fn(args, info)
            except Exception as exc:   # a partition arm must not take the headline down with it
                partition[name] = {"error": f"{type(exc).__name__}: {exc}"}
            if isinstance(partition[name], dict):
                partition[name]["bench_seconds"] = round(time.perf_counter() - t_part, 1)
    if rank != 0:
        return None

    value = world * K / (span_ms / 1e3)
    e2e_value = world * K / (wall_e2e_ms / 1e3)
    alg = algorithmic_bytes(B, M, P, int(prm.substeps), sb)
    if J:
        alg["step"] += int(prm.substeps) * (300 * J + 100 * B) * (sb / 4.0)   # XPBD joint pass + velocity projection, SURVEY 8d
    peaks_path = ROOT / "MEASURED_PEAKS.json"
    if peaks_path.exists():
        peak, peak_src = float(json.loads(peaks_path.read_text())["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    else:
        peak, peak_src = 6650.0, "fallback (B200_PROFILING.md)"
    achieved = alg["step"] / (mega_ms / 1e3) / 1e9
    traffic = None
    tfile = ROOT / "profiles" / "traffic.json"
    if tfile.exists():
        try:
            traffic = json.loads(tfile.read_text()).get(args.scene, {}).get("dram_bytes_per_launch")
        except Exception:
            traffic = None
    sname = "f64" if sb == 8 else "f32"
    cfg = workload_config(sc, prm, B, M, P, J, args.settle, sname, int(prm.solver_iterations))
    cfg.update({"colliders": n_colliders, "existing_pairs": n_existing,
                "new_pairs_per_step": new_pairs, "parallelism": "1 pile per GPU (island sharding of independent scenes), no data-path collective",
                "l2": "inputs larger than L2: constraint planes + columns > 126 MB per step",
                "timing": "value: one CUDA-event span over K back-to-back steps on the library stream; e2e: wall clock between barriers; max over ranks",
                "launch_mode": MODES.get(mode, mode)})
    roof = {"bound": "hbm", "kernel": f"step_megakernel<{'double' if sb == 8 else 'float'}> (whole solver stage, one launch per step)", "achieved": achieved,
            "peak": peak, "unit": "GB/s", "frac": achieved / peak, "traffic": traffic, "peak_source": peak_src, "algorithmic_bytes_per_launch": alg["step"],
            "kernel_ms": mega_ms, "solve_pass_bytes": alg["solve_pass"]}
    if solver_pass is not None:
        pass_gbs = alg["solve_pass"] / (solver_pass["ms_per_pass"] / 1e3) / 1e9
        roof["solver_pass"] = {"kernel": "phase_kernel<OP_SOLVE_BIAS> x active colours (one solver-iteration pass, one launch per colour)",
                               "ms_per_pass": solver_pass["ms_per_pass"], "achieved": pass_gbs, "frac": pass_gbs / peak, "how": solver_pass["how"]}
    host_arm = {"value": e2e_value, "unit": "steps/s", "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h), "ms_per_step": wall_e2e_ms / K,
                "last_step_device_ms": e2e_break, "what": "avn_broadphase + avn_solver_step with the manifold columns of a host narrow phase uploaded every step"}
    if resident is not None and "error" not in resident:
        e2e_block = {"value": world * K / (resident["wall_ms"] / 1e3), "unit": "steps/s", "h2d_bytes_per_step": resident["h2d"], "d2h_bytes_per_step": resident["d2h"],
                     "ms_per_step": resident["wall_ms"] / K, "pipeline": resident["what"], "graph": resident["graph"], "host_manifolds": host_arm}
    else:
        e2e_block = dict(host_arm)
        if resident is not None:
            e2e_block["resident_error"] = resident["error"]
    result = {
        "metric": metric_name(args.scene), "value": value, "unit": "steps/s",
        "n_gpus": world, "steps": K, "warmup": args.warmup, "ms_per_step": span_ms / K, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": sname, "data": "synthetic", "config": cfg,
        "e2e": e2e_block,
        "gpu_launches": int(round(launches_per_step * K)), "clocks": clocks, "roofline": roof,
        "breakdown_ms": {"broad_phase": bp_ms, "solver_stage": mega_ms, "resident_span": span_ms / K, "resident_wall": wall_res_ms / K,
                         "kernel_launches_per_step": launches_per_step},
    }
    if partition is not None:
        result["partition"] = partition
    if not args.no_cpu:
        keep = {}
        result["cpu_baseline"] = cpu_arm(args, prm, b0, m0, aabbs, sample_steps=args.cpu_steps, joints=joints, keep=keep)
        result["parity"] = parity_block(gpu_out, keep)
    return result


def _resident_world(args, ctx):
    """A DeviceGraphWorld of the scene (contact rows, ContactGraph and ConstraintGraph on the device), settled, with every per-step host column
    pinned.  The AABB columns are frozen after the settle steps (like the snapshot of the other arms: the broad phase runs in full and finds the
    pairs it already has); the bodies keep evolving, so contacts start and stop touching and the graphs change on the device every step."""
    from avian_b200 import api, plugins, scenes
    builder, substeps, _ = SCENES[args.scene]
    w = plugins.DeviceGraphWorld(builder(scenes), plugins.PhysicsPlugins(ctx), ctx, substeps=substeps)
    w.params.solver_iterations = args.solver_iterations
    first = None
    for _ in range(args.settle + 2):
        w.step()
        first = first or dict(w.stats)
    pin_columns(ctx, w.bodies)
    mn, mx = w.pipeline.update_aabbs(w.bodies, w.params.dt)
    mn, mx = ctx.pin_like(mn), ctx.pin_like(mx)
    w._shape, w._dims = ctx.pin_like(w._shape), ctx.pin_like(w._dims)
    aabbs = None
    for _ in range(4):                    # until the frozen AABBs bring no new pair; the order is a fixed point then
        aabbs = pin_columns(ctx, w.intervals(mn, mx))
        w.step_from(aabbs, mn, mx)
        if w.new_pairs == 0:
            break
    aabbs = pin_columns(ctx, w.intervals(mn, mx))
    for _ in range(max(2, args.warmup)):
        w.step_from(aabbs, mn, mx)
    return w, aabbs, mn, mx, first


def e2e_resident(args, info, barrier):
    """K steps of DeviceGraphWorld.step_from from pinned host columns; returns wall ms (max over ranks) and the bytes that cross the bus."""
    from avian_b200 import api, parallel
    scalar = np.float64 if args.scene.startswith("spheres") else np.float32
    ctx = api.Context(device=info.local_rank, scalar=scalar)
    try:
        error = None
        try:
            w, aabbs, mn, mx, first = _resident_world(args, ctx)
        except Exception as exc:
            error = f"{type(exc).__name__}: {exc}"
        if parallel.reduce_max([0.0 if error is None else 1.0], info, device="cuda")[0] > 0:     # every rank agrees before the barriers
            return {"error": error or "another rank failed to set the resident world up"}
        barrier()
        changes = rounds = 0
        t0 = time.perf_counter()
        try:
            for _ in range(args.steps):
                st = w.step_from(aabbs, mn, mx)
                changes += st["started_touching"] + st["stopped_touching"] + st["pairs_added"] + st["pairs_removed"]
                rounds = max(rounds, st["colouring_rounds"])
        except Exception as exc:   # a rank that fails must still reach the barrier the others wait at; the arm is then reported as failed
            error = f"{type(exc).__name__}: {exc}"
        barrier()
        wall_ms = parallel.reduce_max([(time.perf_counter() - t0) * 1e3], info, device="cuda")[0]
        if parallel.reduce_max([0.0 if error is None else 1.0], info, device="cuda")[0] > 0:
            return {"error": error or "another rank failed inside the resident arm"}
        b, sb = w.bodies, w.bodies.position.dtype.itemsize
        C = int(aabbs.collider.shape[0])
        # what crosses the bus per step in the steady state: the interval columns of the broad phase; collider poses + AABBs and body velocities of
        # the contact step; position, rotation, velocities (and accelerations) of the solver's bodies.  Shapes and the columns that describe
        # the bodies (mass properties, damping ...) stay on the device (AVN_CONTACTS_SHAPES_UNCHANGED / AVN_BODIES_STATIC_UNCHANGED).
        acc = sum(v.nbytes for k, v in b.__dict__.items() if isinstance(v, np.ndarray) and k in ("linear_acceleration", "angular_acceleration"))
        h2d = sum(v.nbytes for k, v in aabbs.__dict__.items() if isinstance(v, np.ndarray) and k != "order_out") \
            + C * (3 + 4 + 3 + 3) * sb + b.count * (3 + 3) * sb + b.count * (3 + 4 + 3 + 3) * sb + acc
        d2h = b.count * (3 + 4 + 3 + 3) * sb + C * 4 + 35 * 4 + 16
        st = w.stats
        return {"wall_ms": wall_ms, "h2d": int(h2d), "d2h": int(d2h),
                "graph": {"contact_rows": st["rows_live"], "manifolds": st["manifold_count"], "changes_per_step": changes / max(args.steps, 1),
                          "max_colouring_rounds": rounds, "first_frame": {k: first[k] for k in ("pairs_added", "started_touching", "colouring_rounds")}},
                "what": "avn_broadphase (new pairs stay on the device) -> avn_contacts_step (rows, geometry + match_contacts, touching state machine, "
                        "ContactGraph, ConstraintGraph colouring, colour-major list: all on the device) -> avn_solver_upload_resident/run/download"}
    finally:
        ctx.close()


def measure_solver_pass(args, prm, bodies, man, joints, scalar, device):
    """Device time of ONE biased-solve pass over all colours = (T(step with 2 biased iterations) - T(step with 1)) / substeps, both in
    one-launch-per-phase mode (AVN_LAUNCH_MODE=phases: the kernel per colour is phase_kernel<OP_SOLVE_BIAS>, the same per-item routine the
    megakernel runs).  Differencing isolates exactly the launches of the extra pass; the library's own CUDA events time the steps."""
    from avian_b200 import api
    old = os.environ.get("AVN_LAUNCH_MODE")
    os.environ["AVN_LAUNCH_MODE"] = "phases"
    keep_iters = prm.solver_iterations
    try:
        with api.Context(device=device, scalar=scalar) as c2:
            times = {}
            for iters in (1, 2):
                prm.solver_iterations = iters
                c2.solver_upload(prm, bodies, man, joints)
                for _ in range(2):
                    c2.solver_run()
                tot, n = 0.0, 5
                for _ in range(n):
                    c2.solver_run(); c2.solver_download()
                    tot += c2.timings()["total_ms"]
                times[iters] = tot / n
        return {"ms_per_pass": (times[2] - times[1]) / int(prm.substeps),
                "how": f"phase mode: (step with 2 biased passes {times[2]:.3f} ms - step with 1 pass {times[1]:.3f} ms) / {int(prm.substeps)} substeps"}
    finally:
        prm.solver_iterations = keep_iters
        if old is None:
            os.environ.pop("AVN_LAUNCH_MODE", None)
        else:
            os.environ["AVN_LAUNCH_MODE"] = old


# ---------------------------------------------------------------------------------------------------------------------------------------
# ONE scene over the N GPUs
# ---------------------------------------------------------------------------------------------------------------------------------------
def _comm_init(ctx, info):
    """avn_comm_init on every rank: rank 0 draws the NCCL id inside the library, the bytes travel over torch.distributed's object broadcast
    (any host channel would do); the collective itself then lives in libavian_b200.so."""
    if info.world == 1:
        ctx.comm_init(0, 1, None)
        return
    import torch.distributed as dist
    box = [ctx.comm_unique_id() if info.rank == 0 else None]
    dist.broadcast_object_list(box, src=0)
    ctx.comm_init(info.rank, info.world, box[0])


def _partition_loop(args, info, ctx, step, dev):
    """warm-up, then K steps as one CUDA-event span on the library's stream, max over ranks; returns ms per step"""
    import torch
    from avian_b200 import parallel
    K, W = args.partition_steps, 3
    for _ in range(W):
        step()
    timer = StreamTimer(ctx)
    parallel.barrier(info); torch.cuda.synchronize()
    timer.start()
    for _ in range(K):
        step()
    ms = timer.stop_ms()
    parallel.barrier(info); torch.cuda.synchronize()
    return parallel.reduce_max([ms], info, dev)[0] / K


def partition_slab(args, info) -> dict | None:
    """BASELINE configs[4]: 1M spheres f64, one scene cut into `world` x-slabs.  Per step and rank: local slab broad phase + the partitioned
    solver stage with one NCCL all-gather of the packed boundary tables per substep inside the library (avn_solver_step_partitioned)."""
    from avian_b200 import api, parallel
    scene = args.partition_slab_scene
    rank, world = info.rank, info.world
    dev = f"cuda:{info.local_rank}" if world > 1 else "cpu"
    ctx = api.Context(device=info.local_rank, scalar=np.float64 if scene.startswith("spheres") else np.float32)
    try:
        sc, prm, bodies, man, aabbs, joints = build_snapshot(scene, min(SCENES[scene][2], 1), ctx)   # the same global snapshot on every rank
        _comm_init(ctx, info)
        cuts = parallel.body_slab_cuts(bodies, world)
        shard = parallel.shard_solver(bodies, man, cuts, rank, world)
        acuts = parallel.slab_cuts(aabbs.aabb_min[:, 0], world)
        ashard = parallel.shard_aabbs(aabbs, acuts, rank)
        pin_columns(ctx, shard.bodies); pin_columns(ctx, ashard.aabbs)
        if shard.manifolds is not None:
            pin_columns(ctx, shard.manifolds)
        ctx.solver_upload(prm, shard.bodies, shard.manifolds, None)
        ctx.solver_set_boundary(shard.bnd_body, shard.bnd_source, shard.bnd_owner, shard.record_count, rank, world)
        ctx.broadphase_upload(ashard.aabbs)

        def step():
            ctx.broadphase_run()
            ctx.solver_step_partitioned()

        ms = _partition_loop(args, info, ctx, step, dev)
        ctx.solver_download()
        held = parallel.reduce_sum([float(shard.bodies.count), float(0 if shard.manifolds is None else shard.manifolds.count), float(ashard.index.size)], info, dev)
        ctx.comm_destroy()
        if rank != 0:
            return None
        sb = bodies.position.dtype.itemsize
        return {"scene": sc.name, "value": 1e3 / ms, "unit": "steps/s", "ms_per_step": ms, "scaling": "strong", "n_gpus": world, "dtype": "f64" if sb == 8 else "f32",
                "bodies": bodies.count, "manifolds": man.count, "boundary_bodies": shard.slot_count, "bodies_held_all_ranks": int(held[0]),
                "manifolds_all_ranks": int(held[1]), "intervals_held_all_ranks": int(held[2]),
                "collective": "ncclAllGather of the packed boundary tables once per substep, issued by libavian_b200.so on its own stream",
                "exchange_bytes_per_substep_per_rank": shard.record_count * api.BOUNDARY_RECORD_SCALARS * sb,
                "parity": "broad phase bit-exact; solver stage = oracle slab engine at 1e-5 (tests/test_gpu_multi.py), solver tolerance vs the unpartitioned step"}
    finally:
        ctx.close()


def partition_islands(args, info) -> dict | None:
    """BASELINE configs[3]: the ragdoll field dealt out by island (connected components of dynamic bodies): every rank steps its islands with the
    ordinary avn_solver_run — no collective in the data path, results bit-identical to the unsharded step — plus its x-slab of the broad phase."""
    from avian_b200 import api, parallel
    scene = args.partition_island_scene
    rank, world = info.rank, info.world
    dev = f"cuda:{info.local_rank}" if world > 1 else "cpu"
    ctx = api.Context(device=info.local_rank, scalar=np.float32)
    try:
        sc, prm, bodies, man, aabbs, joints = build_snapshot(scene, SCENES[scene][2], ctx)
        labels, n_islands = parallel.find_islands(bodies, man, joints)
        sh = parallel.shard_by_island(bodies, man, joints, world, rank, labels)
        acuts = parallel.slab_cuts(aabbs.aabb_min[:, 0], world)
        ashard = parallel.shard_aabbs(aabbs, acuts, rank)
        pin_columns(ctx, sh.bodies); pin_columns(ctx, ashard.aabbs)
        ctx.solver_upload(prm, sh.bodies, sh.manifolds, sh.joints)
        ctx.broadphase_upload(ashard.aabbs)

        def step():
            ctx.broadphase_run()
            ctx.solver_run()

        ms = _partition_loop(args, info, ctx, step, dev)
        ctx.solver_download()
        mode = ctx.timings()["launch_mode"]
        held = parallel.reduce_sum([float(sh.bodies.count), float(0 if sh.joints is None else sh.joints.count)], info, dev)
        if rank != 0:
            return None
        return {"scene": sc.name, "value": 1e3 / ms, "unit": "steps/s", "ms_per_step": ms, "scaling": "strong", "n_gpus": world, "dtype": "f32",
                "bodies": bodies.count, "joints": 0 if joints is None else joints.count, "manifolds": man.count, "islands": int(n_islands),
                "bodies_held_all_ranks": int(held[0]), "joints_all_ranks": int(held[1]), "collective": "none in the data path (islands are independent)",
                "launch_mode": MODES.get(mode, mode), "parity": "bit-identical to the unsharded step (tests/test_island_cpu.py, tests/test_gpu_multi.py)"}
    finally:
        ctx.close()


def parity_block(gpu_out, keep) -> dict:
    """The GPU step and the CPU oracle step from the SAME full-size snapshot, compared element-wise (tests/helpers.py parity_report):
    relative error with a floor of one unit, bar 1e-5 (BASELINE.json north_star); the broad phase's pair list and persistent order
    bit for bit.  The run FAILS (exit code 1) when the bar is missed."""
    sys.path.insert(0, str(ROOT / "tests"))
    from helpers import BODY_OUT, IMPULSE_OUT, parity_report
    gb, gm, gp, gorder = gpu_out
    ob, om, op, oorder = keep["bodies"], keep["manifolds"], keep["pairs"], keep["order"]
    rep = parity_report(gb, ob, BODY_OUT)
    rep.update(parity_report(gm, om, IMPULSE_OUT))
    pairs_ok = gp.count == op.count and all(np.array_equal(getattr(gp, k)[:gp.count], getattr(op, k)[:op.count]) for k in ("collider1", "collider2", "body1", "body2", "flags"))
    order_ok = gorder is None or oorder is None or bool(np.array_equal(gorder, oorder))
    worst = max(r["max_rel_err"] for r in rep.values())
    return {"max_rel_err_pos": rep["position"]["max_rel_err"], "max_rel_err_rot": rep["rotation"]["max_rel_err"],
            "max_rel_err_vel": max(rep["linear_velocity"]["max_rel_err"], rep["angular_velocity"]["max_rel_err"]),
            "max_rel_err_impulse": max(rep[k]["max_rel_err"] for k in IMPULSE_OUT if k in rep) if any(k in rep for k in IMPULSE_OUT) else 0.0,
            "pairs_bit_exact": bool(pairs_ok), "order_bit_exact": order_ok, "pairs": int(op.count),
            "bit_identical_share": min(r["bit_identical"] for r in rep.values()), "max_ulp": max(r["max_ulp"] for r in rep.values()),
            "definition": "element-wise |gpu - cpu| / max(1, |cpu|) after one full step from the same snapshot; cpu = oracle/ (restated reference)",
            "bar": 1e-5, "ok": bool(worst <= 1e-5 and pairs_ok and order_ok)}


def cpu_arm(args, prm, bodies, man, aabbs, sample_steps: int, joints=None, keep: dict | None = None) -> dict:
    """The oracle (restated reference path, colour-parallel like the reference) on the host cores."""
    sys.path.insert(0, str(ROOT / "tests"))
    import oracle_lib
    from avian_b200 import api
    threads = os.cpu_count() or 1
    t_total = 0.0
    for i in range(sample_steps):
        b, m, j = bodies.copy(), man.copy(), None if joints is None else joints.copy()
        a = api.Aabbs(**{k: (v.copy() if isinstance(v, np.ndarray) else v) for k, v in aabbs.__dict__.items()})
        t0 = time.perf_counter()
        pairs = oracle_lib.broadphase(a, capacity=1 << 20)
        oracle_lib.solver_step(prm, b, m, j, threads=threads)
        t_total += time.perf_counter() - t0
        if keep is not None and i == 0:
            keep.update(bodies=b, manifolds=m, joints=j, pairs=pairs, aabbs=a, order=a.order_out)
    return {"value": sample_steps / t_total, "unit": "steps/s", "cores": threads, "kind": "port",
            "sample": f"{sample_steps} full steps of the same snapshot (SAP single-threaded + solver stage colour-parallel on {threads} threads)",
            "ms_per_step": t_total / sample_steps * 1e3}


def run_reference(args, rank: int, world: int):
    """--impl reference: the reference's CPU implementation of the path = the oracle port (Rust cannot be built here).  Same config, same
    steps / warm-up as the repo arm: every step is one full step of the 100k snapshot (~1 s on the box's cores)."""
    if rank != 0:
        return None
    sc, prm, bodies, man, aabbs, joints = build_snapshot(args.scene, args.settle if args.settle <= 4 else 0, None)
    prm.solver_iterations = args.solver_iterations
    if args.warmup:
        cpu_arm(args, prm, bodies, man, aabbs, args.warmup, joints)
    keep = {}
    cb = cpu_arm(args, prm, bodies, man, aabbs, args.steps, joints, keep=keep)
    if args.dump_outputs:     # every step starts from the same snapshot: the first step's outputs are the last step's
        dump_outputs(args.dump_outputs, step_outputs(keep["bodies"], keep["manifolds"], keep["joints"], keep["pairs"], keep["aabbs"]))
    B, M, P = bodies.count, man.count, int(man.penetration.shape[0])
    sname = "f64" if bodies.position.dtype == np.float64 else "f32"
    cfg = workload_config(sc, prm, B, M, P, 0 if joints is None else joints.count, args.settle, sname, int(prm.solver_iterations))
    cfg["note"] = "restated Avian CPU path (C++ oracle), not Avian itself: no Rust toolchain in this image"
    return {
        "impl": "reference", "metric": metric_name(args.scene), "value": cb["value"], "unit": "steps/s",
        "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": cb["ms_per_step"], "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": sname, "data": "synthetic", "config": cfg,
        "cpu_baseline": cb, "e2e": {"value": cb["value"], "unit": "steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--scene", default="stack100k", choices=sorted(SCENES))
    ap.add_argument("--settle", type=int, default=None, help="full pipeline steps before the snapshot is frozen (default: per scene)")
    ap.add_argument("--solver-iterations", type=int, default=1, help="EXTENSION: biased solve passes per substep (reference semantics = 1)")
    ap.add_argument("--cpu-steps", type=int, default=3, help="bounded CPU sample (full steps) for cpu_baseline")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-partition", action="store_true", help="skip the one-scene-over-N-GPUs arms")
    ap.add_argument("--no-pass", action="store_true", help="skip the single solver-pass roofline measurement")
    ap.add_argument("--no-resident", action="store_true", help="e2e = round 1's host-manifold arm only")
    ap.add_argument("--partition-steps", type=int, default=None, help="timed steps of the partition arms (default: --steps)")
    ap.add_argument("--partition-slab-scene", default="spheres1m", choices=sorted(SCENES))
    ap.add_argument("--partition-island-scene", default="ragdolls5k", choices=sorted(SCENES))
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the timed path computed in its last step as DIR/<name>.npy (float32/float64, at most 64 MB in all)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    args.warmup = max(args.warmup, 3) if args.impl == "b200" else args.warmup
    if args.partition_steps is None:
        args.partition_steps = args.steps
    if args.settle is None:
        args.settle = SCENES[args.scene][2]
    if args.scene != "stack100k":
        args.no_partition = True     # the partition arms accompany the headline run only

    from avian_b200 import parallel
    info = parallel.rank_info()
    if args.impl == "reference":
        res = run_reference(args, info.rank, info.world)
    else:
        if info.world > 1:
            import torch
            torch.cuda.set_device(info.local_rank)
            parallel.init(backend="nccl")
        res = run_gpu(args, info)
        if info.world > 1:
            import torch.distributed as dist
            dist.destroy_process_group()
    if res is not None:
        print(json.dumps(res))
        if isinstance(res.get("parity"), dict) and not res["parity"]["ok"]:
            sys.exit(1)


if __name__ == "__main__":
    main()
