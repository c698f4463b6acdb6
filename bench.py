#!/usr/bin/env python
"""bench.py -- physics steps/s on b3d_many_pyramids (3-D f32), BASELINE.json's metric, on BASELINE.json's
configs[1] (80 pyramids x 20 levels); the reference file's own 14 x 14 x 10 size is reported in `other_configs`.

  python bench.py --gpus 1 --steps K --warmup W            our CUDA path (one JSON line)
  python bench.py --impl reference --steps K --warmup W     CPU arm (oracle port, all host threads)
  torchrun --nproc-per-node N bench.py --gpus N ...         weak scaling: N x the scene, sharded by island

A "step" is one PhysicsPipeline::step of the whole scene.  `value` times steps with all state
resident in HBM (CUDA events on the launching stream, max over ranks); `e2e` times the same steps
through rb_world_step_host with HOST state buffers (H2D of every body state + D2H of the result in
the timed region).  The reference arm is the CPU oracle (`oracle/`, a scalar restatement -- the Rust
reference cannot be built in this image, see DESIGN.md), built -O3 -march=native on the host it runs on and run
with the thread count that is fastest for the scene (swept; the sweep is printed).

bench.py runs the library that `__graft_entry__.build()` left in the tree and writes nothing there (the CPU arm's
host-specific build goes to a temporary directory), so the tree may be read-only.  --dump-outputs DIR writes the body
poses and velocities the last timed step left, as DIR/<scene>_pose.npy (n x 7) and DIR/<scene>_vel.npy (n x 6), float32:
the scenes are fixed, so two builds run with the same arguments can be compared output for output.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

sys.dont_write_bytecode = True   # no __pycache__ in the tree
ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))


def scene_for(name, replicas=1):
    from rapier_b200 import scenes
    if name == "b3d_many_pyramids":
        # reference file examples3d/b3d_many_pyramids.rs: 14 x 14 pyramids, base 10 (10 780 cubes).
        # replicas > 1 (multi-GPU weak scaling): 14*replicas rows of the same arrangement.
        return scenes.pyramids(14 * replicas, 14, 10, name="b3d_many_pyramids" + (f"_x{replicas}" if replicas > 1 else ""))
    if name == "b3d_many_pyramids_80x20":
        return scenes.pyramids(8 * replicas, 10, 20, name="b3d_many_pyramids_80x20")
    return scenes.REGISTRY[name]()


class ClockSampler:
    """Samples nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md)."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index = index
        self.samples = []
        self.stop = False
        self.t = threading.Thread(target=self.run, daemon=True)

    def run(self):
        while not self.stop:
            try:
                out = subprocess.run(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}", "--format=csv,noheader,nounits"],
                                     capture_output=True, text=True, timeout=5).stdout.strip()
                if out:
                    self.samples.append([x.strip() for x in out.split(",")])
            except Exception:
                pass
            time.sleep(0.1)

    def __enter__(self):
        self.t.start()
        return self

    def __exit__(self, *a):
        self.stop = True
        self.t.join(timeout=6)

    def summary(self):
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for s in self.samples:
            try:
                sm.append(float(s[0]))
                mx.append(float(s[1]))
                for n, v in zip(names, s[3:7]):
                    if v.lower().startswith("active"):
                        reasons.add(n)
            except Exception:
                pass
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": max(mx), "reasons": sorted(reasons), "samples": len(sm)}


def host_threads():
    """Cores this process is allowed to run on."""
    try:
        n = len(os.sched_getaffinity(0))
    except Exception:
        n = os.cpu_count() or 1
    return max(1, n)


def best_cpu_world(scene, budget_s=8.0):
    """CPU arm: the oracle sources built as a BASELINE (-O3 -march=native, FMA contraction allowed: oracle/Makefile
    `fast`) on this host, with the thread count that runs this scene fastest -- swept over 1, 8, 16, 32, 64 and all
    cores, because the port's spin-wait stage barriers stop scaling (and then lose) beyond a scene-dependent count.
    Returns (world, threads, sweep) with the world already warmed up."""
    import oracle_lib
    allc = host_threads()
    cand = sorted({t for t in (1, 8, 16, 32, 64, allc) if t <= allc})
    sweep = {}
    best = None
    per = budget_s / max(len(cand), 1)
    for t in cand:
        w = oracle_lib.OracleWorld(scene, threads=t, fast=True)
        w.step(3)
        t0 = time.perf_counter()
        n = 0
        while n < 3 or (time.perf_counter() - t0 < per and n < 200):
            w.step(1)
            n += 1
        rate = n / (time.perf_counter() - t0)
        sweep[t] = round(rate, 2)
        if best is None or rate > best[1]:
            best = (t, rate)
        del w
    w = oracle_lib.OracleWorld(scene, threads=best[0], fast=True)
    w.step(3)
    return w, best[0], sweep


def csrc_sha1():
    """Hash of the kernel sources: ties profiles/traffic.json to the build it was measured on."""
    import hashlib
    h = hashlib.sha1()
    d = os.path.join(ROOT, "rapier_b200", "csrc")
    for f in sorted(os.listdir(d)):
        if f.endswith((".cu", ".cuh")):
            h.update(open(os.path.join(d, f), "rb").read())
    return h.hexdigest()


def algorithmic_bytes(m, b, j):
    """SURVEY.md 8(d) / BASELINE.md 4: streaming model, f32, twist friction, p = 4, S = 4."""
    return 12076 * m + 1608 * b + 6576 * j


def run_reference(args):
    """CPU arm: the oracle sources as a CPU baseline (see best_cpu_world)."""
    from rapier_b200 import scenes  # noqa: F401
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    scene = scene_for(args.scene, 1)
    w, cores, sweep = best_cpu_world(scene)
    # settle the first (broad-phase + full narrow-phase) steps outside the timed region, like the GPU arm
    w.step(max(args.warmup, 3))
    t0 = time.perf_counter()
    w.step(args.steps)
    dt = time.perf_counter() - t0
    c = w.counters()
    value = args.steps / dt
    line = {
        "impl": "reference", "metric": "physics steps/sec on b3d_many_pyramids (3D f32)", "value": value, "unit": "steps/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1000.0 * dt / args.steps,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": workload_name(args.scene, 1), "bodies": c["num_bodies"], "manifolds": c["num_active_manifolds"]},
        "cpu_baseline": {"value": value, "unit": "steps/s", "cores": cores, "kind": "port",
                         "sample": f"{args.steps} consecutive steps of the full scene after {max(args.warmup, 3)} warm-up steps; -O3 -march=native build of the oracle sources, best of the thread sweep",
                         "thread_sweep_steps_per_s": sweep, "host_cores": host_threads()},
        "e2e": {"value": value, "unit": "steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "note": "CPU restatement (oracle/), not the reference binary: no Rust toolchain in this image. value = steps/s of ONE replica of the workload on all host threads; under weak scaling (N replicas) a CPU's replica-steps/s stay the same, so it is the comparable whole-job figure for every N",
    }
    print(json.dumps(line), flush=True)


def workload_name(scene, replicas):
    base = {"b3d_many_pyramids": "b3d_many_pyramids (reference file examples3d/b3d_many_pyramids.rs: 14x14 pyramids, base 10, 10780 cubes)",
            "b3d_many_pyramids_80x20": "b3d_many_pyramids, BASELINE.json configs[1]: 80 pyramids x 20 levels = pyramids(8, 10, 20) of examples3d/b3d_many_pyramids.rs, 16800 cubes"}.get(scene, scene)
    return base if replicas == 1 else f"{replicas} x {base}, one replica per GPU"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=300)
    ap.add_argument("--warmup", type=int, default=30)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--scene", default="b3d_many_pyramids_80x20",
                    help="b3d_many_pyramids_80x20 = BASELINE.json configs[1] (headline); b3d_many_pyramids = the reference file's 14x14x10")
    ap.add_argument("--l2", default="flush", choices=["flush", "keep"])
    ap.add_argument("--cpu-seconds", type=float, default=12.0, help="budget of the cpu_baseline leg")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the body states of each timed scene after its last timed step to DIR/<scene>_{pose,vel}.npy")
    args = ap.parse_args()
    args.warmup = max(args.warmup, 3)
    if args.impl == "reference":
        run_reference(args)
        return

    import numpy as np
    import torch
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world_size = int(os.environ.get("WORLD_SIZE", "1"))
    if world_size != args.gpus:
        raise SystemExit(f"--gpus {args.gpus} but WORLD_SIZE={world_size}: launch with torchrun --nproc-per-node {args.gpus}")
    dist = None
    if world_size > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
        dist.barrier()
    torch.cuda.set_device(local_rank)
    from rapier_b200.world import PhysicsWorld

    scene = scene_for(args.scene, world_size)
    w = PhysicsWorld(scene, device=local_rank)
    w._flush()
    pipe = w.physics_pipeline
    stream = torch.cuda.current_stream()
    pipe.set_stream(stream.cuda_stream)
    nb = len(scene.bodies)
    gravity = scene.gravity

    # ---- multi-GPU: shard whole connected components (islands) across ranks ----
    exchange = None
    if world_size > 1:
        from rapier_b200.sharding import IslandShard
        shard = IslandShard(pipe, dist, rank, world_size, torch.device("cuda", local_rank),
                            refresh_every=int(os.environ.get("RB_SHARD_REFRESH", "128")))   # halo states every step, everything every 128 steps
        exchange = shard.exchange

    flush_buf = torch.empty(256 << 20, dtype=torch.uint8, device=f"cuda:{local_rank}") if args.l2 == "flush" else None

    def one_step():
        pipe.step(gravity, 1, sync=False)
        if exchange is not None:
            exchange()

    def timed_steps(k):
        """CUDA events around each step on the launching stream; L2 flushed between steps."""
        evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(k)]
        for a, b in evs:
            if flush_buf is not None:
                flush_buf.zero_()
            a.record(stream)
            one_step()
            b.record(stream)
        torch.cuda.synchronize()
        return sum(a.elapsed_time(b) for a, b in evs)

    def dump_outputs(name):
        """The body states as a caller of the timed path receives them (float32 pose n x 7, velocity n x 6)."""
        if args.dump_outputs and rank == 0:
            pose, vel = pipe.body_states()
            os.makedirs(args.dump_outputs, exist_ok=True)
            np.save(os.path.join(args.dump_outputs, f"{name}_pose.npy"), pose)
            np.save(os.path.join(args.dump_outputs, f"{name}_vel.npy"), vel)

    for _ in range(args.warmup):
        one_step()
    torch.cuda.synchronize()
    if dist is not None:
        dist.barrier()
    torch.cuda.synchronize()
    k0 = pipe.counters()["kernels_launched"]
    with ClockSampler(local_rank) as clk:
        ms = timed_steps(args.steps)
        k1 = pipe.counters()["kernels_launched"]
        torch.cuda.synchronize()
        if dist is not None:
            dist.barrier()
        # per-launch-group device times for the roofline (events inside the library, same stream)
        if exchange is not None:
            shard.finish()   # no gather may be in flight while steps run without exchange() in between
        dump_outputs(args.scene)   # after finish(): rank 0 holds the states of every body
        pipe.enable_profiling(True)
        prof = {"collision_detection_ms": 0.0, "solver_ms": 0.0}
        nprof = min(args.steps, 100)
        for _ in range(nprof):   # same conditions as the timed region: L2 flushed before every step
            if flush_buf is not None:
                flush_buf.zero_()
            pipe.step(gravity, 1, sync=True)
            c1 = pipe.counters()
            prof["collision_detection_ms"] += c1["collision_detection_ms"] / nprof
            prof["solver_ms"] += c1["solver_ms"] / nprof
        pipe.enable_profiling(False)
        # ---- e2e: host buffers in / out every step through the public C-ABI call ----
        if exchange is not None:
            shard.finish()
        e2e_steps = min(args.steps, 200)
        pose, vel = pipe.body_states()
        # host-side state buffers of the caller: page-locked (the library DMAs them directly)
        st_in = torch.empty((nb, 13), dtype=torch.float32, pin_memory=True).numpy()
        st_out = torch.empty((nb, 13), dtype=torch.float32, pin_memory=True).numpy()
        st_in[:] = np.concatenate([pose, vel], axis=1)
        for _ in range(3):
            pipe.step_host(gravity, st_in, st_out)
            st_in, st_out = st_out, st_in
        if dist is not None:
            dist.barrier()
        t0 = time.perf_counter()
        for _ in range(e2e_steps):
            pipe.step_host(gravity, st_in, st_out)
            st_in, st_out = st_out, st_in
            if exchange is not None:
                exchange()
        torch.cuda.synchronize()
        e2e_s = time.perf_counter() - t0
    clocks = clk.summary()
    shard_check = None
    if dist is not None:   # after draining the exchange every rank must hold bit-identical states of ALL bodies
        shard.finish()
        torch.cuda.synchronize()
        from rapier_b200.sharding import state_tensor
        mine = state_tensor(pipe, torch.device("cuda", local_rank)).clone()
        ref0 = mine.clone()
        dist.broadcast(ref0, src=0)
        diff = (mine.view(torch.int32) != ref0.view(torch.int32)).sum().to(torch.float64)
        dist.all_reduce(diff, op=dist.ReduceOp.MAX)
        shard_check = {"state_words_differing_from_rank0_max_over_ranks": int(diff.item()), "finite": bool(torch.isfinite(mine).all().item())}

    t = torch.tensor([ms, e2e_s], device=f"cuda:{local_rank}", dtype=torch.float64)
    if dist is not None:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms, e2e_s = float(t[0]), float(t[1])

    c = pipe.counters()
    per_rank_bodies = (nb - 1) // world_size
    M = c["num_active_manifolds"]
    # whole-job value: steps of the base scene per second (each rank advances one base-scene replica per step)
    value = world_size * args.steps / (ms / 1000.0)
    e2e_value = world_size * e2e_steps / e2e_s
    solve_ms = prof["solver_ms"]
    a_bytes = algorithmic_bytes(M, per_rank_bodies, 0)
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    peak = float(peaks.get("hbm_gbs", 6650.0))
    achieved = a_bytes / (solve_ms * 1e-3) / 1e9 if solve_ms > 0 else None
    traffic = None
    st = pipe.debug_read("state", np.int32)
    kernel_name = "k_solve_coop_big" if int(st[19]) > 0 else "k_solve_coop"   # streamed items => the big launch shape ran
    try:   # ncu dram bytes of THIS build (profiles/traffic.json carries the hash of the kernel sources it was captured from), else null
        tj = json.load(open(os.path.join(ROOT, "profiles", "traffic.json")))
        if tj.get("csrc_sha1") == csrc_sha1():
            traffic = tj.get(f"{kernel_name}_dram_bytes_per_launch:{args.scene}")
    except Exception:
        pass

    # the reference file's own size of the same scene (14 x 14 pyramids of base 10), reported beside the headline
    other = None
    if world_size == 1 and args.scene == "b3d_many_pyramids_80x20":
        del w
        w2 = PhysicsWorld(scene_for("b3d_many_pyramids", 1), device=local_rank)
        w2._flush()
        pipe = w2.physics_pipeline
        pipe.set_stream(stream.cuda_stream)
        for _ in range(args.warmup):
            one_step()
        torch.cuda.synchronize()
        k2 = min(args.steps, 100)
        ms2 = timed_steps(k2)
        dump_outputs("b3d_many_pyramids")
        c2 = pipe.counters()
        other = {"workload": workload_name("b3d_many_pyramids", 1), "value": k2 / (ms2 / 1000.0), "unit": "steps/s",
                 "ms_per_step": ms2 / k2, "steps": k2, "bodies": c2["num_bodies"] - 1, "manifolds": c2["num_active_manifolds"]}

    if rank == 0:
        cpu = None
        try:
            ow, cores, sweep = best_cpu_world(scene_for(args.scene, 1))
            t0 = time.perf_counter()
            n = 0
            while time.perf_counter() - t0 < args.cpu_seconds and n < 400:
                ow.step(5)
                n += 5
            cdt = time.perf_counter() - t0
            cpu = {"value": n / cdt, "unit": "steps/s", "cores": cores, "kind": "port",
                   "sample": f"{n} consecutive steps of the full {args.scene} scene (after warm-up), oracle sources built -O3 -march=native, {cores} host threads = best of the sweep",
                   "thread_sweep_steps_per_s": sweep, "host_cores": host_threads()}
        except Exception as e:  # the oracle is a checker, its absence must not hide the GPU number
            cpu = {"value": None, "unit": "steps/s", "cores": 0, "kind": "port", "sample": f"unavailable: {e}"}
        line = {
            "metric": "physics steps/sec on b3d_many_pyramids (3D f32)", "value": value, "unit": "steps/s",
            "n_gpus": world_size, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms / args.steps,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": workload_name(args.scene, world_size), "bodies_per_gpu": per_rank_bodies,
                       "manifolds_per_gpu": M, "substeps": 4, "sweeps_per_substep": 3,
                       "l2": "flushed between steps (256 MiB memset)" if args.l2 == "flush" else "not flushed",
                       "parallelism": "1 GPU" if world_size == 1 else f"islands sharded over {world_size} GPUs; NCCL all-gather of the boundary (halo) body states every step -- none in this scene: {shard.halo_steps} steps needed it --, of all body states every {shard.refresh_every} steps and at the end"},
            "e2e": {"value": e2e_value, "unit": "steps/s", "h2d_bytes_per_step": nb * 13 * 4, "d2h_bytes_per_step": nb * 13 * 4,
                    "steps": e2e_steps},
            "gpu_launches": int(k1 - k0),
            "clocks": clocks,
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s",
                         "frac": (achieved / peak) if achieved else None, "traffic": traffic,
                         "kernel": kernel_name, "kernel_ms": solve_ms, "algorithmic_bytes_per_launch": a_bytes,
                         "peak_source": "MEASURED_PEAKS.json hbm_gbs (of measured)" if peaks else "fallback 6650 GB/s (of fallback)",
                         "note": "algorithmic bytes = streaming model of SURVEY 8(d); the working set is L2/shared-memory resident, see DESIGN.md"},
            "cpu_baseline": cpu,
            "stage_ms": {"collide": prof["collision_detection_ms"], "solve": prof["solver_ms"]},
            "other_configs": [other] if other else [],
            "shard_check": shard_check,
        }
        print(json.dumps(line), flush=True)
    if dist is not None:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
