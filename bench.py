#!/usr/bin/env python
"""bench.py - headline benchmark: env-steps/s of the collide -> SolverXPBD.step substep loop.

Workload (BASELINE.json configs[2], the config the metric is quoted on): 4096 Anymal-class quadruped
environments (13 bodies / 13 joints / 18 dofs each, vendored-URDF topology built by newton_b200.scenes),
SolverXPBD(iterations=8), 4 substeps per frame at 50 fps (dt = 5 ms), fp32, synthetic per-env perturbation
(default_rng(1)).  One bench "step" = one frame = 4 x (clear_forces, collide, solver.step, swap) for every env,
replayed as one CUDA graph exactly as the reference examples do (example_basic_urdf.py:112-143).

  python bench.py --gpus N --steps K --warmup W          # N>1: launched by torchrun, one rank per GPU
  python bench.py --impl reference ...                   # the CPU oracle (reference restatement) on host cores
  python bench.py ... --dump-outputs DIR                 # also writes the last timed frame's state and contacts as DIR/<name>.npy

Prints ONE JSON line (see the task contract): whole-job env-steps/s, e2e (host buffers through the public API),
roofline of the dominant kernel, cpu_baseline, clocks.
"""

from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

ENVS_PER_GPU = 4096
ITERATIONS = 8
METRIC = "env_steps_per_sec"
UNIT = "env-steps/s"

# The headline (default) workload is BASELINE.json configs[2]; the other two configs that fit one GPU are selectable
# with --workload for the per-config numbers recorded in profiles/ (they are not the bench line the driver reads).
WORKLOADS = {
    "quadruped_xpbd": dict(
        config="BASELINE.json configs[2]", scene="quadruped", solver="xpbd", envs=4096, substeps=4, fps=50, kernel="xpbd_step_kernel",
        text="quadruped (Anymal-class, 13 bodies/18 dofs) envs, SolverXPBD iterations=8",
        # SURVEY.md §8(d): B_state 1884 (state in 13 x 76 B + out 13 x 52 B + control 220 B) + one read of each 80-byte
        # contact + B_model 4001 (per-env model constants: the reference layout replicates them per world and the kernel
        # reads them every substep)
        alg_bytes=lambda n_c: 1884.0 + 80.0 * n_c + 4001.0, model_bytes=4001.0),
    "quadruped_xpbd_stock": dict(
        config="BASELINE.json configs[2] scene with the stock example's loop (example_basic_urdf.py:28-33: 100 fps, 10 substeps, "
               "iterations=2)", scene="quadruped", solver="xpbd", envs=4096, substeps=10, fps=100, iterations=2,
        kernel="xpbd_step_kernel", text="quadruped (Anymal-class, 13 bodies/18 dofs) envs, SolverXPBD iterations=2",
        alg_bytes=lambda n_c: 1884.0 + 80.0 * n_c + 4001.0, model_bytes=4001.0),
    "box_stacks_xpbd": dict(
        config="BASELINE.json configs[1]", scene="stacks", solver="xpbd", envs=512, substeps=4, fps=60, kernel="xpbd_step_kernel",
        text="5-box stack envs (box-box MPR manifolds + plane-box), SolverXPBD iterations=8",
        alg_bytes=lambda n_c: 5 * 76.0 + 5 * 52.0 + 80.0 * n_c + 5 * 100.0, model_bytes=500.0),
    "quadruped_featherstone": dict(
        config="BASELINE.json configs[3]", scene="quadruped", solver="featherstone", envs=4096, substeps=10, fps=100,
        kernel="featherstone_step_kernel",
        text="quadruped (Anymal-class, 13 bodies/18 dofs) envs, SolverFeatherstone (dense H = J^T M J, Cholesky), penalty contacts",
        # joint_q/qd in+out (2 x 148 B) + body_f in (312) + body_q/qd out (676) + control (220) + 112-byte contacts + B_model
        alg_bytes=lambda n_c: 296.0 + 312.0 + 676.0 + 220.0 + 112.0 * n_c + 4001.0, model_bytes=4001.0),
}
WL = WORKLOADS["quadruped_xpbd"]
SUBSTEPS = WL["substeps"]
FPS = WL["fps"]
DT = 1.0 / FPS / SUBSTEPS


def select_workload(name):
    global WL, SUBSTEPS, FPS, DT
    WL = WORKLOADS[name]
    SUBSTEPS, FPS = WL["substeps"], WL["fps"]
    DT = 1.0 / FPS / SUBSTEPS


def build_scene(envs, seed):
    from newton_b200 import scenes

    if WL["scene"] == "quadruped":
        return scenes.quadruped_model(envs, device="cpu", seed=seed)
    return scenes.box_stack_model(envs, device="cpu", seed=seed)


def make_solver(pkg, model):
    """pkg is newton_b200.solvers (product) or the oracle module (CPU checker)."""
    if WL["solver"] == "xpbd":
        return pkg.SolverXPBD(model, iterations=WL.get("iterations", ITERATIONS))
    return pkg.SolverFeatherstone(model)


def parse_args():
    p = argparse.ArgumentParser()
    p.add_argument("--gpus", type=int, default=1)
    p.add_argument("--steps", type=int, default=1000)
    p.add_argument("--warmup", type=int, default=20)
    p.add_argument("--impl", default="native", choices=["native", "reference"])
    p.add_argument("--envs", type=int, default=None, help="environments per GPU (weak scaling); default: the workload's")
    p.add_argument("--workload", default="quadruped_xpbd", choices=sorted(WORKLOADS))
    p.add_argument("--fast-fp", action="store_true", help="use the FMA-contracted twin library (not bit-exact vs the oracle)")
    p.add_argument("--no-cpu-baseline", action="store_true")
    p.add_argument("--no-fast-twin", action="store_true", help="skip the secondary measurement with the FMA-contracted twin library")
    p.add_argument("--no-export-contacts", action="store_true",
                   help="CollisionPipeline(export_contacts=False): the solver reads the contact blocks, the reference-layout Contacts arrays "
                        "are not written (an RL loop that never looks at them); NOT the default, the headline keeps the export")
    p.add_argument("--gather", default="peer", choices=["peer", "nccl"], help="N > 1: end-of-frame state gather mechanism")
    p.add_argument("--dump-outputs", metavar="DIR", default=None,
                   help="after the timed steps, write what the last timed step computed as DIR/<name>.npy, for comparing two builds")
    a = p.parse_args()
    if a.steps < 1:
        p.error("--steps must be at least 1")
    select_workload(a.workload)
    if a.envs is None:
        a.envs = WL["envs"]
    return a


def workload_config(envs, n_gpus):
    return {
        "workload": f"{envs * n_gpus} {WL['text']}, "
                    f"{SUBSTEPS} substeps/frame @ {FPS} fps, explicit broad phase, ground plane; {WL['config']}"
                    + ("" if n_gpus == 1 else f" sharded {envs}/GPU (configs[4] layout)"),
        "envs_per_gpu": envs,
        "substeps_per_step": SUBSTEPS,
        "iterations": WL.get("iterations", ITERATIONS) if WL["solver"] == "xpbd" else None,
        "dt": DT,
        "parallelism": f"env-sharded x{n_gpus}" if n_gpus > 1 else "single GPU",
        "l2": "flushed between timed steps (256 MiB memset outside the timed events)",
    }


# ------------------------------------------------------------------------------------------------ clocks
class ClockSampler:
    """Samples nvidia-smi during the timed region (profiling recipe's clocks line)."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.gpu = gpu_index
        self.proc = None
        self.lines: list[str] = []

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100", "-i", str(self.gpu)],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True,
            )
            threading.Thread(target=self._pump, daemon=True).start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self) -> dict:
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm, smax, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1]))
                smax.append(float(f[2]))
            except ValueError:
                continue
            for name, val in zip(names, f[5:9]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        return {
            "sm_mhz": float(np.median(sm)) if sm else None,
            "sm_max_mhz": float(max(smax)) if smax else None,
            "samples": len(sm),
            "reasons": sorted(reasons),
        }


# ------------------------------------------------------------------------------------------------ native arm
def run_native(args):
    import torch.distributed as dist

    if args.fast_fp:  # the library is chosen when newton_b200._lib is imported: set the switch BEFORE the import
        os.environ.pop("NB2_LIB", None)
        os.environ["NB2_FP"] = "fast"
    import newton_b200
    from newton_b200 import _lib, scenes

    if args.fast_fp:
        assert _lib.LIB_PATH.endswith("libnewton_b200_fast.so"), _lib.LIB_PATH

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if world != args.gpus:
        if world == 1 and args.gpus > 1:
            raise SystemExit("--gpus N > 1 must be launched through torch.distributed.run (one rank per GPU)")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    envs = args.envs
    # every rank owns `envs` worlds (weak scaling); per-rank seed so shards differ like slices of one big scene
    model = build_scene(envs, seed=1 + rank).to(dev)
    pipeline = newton_b200.CollisionPipeline(model, export_contacts=not args.no_export_contacts)
    solver = make_solver(newton_b200.solvers, model)
    state_0, state_1 = model.state(), model.state()
    control = model.control()
    contacts = pipeline.contacts()

    def simulate():
        nonlocal state_0, state_1
        for _ in range(SUBSTEPS):
            state_0.clear_forces()
            pipeline.collide(state_0, contacts)
            solver.step(state_0, state_1, control, contacts, DT)
            state_0, state_1 = state_1, state_0

    # settle the robots on the ground first (untimed) so the timed frames carry the steady-state contact load
    stream = torch.cuda.Stream(device=dev)
    with torch.cuda.stream(stream):
        for _ in range(int(round(1.2 * FPS))):  # 1.2 s of simulated time
            simulate()
    torch.cuda.synchronize()
    launches_before = _lib.kernel_launch_count()
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph, stream=stream):
        simulate()
    launches_per_step = _lib.kernel_launch_count() - launches_before  # kernels captured in one frame graph
    assert SUBSTEPS % 2 == 0  # state_0/state_1 swap parity: the graph ends where it began

    gathered_q = gathered_qd = snap_q = snap_qd = None
    pending = []  # NCCL work handles of the previous frame's gather
    peer = None
    gather_mode = "none"
    if world > 1:  # end-of-frame state gather over NVLink (SURVEY.md §8(e)); part of every timed step
        if args.gather == "peer":
            try:
                from newton_b200.sim.sharding import PeerStateGather

                peer = PeerStateGather([state_0.body_q, state_0.body_qd])
                gather_mode = "peer writes on the copy engines (nb2_peer_gather_*: CUDA IPC + cudaMemcpyAsync + stream wait-value)"
            except Exception as e:  # no P2P / IPC on this box: the NCCL path below still gives a valid number
                peer = None
                print(f"[bench] peer gather unavailable ({type(e).__name__}: {e}); falling back to NCCL", file=sys.stderr)
            ok = torch.tensor([1 if peer is not None else 0], device=dev)
            dist.all_reduce(ok, op=dist.ReduceOp.MIN)
            if int(ok.item()) == 0:
                peer = None
        if peer is None:
            gather_mode = "NCCL all_gather_into_tensor"
            gathered_q = torch.empty((world * state_0.body_q.shape[0], 7), dtype=torch.float32, device=dev)
            gathered_qd = torch.empty((world * state_0.body_qd.shape[0], 6), dtype=torch.float32, device=dev)
            snap_q, snap_qd = torch.empty_like(state_0.body_q), torch.empty_like(state_0.body_qd)

    def drain():
        if peer is not None:
            peer.wait()  # stream-level wait until every rank's slice of the last push has landed here
            return
        for w in pending:
            w.wait()  # stream-level wait (no host sync)
        pending.clear()

    def step_device():
        """One frame.  N > 1: the frame's body_q / body_qd are snapshotted (2.8 MB D2D) and gathered on a side stream while the
        next frame computes (SURVEY.md §8(e): "on a dedicated stream, overlapped with the next frame"); the snapshot is recycled
        only after the previous gather has read it, and the last gather is drained inside the timed region."""
        graph.replay()
        if world > 1:
            if peer is not None:
                peer.push([state_0.body_q, state_0.body_qd])
                return
            drain()
            snap_q.copy_(state_0.body_q)
            snap_qd.copy_(state_0.body_qd)
            pending.append(dist.all_gather_into_tensor(gathered_q, snap_q, async_op=True))
            pending.append(dist.all_gather_into_tensor(gathered_qd, snap_qd, async_op=True))

    flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device=dev)
    extra_drains = []  # stream-level waits appended to drain() (the pipelined e2e loop's last download)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps, warmup, sampler=None):
        if sampler:
            sampler.start()  # before the warm-up and the barrier: forking nvidia-smi costs rank 0 several ms - inside the synchronised
            #                  region that start-up skew is what every other rank then waits for in the final drain (N = 4: 5 ms / 50 frames)
        for _ in range(warmup):
            fn()
        barrier()
        ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
        for a, b in ev:
            flush.zero_()  # evict L2 (126 MB) between timed steps; not inside the timed events
            a.record()
            fn()
            b.record()
        d0, d1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        d0.record()
        drain()  # the last frame's gather is part of the job
        for f in extra_drains:
            f()
        d1.record()
        barrier()
        clocks = sampler.stop() if sampler else None
        per_step = [a.elapsed_time(b) for a, b in ev]
        per_step[-1] += d0.elapsed_time(d1)
        timed.last_per_step = per_step
        ms = sum(per_step)
        t = torch.tensor([ms], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item()), clocks

    sampler = ClockSampler(local_rank) if rank == 0 else None
    total_ms, clocks = timed(step_device, args.steps, max(args.warmup, 3), sampler)
    outputs = None
    if args.dump_outputs and rank == 0:  # taken now: the e2e and kernel timings below keep stepping the simulation
        if world == 1:
            body_q, body_qd = state_0.body_q, state_0.body_qd
        elif peer is not None:
            body_q, body_qd = (g.reshape(-1, g.shape[-1]) for g in peer.gathered())
        else:
            body_q, body_qd = gathered_q, gathered_qd
        outputs = last_step_outputs(body_q, body_qd, state_0, contacts if pipeline.export_contacts else None)
    env_steps = envs * world * SUBSTEPS * args.steps
    value = env_steps / (total_ms * 1e-3)
    frame_ms = np.asarray(timed.last_per_step)  # rank-local per-frame device times (SURVEY.md §8(d) extras)
    extras = {
        "us_per_substep": float(total_ms / args.steps / SUBSTEPS * 1e3),
        "p50_frame_ms": float(np.percentile(frame_ms, 50)), "p95_frame_ms": float(np.percentile(frame_ms, 95)),
        "realtime_factor": float((1.0 / FPS) / (total_ms / args.steps * 1e-3)),
    }

    # ---- e2e: host buffers through the public API (H2D of the step's control inputs, D2H of the resulting state)
    h_target = model.joint_target_q.cpu().pin_memory()
    h_jf = torch.zeros_like(control.joint_f, device="cpu").pin_memory()
    h_q = torch.empty_like(state_0.body_q, device="cpu").pin_memory()
    h_qd = torch.empty_like(state_0.body_qd, device="cpu").pin_memory()

    def step_e2e_serial():
        """everything in stream order: H2D of the inputs, the frame, D2H of the result"""
        control.joint_target_q.copy_(h_target, non_blocking=True)
        control.joint_f.copy_(h_jf, non_blocking=True)
        step_device()
        h_q.copy_(state_0.body_q, non_blocking=True)
        h_qd.copy_(state_0.body_qd, non_blocking=True)

    # Pipelined variant (what a training loop does): the PCIe copies ride on two copy streams - the inputs of frame k+1 go up into a
    # device staging buffer while frame k computes, the result of frame k comes down from a device snapshot while frame k+1 computes.
    # Every frame's inputs are still copied from pinned host memory and every frame's result still lands in pinned host memory
    # inside the timed region (the last download is drained before the clock stops).  On the compute stream a frame pays two
    # device-to-device copies of the controls (0.6 MB) and two of the state snapshot (2.8 MB) instead of the PCIe time.
    up, down = torch.cuda.Stream(device=dev), torch.cuda.Stream(device=dev)
    st_target, st_jf = torch.empty_like(control.joint_target_q), torch.empty_like(control.joint_f)
    e2e_snap_q, e2e_snap_qd = torch.empty_like(state_0.body_q), torch.empty_like(state_0.body_qd)
    ev_up_done, ev_stage_free = torch.cuda.Event(), torch.cuda.Event()
    ev_snap_ready, ev_down_done = torch.cuda.Event(), torch.cuda.Event()
    pipe = {"primed": False}

    def upload_next():
        up.wait_event(ev_stage_free)  # the compute stream has consumed the previous staging contents
        with torch.cuda.stream(up):
            st_target.copy_(h_target, non_blocking=True)
            st_jf.copy_(h_jf, non_blocking=True)
            ev_up_done.record(up)

    def step_e2e_pipelined():
        main = torch.cuda.current_stream()
        if not pipe["primed"]:
            ev_stage_free.record(main)
            ev_down_done.record(down)
            upload_next()
            pipe["primed"] = True
        main.wait_event(ev_up_done)  # this frame's inputs are on the device
        control.joint_target_q.copy_(st_target, non_blocking=True)
        control.joint_f.copy_(st_jf, non_blocking=True)
        ev_stage_free.record(main)
        upload_next()  # the NEXT frame's inputs travel while this frame computes
        step_device()
        main.wait_event(ev_down_done)  # the previous download has finished reading the snapshot
        e2e_snap_q.copy_(state_0.body_q, non_blocking=True)
        e2e_snap_qd.copy_(state_0.body_qd, non_blocking=True)
        ev_snap_ready.record(main)
        down.wait_event(ev_snap_ready)
        with torch.cuda.stream(down):
            h_q.copy_(e2e_snap_q, non_blocking=True)
            h_qd.copy_(e2e_snap_qd, non_blocking=True)
            ev_down_done.record(down)

    def drain_e2e():
        torch.cuda.current_stream().wait_event(ev_down_done)  # the last frame's result is in host memory
        torch.cuda.current_stream().wait_event(ev_up_done)

    e2e_serial_ms, _ = timed(step_e2e_serial, args.steps, 3)
    extra_drains.append(drain_e2e)
    e2e_ms, _ = timed(step_e2e_pipelined, args.steps, 3)
    extra_drains.clear()
    torch.cuda.synchronize()
    assert torch.equal(h_q, state_0.body_q.cpu()), "pipelined e2e: the downloaded state is not the last frame's"
    e2e_value = env_steps / (e2e_ms * 1e-3)
    h2d = h_target.numel() * 4 + h_jf.numel() * 4
    d2h = h_q.numel() * 4 + h_qd.numel() * 4

    # ---- roofline of the dominant kernel (the fused solver kernel): CUDA events around single launches on this stream
    n_c = float(contacts.rigid_contact_count.item()) / envs
    reps = 40
    evs = []
    for _ in range(5):
        pipeline.collide(state_0, contacts)
        solver.step(state_0, state_1, control, contacts, DT)
    for _ in range(reps):
        # same cache state as inside a frame (collide has just written the contact blocks): the kernel's share of the frame
        # then matches the ncu launch list (profiles/*launch_list*); the frame-level timing above is the L2-flushed one
        pipeline.collide(state_0, contacts)
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        solver.step(state_0, state_1, control, contacts, DT)
        b.record()
        evs.append((a, b))
    torch.cuda.synchronize()
    kern_ms = float(np.mean([a.elapsed_time(b) for a, b in evs]))
    # algorithmic bytes per env-substep of the solver kernel (SURVEY.md §8(d), DESIGN.md §6); the matching contact
    # write belongs to the collide kernel
    alg_bytes_env = WL["alg_bytes"](n_c)
    achieved = alg_bytes_env * envs / (kern_ms * 1e-3) / 1e9
    peaks = {}
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            peaks = json.load(f)
    except Exception:
        pass
    peak = float(peaks.get("hbm_gbs", 6650.0))
    # measured DRAM traffic of ONE launch of the dominant kernel: dram__bytes_read.sum + dram__bytes_write.sum of the committed
    # `ncu --set full` capture for this workload (profiles/traffic.json names the report it was read from); null when no capture
    # of the current kernel at this size is committed
    traffic = traffic_src = None
    try:
        with open(os.path.join(ROOT, "profiles", "traffic.json")) as f:
            t = json.load(f).get(f"{args.workload}:{envs}")
        if t:
            traffic, traffic_src = float(t["dram_bytes"]), t["source"]
    except Exception:
        pass
    no_model = (alg_bytes_env - WL["model_bytes"]) * envs / (kern_ms * 1e-3) / 1e9
    roofline = {
        "bound": "hbm", "kernel": WL["kernel"], "achieved": achieved, "peak": peak, "unit": "GB/s",
        "frac": achieved / peak, "traffic": traffic, "traffic_source": traffic_src,
        "peak_source": "measured" if peaks else "fallback",
        "algorithmic_bytes_per_env_substep": alg_bytes_env, "kernel_ms": kern_ms, "contacts_per_env": n_c,
        # SURVEY.md §8(d) asks for both: with the per-env model constants (read every substep; what DRAM traffic shows) and
        # without them (state + control + contacts only)
        "achieved_no_model_constants": no_model, "frac_no_model_constants": no_model / peak,
        "algorithmic_bytes_no_model_constants": alg_bytes_env - WL["model_bytes"],
        "kernel_share_of_step": kern_ms * SUBSTEPS / (total_ms / args.steps),
    }

    cpu_baseline = None
    if rank == 0 and not args.no_cpu_baseline:
        cpu_baseline = oracle_throughput(envs, frames=20, threads=host_threads()[0])

    # Secondary figure, N = 1 only: the same workload on the FMA-contracted twin library (NB2_FP=fast - same sources, nvcc's default
    # contraction; contact counts identical and body_q within the north-star's 1e-5 after 100 substeps, tests/test_gpu_fast_fp.py),
    # measured in a child process because a process loads one library.  The headline `value` stays the strict, bit-exact build.
    fast_twin = None
    if rank == 0 and world == 1 and not args.fast_fp and not args.no_fast_twin:
        fast_twin = fast_twin_measurement(args, envs)

    if rank == 0:
        out = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3),
            "ms_per_step": total_ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic", "config": workload_config(envs, world), "impl": "native",
            "fp_mode": "fast(fma)" if args.fast_fp else "strict (bit-exact vs oracle)",
            "contacts_exported": not args.no_export_contacts,
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                    "ms_per_step": e2e_ms / args.steps, "mode": "copies pipelined on two copy streams (inputs of frame k+1 up / result of "
                    "frame k down while a frame computes; last download drained inside the timed region)",
                    "serial_value": env_steps / (e2e_serial_ms * 1e-3), "serial_ms_per_step": e2e_serial_ms / args.steps},
            "gpu_launches": int(launches_per_step * args.steps),
            "gpu_launches_per_step": int(launches_per_step), "frame_stats": extras,
            "roofline": roofline, "cpu_baseline": cpu_baseline, "clocks": clocks, "fast_fp": fast_twin,
            "comm": {"backend": "nccl" if world > 1 else None, "nranks": world, "gather": gather_mode,
                     "gather_bytes_per_rank_per_step": int(state_0.body_q.numel() * 4 + state_0.body_qd.numel() * 4) if world > 1 else 0},
        }
        if outputs is not None:
            write_outputs(args.dump_outputs, outputs)
        print(json.dumps(out))
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


CONTACT_FIELDS = ("shape0", "shape1", "point0", "point1", "offset0", "offset1", "normal", "margin0", "margin1")
DUMP_BYTES = 60 << 20  # leaves room for the .npy headers under 64 MB in all


def last_step_outputs(body_q, body_qd, state, contacts):
    """Host copies of what a caller of the timed frame receives: the body state (gathered over all ranks when N > 1), the joint
    state for Featherstone (XPBD does not write it) and, when exported, the last substep's contacts of this rank.  The contacts
    are put in (shape0, shape1, emission) order, so a build that emits the same contacts in another order compares equal."""
    out = {"body_q": body_q, "body_qd": body_qd}
    if WL["solver"] == "featherstone":
        out["joint_q"], out["joint_qd"] = state.joint_q, state.joint_qd
    out = {k: v.cpu().numpy() for k, v in out.items()}
    if contacts is not None:
        n = min(int(contacts.rigid_contact_count.item()), contacts.rigid_contact_max)
        c = {k: getattr(contacts, "rigid_contact_" + k)[:n].cpu().numpy() for k in CONTACT_FIELDS}
        order = np.lexsort((np.arange(n), c["shape1"], c["shape0"]))
        out["contact_count"] = np.array([n])
        out.update({"contact_" + k: v[order] for k, v in c.items()})
    return {k: v if v.dtype == np.float32 else v.astype(np.float64) for k, v in out.items()}


def write_outputs(directory, outputs):
    """``DIR/<name>.npy`` for every output.  Above DUMP_BYTES in all, each array keeps the same share of its rows, chosen by a
    fixed seed from its length alone: arrays of one length (the contact fields) keep the same rows, and two runs the same sample."""
    total = sum(v.nbytes for v in outputs.values())
    keep = min(1.0, DUMP_BYTES / total) if total else 1.0
    os.makedirs(directory, exist_ok=True)
    for name, v in outputs.items():
        if keep < 1.0 and len(v) > 1:
            v = v[np.sort(np.random.default_rng(0).choice(len(v), int(len(v) * keep), replace=False))]
        np.save(os.path.join(directory, name + ".npy"), v)


def fast_twin_measurement(args, envs):
    import subprocess

    steps = int(args.steps)
    cmd = [sys.executable, os.path.abspath(__file__), "--fast-fp", "--steps", str(steps), "--warmup", str(max(args.warmup, 3)),
           "--workload", args.workload, "--envs", str(envs), "--no-cpu-baseline", "--no-fast-twin"]
    if args.no_export_contacts:
        cmd.append("--no-export-contacts")
    try:
        env = dict(os.environ)
        env.pop("NB2_LIB", None)
        p = subprocess.run(cmd, capture_output=True, text=True, timeout=300, env=env, cwd=ROOT)
        line = [ln for ln in p.stdout.splitlines() if ln.startswith("{")][-1]
        r = json.loads(line)
        return {"value": r["value"], "unit": r["unit"], "e2e_value": r["e2e"]["value"], "ms_per_step": r["ms_per_step"],
                "kernel_ms": r["roofline"]["kernel_ms"], "steps": steps, "library": "libnewton_b200_fast.so (NB2_FP=fast)",
                "parity": "contact counts identical, body_q within 1e-5 relative after 100 substeps vs the oracle "
                          "(tests/test_gpu_fast_fp.py); NOT the headline"}
    except Exception as e:  # noqa: BLE001 - a missing secondary figure must not cost the headline
        return {"unavailable": f"{type(e).__name__}: {e}"[:200]}


# ------------------------------------------------------------------------------------------------ CPU arm
def host_threads() -> tuple[int, float | None]:
    """(threads to use, CPU quota of this container in cores or None).  The GPU boxes report 128 logical CPUs but run the
    container under a CFS quota (cpu.max, measured 16 cores): more runnable threads than the quota only add throttling stalls."""
    n = os.cpu_count() or 1
    quota = None
    try:
        with open("/sys/fs/cgroup/cpu.max") as f:
            a, b = f.read().split()
        if a != "max":
            quota = float(a) / float(b)
    except Exception:
        pass
    try:
        n = min(n, len(os.sched_getaffinity(0)))
    except Exception:
        pass
    if quota is not None:
        n = max(1, min(n, int(round(quota))))
    return n, quota


ENVS_PER_SHARD = 32  # >= 32 environments per unit of CPU work; shards are handed to the threads dynamically


class CpuArm:
    """The reference's CPU path for the SAME workload (all `envs` environments of the stated config): the oracle - a C++
    restatement of the reference's Warp-CPU kernels - running the substep loop of independent world shards on a persistent
    pool of native threads (oracle.FramePool, created and settled BEFORE any timer; no Python inside the timed region)."""

    def __init__(self, envs: int, threads: int):
        import oracle

        oracle.build()
        base = build_scene(envs, seed=1)
        n_shards = max(1, envs // ENVS_PER_SHARD)
        while envs % n_shards:  # Model.shard splits the world range evenly
            n_shards -= 1
        self.envs, self.threads, self.n_shards = envs, max(1, min(threads, n_shards)), n_shards
        models = [base.shard(r, n_shards) for r in range(n_shards)] if n_shards > 1 else [base]
        self.pool = oracle.FramePool(models, lambda m: make_solver(oracle, m), substeps=SUBSTEPS, dt=DT, threads=self.threads)
        # one more pool with a single thread over ONE shard: what the reference's Warp-CPU device gives (kernels run serially
        # on one host thread, SURVEY.md §8(d))
        self.single = oracle.FramePool(models[:1], lambda m: make_solver(oracle, m), substeps=SUBSTEPS, dt=DT, threads=1)
        self.single_envs = envs // n_shards
        self.settled = False

    def settle(self):
        """Same untimed lead-in as the native arm: 1.2 s of simulated time so the timed frames carry standing contacts."""
        if not self.settled:
            n = int(round(1.2 * FPS))
            self.pool.run_frames(n)
            self.single.run_frames(n)
            self.settled = True

    def frame(self) -> float:
        """One frame (= one bench step) of all envs; returns seconds."""
        return self.pool.run_frames(1)

    def describe(self, value, seconds, frames, single_value) -> dict:
        phys = None
        try:
            import psutil

            phys = psutil.cpu_count(logical=False)
        except Exception:
            pass
        return {
            "value": value, "unit": UNIT, "cores": self.threads, "physical_cores": phys, "logical_cpus": os.cpu_count(),
            "cpu_quota_cores": host_threads()[1], "kind": "port",
            "all_cores": value, "single_thread": single_value,
            "sample": f"{self.envs} envs x {frames} frames x {SUBSTEPS} substeps of the bench workload (same scene, seed and solver "
                      f"settings, settled 1.2 s first), oracle C++ port of the reference kernels; {self.n_shards} shards of "
                      f"{self.envs // self.n_shards} envs on a persistent pool of {self.threads} native threads (no Python in the timed "
                      f"region); single_thread = one shard of {self.single_envs} envs on one thread; the reference itself (Warp) "
                      f"cannot run here",
            "seconds": seconds,
        }

    def single_thread_value(self, frames: int) -> float:
        sec = self.single.run_frames(frames)
        return self.single_envs * SUBSTEPS * frames / sec

    def close(self):
        self.pool.close()
        self.single.close()


def oracle_throughput(envs: int, frames: int, threads: int) -> dict:
    """cpu_baseline of the native arm: `frames` timed frames of the full workload on all host threads (bounded: 4096 envs x
    20 frames x 4 substeps is ~20 s of CPU work)."""
    arm = CpuArm(envs, threads)
    arm.settle()
    for _ in range(2):
        arm.frame()
    sec = sum(arm.frame() for _ in range(frames))
    single = arm.single_thread_value(max(2, frames // 4))
    out = arm.describe(envs * SUBSTEPS * frames / sec, sec, frames, single)
    arm.close()
    return out


def run_reference(args):
    """`--impl reference`: the same config, metric and unit as the native arm, K timed steps after W warm-up steps, one step =
    one frame of ALL `envs` environments (4 substeps) on the host cores."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    threads = host_threads()[0]
    steps, warm = max(1, args.steps), max(0, args.warmup)
    arm = CpuArm(args.envs, threads)
    arm.settle()
    for _ in range(warm):
        arm.frame()
    per_step = [arm.frame() for _ in range(steps)]
    sec = float(sum(per_step))
    value = args.envs * SUBSTEPS * steps / sec
    single = arm.single_thread_value(max(2, min(steps, 5)))
    cb = arm.describe(value, sec, steps, single)
    arm.close()
    cfg = workload_config(args.envs, 1)
    cfg["l2"] = "n/a (CPU)"
    cfg["parallelism"] = f"{cb['cores']} host threads, {arm.n_shards} world shards"
    out = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": steps, "warmup": warm,
        "ms_per_step": sec / steps * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
        "data": "synthetic", "config": cfg, "impl": "reference", "cpu_baseline": cb,
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
        "note": "reference arm = CPU oracle (C++ restatement of the reference's Warp kernels) on all host threads; the unmodified "
                "reference needs NVIDIA Warp, which is not installed and cannot be installed offline (see DESIGN.md).  The "
                "reference's own Warp-CPU device runs kernels on ONE host thread: that figure is cpu_baseline.single_thread",
    }
    print(json.dumps(out))


if __name__ == "__main__":
    a = parse_args()
    if a.impl == "reference":
        run_reference(a)
    else:
        run_native(a)
