#!/usr/bin/env python
"""bench.py — the headline benchmark of solver2d-b200 (contract: see the task statement and DESIGN.md §measurement).

Metric (BASELINE.json): constraint-iterations / second on the 100k-box TGS_Soft pyramid.
  * workload  : Pyramid recipe (reference samples/collection/sample_contact.cpp:499-561), baseCount = 447
                -> 100 128 boxes, ~299 490 contact constraints; s2_solverTGS_Soft, dt = 1/60, 4 sub-steps, 2 relax
                iterations, warm starting on. Deterministic lattice ("data": "synthetic").
  * a "step"  : one s2World_Step (pair update, narrow phase, solver, finalize), all of it inside the timed region.
  * unit of work: constraint-iteration = one execution of the per-constraint solve body on one manifold or joint
                (SURVEY.md §8d): per step (manifolds with >= 1 point + joints) x sub-steps x (1 + [relax > 0]); counted
                by a device-side meter inside the solver stage.
  * value     : constraint-iterations / device time, state resident in HBM, whole step timed with CUDA events on the
                world's stream, L2 evicted between timed steps.
  * e2e       : same metric through the public C API with host buffers: every step applies a force to every box
                (host -> device), steps, and reads every body transform back (device -> host), wall clock.
  * roofline  : persistent solver kernel (the dominant kernel): algorithmic bytes of SURVEY.md §8d / its device time,
                against the measured HBM copy bandwidth of MEASURED_PEAKS.json.
  * cpu_baseline: the unmodified reference (oracle/_ref, compiled from /root/reference) on one host core, bounded sample.

`--impl reference` times the reference's own CPU implementation on the same workload (bounded sample per step).
N > 1 (`torchrun`): the 100k-box pyramid is ONE island and does not shard (SURVEY.md §8e) -> one replica per GPU
("replicas only", weak scaling) with the per-step NCCL all-gather of packed body state north_star asks for.
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

DT = 1.0 / 60.0


def _peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            p = json.load(f)
        return float(p["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """nvidia-smi SM clock / throttle reasons sampled every 20 ms while the timed region runs (the region is tens of
    milliseconds long). start() returns once the first sample has arrived: nvidia-smi's start-up query stalls kernel
    launches for milliseconds and must not land inside the timed region."""

    QUERY = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.gpu_index = gpu_index
        self.lines = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.QUERY}", "--format=csv,noheader,nounits",
                                          "-i", str(self.gpu_index), "-lms", "20"], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._pump, daemon=True).start()
            t0 = time.perf_counter()
            while not self.lines and time.perf_counter() - t0 < 5.0:
                time.sleep(0.02)
            self.warm_lines = len(self.lines)
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self) -> dict:
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["unavailable"]}
        time.sleep(0.05)
        self.proc.terminate()
        sm, smax, reasons = [], [], set()
        for line in self.lines[getattr(self, "warm_lines", 0):] or self.lines:
            parts = [p.strip() for p in line.split(",")]
            if len(parts) < 9:
                continue
            try:
                sm.append(float(parts[1]))
                smax.append(float(parts[2]))
            except ValueError:
                continue
            for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), parts[5:9]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(smax) if smax else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def algorithmic_bytes_per_step(constraints: int, bodies: int, substeps: int, relax: bool) -> float:
    """SURVEY.md §8d: S*[C*(152 + 208*(1+[E>0])) + Nb*100] + C*(250 + 16) + Nb*32 for one TGS_Soft solver stage."""
    passes = 1 + (1 if relax else 0)
    return substeps * (constraints * (152.0 + 208.0 * passes) + bodies * 100.0) + constraints * (250.0 + 16.0) + bodies * 32.0


def _traffic(which: str):
    """DRAM bytes per launch (dram__bytes_read.sum + dram__bytes_write.sum) of the named kernel from the committed
    `ncu --set full` capture of this workload (profiles/traffic.json), or None."""
    try:
        with open(os.path.join(os.path.dirname(os.path.abspath(__file__)), "profiles", "traffic.json")) as fh:
            return json.load(fh).get(which, {}).get("dram_bytes_per_launch")
    except Exception:
        return None


def build_scene(lib, base_count: int, workload: str = "pyramid", rank: int = 0, world_size: int = 1, field_count: int = 256):
    """pyramid: the headline workload (one replica per rank). field: SURVEY §8d config 5 — `field_count` independent
    pyramid worlds of `base_count` rows batched into one s2World per rank; world k lives on rank k mod world_size."""
    from solver2d_b200 import scenes
    if workload == "field":
        mine = len(range(rank, field_count, world_size))
        return scenes.pyramid_field(lib, "TGS_Soft", count=mine, base_count=base_count, first=0)
    return scenes.pyramid(lib, "TGS_Soft", base_count=base_count)


def run_reference(args, rank: int, world_size: int):
    """The reference's own CPU implementation of the path (oracle/_ref), one host thread (it is single-threaded)."""
    if rank != 0:
        return
    from oracle import ref
    if not ref.available():
        ref.build_ref()
    R = ref.load()
    sc = build_scene(R, args.base, args.workload, 0, 1, args.field_count)
    nb = len(sc.bodies)
    idx = np.array([b.index for b in sc.bodies[1:]], dtype=np.int32)
    forces = np.zeros((len(idx), 2), dtype=np.float32)
    forces[:, 0] = 0.01
    caps = R.capacities(sc.world)
    transforms = np.zeros((caps["bodyCap"], 4), dtype=np.float32)
    t0 = time.perf_counter()
    sc.step(DT, args.substeps, args.relax, True)  # first step: all-pairs broad phase, reported apart
    first = time.perf_counter() - t0
    for _ in range(max(args.warmup - 1, 0)):
        sc.step(DT, args.substeps, args.relax, True)
    work = 0
    total = 0.0
    for _ in range(args.steps):
        # constraints of this step are those of the manifolds as they stand after the step's own narrow phase; the
        # count after the step is the same set (manifold geometry is fixed before the solver runs)
        total += R.timed_e2e_steps(sc.world, 1, DT, args.substeps, args.relax, True, idx, forces, transforms)
        c, j = R.constraint_counts(sc.world)
        work += (c + j) * args.substeps * (1 + (1 if args.relax > 0 else 0))
    value = work / total
    line = {
        "impl": "reference", "metric": "constraint_iters_per_sec", "value": value, "unit": "constraint-iters/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * total / args.steps,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": (f"field{args.field_count}x_pyramid{args.base}" if args.workload == "field" else f"pyramid{args.base}")
                   + f"_tgs_soft_s{args.substeps}_e{args.relax}", "boxes": nb - 1,
                   "dt": DT, "note": "reference CPU path, 1 thread (the reference is single-threaded)"},
        "cpu_baseline": {"value": value, "unit": "constraint-iters/s", "cores": 1, "kind": "reference",
                         "sample": f"{args.steps} steps after {args.warmup} warm-up; first step {first:.3f} s"},
        "e2e": {"value": value, "unit": "constraint-iters/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


def aggregate_over_ranks(dist, device, total_ms, e2e_time, work, e2e_work):
    """Whole-job numbers of an N-rank run: the time of the job is the MAX over ranks, its work the SUM (weak scaling:
    every rank steps its own replica). dist = torch.distributed or None for a single process."""
    import torch
    t_vals = torch.tensor([total_ms, e2e_time], dtype=torch.float64, device=device)
    w_vals = torch.tensor([float(work), float(e2e_work)], dtype=torch.float64, device=device)
    if dist is not None:
        dist.all_reduce(t_vals, op=dist.ReduceOp.MAX)
        dist.all_reduce(w_vals, op=dist.ReduceOp.SUM)
    total_ms_max, e2e_time_max = t_vals.tolist()
    work_all, e2e_work_all = w_vals.tolist()
    return total_ms_max, e2e_time_max, work_all, e2e_work_all


def measure_field(args, P, dev, dist, rank: int, world_size: int, local_rank: int, shard: bool):
    """SURVEY §8d config 5 / north_star: `--field-count` independent pyramid worlds of `--field-base` rows. shard=True: world k
    lives on rank k mod N (rank r batches worlds r, r+N, ... into ONE s2World: disconnected islands of one constraint graph,
    one set of launches), no data-path collective; the one NCCL all-gather of packed body state per step runs on a side
    stream behind the step. shard=False: this rank steps all the worlds alone (the 1-GPU point of the strong-scaling curve).
    Returns (device ms over the timed steps, constraint-iterations done, boxes, constraints) of THIS rank."""
    import torch
    from solver2d_b200 import device, scenes
    L = P.lib
    mine = len(range(rank, args.field_count, world_size)) if shard else args.field_count
    if shard and args.field_single_world and world_size > 1:
        # ONE s2World holding every pile, sharded by ISLAND: every rank builds the whole world, asks the device for the islands
        # of its constraint graph (s2b_download_islands) and keeps island k mod N == rank (static bodies stay everywhere)
        sc = scenes.pyramid_field(P, "TGS_Soft", count=args.field_count, base_count=args.field_base, first=0)
        sc.step(DT, args.substeps, args.relax, True)
        dw = device.DeviceWorld.attach(dev, sc.world)
        labels, _ = dw.islands()
        ids = np.array([b.index for b in sc.bodies])
        dynamic = np.array([P.s2Body_GetType(b) == 2 for b in sc.bodies])
        roots = np.unique(labels[ids[dynamic]])
        owner = {int(r): k % world_size for k, r in enumerate(roots)}
        keep = []
        for b, dyn in zip(sc.bodies, dynamic):
            if dyn and owner[int(labels[b.index])] != rank:
                P.s2DestroyBody(b)
            else:
                keep.append(b)
        sc.bodies = keep
        mine = int(sum(1 for r in roots if owner[int(r)] == rank))
    else:
        sc = scenes.pyramid_field(P, "TGS_Soft", count=mine, base_count=args.field_base, first=0)
        dw = device.DeviceWorld.attach(dev, sc.world)
    nb = len(sc.bodies)
    gather_in = gather_out = ext_stream = side_stream = None
    state = {"done": None}
    if dist is not None and shard:
        most_t = torch.tensor([nb], dtype=torch.int64, device="cuda")
        dist.all_reduce(most_t, op=dist.ReduceOp.MAX)  # equal payload on every rank: the largest body count
        most = int(most_t.item())
        gather_in = torch.zeros((most + 8) * 8, dtype=torch.float32, device="cuda")
        gather_out = torch.empty(world_size * (most + 8) * 8, dtype=torch.float32, device="cuda")
        L.s2b_get_stream.restype = C.c_void_p
        L.s2b_get_stream.argtypes = [C.c_void_p]
        ext_stream = torch.cuda.ExternalStream(int(L.s2b_get_stream(dw.h)), device=torch.device("cuda", local_rank))
        side_stream = torch.cuda.Stream(device=torch.device("cuda", local_rank))

    def exchange():
        if gather_in is None:
            return
        if state["done"] is not None:
            ext_stream.wait_event(state["done"])
        L.s2b_pack_body_state(dw.h, 0, nb, C.c_void_p(gather_in.data_ptr()))
        packed = torch.cuda.Event()
        packed.record(ext_stream)
        side_stream.wait_event(packed)
        with torch.cuda.stream(side_stream):
            dist.all_gather_into_tensor(gather_out, gather_in)
            done = torch.cuda.Event()
            done.record(side_stream)
        state["done"] = done

    for _ in range(max(args.warmup, 3)):
        sc.step(DT, args.substeps, args.relax, True)
        exchange()
    dw.sync()
    out = (C.c_uint64 * 2)()
    L.s2b_get_work(dw.h, out, 1)
    if dist is not None and shard:
        dist.barrier()
    torch.cuda.synchronize()
    total_ms = 0.0
    if gather_in is None:
        for _ in range(args.steps):
            total_ms += float(L.s2World_TimedSteps(sc.world, 1, DT, args.substeps, args.relax, True, 1 if args.flush_l2 else 0))
    else:
        pairs = []
        for _ in range(args.steps):
            if args.flush_l2:
                L.s2b_flush_l2(dw.h)
            e0 = torch.cuda.Event(enable_timing=True)
            e1 = torch.cuda.Event(enable_timing=True)
            e0.record(ext_stream)
            sc.step(DT, args.substeps, args.relax, True)
            exchange()
            e1.record(ext_stream)
            pairs.append((e0, e1))
        tail = torch.cuda.Event(enable_timing=True)
        ext_stream.wait_event(state["done"])
        tail.record(ext_stream)
        torch.cuda.synchronize()
        total_ms = sum(a.elapsed_time(b) for a, b in pairs) + pairs[-1][1].elapsed_time(tail)
    torch.cuda.synchronize()
    L.s2b_get_work(dw.h, out, 1)
    c = dw.counters()
    boxes = sum(1 for b in sc.bodies if P.s2Body_GetType(b) == 2) if args.field_single_world else nb - mine
    res = (total_ms, int(out[0]), boxes, c.constraintCount, c.regionCount, c.cutCount)
    sc.destroy()
    return res


def field_report(args, P, dev, dist, rank: int, world_size: int, local_rank: int) -> dict | None:
    """The sharded config-5 numbers attached to the bench line (key "field"). At N > 1 rank 0 also steps the whole field
    alone afterwards: the 1-GPU point the strong-scaling efficiency is quoted against, measured in the same run."""
    import torch
    ms, work, boxes, constraints, regions, cut = measure_field(args, P, dev, dist, rank, world_size, local_rank, True)
    t = torch.tensor([ms], dtype=torch.float64, device="cuda")
    w = torch.tensor([float(work), float(boxes), float(constraints)], dtype=torch.float64, device="cuda")
    if dist is not None:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dist.all_reduce(w, op=dist.ReduceOp.SUM)
    ms_max = float(t.item())
    work_all, boxes_all, constraints_all = w.tolist()
    rep = None
    if rank == 0:
        rep = {"workload": f"field{args.field_count}x_pyramid{args.field_base}_tgs_soft_s{args.substeps}_e{args.relax}",
               "value": work_all / (ms_max * 1e-3), "unit": "constraint-iters/s", "ms_per_step": ms_max / args.steps,
               "scaling": "strong", "worlds_per_rank": len(range(0, args.field_count, world_size)), "boxes": int(boxes_all),
               "contact_constraints": int(constraints_all), "regions_rank0": regions, "cut_constraints_rank0": cut,
               "partition": "world k -> rank k mod N, a rank's worlds batched into one s2World; no data-path collective; "
                            "one NCCL all-gather of packed body state per step on a side stream" if world_size > 1 else
                            "all worlds batched into one s2World on one GPU"}
    if world_size > 1:
        if rank == 0 and not args.no_field_n1:
            ms1, work1, *_ = measure_field(args, P, dev, None, 0, 1, local_rank, False)
            rep["n1_value_same_run"] = work1 / (ms1 * 1e-3)
            rep["n1_ms_per_step_same_run"] = ms1 / args.steps
            rep["efficiency_vs_n1"] = rep["value"] / (world_size * rep["n1_value_same_run"])
        dist.barrier()
    return rep


def run_ours(args, rank: int, world_size: int, local_rank: int):
    os.environ["S2B_DEVICE"] = str(local_rank)  # worlds of this process live on its own GPU
    import torch
    dist = None
    if world_size > 1:
        import torch.distributed as dist_mod
        dist = dist_mod
        torch.cuda.set_device(local_rank)
        # (NCCL prints its version banner to STDOUT at this level; the one line this script owes the driver is JSON)
        if os.environ.get("NCCL_DEBUG", "VERSION").upper() == "VERSION":
            os.environ["NCCL_DEBUG"] = "WARN"
        dist.init_process_group(backend="nccl", device_id=torch.device("cuda", local_rank))
    else:
        torch.cuda.set_device(local_rank)

    from solver2d_b200 import capi, device
    P = capi.Solver2D(device.LIB_PATH)
    dev = device.Device()
    L = P.lib
    L.s2World_TimedSteps.restype = C.c_float
    L.s2World_TimedSteps.argtypes = [capi.WorldId, C.c_int32, C.c_float, C.c_int32, C.c_int32, C.c_bool, C.c_int32]
    L.s2World_ApplyForcesToCenters.argtypes = [capi.WorldId, C.c_void_p, C.c_void_p, C.c_int32]
    L.s2World_GetBodyTransforms.restype = C.c_int32
    L.s2World_GetBodyTransforms.argtypes = [capi.WorldId, C.c_void_p, C.c_int32]
    L.s2b_get_work.argtypes = [C.c_void_p, C.c_void_p, C.c_int]
    L.s2b_last_solve_kernel_ms.restype = C.c_float
    L.s2b_last_solve_kernel_ms.argtypes = [C.c_void_p]
    L.s2b_flush_l2.argtypes = [C.c_void_p]

    sc = build_scene(P, args.base, args.workload, rank, world_size, args.field_count)
    dw = device.DeviceWorld.attach(dev, sc.world)
    nb = len(sc.bodies)

    def get_work(reset=False):
        out = (C.c_uint64 * 2)()
        L.s2b_get_work(dw.h, out, 1 if reset else 0)
        return int(out[0]), int(out[1])

    # per-step NCCL all-gather of packed body state (north_star) when several GPUs run replicas
    gather_in = gather_out = None
    if dist is not None:
        gather_in = torch.empty((nb + 8) * 8, dtype=torch.float32, device="cuda")
        gather_out = torch.empty(world_size * (nb + 8) * 8, dtype=torch.float32, device="cuda")

    ext_stream = None
    if dist is not None:
        L.s2b_get_stream.restype = C.c_void_p
        L.s2b_get_stream.argtypes = [C.c_void_p]
        # the collective is enqueued on the world's own stream, right behind the step: no host synchronisation
        ext_stream = torch.cuda.ExternalStream(int(L.s2b_get_stream(dw.h)), device=torch.device("cuda", local_rank))

    side_stream = torch.cuda.Stream(device=torch.device("cuda", local_rank)) if dist is not None else None
    ex_state = {"done": None}

    def exchange():
        """Pack this rank's body state on the world's stream, then all-gather it on a side stream: the collective runs
        while the next step is already executing (nothing in a step depends on the other replicas' bodies). The next pack
        waits for the previous all-gather to have consumed the buffer."""
        if dist is None:
            return
        if ex_state["done"] is not None:
            ext_stream.wait_event(ex_state["done"])
        L.s2b_pack_body_state(dw.h, 0, nb, C.c_void_p(gather_in.data_ptr()))
        packed = torch.cuda.Event()
        packed.record(ext_stream)
        side_stream.wait_event(packed)
        with torch.cuda.stream(side_stream):
            dist.all_gather_into_tensor(gather_out, gather_in)
            done = torch.cuda.Event()
            done.record(side_stream)
        ex_state["done"] = done

    # ---- warm-up (includes the first-step all-pairs broad phase) ----
    for _ in range(max(args.warmup - 3, 0)):
        sc.step(DT, args.substeps, args.relax, True)
        exchange()
    dw.sync()

    # ---- value: device-resident, CUDA events per step, L2 flushed between steps ----
    sampler = ClockSampler(local_rank)
    if rank == 0 and os.environ.get("BENCH_NO_SAMPLER") is None:
        sampler.start()
    # the last warm-up steps go through the timed entry point so that its one-off costs (L2-flush buffer) are paid here
    for _ in range(min(3, args.warmup)):
        L.s2World_TimedSteps(sc.world, 1, DT, args.substeps, args.relax, True, 1 if args.flush_l2 else 0)
        exchange()
    dw.sync()
    get_work(reset=True)
    c0 = dw.counters()
    launches0, captures0 = c0.kernelLaunches, c0.graphCaptures
    if dist is not None:
        dist.barrier()
    torch.cuda.synchronize()
    t_wall0 = time.perf_counter()
    solve_kernel_ms = []
    step_ms = []
    total_ms = 0.0
    if dist is None:
        host_ms = []
        for _ in range(args.steps):
            th = time.perf_counter()
            step_ms.append(float(L.s2World_TimedSteps(sc.world, 1, DT, args.substeps, args.relax, True, 1 if args.flush_l2 else 0)))
            host_ms.append(1e3 * (time.perf_counter() - th))
            total_ms += step_ms[-1]
            solve_kernel_ms.append(float(L.s2b_last_solve_kernel_ms(dw.h)))
        if os.environ.get("BENCH_DEBUG"):
            st = dw.stage_ms()
            print("debug first steps: device ms", [round(x, 3) for x in step_ms[:4]], "host ms of the call", [round(x, 3) for x in host_ms[:4]],
                  file=sys.stderr)
    else:
        # per step: [L2 flush] e0 | step | pack | e1 ; the all-gather overlaps the next step on the side stream, only its
        # tail after the last step is exposed and is added at the end
        pairs = []
        for _ in range(args.steps):
            if args.flush_l2:
                L.s2b_flush_l2(dw.h)
            e0 = torch.cuda.Event(enable_timing=True)
            e1 = torch.cuda.Event(enable_timing=True)
            e0.record(ext_stream)
            sc.step(DT, args.substeps, args.relax, True)
            exchange()
            e1.record(ext_stream)
            pairs.append((e0, e1))
        tail = torch.cuda.Event(enable_timing=True)
        ext_stream.wait_event(ex_state["done"])
        tail.record(ext_stream)
        torch.cuda.synchronize()
        step_ms = [a.elapsed_time(b) for a, b in pairs]
        total_ms = sum(step_ms) + pairs[-1][1].elapsed_time(tail)
        solve_kernel_ms.append(float(L.s2b_last_solve_kernel_ms(dw.h)))
    torch.cuda.synchronize()
    if dist is not None:
        dist.barrier()
    wall = time.perf_counter() - t_wall0
    clocks = sampler.stop() if rank == 0 else None
    work, solves = get_work(reset=True)
    launches = dw.counters().kernelLaunches - launches0
    counters = dw.counters()
    stage_ms = dw.stage_ms()
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, dw, sc, counters.bodyCapacity)

    # ---- e2e: public API with host buffers, H2D + D2H inside the timed region ----
    idx = np.array([b.index for b in sc.bodies[1:]], dtype=np.int32)
    forces = np.zeros((len(idx), 2), dtype=np.float32)
    forces[:, 0] = 0.01
    # the caller's buffers are page-locked host memory (the library's own allocator for that, s2b_host_alloc)
    L.s2b_host_alloc.restype = C.c_void_p
    L.s2b_host_alloc.argtypes = [C.c_size_t]
    xf_bytes = counters.bodyCapacity * 16
    xf_ptr = L.s2b_host_alloc(xf_bytes)
    transforms = np.frombuffer((C.c_char * xf_bytes).from_address(xf_ptr), dtype=np.float32).reshape(counters.bodyCapacity, 4)
    e2e_steps = max(args.steps // 2, 3)
    for _ in range(2):
        L.s2World_ApplyForcesToCenters(sc.world, idx.ctypes.data, forces.ctypes.data, len(idx))
        sc.step(DT, args.substeps, args.relax, True)
        L.s2World_GetBodyTransforms(sc.world, transforms.ctypes.data, counters.bodyCapacity)
    get_work(reset=True)
    if dist is not None:
        dist.barrier()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    e2e_parts = [0.0, 0.0, 0.0]
    for s in range(e2e_steps):
        f = forces if (s & 1) == 0 else -forces
        ta = time.perf_counter()
        L.s2World_ApplyForcesToCenters(sc.world, idx.ctypes.data, f.ctypes.data, len(idx))
        tb = time.perf_counter()
        sc.step(DT, args.substeps, args.relax, True)
        tc = time.perf_counter()
        L.s2World_GetBodyTransforms(sc.world, transforms.ctypes.data, counters.bodyCapacity)
        td = time.perf_counter()
        e2e_parts[0] += tb - ta
        e2e_parts[1] += tc - tb
        e2e_parts[2] += td - tc
        exchange()
    torch.cuda.synchronize()
    e2e_time = time.perf_counter() - t0
    e2e_work, _ = get_work(reset=True)

    total_ms_max, e2e_time_max, work_all, e2e_work_all = aggregate_over_ranks(dist, "cuda", total_ms, e2e_time, work, e2e_work)

    if rank == 0:
        value = work_all / (total_ms_max * 1e-3)
        e2e_value = e2e_work_all / e2e_time_max
        peak, peak_src = _peaks()
        constraints = counters.constraintCount
        alg = algorithmic_bytes_per_step(constraints, nb, args.substeps, args.relax > 0)
        k_ms = float(np.mean(solve_kernel_ms)) if solve_kernel_ms else 0.0
        achieved = (alg / (k_ms * 1e-3)) / 1e9 if k_ms > 0 else 0.0
        line = {
            "metric": "constraint_iters_per_sec", "value": value, "unit": "constraint-iters/s", "n_gpus": world_size,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": total_ms_max / args.steps,
            "higher_is_better": True, "scaling": "strong" if args.workload == "field" else "weak", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic",
            "config": {"workload": (f"field{args.field_count}x_pyramid{args.base}" if args.workload == "field" else f"pyramid{args.base}")
                       + f"_tgs_soft_s{args.substeps}_e{args.relax}", "boxes": nb - 1,
                       "contact_constraints": constraints, "colours": counters.groupCount, "dt": DT,
                       "l2": "flushed between timed steps" if args.flush_l2 else "not flushed (working set < L2)",
                       "parallelism": "single island: replicas only" + ("" if world_size == 1 else
                                                                        f", x{world_size} + NCCL all-gather of body state"),
                       "schedule": "graph colouring, persistent cooperative solver kernel"},
            "stage_ms_last_step": {"pairs": stage_ms[0], "contacts": stage_ms[1], "solve": stage_ms[2], "finalize": stage_ms[3]},
            "step_ms_stats": {"min": float(np.min(step_ms)), "median": float(np.median(step_ms)), "max": float(np.max(step_ms)), "argmax": int(np.argmax(step_ms)),
                              "over_2x_median": [round(float(x), 3) for x in step_ms if x > 2 * np.median(step_ms)],
                              "pair_passes_total": int(counters.pairPassCount),
                              "graph_captures_in_timed_region": int(counters.graphCaptures - captures0),
                              "graph_replays_total": int(counters.graphReplays)},
            "e2e": {"value": e2e_value, "unit": "constraint-iters/s", "ms_per_step": 1e3 * e2e_time_max / e2e_steps,
                    "h2d_bytes_per_step": int(len(idx) * 12), "d2h_bytes_per_step": int(nb * 16),
                    "steps": e2e_steps, "clock": "host wall clock, synchronised on both sides",
                    "host_ms_per_step": {"apply_forces": 1e3 * e2e_parts[0] / e2e_steps, "step_call": 1e3 * e2e_parts[1] / e2e_steps,
                                         "get_transforms_incl_wait": 1e3 * e2e_parts[2] / e2e_steps}},
            "gpu_launches": int(launches),
            "roofline": {"kernel": "s2bPersistentSolveT<7> (TGS_Soft instantiation; the whole solver stage of one step)", "bound": "hbm",
                         "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak if peak else None,
                         "traffic": _traffic("persistent_solve"),
                         "traffic_source": "profiles/traffic.json: dram__bytes_read.sum + dram__bytes_write.sum of one `ncu --set full` "
                                           "capture of this workload (committed), not measured in this run",
                         "algorithmic_bytes_per_launch": alg, "kernel_ms": k_ms, "peak_source": peak_src},
            "clocks": clocks,
            "wall_s_timed_region": wall,
        }
        if not args.no_colour_probe and world_size == 1:
            # the hot kernel on its own, at a size where one colour exceeds L2 (see tools/color_kernel_probe.py)
            try:
                sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "tools"))
                from color_kernel_probe import probe
                pr = probe(args.probe_base)
                line["roofline_colour_kernel"] = {
                    "kernel": "s2bTgsSoftColorKernel (TGS_Soft relax pass over the largest colour, L2 evicted before each launch)",
                    "workload": f"pyramid{args.probe_base}: {pr['boxes']} boxes, {pr['contact_constraints']} constraints, "
                                f"{pr['colours']} colours, largest colour {pr['largest_colour_constraints']}",
                    "bound": "hbm", "achieved": pr.get("achieved_GBps"), "peak": peak, "unit": "GB/s",
                    "frac": (pr.get("achieved_GBps", 0.0) / peak) if peak else None, "kernel_ms": pr["kernel_ms"],
                    "algorithmic_bytes_per_launch": pr.get("algorithmic_bytes"), "traffic": _traffic("colour_kernel")}
            except Exception as e:  # the probe is additional evidence, never a reason to lose the bench line
                line["roofline_colour_kernel"] = {"error": repr(e)}
        if not args.no_cpu_baseline and world_size == 1:
            line["cpu_baseline"] = cpu_baseline(args)
    sc.destroy()
    sc = None
    # config 5 (the configuration that shards): every rank takes part, rank 0 reports
    field = None
    if not args.no_field and args.workload == "pyramid":
        try:
            field = field_report(args, P, dev, dist, rank, world_size, local_rank)
        except Exception as e:  # additional evidence, never a reason to lose the bench line
            field = {"error": repr(e)}
    if rank == 0:
        if field is not None:
            line["field"] = field
        print(json.dumps(line), flush=True)
    if dist is not None:
        dist.barrier()
        dist.destroy_process_group()


DUMP_BUDGET_BYTES = 64 << 20
DUMP_FIELDS = (("body_origin", "origin"), ("body_rotation", "rot"), ("body_linear_velocity", "linearVelocity"),
               ("body_angular_velocity", "angularVelocity"))


def dump_outputs(out_dir: str, dw, sc, body_capacity: int) -> None:
    """The body state a caller of the timed step reads back after its last step: body origin (what s2Body_GetPosition and
    s2World_GetBodyTransforms return), rotation (sin, cos), linear and angular velocity, one row per body of the scene in
    creation order (the static ground first), as float32 .npy files; body_index.npy (float64) names each row's body.
    36 bytes per body: above 64 MB a fixed, seeded sample of the bodies is written, in creation order."""
    n = len(sc.bodies)
    keep = np.arange(n)
    per_body = 4 * 7 + 8
    if n * per_body > DUMP_BUDGET_BYTES:
        keep = np.sort(np.random.default_rng(0).choice(n, DUMP_BUDGET_BYTES // per_body, replace=False))
    rows = dw.download_all_bodies(body_capacity)
    rows = rows[np.array([sc.bodies[k].index for k in keep], dtype=np.int64)]
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "body_index.npy"), keep.astype(np.float64))
    for name, field in DUMP_FIELDS:
        np.save(os.path.join(out_dir, f"{name}.npy"), np.ascontiguousarray(rows[field], dtype=np.float32))


def cpu_baseline(args) -> dict:
    """Bounded sample of the same workload on the unmodified reference, one host core."""
    from oracle import ref
    if not ref.available() and not ref.build_ref():
        return {"value": None, "unit": "constraint-iters/s", "cores": 1, "kind": "reference", "sample": "oracle/_ref missing"}
    R = ref.load()
    sc = build_scene(R, args.base, args.workload, 0, 1, args.field_count)
    t0 = time.perf_counter()
    sc.step(DT, args.substeps, args.relax, True)
    first = time.perf_counter() - t0
    for _ in range(2):
        sc.step(DT, args.substeps, args.relax, True)
    steps = args.cpu_steps
    total = R.timed_steps(sc.world, steps, DT, args.substeps, args.relax, True)
    c, j = R.constraint_counts(sc.world)
    work = (c + j) * args.substeps * (1 + (1 if args.relax > 0 else 0)) * steps
    sc.destroy()
    return {"value": work / total, "unit": "constraint-iters/s", "cores": 1, "kind": "reference",
            "ms_per_step": 1e3 * total / steps,
            "sample": f"{steps} steady steps of the same workload after 3 warm-up steps (first step {first:.2f} s); host has "
                      f"{os.cpu_count()} cores, the reference uses 1"}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=30)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--impl", choices=["ours", "reference"], default="ours")
    ap.add_argument("--base", type=int, default=447, help="pyramid base count (447 -> 100 128 boxes)")
    ap.add_argument("--workload", choices=["pyramid", "field"], default="pyramid",
                    help="pyramid = headline (replica per rank); field = config 5: --field-count worlds of --base rows, sharded over ranks")
    ap.add_argument("--field-count", type=int, default=256)
    ap.add_argument("--field-base", type=int, default=45, help="rows of each world of the sharded config-5 measurement (45 -> 1 035 boxes)")
    ap.add_argument("--field-single-world", action="store_true",
                    help="config 5 built as ONE s2World on every rank and sharded by island (s2b_download_islands) instead of by construction")
    ap.add_argument("--no-field", action="store_true", help="skip the sharded config-5 measurement attached as key 'field'")
    ap.add_argument("--no-field-n1", action="store_true", help="at N > 1: skip rank 0's single-GPU run of the whole field")
    ap.add_argument("--substeps", type=int, default=4)
    ap.add_argument("--relax", type=int, default=2)
    ap.add_argument("--no-flush-l2", dest="flush_l2", action="store_false")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-colour-probe", action="store_true")
    ap.add_argument("--probe-base", type=int, default=2600, help="pyramid base of the per-colour kernel roofline probe")
    ap.add_argument("--cpu-steps", type=int, default=20)
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write the body state of the last one to DIR/<name>.npy (at most 64 MB)")
    args = ap.parse_args()
    args.warmup = max(args.warmup, 3)

    rank = int(os.environ.get("RANK", "0"))
    world_size = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))

    if args.impl == "reference":
        run_reference(args, rank, world_size)
    else:
        run_ours(args, rank, world_size, local_rank)


if __name__ == "__main__":
    main()
