#!/usr/bin/env python
"""bench.py -- simulation steps/s of the Eulerian fluid step (BASELINE.json metric) on N B200s.

Contract: `python bench.py --gpus N --steps K --warmup W` prints ONE JSON line (rank 0).
One *step* = one `tfluids.simulate` call (torch/lib/simulate.lua:175-327) on a 128^3 MAC
grid: MacCormack("maccormackOurs") advection of density and velocity, plume BCs, buoyancy,
vorticity confinement and the CNN pressure projection -- BASELINE.json configs[2]
(configs[1], 64^3 CNN forward only, is a parity-test case).

  value     whole-job steps/s with the state resident in HBM (CUDA events on the launch stream), the step replayed
            from a CUDA graph (tfl_step_graph_launch); `ungraphed` = the same step launched kernel by kernel
  e2e       the same step through the C-ABI host-buffer call (tfl_host_sim_step): pinned
            host p/U/density copied in, step, copied back, every step
  roofline  the dominant kernel's ALGORITHMIC bytes / its measured mean duration vs the
            measured HBM copy bandwidth (MEASURED_PEAKS.json)
  cpu_baseline  the reference's own CPU operators (oracle/_ref, compiled in place) -- or the C
            restatement when that is absent -- timed on this box's host cores on a bounded
            sample (one full 128^3 step without the conv stack is ~1 s on 8 cores; the sample
            used is stated)

`--impl reference` times that CPU path alone and prints the same line shape.
`--dump-outputs DIR` writes the state the last timed step left (pDiv, UDiv, density) as DIR/<name>.npy, float32;
the inputs are seeded, so two builds run with the same arguments can be compared output for output.
Multi-GPU (N > 1, launched with torchrun): weak scaling -- every rank advances an
independent 128^3 grid (the batch-of-grids decomposition north_star allows); no data-path
collective; time = max over ranks.
"""
import argparse
import ctypes
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

N_GRID = 128
# SURVEY.md section 8(d): algorithmic bytes per voxel of one C3 step (fp32, flags as fp32).
BYTES_PER_VOXEL_STEP = 364
# dominant kernels' algorithmic bytes per voxel (DESIGN.md "Kernels"): filled per kernel name
ALGO_BYTES = {
    "advect_vel": 28,       # U 12 + flags 4 read, U 12 written   (both MacCormack passes)
    "advect_scalar": 24,    # s 4 + U 12 + flags 4 read, s 4 written
    "cnn": 36,              # pDiv 4 + UDiv 12 + flags 4 read, p 4 + U 12 written
}
# --dump-outputs writes at most this many bytes of array data (a 128^3 step's state is 42 MB)
DUMP_LIMIT_BYTES = 60 * 10 ** 6


def dump_outputs(directory, arrays):
    """Writes each array as <directory>/<name>.npy in float32.  Above DUMP_LIMIT_BYTES in all, each array is cut
    to a fixed, seeded sample of its flat indices, sized to its share of the limit."""
    os.makedirs(directory, exist_ok=True)
    total = sum(a.size * 4 for a in arrays.values())
    for name, a in arrays.items():
        a = np.ascontiguousarray(a, np.float32)
        if total > DUMP_LIMIT_BYTES:
            k = a.size * DUMP_LIMIT_BYTES // total
            a = a.reshape(-1)[np.sort(np.random.default_rng(0).integers(0, a.size, k))]
        np.save(os.path.join(directory, name + ".npy"), a)


def use_all_host_cores():
    """The CPU arm uses every host core whatever the launcher exported (torchrun sets OMP_NUM_THREADS=1)."""
    n = os.cpu_count() or 1
    os.environ["OMP_NUM_THREADS"] = str(n)
    try:
        ctypes.CDLL("libgomp.so.1").omp_set_num_threads(n)      # the runtime may already be initialised
    except OSError:
        pass
    return n


def ncu_traffic(kernel_regexes, path=None):
    """dram read + write bytes per launch of the named kernels, summed, from the tracked ncu raw table of the
    current build (profiles/r02_advect_ncu_raw.csv: `ncu -i ... --page raw --csv`); None when absent."""
    import csv
    import re
    path = path or os.path.join(ROOT, "profiles", "r02_advect_ncu_raw.csv")
    if not os.path.exists(path):
        return None, None
    rows = list(csv.reader(open(path)))
    hdr = next((r for r in rows if "Kernel Name" in r), None)
    if hdr is None:
        return None, None
    ki = hdr.index("Kernel Name")
    cols = [i for i, h in enumerate(hdr) if h in ("dram__bytes_read.sum", "dram__bytes_write.sum")]
    units = rows[rows.index(hdr) + 1]
    scale = {"byte": 1.0, "Kbyte": 1e3, "Mbyte": 1e6, "Gbyte": 1e9}
    total = 0.0
    for rx in kernel_regexes:
        vals = []
        for r in rows[rows.index(hdr) + 2:]:
            if len(r) > ki and re.search(rx, r[ki]):
                vals.append(sum(float(r[i].replace(",", "")) * scale.get(units[i], 1.0) for i in cols))
        if not vals:
            return None, None
        total += sum(vals) / len(vals)
    return total, os.path.relpath(path, ROOT)


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return d.get("hbm_gbs", 6650.0), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler(threading.Thread):
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md)."""

    def __init__(self, gpu_index):
        super().__init__(daemon=True)
        self.idx = gpu_index
        self.stop_flag = threading.Event()
        self.samples = []
        self.reasons = set()
        self.max_mhz = None

    def run(self):
        q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        while not self.stop_flag.is_set():
            try:
                out = subprocess.run(["nvidia-smi", "-i", str(self.idx), "--query-gpu=" + q,
                                      "--format=csv,noheader,nounits"], capture_output=True, text=True,
                                     timeout=5).stdout.strip()
                parts = [x.strip() for x in out.split(",")]
                self.samples.append(float(parts[0]))
                self.max_mhz = float(parts[1])
                for nm, v in zip(names, parts[2:]):
                    if v.lower().startswith("active"):
                        self.reasons.add(nm)
            except Exception:
                pass
            self.stop_flag.wait(0.2)

    def summary(self):
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": ["unsampled"]}
        return {"sm_mhz": float(np.median(self.samples)), "sm_max_mhz": self.max_mhz,
                "reasons": sorted(self.reasons)}


def make_problem(n=N_GRID, velocity="smooth"):
    """velocity: "smooth" (band-limited, +-2 cells/s) or "random" (SURVEY.md 8d: uniform in [-2, 2] per face)."""
    import torch
    from fluidnet_b200 import synth, simulate
    flags = synth.make_flags(n, n, n, True, nb=1, geometry=True)
    U = (synth.make_smooth_velocity if velocity == "smooth" else synth.make_velocity)(flags, True, amp=2.0)
    density = synth.make_density(flags)
    batch = {"pDiv": np.zeros_like(flags), "UDiv": U, "flags": flags, "density": density}
    # Plume inflow BCs from the product's own host mirror of tfluids.createPlumeBCs (lib/simulate.lua:47-123);
    # nothing under oracle/ is touched on this arm's input path.
    tb = {k: torch.from_numpy(v) for k, v in batch.items()}
    simulate.createPlumeBCs(tb, [1.0], n / 128.0, 0.15)
    for k in ("UBC", "UBCInvMask", "densityBC", "densityBCInvMask"):
        batch[k] = tb[k].numpy()
    # fluid_net_3d_sim.lua:73-87
    mconf = dict(dt=0.1, advectionMethod="maccormackOurs", maccormackStrength=0.6,
                 buoyancyScale=2.0 * n / 128.0, gravityScale=0.0, gravity=None,
                 vorticityConfinementAmp=3.0, simMethod="convnet", maxIter=None, is3D=True,
                 normalizeInputThreshold=1e-5)
    return batch, mconf, synth.make_model(True)


def cpu_step_ops(be, batch, mconf, with_cnn_model=None):
    """One step with the CPU reference operators (conv stack optional: it is not reference
    code, lib/model.lua's cuDNN layers have no CPU source in the tree)."""
    import oracle
    if with_cnn_model is not None:
        oracle.simulate(be, mconf, batch, with_cnn_model)
    else:
        m = dict(mconf)
        m["simMethod"] = "jacobi"
        m["maxIter"] = 1
        oracle.simulate(be, m, batch, None)


def run_reference(args):
    """--impl reference: the reference's own CPU implementation of the path on the host cores."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    use_all_host_cores()
    import oracle
    oracle.build()
    be = oracle.Reference() if oracle.have_reference() else oracle.Oracle()
    n = N_GRID
    batch, mconf, mnp = make_problem(n)
    # bounded sample: advection + forces + BCs + wall/divergence/1 Jacobi sweep/velocity update
    # of the full 128^3 grid (everything the reference has CPU code for); the conv stack is
    # excluded from the reference arm because its CPU source is not in the reference tree.
    times = []
    for it in range(args.warmup + args.steps):
        t0 = time.perf_counter()
        cpu_step_ops(be, batch, mconf, None)
        dt = time.perf_counter() - t0
        if it >= args.warmup:
            times.append(dt)
    T = float(np.mean(times))
    v = 1.0 / T
    line = {"impl": "reference", "metric": "sim steps/sec on 128^3 MAC grid (CNN proj)", "value": v,
            "unit": "steps/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": T * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic",
            "config": {"workload": "3D 128^3 MAC grid, maccormackOurs advection + buoyancy + vorticity "
                                   "confinement + projection", "grid": [n, n, n]},
            "cpu_baseline": {"value": v, "unit": "steps/s", "cores": be.num_threads(),
                             "kind": "reference" if be.name == "reference" else "port",
                             "sample": "full 128^3 step of the reference CPU operators; the CNN conv stack "
                                       "(no CPU source in the reference) replaced by 1 Jacobi sweep"},
            "e2e": {"value": v, "unit": "steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line))
    return 0


def measure_slab(n, steps, warmup, world, rank, local):
    """BASELINE config 5: ONE n^3 domain split in z across the ranks, stepped by tfl_slab_sim_step (the library
    owns the NCCL communicator; neighbour ncclSend / ncclRecv straight on the field arrays).  Strong scaling.
    Returns the record (rank 0) or None."""
    import torch
    import torch.distributed as dist
    from fluidnet_b200.slab import NativeSlabSimulator
    batch_np, mconf, mnp = make_problem(n)
    tb = {k: torch.from_numpy(v) for k, v in batch_np.items()}
    sim = NativeSlabSimulator(tb, mconf, mnp["layers"], torch.device("cuda", local), rank, world)
    del tb
    warmup = max(warmup, 3)
    for _ in range(warmup):
        sim.step()
    sim.check()
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    stream = torch.cuda.current_stream()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    l0 = sim.ctx.launch_count()
    e0.record(stream)
    for _ in range(steps):
        sim.step()
    e1.record(stream)
    torch.cuda.synchronize()
    launches = sim.ctx.launch_count() - l0
    if world > 1:
        dist.barrier()
    t = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device="cuda")
    ex_ms, ex_bytes = sim.exchange_stats()
    ex = torch.tensor(ex_ms, dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dist.all_reduce(ex, op=dist.ReduceOp.MAX)
    sim.check()
    transport = {"nccl": "one packed ncclSend / ncclRecv per neighbour and direction, grouped per phase"}.get(
        sim.halo_transport, "push / pull kernels over peer memory (CUDA IPC handles, remote stores over NVLink, "
                            "system-scope step counters)") if world > 1 else "none (single rank)"
    sim.close()
    if rank != 0:
        return None
    ms = t.item() / steps
    ex = [float(v) for v in ex.tolist()]
    names = ["U+density, %d planes (before the advection)" % (2 * 2 + 2), "U+density, 4 planes (before the forces)",
             "U+p, 5 planes (before the projection)"]
    limiting = names[max(range(3), key=lambda i: ex[i])] if world > 1 else None
    return {"metric": "sim steps/sec on ONE %d^3 MAC grid (CNN proj), z-slab decomposed" % n, "value": 1000.0 / ms,
            "unit": "steps/s", "n_gpus": world, "steps": steps, "warmup": warmup, "ms_per_step": ms,
            "scaling": "strong", "grid": [n, n, n],
            "parallelism": "z-slab x%d; per step 3 neighbour halo exchanges + one 2-double ncclAllReduce, all issued by "
                           "libtfl (tfl_slab_sim_step); halo transport: %s" % (world, transport),
            "halo_bytes_sent_per_rank_step": int(sum(ex_bytes)),
            "exchange_ms_last_step_max_over_ranks": {"halo_advect": ex[0], "halo_forces": ex[1],
                                                     "halo_projection": ex[2], "allreduce": ex[3]},
            "limiting_exchange": limiting,
            "l2": "working set %d MB per rank; no flush between steps" % (60 * (n / 128.0) ** 3 / world),
            "gpu_launches": int(launches)}


def run_slab(args, world, rank, local):
    """--mode slab: only the z-slab measurement, as its own JSON line."""
    import torch.distributed as dist
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    rec = measure_slab(args.grid, args.steps, args.warmup, world, rank, local)
    if rank == 0:
        sampler.stop_flag.set()
        rec.update({"higher_is_better": True, "vs_baseline": None, "dtype": "f32", "data": "synthetic",
                    "config": {"workload": "ONE 3D %d^3 MAC grid split in z over %d GPU(s): maccormackOurs advection + "
                                           "plume BCs + buoyancy + vorticity confinement + CNN projection" % (args.grid, world),
                               "grid": rec["grid"], "parallelism": rec["parallelism"]},
                    "clocks": sampler.summary()})
        print(json.dumps(rec))
    if world > 1:
        dist.destroy_process_group()
    return 0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200")
    ap.add_argument("--grid", type=int, default=N_GRID)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-slab", action="store_true", help="skip the 256^3 z-slab (BASELINE config 5) sub-record")
    ap.add_argument("--slab-grid", type=int, default=256)
    ap.add_argument("--no-extra", action="store_true", help="skip the Jacobi / PCG side measurements (kernel experiments)")
    ap.add_argument("--mode", default="grids", choices=["grids", "slab"],
                    help="grids: one independent --grid^3 domain per GPU (weak scaling, the default and the "
                         "BASELINE metric); slab: ONE --grid^3 domain z-slab decomposed over the GPUs with NCCL "
                         "halo exchange (strong scaling, BASELINE config 5)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write pDiv, UDiv and density after the last timed step as DIR/<name>.npy (rank 0)")
    args = ap.parse_args()
    if args.dump_outputs and (args.impl == "reference" or args.mode == "slab"):
        ap.error("--dump-outputs applies to the default GPU measurement (--impl b200 --mode grids)")
    if args.impl == "reference":
        return run_reference(args)

    import torch
    import torch.distributed as dist
    from fluidnet_b200 import tfluids, simulate, model as fmodel

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    n = args.grid
    if args.mode == "slab":
        return run_slab(args, world, rank, local)
    batch_np, mconf, mnp = make_problem(n)
    stream = torch.cuda.Stream()
    with torch.cuda.stream(stream):
        gb = {k: torch.from_numpy(v.copy()).cuda() for k, v in batch_np.items()}
        gm = fmodel.ProjectionModel(mnp["layers"], True)
        ctx = tfluids.context()
        # L2 flush buffer (> 126 MB) written between timed iterations.
        flush = torch.empty(256 * 1024 * 1024 // 4, dtype=torch.float32, device="cuda")

        def timed_steps(state, steps, warmup):
            """Per-step CUDA events on the launch stream, L2 flushed before each step; returns total ms."""
            for _ in range(warmup):
                simulate.simulate_fused(None, mconf, state, gm)
            stream.synchronize()
            if world > 1:
                dist.barrier()
            torch.cuda.synchronize()
            evs = []
            lc0 = ctx.launch_count()
            for _ in range(steps):
                flush.fill_(0.0)
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record(stream)
                simulate.simulate_fused(None, mconf, state, gm)
                e1.record(stream)
                evs.append((e0, e1))
            stream.synchronize()
            torch.cuda.synchronize()
            return sum(a.elapsed_time(b) for a, b in evs), ctx.launch_count() - lc0

        def timed_graph_steps(state, steps):
            """The same step replayed from a CUDA graph (tfl_step_graph_*): one launch per step."""
            graph = simulate.StepGraph(mconf, state, gm)
            for _ in range(2):
                graph.launch()
            stream.synchronize()
            evs = []
            for _ in range(steps):
                flush.fill_(0.0)
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record(stream)
                graph.launch()
                e1.record(stream)
                evs.append((e0, e1))
            stream.synchronize()
            ms = sum(a.elapsed_time(b) for a, b in evs)
            graph.close()
            return ms

        sampler = ClockSampler(local)
        if rank == 0:
            sampler.start()
        total_ms, launches = timed_steps(gb, args.steps, max(args.warmup, 3))
        lg0 = ctx.launch_count()
        graph_error = None
        try:
            graph_ms = timed_graph_steps(gb, args.steps)
            # kernels inside the timed graph region: the 2 untimed warm-up replays are subtracted
            graph_launches = (ctx.launch_count() - lg0) * args.steps // (args.steps + 2)
        except Exception as e:                      # a box that cannot capture: the kernel-by-kernel number is the headline
            graph_error = "%s: %s" % (type(e).__name__, e)
            graph_ms, graph_launches = total_ms, launches
        if args.dump_outputs and rank == 0:
            dump_outputs(args.dump_outputs, {k: gb[k].cpu().numpy() for k in ("pDiv", "UDiv", "density")})
        # trace-length regime of the timed steps (the advection cost is data dependent)
        max_u_dt = float(gb["UDiv"].abs().max().item()) * mconf["dt"]
        if world > 1:
            dist.barrier()
        if rank == 0:
            sampler.stop_flag.set()
        t = torch.tensor([total_ms], dtype=torch.float64, device="cuda")
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        total_ms = t.item()
        tg = torch.tensor([graph_ms], dtype=torch.float64, device="cuda")
        if world > 1:
            dist.all_reduce(tg, op=dist.ReduceOp.MAX)
        graph_ms = tg.item()
        assert ctx.trace_faults() == 0, "line traces left the domain / hit a hard-error path"

        # ---- SURVEY.md 8(d) variant: uniform-random +-2 velocity (incoherent gathers), same step ----
        variant = None
        if not args.no_extra:
            b_r, _, _ = make_problem(n, velocity="random")
            g_r = {k: torch.from_numpy(v.copy()).cuda() for k, v in b_r.items()}
            vsteps = max(3, min(args.steps, 10))
            ms_r, _ = timed_steps(g_r, vsteps, 3)
            tr = torch.tensor([ms_r], dtype=torch.float64, device="cuda")
            if world > 1:
                dist.all_reduce(tr, op=dist.ReduceOp.MAX)
            variant = {"velocity": "uniform random in [-2, 2] cells/s per face at step 0 (SURVEY.md 8d)",
                       "value": world * 1000.0 * vsteps / tr.item(), "unit": "steps/s", "steps": vsteps,
                       "max_u_dt_cells": float(g_r["UDiv"].abs().max().item()) * mconf["dt"]}
            del g_r

        # ---- e2e: host buffers through the C-ABI host-sim call -----------------------------
        import ctypes as C
        lib = ctx.lib
        hs = C.c_void_p()
        fl = np.ascontiguousarray(batch_np["flags"])
        arrs = [np.ascontiguousarray(batch_np[k]) for k in ("UBC", "UBCInvMask", "densityBC", "densityBCInvMask")]
        ctx.check(lib.tfl_host_sim_create(ctx.h, 1, n, n, n, 1, fl.ctypes.data, arrs[0].ctypes.data,
                                          arrs[1].ctypes.data, arrs[2].ctypes.data, arrs[3].ctypes.data,
                                          C.byref(hs)))
        hp = torch.zeros(1, 1, n, n, n).pin_memory()
        hU = torch.from_numpy(batch_np["UDiv"].copy()).pin_memory()
        hd = torch.from_numpy(batch_np["density"].copy()).pin_memory()
        mc = simulate.make_mconf(mconf)
        e2e_steps = max(3, min(args.steps, 20))
        for _ in range(2):
            ctx.check(lib.tfl_host_sim_step(ctx.h, hs, hp.data_ptr(), hU.data_ptr(), hd.data_ptr(), C.byref(mc), gm.h))
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for _ in range(e2e_steps):
            ctx.check(lib.tfl_host_sim_step(ctx.h, hs, hp.data_ptr(), hU.data_ptr(), hd.data_ptr(), C.byref(mc), gm.h))
        torch.cuda.synchronize()
        e2e_s = time.perf_counter() - t0
        t = torch.tensor([e2e_s], dtype=torch.float64, device="cuda")
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        e2e_s = t.item()
        lib.tfl_host_sim_destroy(ctx.h, hs)
        bytes_io = 5 * n ** 3 * 4

        # ---- roofline of the dominant kernel (advectVel, both passes), timed alone --------
        peak, peak_src = peaks()
        U = gb["UDiv"]
        Ud = torch.empty_like(U)
        reps = 10
        for _ in range(3):
            tfluids.advectVel(0.1, U, gb["flags"], "maccormackOurs", Ud, 0.6)
        # CUDA events right around the kernel's launch, on the stream it is launched on (the library records them
        # when asked to: the operator call around it also refreshes the flag bytes, which is not this kernel)
        lib.tfl_debug_time_advect_kernel.argtypes = [ctypes.c_void_p, ctypes.c_int]
        lib.tfl_debug_last_advect_kernel_ms.argtypes = [ctypes.c_void_p]
        lib.tfl_debug_last_advect_kernel_ms.restype = ctypes.c_float
        lib.tfl_debug_time_advect_kernel(ctx.h, 1)
        ks, ops = [], []
        for _ in range(reps):
            flush.fill_(0.0)
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record(stream)
            tfluids.advectVel(0.1, U, gb["flags"], "maccormackOurs", Ud, 0.6)
            b.record(stream)
            stream.synchronize()
            ks.append(float(lib.tfl_debug_last_advect_kernel_ms(ctx.h)))
            ops.append(a.elapsed_time(b))
        lib.tfl_debug_time_advect_kernel(ctx.h, 0)
        op_ms = float(np.mean(ops))
        k_ms = float(np.mean(ks)) if min(ks) > 0 else op_ms
        algo_bytes = ALGO_BYTES["advect_vel"] * n ** 3
        achieved = algo_bytes / (k_ms * 1e-3) / 1e9
        traffic, traffic_src = ncu_traffic([r"k_advect_vel_tile"]) if n == 128 else (None, None)

        # ---- BASELINE config 4: 100-iteration Jacobi sweep (stencil HBM roofline) ----------
        extra = []
        if rank == 0 and not args.no_extra:
            from fluidnet_b200 import synth as _synth
            for nj in (128, 256):
                fl = torch.from_numpy(_synth.make_flags(nj, nj, nj, True, nb=1, geometry=True)).cuda()
                dv = torch.randn(1, 1, nj, nj, nj, device="cuda") * (fl == 1)
                pj = torch.zeros_like(fl)
                lib.tfl_solve_linear_system_jacobi(ctx.h, tfluids._grid(pj), tfluids._grid(fl), tfluids._grid(dv),
                                                   1, 0.0, 100, None, None)
                a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                flush.fill_(0.0)
                a.record(stream)
                ctx.check(lib.tfl_solve_linear_system_jacobi(ctx.h, tfluids._grid(pj), tfluids._grid(fl),
                                                             tfluids._grid(dv), 1, 0.0, 100, None, None))
                b.record(stream)
                stream.synchronize()
                ms_j = a.elapsed_time(b)
                ach = 16.0 * nj ** 3 * 100 / (ms_j * 1e-3) / 1e9
                extra.append({"kernel": "Jacobi x100 (k_jacobi_mask + %s), %d^3"
                                        % ("100 x k_jacobi_march" if nj >= 256 else
                                           "k_jacobi_resident: 99 sweeps in one cooperative launch + 1 x k_jacobi_iter4", nj),
                              "bound": "hbm", "achieved": ach, "peak": peak, "unit": "GB/s", "frac": ach / peak,
                              "ms": ms_j, "algorithmic_bytes_per_voxel_iter": 16})
                if nj == 128:
                    # ---- BASELINE config 4, second half: PCG, ic0, tol 1e-4, maxIter 100 (lib/simulate.lua:280-286).
                    # Right-hand side = divergence of a wall-conditioned smooth velocity (compatible per component).
                    Uj = torch.from_numpy(_synth.make_smooth_velocity(fl.cpu().numpy(), True, amp=2.0)).cuda()
                    tfluids.setWallBcsForward(Uj, fl)
                    tfluids.velocityDivergenceForward(Uj, fl, dv)
                    res_p, it_p = ctypes.c_float(0), ctypes.c_int(0)
                    for _ in range(2):
                        flush.fill_(0.0)
                        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                        a.record(stream)
                        ctx.check(lib.tfl_solve_linear_system_pcg(ctx.h, tfluids._grid(pj), tfluids._grid(fl),
                                                                  tfluids._grid(dv), 1, 2, 1e-4, 100,
                                                                  ctypes.byref(res_p), ctypes.byref(it_p)))
                        b.record(stream)
                        stream.synchronize()
                    extra.append({"kernel": "PCG ic0 tol 1e-4 maxIter 100 (k_sweep + k_direction_spmv + k_update per "
                                            "iteration), 128^3", "bound": "latency (wavefront-sequential triangular solves)",
                                  "ms": a.elapsed_time(b), "iterations": it_p.value, "residual": res_p.value,
                                  "ms_per_iteration": a.elapsed_time(b) / max(it_p.value, 1)})
                    del Uj
                del fl, dv, pj

    # ---- BASELINE config 5 beside the headline: ONE 256^3 domain in z-slabs over the same ranks (strong scaling)
    slab = None
    if not args.no_slab:
        del gb
        torch.cuda.empty_cache()
        try:
            slab = measure_slab(args.slab_grid, max(3, min(args.steps, 10)), 3, world, rank, local)
        except Exception as e:                      # the sub-record must not take the headline down with it
            slab = {"error": "%s: %s" % (type(e).__name__, e)} if rank == 0 else None

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return 0

    cpu = None
    if not args.no_cpu_baseline and world == 1:
        use_all_host_cores()
        import oracle
        be = oracle.Reference() if oracle.have_reference() else oracle.Oracle()
        b2, m2, _ = make_problem(n)
        ts = []
        for it in range(4):                    # 1 warm-up + 3 timed steps, median
            t0 = time.perf_counter()
            cpu_step_ops(be, b2, m2, None)
            if it > 0:
                ts.append(time.perf_counter() - t0)
        t1 = float(np.median(ts))
        cpu = {"value": 1.0 / t1, "unit": "steps/s", "cores": be.num_threads(),
               "kind": "reference" if be.name == "reference" else "port",
               "sample": "median of 3 full %d^3 steps (after 1 warm-up) of the reference CPU operators (advection, "
                         "BCs, buoyancy, vorticity, wall BCs, divergence, velocity update; CNN conv stack replaced "
                         "by 1 Jacobi sweep: no CPU conv source in the reference)" % n}

    # Headline: the step replayed from a CUDA graph (tfl_step_graph_launch: the same kernels, one launch per step,
    # results bit-identical to tfl_simulate_step -- tests/test_gpu_step.py); the kernel-by-kernel launch of the same
    # step is reported beside it (it depends on how fast the box's host enqueues ~25 stream operations per step).
    ms_direct = total_ms / args.steps
    ms = graph_ms / args.steps
    line = {
        "metric": "sim steps/sec on 128^3 MAC grid (CNN proj)",
        "value": world * 1000.0 / ms, "unit": "steps/s", "n_gpus": world, "steps": args.steps,
        "warmup": max(args.warmup, 3), "ms_per_step": ms, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": "3D %d^3 MAC grid per GPU, maccormackOurs advection (density+velocity) + plume "
                               "BCs + buoyancy + vorticity confinement + CNN projection (3-D default net), "
                               "1 tfluids.simulate per step" % n,
                   "grid": [n, n, n], "batch_per_gpu": 1, "parallelism": "independent grid per GPU",
                   "l2": "256 MB buffer written between timed steps (L2 flush)",
                   "velocity": "band-limited (4 Fourier modes per component), +-2 cells/s at step 0",
                   "max_u_dt_cells_at_end": max_u_dt},
        "launch_mode": ("CUDA graph replay (tfl_step_graph_launch), one launch per step" if graph_error is None else
                        "kernel by kernel (graph capture failed: %s)" % graph_error),
        "ungraphed": {"value": world * 1000.0 / ms_direct, "unit": "steps/s", "ms_per_step": ms_direct,
                      "what": "the same step through tfl_simulate_step, kernel by kernel"},
        "variant_random_velocity": variant,
        "hbm_gbs_algorithmic": BYTES_PER_VOXEL_STEP * n ** 3 / (ms * 1e-3) / 1e9,
        "e2e": {"value": world * e2e_steps / e2e_s, "unit": "steps/s", "h2d_bytes_per_step": bytes_io,
                "d2h_bytes_per_step": bytes_io},
        "gpu_launches": int(graph_launches),
        "roofline": {"bound": "hbm", "kernel": "k_advect_vel_tile (advectVel, maccormackOurs): the step's longest kernel, timed "
                                                  "alone with CUDA events around its launch",
                     "operator_ms": op_ms,
                     "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                     "traffic": traffic, "traffic_source": traffic_src,
                     "algorithmic_bytes": algo_bytes, "peak_source": peak_src, "kernel_ms": k_ms,
                     "limiter": "instruction issue, not HBM: 1567 warp-instructions per 32 voxels at 72 % issue-active "
                                "(profiles/r02_advect_tile_*)"},
        "roofline_extra": extra,
        "slab": slab,
        "cpu_baseline": cpu,
        "clocks": sampler.summary(),
    }
    print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    # The contract is ONE JSON line on stdout: libraries that write to fd 1 (NCCL prints its version there when a
    # communicator is created) are sent to stderr; only print() below reaches the real stdout.
    sys.stdout.flush()
    _real = os.dup(1)
    os.dup2(2, 1)
    sys.stdout = os.fdopen(_real, "w")
    rc = main()
    sys.stdout.flush()
    sys.exit(rc)
