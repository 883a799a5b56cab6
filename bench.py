#!/usr/bin/env python
"""bench.py -- ns/day of the B200-native OpenMM hot path (BASELINE.json metric) + roofline of the dominant kernel.

    python bench.py --gpus N --steps K --warmup W            # our arm (CUDA, through the C-ABI)
    python bench.py --impl reference --gpus N --steps K ...  # the reference's own CPU platform on the host cores

One bench "step" = `--md-steps` MD steps (default 500 = 1 ps at 2 fs) of the workload: force evaluation (tile list
check/rebuild, direct-space tile kernel, PME spread + bespoke FFT/convolution + gather, exclusion corrections) and the
fused Langevin+SETTLE/SHAKE update.  Default workload `dhfr` = BASELINE.json configs[1]: the real DHFR benchmark system
(23,558 atoms, amber99sb + tip3p, PME 0.9 nm, 56^3 grid, HBonds + rigid water, Langevin 2 fs) from data/dhfr.npz, which
tools/make_benchmark_systems.py builds with the reference's own forcefield.py.  Others: `apoa1` (92,224 atoms, 88^3),
`water24k` (S1 of SURVEY.md 8d), `water1m` (S4).
N > 1 (torchrun, one process per GPU): the SAME system on N GPUs by force decomposition -> "scaling": "strong".
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
import numpy as np  # noqa: E402


# what the inputs are: the real benchmark structures where the reference ships them (built here by the reference's own
# forcefield.py, tools/make_benchmark_systems.py), synthetic water boxes otherwise; velocities are always synthetic
DATA_NOTE = {"dhfr": "real DHFR benchmark system of the reference (5dfr_solv-cube_equil.pdb, amber99sb+tip3p via the reference's forcefield.py); synthetic velocities",
             "apoa1": "real ApoA1 benchmark system of the reference (apoa1.pdb, amber14+lipid17+tip3p via the reference's forcefield.py); synthetic velocities",
             "water24k": "synthetic", "water1m": "synthetic"}


def load_workload(name):
    from openmm_b200 import systems
    if name == "water24k":
        return systems.water_box(20, cutoff=0.9).rounded()
    if name == "water1m":
        d = systems.water_box(69, cutoff=0.9).rounded()      # 985,527 atoms (SURVEY.md 8d S4)
        d.pme_alpha, d.pme_grid = d.pme_parameters()[0], (128, 128, 128)
        return d
    path = os.path.join(ROOT, "data", name + ".npz")
    if os.path.exists(path):
        return systems.SystemDesc.load(path).rounded()
    raise SystemExit("unknown workload %s (no %s)" % (name, path))


class ClockSampler(threading.Thread):
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md)."""
    Q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.rows, self.stop_flag = index, [], False

    def run(self):
        while not self.stop_flag:
            try:
                out = subprocess.run(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits"],
                                     capture_output=True, text=True, timeout=5).stdout.strip()
                if out:
                    self.rows.append([x.strip() for x in out.split(",")])
            except Exception:
                pass
            time.sleep(0.2)

    def summary(self):
        if not self.rows:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["unavailable"]}
        sm = sorted(float(r[0]) for r in self.rows if r[0].replace(".", "").isdigit())
        reasons = set()
        for r in self.rows:
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": sm[len(sm)//2] if sm else None, "sm_max_mhz": float(self.rows[0][1]) if self.rows[0][1].isdigit() else None,
                "power_w_max": max(float(r[2]) for r in self.rows if r[2].replace(".", "").isdigit()), "samples": len(self.rows),
                "reasons": sorted(reasons)}


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        return json.load(open(p))["hbm_gbs"], "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


def run_reference(args, rank, world):
    """The reference's own CPU implementation of the path (platforms/cpu, all host threads) through the reference's
    public API (Context / LangevinIntegrator.step), oracle/_ref build of the unmodified sources."""
    if rank != 0:
        return
    from oracle import omm
    from openmm_b200 import systems
    d = load_workload(args.workload)
    omm.load_plugin(os.path.join(ROOT, "oracle", "_ref", "libOpenMMCPU.so"))
    cores = os.cpu_count()
    md = args.ref_md_steps
    sim = omm.Simulation(d, "CPU", integrator=(systems.INT_LANGEVIN, 300.0, 1.0, args.dt), seed=7, pme=d.pme_parameters(), props="Threads=%d" % cores)
    for _ in range(args.warmup):
        sim.step(md)
    sim.state(energy=True)
    t0 = time.time()
    for _ in range(args.steps):
        sim.step(md)
    sim.state(energy=True)
    sec = time.time() - t0
    nsday = args.dt*1e-3*md*args.steps*86400/sec
    line = {"impl": "reference", "metric": "ns/day", "value": nsday, "unit": "ns/day", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": 1e3*sec/args.steps, "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32",
            "data": DATA_NOTE.get(args.workload, "synthetic"), "config": {"workload": args.workload, "atoms": d.natoms, "md_steps_per_step": md, "dt_fs": args.dt*1e3,
                                            "platform": "reference CPU platform (platforms/cpu), reference PME (no FFTW)", "pme_grid": list(d.pme_parameters()[1:])},
            "cpu_baseline": {"value": nsday, "unit": "ns/day", "cores": cores, "kind": "reference", "sample": "%d x %d MD steps" % (args.steps, md)},
            "e2e": {"value": nsday, "unit": "ns/day", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}, "gpu_launches": 0}
    print(json.dumps(line), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default=os.environ.get("B200MD_WORKLOAD"),
                    help="dhfr (default on 1 GPU: BASELINE.json configs[1]), apoa1 (default on N > 1 GPUs: configs[3]), water24k, water1m")
    ap.add_argument("--via", default="plugin", choices=["plugin", "cabi"],
                    help="e2e leg: through the OpenMM Platform plugin (Context + LangevinIntegrator.step) or through the bare C-ABI")
    ap.add_argument("--md-steps", type=int, default=500)
    ap.add_argument("--ref-md-steps", type=int, default=10)
    ap.add_argument("--dt", type=float, default=0.002)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the last timed step, write DIR/positions.npy and DIR/velocities.npy (nm, nm/ps; float64)")
    args = ap.parse_args()
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if args.workload is None:
        args.workload = "dhfr" if max(world, args.gpus) == 1 else "apoa1"
    if args.impl == "reference":
        return run_reference(args, rank, world)

    import torch
    import torch.distributed as dist
    from openmm_b200 import systems, Engine, _lib
    import ctypes as C
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the B200 hot path has no CPU fallback")
    torch.cuda.set_device(local)
    comm = None
    if world > 1:
        # control plane on gloo (CPU tensors), data plane = the engine's own NCCL communicator: torch never enqueues an NCCL
        # kernel next to the engine's in-graph collectives (two communicators racing on one GPU can deadlock)
        dist.init_process_group("gloo")
        os.environ.setdefault("B200MD_NCCL_LIB", os.path.join(os.path.dirname(torch.__file__), "..", "nvidia", "nccl", "lib", "libnccl.so.2"))
        uid = torch.zeros(128, dtype=torch.uint8)
        if rank == 0:
            buf = C.create_string_buffer(128)
            assert _lib.load().b200md_comm_unique_id(C.cast(buf, C.c_void_p)) == 0
            uid = torch.frombuffer(bytearray(buf.raw), dtype=torch.uint8).clone()
        dist.broadcast(uid, 0)                       # CPU tensor -> gloo
        comm = (rank, world, bytes(uid.numpy().tobytes()))

    d = load_workload(args.workload)
    # N > 1: the SAME workload on ONE GPU, measured by rank 0 in this very run, so that a scaling efficiency can be formed on a
    # like-for-like basis (the driver's own N=1 run uses the N=1 default workload, DHFR)
    n1 = None
    if world > 1:
        if rank == 0:
            e1 = Engine(d, device=local)
            e1.set_integrator(systems.INT_LANGEVIN, args.dt, 300.0, 1.0, 7, 1e-5)
            e1.step(300 + args.md_steps); e1.synchronize()
            s1 = torch.cuda.ExternalStream(e1.stream(), device=local)
            a0, a1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a0.record(s1); e1.step(2*args.md_steps); a1.record(s1); e1.synchronize()
            ms1 = a0.elapsed_time(a1)/2
            n1 = {"workload": args.workload, "n_gpus": 1, "value": args.dt*1e-3*args.md_steps*86400/(ms1*1e-3), "unit": "ns/day", "us_per_md_step": 1e3*ms1/args.md_steps,
                  "note": "same workload, single-GPU engine, rank 0 of this run, %d MD steps device-timed" % (2*args.md_steps)}
            e1.close()
        dist.all_reduce(torch.zeros(1))
    eng = Engine(d, device=local, comm=comm)
    eng.set_integrator(systems.INT_LANGEVIN, args.dt, 300.0, 1.0, 7, 1e-5)
    stream = torch.cuda.ExternalStream(eng.stream(), device=local)
    flush = torch.empty(256*1024*1024, dtype=torch.uint8, device="cuda")      # > 126 MB L2

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.all_reduce(torch.zeros(1))          # gloo barrier (CPU tensor)
        torch.cuda.synchronize()

    md = args.md_steps
    # equilibrate off the lattice so that the timed region is steady-state MD
    eng.step(300)
    for _ in range(args.warmup):
        with torch.cuda.stream(stream):
            flush.zero_()                     # also warms torch's lazily loaded fill kernel outside the timed region
        eng.step(md)
    eng.synchronize()
    st0 = eng.stats()
    sampler = ClockSampler(local)
    sampler.start()
    barrier()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record(stream)
    for _ in range(args.steps):
        with torch.cuda.stream(stream):
            flush.zero_()                     # L2 flush between timed iterations (inside the timed region)
        eng.step(md)
    ev1.record(stream)
    barrier()
    ms = ev0.elapsed_time(ev1)
    sampler.stop_flag = True
    st1 = eng.stats()
    if world > 1:
        t = torch.tensor([ms])
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t.item())
    nsday = args.dt*1e-3*md*args.steps*86400/(ms*1e-3)

    # ---- end to end with HOST buffers: upload the state, run, read back positions + velocities + energy ----
    # --via plugin (default, single GPU): through the reference's public API -- Context.setPositions/setVelocities,
    # LangevinIntegrator.step(md), Context.getState -- on the B200 Platform plugin (libOpenMMB200.so, plugin/, loaded into the
    # unmodified libOpenMM.so as its host application); --via cabi (and N > 1): the same calls on the bare C-ABI.
    x = eng.get_positions()
    v = eng.get_velocities()
    if args.dump_outputs and rank == 0:
        # every rank holds the same state; 48 bytes per atom, 47 MB for the largest workload (water1m)
        os.makedirs(args.dump_outputs, exist_ok=True)
        np.save(os.path.join(args.dump_outputs, "positions.npy"), x)
        np.save(os.path.join(args.dump_outputs, "velocities.npy"), v)
    via = args.via if world == 1 else "cabi"
    e2e_launches = 0
    e2e_sec = None
    plugin_lib = os.path.join(ROOT, "oracle", "_ref", "plugins", "libOpenMMB200.so")
    if via == "plugin" and not os.path.exists(plugin_lib):
        pass                                  # the plugin needs the reference headers to build; reported as not measured below
    elif via == "plugin":
        from oracle import omm                # the host application (reference libOpenMM.so + ctypes shim); compute is the plugin's
        omm.load_plugin(plugin_lib)
        sim = omm.Simulation(d, "B200", integrator=(systems.INT_LANGEVIN, 300.0, 1.0, args.dt), seed=7, constraint_tol=1e-5, pme=d.pme_parameters(),
                             props="DeviceIndex=%d" % local)
        assert sim.platform() == "B200"
        sim.set_positions(x); sim.set_velocities(v)
        sim.step(md)                          # captures the step graph outside the timed region
        sim.state(energy=True)
        t0 = time.perf_counter()
        for _ in range(args.steps):
            sim.set_positions(x)
            sim.set_velocities(v)
            sim.step(md)
            st = sim.state(positions=True, velocities=True)
            x, v = st["positions"], st["velocities"]
        e_final = sim.state(energy=True)["potential"]
        e2e_sec = time.perf_counter() - t0
        sim.close()
    else:
        barrier()
        t0 = time.perf_counter()
        for _ in range(args.steps):
            eng.set_positions(x)
            eng.set_velocities(v)
            eng.step(md)
            x = eng.get_positions()
            v = eng.get_velocities()
        e_final = eng.compute()
        barrier()
        e2e_sec = time.perf_counter() - t0
    if world > 1:
        t = torch.tensor([e2e_sec])
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        e2e_sec = float(t.item())
    e2e_nsday = args.dt*1e-3*md*args.steps*86400/e2e_sec if e2e_sec is not None else None
    nbytes = d.natoms*3*8

    if world > 1:
        barrier()
        dist.destroy_process_group()
    if rank != 0:
        return
    # ---- roofline of the dominant kernel (the direct-space tile kernel), timed live with CUDA events on its stream ----
    pair_ms = eng.time_phase("pair", 50)
    st = eng.stats()
    T, X, NP = st["num_tiles"], st["num_mask_tiles"], st["padded_atoms"]
    alg_bytes = T*(32*4 + 4 + 4) + X*32*4 + NP*(16 + 8) + NP*24       # tiles (j list, i block, mask idx) + masks + posq/sigeps read + force write
    peak, peak_src = peaks()
    achieved = alg_bytes/(pair_ms*1e-3)/1e9
    # dram__bytes_read.sum + dram__bytes_write.sum of one `ncu --set full` capture of this kernel ON THIS WORKLOAD
    # (tools/summarize_profile.py writes profiles/r02_<workload>_k_pair_summary.json); null when no capture exists
    traffic = None
    tpath = os.path.join(ROOT, "profiles", "r02_%s_k_pair_summary.json" % args.workload)
    if os.path.exists(tpath):
        tj = json.load(open(tpath))
        traffic = tj["dram_bytes_read"] + tj["dram_bytes_write"]
    phases = {ph: round(eng.time_phase(ph, 30)*1e3, 2) for ph in ("pair", "pme_spread", "pme_fft_conv", "pme_gather", "bonded", "integrate", "list_build")}
    flops = T*1024*60.0
    line = {"metric": "ns/day", "value": nsday, "unit": "ns/day", "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms/args.steps,
            "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": DATA_NOTE.get(args.workload, "synthetic"),
            "config": {"workload": args.workload, "atoms": d.natoms, "md_steps_per_step": md, "dt_fs": args.dt*1e3, "integrator": "Langevin 300K 1/ps + SETTLE/SHAKE (HBonds)",
                       "cutoff_nm": d.cutoff, "pme_grid": st["pme_grid"], "parallelism": ("owner decomposition over %d ranks, peer-memory data plane: tiles by i-block, forces reduced to the owners and positions "
                                       "published by the integrate kernel through NVLink stores, x-slab-decomposed PME FFT with the transposes fused into the FFT kernels' stores; "
                                       "no NCCL call on the step path" % world) if world > 1 and os.environ.get("B200MD_MGPU", "p2p") != "nccl" else
                                      (("replicated atoms: %d direct-space ranks + 1 PME rank, int64 force all-reduce (NCCL)" % (world-1)) if world > 1 else "single GPU"),
                       "l2": "256 MiB buffer written between timed iterations (inside the timed region)", "us_per_md_step": 1e3*ms/(args.steps*md)},
            "clocks": sampler.summary(),
            "e2e": {"value": e2e_nsday, "unit": "ns/day", "h2d_bytes_per_step": 2*nbytes, "d2h_bytes_per_step": 2*nbytes + 8,
                    "via": "OpenMM Platform plugin: Context.setPositions/setVelocities + LangevinIntegrator.step + Context.getState (libOpenMMB200.so)" if via == "plugin" else "C-ABI (b200md_set_positions/.../b200md_step)",
                    "note": ("per bench step: positions+velocities from host doubles, %d MD steps, positions+velocities back; final energy %.1f" % (md, e_final))
                    if e2e_sec is not None else "not measured: the plugin library %s is not built" % os.path.relpath(plugin_lib, ROOT)},
            "gpu_launches": int(st1["kernel_launches"] - st0["kernel_launches"]),
            "roofline": {"kernel": "k_pair (direct-space 32x32 tile kernel)", "bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved/peak,
                         "traffic": traffic, "peak_source": peak_src, "algorithmic_bytes_per_launch": alg_bytes, "kernel_ms": pair_ms,
                         "tiles": T, "pairs_in_cutoff": st["pairs_in_cutoff"], "tile_fill": st["pairs_in_cutoff"]/(T*1024.0),
                         "fp32_tflops_all_slots": flops/(pair_ms*1e-3)/1e12,       # 60 flop x every evaluated slot, in or out of the cutoff
                         "fp32_tflops_useful_pairs": st["pairs_in_cutoff"]*60.0/(pair_ms*1e-3)/1e12,
                         "note": "compute (FP32/SFU) bound kernel: arithmetic intensity ~%.0f flop/B; see DESIGN.md" % (flops/alg_bytes)},
            "phases_us": phases, "list_builds_in_timed_region": int(st1["list_builds"] - st0["list_builds"])}
    if n1 is not None:
        line["scaling_basis"] = ("N > 1 runs ApoA1 (BASELINE.json configs[3]); the N = 1 default of this bench is DHFR (configs[1]), so a scaling "
                                 "efficiency must be formed against single_gpu_same_workload (ApoA1 on ONE GPU, measured by rank 0 in this run)")
        line["single_gpu_same_workload"] = n1
        line["speedup_vs_single_gpu_same_workload"] = nsday/n1["value"]
    if not args.no_cpu_baseline and world == 1:          # the CPU baseline is a rank-0, N = 1 leg (the reference arm covers N > 1)
        try:
            from oracle import omm
            omm.load_plugin(os.path.join(ROOT, "oracle", "_ref", "libOpenMMCPU.so"))
            cores = os.cpu_count()
            sim = omm.Simulation(d, "CPU", integrator=(systems.INT_LANGEVIN, 300.0, 1.0, args.dt), seed=7, pme=d.pme_parameters(), props="Threads=%d" % cores)
            sim.step(5)
            t0 = time.time()
            n = 0
            while time.time() - t0 < 12.0:
                sim.step(10)
                n += 10
            sim.state(energy=True)
            sec = time.time() - t0
            line["cpu_baseline"] = {"value": args.dt*1e-3*n*86400/sec, "unit": "ns/day", "cores": cores, "kind": "reference",
                                    "sample": "%d MD steps of the same workload on the reference CPU platform (platforms/cpu, %d threads)" % (n, cores)}
        except Exception as ex:       # the baseline is a reported number, never the product path
            line["cpu_baseline"] = {"value": None, "unit": "ns/day", "cores": os.cpu_count(), "kind": "reference", "sample": "failed: %s" % ex}
    print(json.dumps(line), flush=True)


if __name__ == "__main__":
    main()
