#!/usr/bin/env python
"""bench.py — f64 lattice updates/s (GLUPS) of the imaginary-time FDTD hot path.

  python bench.py --gpus N --steps K --warmup W          # B200 arm (this repo's CUDA path)
  python bench.py --impl reference --gpus N ...          # reference arm: the CPU restatement of the
                                                         # reference's rayon path on the host cores
  python bench.py --workload C5 --gpus N ...             # weak-scaling config (2048 x 2048 x 256 per GPU)

Workload C4 (BASELINE.json configs[3], the default): 1024^3, ThreePoint, gen_potential.py's Poschl-Teller
potential, Boolean initial condition, ground state; x-slab decomposed over N GPUs of one box (strong scaling).
One "step" is one `evolve(wnum=0, screen_update)` call = SWEEPS lattice sweeps (grid.rs:544-687; default 1000 =
wafer.yaml:98).  `value` counts nx*ny*nz*SWEEPS*K updates over the max-over-ranks device time; `e2e` adds, every
step, the host->device copy of psi before evolve, one observables check (grid.rs:127-135) and the device->host copy
of the evolved psi after it (what a stateless drop-in of the reference's loop body has to do).  `parity` compares
the measured path bit-for-bit with an independent path of the same library (N = 1: the one-step register-queue
kernel; N > 1: a single-GPU run of the whole lattice) through wafer_phi_checksum.  Prints ONE JSON line on rank 0.

  python bench.py --gpus 1 --steps K --warmup W --dump-outputs DIR

also writes DIR/phi.npy: psi as the last timed step left it, sampled at a fixed set of work sites (see dump_outputs).
The inputs are generated on the device from the arguments alone, so two builds run with the same arguments can be
compared output for output.
"""
import argparse
import json
import os
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

BYTES_PER_UPDATE = 32.0  # SURVEY.md §8(d): read psi, A, B + write psi', 8 B each
FALLBACK_HBM_GBS = 6650.0  # /opt/skills/guides/B200_PROFILING.md fallback


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="C4", choices=["C4", "C5"],
                    help="C4: 1024^3 Poschl-Teller, strong scaling (default); C5: 2048 x 2048 x (256 per GPU) harmonic, weak scaling")
    ap.add_argument("--grid", type=int, default=0, help="lattice edge N (N^3 work sites); default from --workload")
    ap.add_argument("--nx", type=int, default=0,
                    help="x extent (the decomposed axis) if not N: e.g. --grid 2048 --nx 256 is one GPU's share of C5")
    ap.add_argument("--sweeps", type=int, default=1000,
                    help="lattice sweeps per step = output.screen_update; 1000 is the reference's default (wafer.yaml:98)")
    ap.add_argument("--stencil", default="ThreePoint", choices=["ThreePoint", "FivePoint", "SevenPoint"])
    ap.add_argument("--flags", type=int, default=0, help="wafer_params.flags (1 = A/B arrays, 4 = simple sweep)")
    ap.add_argument("--no-p2p", action="store_true", help="multi-GPU: NCCL send/recv halos instead of fused peer stores")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-512", action="store_true")
    ap.add_argument("--no-parity", action="store_true")
    ap.add_argument("--parity-sweeps", type=int, default=200)
    ap.add_argument("--cpu-grid", type=int, default=512, help="edge of the CPU sample lattice when the full one does not fit")
    ap.add_argument("--cpu-lattice", default="auto", choices=["auto", "sample"],
                    help="reference arm: auto = the workload's own lattice when 1.5x its five fields fit in free host memory")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="single GPU: after the timed steps write DIR/phi.npy, a fixed float64 sample of the evolved psi")
    a = ap.parse_args()
    if a.steps < 1 or a.warmup < 0:
        ap.error("--steps must be >= 1 and --warmup >= 0")
    world = int(os.environ.get("WORLD_SIZE", "1")) if a.impl == "b200" else max(a.gpus, 1)
    if a.dump_outputs and (a.impl != "b200" or world > 1):
        ap.error("--dump-outputs needs the B200 arm on a single GPU")
    if a.workload == "C5":
        a.grid = a.grid or 2048
        a.nx = a.nx or 256 * world
        a.potential, a.scaling = "Harmonic", "weak"
    else:
        a.grid = a.grid or 1024
        a.potential, a.scaling = "PoschlTeller", "strong"
    return a


def physical_params(args, n):
    """dn, dt, mass.  C4: box of width 10.24 (dn 0.01 at 1024), dt = 0.3 dn^2; C5: SURVEY §8(d) dn 0.005, dt 8e-6."""
    if args.workload == "C5" and n == args.grid:
        return 0.005, 8e-6, 1.0
    dn = 10.24 / n
    return dn, 0.3 * dn * dn, 1.0


def physical_cores():
    """the reference sizes its rayon pool with num_cpus::get_physical() (main.rs:190-192)"""
    try:
        import psutil
        return psutil.cpu_count(logical=False) or os.cpu_count() or 1
    except Exception:
        return os.cpu_count() or 1


# ------------------------------------------------------------------------------------------------- clocks
class ClockSampler:
    """Samples SM clock and throttle reasons of one GPU during the timed region (NVML, 100 ms period)."""
    REASONS = {0x8: "hw_slowdown", 0x40: "hw_thermal_slowdown", 0x20: "sw_thermal_slowdown", 0x4: "sw_power_cap",
               0x80: "hw_power_brake_slowdown"}

    def __init__(self, index):
        self.samples, self.reasons, self.max_mhz, self._stop, self._t = [], set(), None, threading.Event(), None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self.nv = None

    def _run(self):
        while not self._stop.is_set():
            try:
                self.samples.append(self.nv.nvmlDeviceGetClockInfo(self.h, self.nv.NVML_CLOCK_SM))
                mask = self.nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                for bit, name in self.REASONS.items():
                    if mask & bit:
                        self.reasons.add(name)
            except Exception:
                pass
            self._stop.wait(0.1)

    def start(self):
        if self.nv:
            self._t = threading.Thread(target=self._run, daemon=True)
            self._t.start()

    def stop(self):
        self._stop.set()
        if self._t:
            self._t.join()
        s = sorted(self.samples)
        return {"sm_mhz": s[len(s) // 2] if s else None, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons),
                "samples": len(s)}


# ------------------------------------------------------------------------------------------------- CPU arm
def cpu_arm(args, steps, warmup, budget_s, full_lattice):
    """The reference's CPU path (its Rust cannot be built here — SURVEY F2/F3 — so: the C++ restatement with the
    reference's own pass structure, oracle/wafer_oracle.cpp) timed on the host's physical cores on a bounded sample:
    each step is a few of the workload's `sweeps` sweeps.  full_lattice: use the workload's real lattice when host
    memory allows (5 fields of it), else a --cpu-grid^3 sub-lattice; the choice is written into `sample`."""
    import numpy as np

    from oracle import binding as oracle
    n = args.grid
    nx = args.nx or n
    need = 5.2 * nx * n * n * 8
    avail = 0
    try:
        import psutil
        avail = psutil.virtual_memory().available
    except Exception:
        pass
    if not full_lattice or args.cpu_lattice == "sample" or avail < need * 1.5:
        nx = n = args.cpu_grid
    dn, dt, mass = physical_params(args, args.grid)
    ext = {"ThreePoint": 1, "FivePoint": 2, "SevenPoint": 3}[args.stencil]
    cores = physical_cores()
    oracle.set_num_threads(cores)
    g = oracle.make_grid(nx, n, n, ext=ext, dn=dn, dt=dt, mass=mass)
    v = oracle.potential(g, args.potential)
    a, b = oracle.build_ab(v, dt)
    del v
    phi = oracle.initial_condition(g, "Boolean")
    work = np.zeros(g.work_shape)  # grid.rs:560, allocated once per 1000-sweep evolve call in the reference
    t0 = time.perf_counter()
    oracle.evolve(g, phi, a, b, 1, work=work)   # also faults the pages in
    oracle.evolve(g, phi, a, b, 1, work=work)
    t1 = (time.perf_counter() - t0) / 2
    per_step = max(1, min(50, int(budget_s / max(steps + warmup, 1) / max(t1, 1e-3))))
    for _ in range(warmup):
        oracle.evolve(g, phi, a, b, per_step, work=work)
    times = []
    for _ in range(steps):
        t0 = time.perf_counter()
        oracle.evolve(g, phi, a, b, per_step, work=work)
        times.append(time.perf_counter() - t0)
    el = sum(times)
    sites_ = nx * n * n
    rate = lambda t: sites_ * per_step / t / 1e9
    ts = sorted(times)
    return {"value": sites_ * per_step * steps / el / 1e9, "unit": "GLUPS", "cores": oracle.num_threads(), "kind": "port",
            "sample": "%dx%dx%d lattice (%s), %d steps x %d of the step's %d sweeps of oracle evolve (stencil into work + "
                      "copy-back, grid.rs:560-673; work array pre-allocated as the reference amortises it over the whole "
                      "call), OpenMP on %d threads = physical cores (main.rs:190-192)"
                      % (nx, n, n, "the workload's own lattice" if (nx, n) == (args.nx or args.grid, args.grid) else "sub-lattice of the workload: host memory",
                         steps, per_step, args.sweeps, oracle.num_threads()),
            "spread": {"min": rate(ts[-1]), "median": rate(ts[len(ts) // 2]), "max": rate(ts[0]), "repetitions": len(ts)},
            "ms_per_step": el / steps * 1e3, "sweeps_per_step": per_step, "lattice": [nx, n, n]}


def reference_main(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cb = cpu_arm(args, args.steps, args.warmup, budget_s=75.0, full_lattice=True)
    cfg = workload_config(args, args.gpus)
    cfg["reference_sample"] = {"lattice": cb["lattice"], "sweeps_per_step": cb["sweeps_per_step"],
                               "note": "a CPU step is a bounded sample (sweeps_per_step of the workload's %d sweeps per "
                                       "step); the value is a rate, so it compares with the GPU arm's" % args.sweeps}
    line = {
        "impl": "reference", "metric": "f64 lattice updates/s", "value": cb["value"], "unit": "GLUPS",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": cb["ms_per_step"],
        "higher_is_better": True, "scaling": args.scaling, "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": cfg,
        "cpu_baseline": {k: cb[k] for k in ("value", "unit", "cores", "kind", "sample", "spread")},
        "e2e": {"value": cb["value"], "unit": "GLUPS", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


def workload_config(args, world):
    n = args.grid
    nx = args.nx or n
    pot = {"PoschlTeller": "Poschl-Teller (gen_potential.py formula, lam=6)", "Harmonic": "Harmonic (potential.rs:270-274)"}[args.potential]
    return {"workload": "%s: %dx%dx%d %s, %s, Boolean IC, ground state; step = evolve(wnum=0, screen_update=%d)"
                        % (args.workload, nx, n, n, args.stencil, pot, args.sweeps),
            "grid": [nx, n, n], "stencil": args.stencil, "sweeps_per_step": args.sweeps,
            "decomposition": ("x-slab x%d, halo: %s" % (world, "NCCL send/recv" if args.no_p2p else "fused peer stores (CUDA IPC over NVLink)"))
            if world > 1 else "single GPU",
            "l2": "inputs larger than L2 (%.1f GB per field per GPU vs 126 MB)" % (nx * n * n * 8 / world / 1e9)}


# ------------------------------------------------------------------------------------------------- B200 arm
def measure(lat, args, nsites, dist, steps, warmup, sampler=None):
    """W untimed + K timed evolve(0, sweeps) calls, device-timed with CUDA events on the library's stream."""
    for _ in range(warmup):
        lat.evolve(0, args.sweeps)
    lat.synchronize()
    if dist is not None:
        dist.barrier()
    if sampler:
        sampler.start()
    launches0 = lat.kernel_launches
    lat.timer_begin()
    for _ in range(steps):
        lat.evolve(0, args.sweeps)
    ms = lat.timer_end()
    lat.synchronize()
    launches = lat.kernel_launches - launches0
    clocks = sampler.stop() if sampler else None
    if dist is not None:
        import torch
        t = torch.tensor([ms], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dist.barrier()
        ms = float(t.item())
    glups = nsites * args.sweeps * steps / (ms * 1e-3) / 1e9
    return glups, ms, launches, clocks


DUMP_SITES = 1 << 22  # 32 MB of float64
DUMP_SEED = 0


def dump_outputs(lat, out_dir):
    """Writes out_dir/phi.npy: the float64 values of psi (what get_phi hands a caller of evolve) at DUMP_SITES work
    sites drawn without replacement with seed DUMP_SEED, in C order of the work area (every site when there are
    fewer).  The sites depend only on the lattice shape, so dumps of two builds line up value for value."""
    import numpy as np
    nx, ny, nz = lat.size
    e = lat.ext
    total = nx * ny * nz
    if total <= DUMP_SITES:
        idx = np.arange(total)
    else:
        idx = np.sort(np.random.default_rng(DUMP_SEED).choice(total, DUMP_SITES, replace=False))
    x, yz = np.divmod(idx, ny * nz)
    y, z = np.divmod(yz, nz)
    phi = lat.get_phi()[x + e, y + e, z + e]
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "phi.npy"), phi)


def hbm_peak():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return FALLBACK_HBM_GBS, "fallback (B200_PROFILING.md)"


def ncu_traffic(variant, updates_per_launch):
    """dram__bytes_read+write per launch of the sweep kernel, from the committed `ncu --set full` capture of the
    same kernel (profiles/ncu_traffic.json: measured at 512^3, scaled by updates per launch)."""
    try:
        with open(os.path.join(ROOT, "profiles", "ncu_traffic.json")) as f:
            for rec in json.load(f):
                if variant.startswith(rec["variant"]):
                    return rec["dram_bytes_per_update"] * updates_per_launch, rec["note"]
    except Exception:
        pass
    return None, None


def connect_p2p(lat, dist, rank, world):
    """fused halo: boundary CTAs store into the neighbours' ghost planes through CUDA-IPC mapped peer memory"""
    import torch
    mine = torch.tensor(list(lat.p2p_export()), dtype=torch.uint8, device="cuda")
    blobs = [torch.zeros(192, dtype=torch.uint8, device="cuda") for _ in range(world)]
    dist.all_gather(blobs, mine)
    blobs = [bytes(b.cpu().tolist()) for b in blobs]
    lat.p2p_connect(blobs[rank - 1] if rank > 0 else None, blobs[rank + 1] if rank < world - 1 else None)


def parity_leg(lat, args, shape, phys, local_rank, rank, world, dist):
    """Bit-for-bit comparison of the measured path with an independent one, at the workload's full size.
    N = 1: the time-tiled TMA kernel against the plain one-step register-queue kernel (WAFER_FLAG_SIMPLE_SWEEP).
    N > 1: this rank's slab of the decomposed run against the same planes of a single-GPU run of the WHOLE lattice
    (every rank runs its own copy on its own GPU), after `parity_sweeps` sweeps — long enough for the ranks to
    drift apart — followed by one observables check on both (the check reads the ghost planes)."""
    import wafer_b200
    dn, dt, mass = phys
    s = args.parity_sweeps
    other_flags = wafer_b200.FLAG_SIMPLE_SWEEP if world == 1 else args.flags
    # the comparison run holds the WHOLE lattice on this GPU next to the slab: skip (and say so) when that cannot fit
    field = (shape[0] + 4) * (shape[1] + 2) * (shape[2] + 16) * 8
    need = 4.2 * field + 4.2 * field / world
    total = lat.device_info()["mem_bytes"]
    if need > 0.92 * total:
        return {"skipped": "a single-GPU run of the whole %dx%dx%d lattice (%.0f GB with the slab) does not fit one GPU's %.0f GB"
                           % (shape + (need / 1e9, total / 1e9)), "ok": None}
    x0, x1 = lat.slab
    lat.generate_potential(args.potential)
    lat.set_initial_conditions("Boolean")
    lat.check(0)
    lat.evolve(0, s)
    mine = lat.phi_checksum(x0, x1)
    o_mine = lat.check(0)
    with wafer_b200.Lattice(shape, args.stencil, dn=dn, dt=dt, mass=mass, device=local_rank, flags=other_flags) as ref:
        ref.generate_potential(args.potential)
        ref.set_initial_conditions("Boolean")
        ref.check(0)
        ref.evolve(0, s)
        theirs = ref.phi_checksum(x0, x1)
        o_ref = ref.check(0)
        ref_variant = ref.sweep_variant
    e_mine, e_ref = o_mine["energy"] / o_mine["norm2"], o_ref["energy"] / o_ref["norm2"]
    bit = mine == theirs
    rel = abs(e_mine - e_ref) / abs(e_ref)
    if dist is not None:
        import torch
        t = torch.tensor([0.0 if bit else 1.0, rel], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        bit, rel = bool(t[0].item() == 0.0), float(t[1].item())
    return {"psi_bitwise_equal": bit, "energy_rel_diff": rel, "energy": e_mine, "sweeps": s,
            "against": ("single-GPU run of the whole lattice (%s) on every rank's GPU, compared per slab" % ref_variant) if world > 1
            else "one-step register-queue kernel (%s) on the same GPU" % ref_variant,
            "method": "wafer_phi_checksum (position-sensitive 128-bit sum/xor of per-site hashes) after evolve(0, %d); "
                      "energy from wafer_check on both; tolerance 1e-9 relative (north_star)" % s,
            "ok": bool(bit and rel <= 1e-9)}


def e2e_leg(lat, args, nsites, world, dist, pinned):
    """set_phi_owned(host) -> evolve -> check -> get_phi_slab(host) per step; the state travels through HOST buffers.
    pinned = False: ordinary pageable numpy arrays, which is what the reference's Array3::as_ptr() would hand over;
    pinned = "registered": the same caller-owned arrays page-locked once with wafer_host_register."""
    import numpy as np

    import wafer_b200
    q0, q1 = lat.slab_planes(1)
    shp = (q1 - q0,) + lat.padded_shape[1:]
    if pinned is True:
        h_in, h_out = wafer_b200.pinned_empty(shp), wafer_b200.pinned_empty(shp)
    else:
        h_in, h_out = np.empty(shp), np.empty(shp)
        if pinned == "registered":
            wafer_b200.pin(h_in)
            wafer_b200.pin(h_out)
    lat.get_phi_slab(h_in)
    e_steps, e_warm = (min(args.steps, 3), 1) if pinned is True else (min(args.steps, 2), 1)
    tot, obs = 0.0, None
    for it in range(e_warm + e_steps):
        if dist is not None:
            dist.barrier()
        t0 = time.perf_counter()
        lat.timer_begin()
        lat.set_phi_owned(h_in)     # owned planes from the host; ghost planes re-fetched from the neighbours
        lat.evolve(0, args.sweeps)
        obs = lat.check(0)          # the loop body of grid.rs:126-221: observables + normalise, 4 scalars back to the host
        lat.get_phi_slab(h_out)
        ms_e = lat.timer_end()
        wall = (time.perf_counter() - t0) * 1e3
        ms_e = max(ms_e, wall)      # the copies synchronise the host: count whichever clock saw more
        if dist is not None:
            import torch
            t = torch.tensor([ms_e], dtype=torch.float64, device="cuda")
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms_e = float(t.item())
        if it >= e_warm:
            tot += ms_e
        h_in, h_out = h_out, h_in   # the evolved state is the next step's input
    out = {"value": nsites * args.sweeps * e_steps / (tot * 1e-3) / 1e9, "unit": "GLUPS",
           "h2d_bytes_per_step": int(h_in.size * 8 * world), "d2h_bytes_per_step": int(h_out.size * 8 * world),
           "steps": e_steps, "ms_per_step": tot / e_steps, "host_memory": {True: "pinned (wafer_host_alloc)", False: "pageable (numpy)",
                           "registered": "caller-owned numpy arrays page-locked once (wafer_host_register)"}[pinned],
           "call": "wafer_set_phi_owned(host) -> wafer_evolve(0, %d) -> wafer_check(0) -> wafer_get_phi_slab(host)" % args.sweeps,
           "last_energy": obs["energy"] / obs["norm2"], "checks_seen": e_warm + e_steps}
    if pinned is True:
        wafer_b200.pinned_free(h_in)
        wafer_b200.pinned_free(h_out)
    elif pinned == "registered":
        wafer_b200.unpin(h_in)
        wafer_b200.unpin(h_out)
    return out


def b200_main(args):
    import wafer_b200

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    dist = None
    nccl_id = None
    if world > 1:
        import torch
        import torch.distributed as td
        torch.cuda.set_device(local_rank)
        td.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
        dist = td
        idt = torch.zeros(128, dtype=torch.uint8, device="cuda")
        if rank == 0:
            idt = torch.tensor(list(wafer_b200.nccl_unique_id()), dtype=torch.uint8, device="cuda")
        td.broadcast(idt, 0)
        nccl_id = bytes(idt.cpu().tolist())
    if world != args.gpus and rank == 0:
        sys.stderr.write("warning: --gpus %d but WORLD_SIZE %d; using WORLD_SIZE\n" % (args.gpus, world))

    n = args.grid
    shape = (args.nx or n, n, n)
    phys = physical_params(args, n)
    dn, dt, mass = phys
    nsites = shape[0] * n * n
    lat = wafer_b200.Lattice(shape, args.stencil, dn=dn, dt=dt, mass=mass, device=local_rank, rank=rank, world=world,
                             nccl_id=nccl_id, flags=args.flags)
    if world > 1 and not args.no_p2p:
        connect_p2p(lat, dist, rank, world)

    parity = None
    if not args.no_parity:
        parity = parity_leg(lat, args, shape, phys, local_rank, rank, world, dist)

    lat.generate_potential(args.potential)
    lat.set_initial_conditions("Boolean")
    lat.check(0)  # normalise once so that thousands of sweeps stay in range

    sampler = ClockSampler(local_rank) if rank == 0 else None
    glups, ms, launches, clocks = measure(lat, args, nsites, dist, args.steps, args.warmup, sampler)
    if args.dump_outputs:
        dump_outputs(lat, args.dump_outputs)  # before the e2e legs below replace psi
    sweeps_total = args.sweeps * args.steps

    peak, peak_src = hbm_peak()
    # dominant kernel = the sweep.  The time-tiled kernel advances TWO lattice steps per launch, the plain one a
    # single step; multi-GPU runs add two small boundary-plane launches per pass on the halo stream.  The figure is
    # per main-stream launch: the timed region holds nothing but back-to-back sweep launches.
    steps_per_launch = 2 if lat.sweep_variant.startswith("tb2") else 1
    n_main = sweeps_total // steps_per_launch + sweeps_total % steps_per_launch
    launch_ms = ms / n_main
    updates_per_launch = nsites / world * sweeps_total / n_main
    achieved = BYTES_PER_UPDATE * updates_per_launch / (launch_ms * 1e-3) / 1e9
    traffic, traffic_note = ncu_traffic(lat.sweep_variant, updates_per_launch)
    roofline = {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                "traffic": traffic, "traffic_note": traffic_note, "peak_source": peak_src, "kernel": lat.sweep_variant,
                "algorithmic_bytes_per_update": BYTES_PER_UPDATE, "updates_per_launch": updates_per_launch,
                "steps_per_launch": steps_per_launch, "launch_ms": launch_ms,
                "dram_frac_of_peak": (traffic / (launch_ms * 1e-3) / 1e9 / peak) if traffic else None,
                "frac_of_nominal_8TBps": achieved / 8000.0}

    # ---- e2e: host buffers in and out of every step, through the C ABI
    e2e = None
    if not args.no_e2e:
        e2e = e2e_leg(lat, args, nsites, world, dist, pinned=True)
        keep = ("value", "unit", "ms_per_step", "steps", "host_memory", "last_energy")
        e2e["pageable"] = {k: v for k, v in e2e_leg(lat, args, nsites, world, dist, pinned=False).items() if k in keep}
        e2e["registered"] = {k: v for k, v in e2e_leg(lat, args, nsites, world, dist, pinned="registered").items() if k in keep}

    info = lat.device_info()
    variant = lat.sweep_variant
    lat.close()

    extra = {}
    if rank == 0 and world == 1 and not args.no_512 and n != 512 and not args.nx and args.workload == "C4":
        # BASELINE metric's other quoted point: 512^3 on one GPU
        a2 = argparse.Namespace(**vars(args))
        a2.grid = 512
        dn2, dt2, m2 = physical_params(a2, 512)
        with wafer_b200.Lattice((512,) * 3, args.stencil, dn=dn2, dt=dt2, mass=m2, device=local_rank, flags=args.flags) as l2:
            l2.generate_potential(args.potential)
            l2.set_initial_conditions("Boolean")
            l2.check(0)
            g512, ms512, _, _ = measure(l2, a2, 512 ** 3, None, max(args.steps, 3), 3)
        extra["glups_512cubed_1gpu"] = g512
        extra["hbm_frac_512cubed"] = g512 * BYTES_PER_UPDATE / peak

    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu:
        cpu = cpu_arm(args, steps=3, warmup=1, budget_s=15.0, full_lattice=False)
        cpu = {k: cpu[k] for k in ("value", "unit", "cores", "kind", "sample", "spread")}

    if rank == 0:
        line = {
            "metric": "f64 lattice updates/s", "value": glups, "unit": "GLUPS", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": args.scaling,
            "vs_baseline": None, "dtype": "f64", "data": "synthetic", "config": workload_config(args, world),
            "roofline": roofline, "cpu_baseline": cpu, "e2e": e2e, "parity": parity, "gpu_launches": int(launches),
            "clocks": clocks, "device": info["name"], "sweep_variant": variant, "extra": extra,
        }
        print(json.dumps(line), flush=True)
    if dist is not None:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    a = parse_args()
    if a.impl == "reference":
        reference_main(a)
    else:
        b200_main(a)
