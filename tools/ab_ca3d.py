#!/usr/bin/env python
"""tools/ab_ca3d.py -- A/B of the ca3d row loops inside ONE process: the interior row loop (the default) against the
general row step on every row (CLAPCA_ROWLOOP=generic), on the bench workload -- 2048^3 synthetic seed
(clap_b200/synth.py), 50 generations of ca_coral.  The arms alternate run by run; every run starts from the same
seed (device-to-device upload).  Both arms must leave the SAME volume: the per-plane fingerprints
(clapca_hash_planes, on the device) of each arm's last run are compared.  Prints the median and spread of the sweep
kernel time (CUDA events inside the library) and of the step time per arm, with the card's name, power limit and SM
clock read in the same process.

    python tools/ab_ca3d.py [runs [side [generations]]] [--profile FILE]

--profile FILE: afterwards one more run per arm under torch.profiler (CUDA activities), its kernel-time table to FILE.
"""
import os
import statistics
import subprocess
import sys
import time

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import clap_b200                                         # noqa: E402
from clap_b200 import synth                              # noqa: E402
from clap_b200.ca import hash_planes                     # noqa: E402
from clap_b200.rules import ca3d_rule                    # noqa: E402

CORAL = 7
ARMS = [("generic", "generic"), ("interior", None)]     # (name, CLAPCA_ROWLOOP)


def card():
    q = "name,power.limit,clocks.sm,clocks.max.sm,temperature.gpu"
    try:
        r = subprocess.run(["nvidia-smi", "-i", os.environ.get("CUDA_VISIBLE_DEVICES", "0").split(",")[0],
                            f"--query-gpu={q}", "--format=csv,noheader"], capture_output=True, text=True, timeout=30)
        return f"{q}: {r.stdout.strip()}"
    except (OSError, subprocess.SubprocessError) as e:
        return f"{torch.cuda.get_device_name(0)} (nvidia-smi unavailable: {e})"


def spread(v):
    return f"median {statistics.median(v):8.3f}  min {min(v):8.3f}  max {max(v):8.3f}  (max-min {max(v) - min(v):6.3f})"


def set_arm(val):
    if val is None:
        os.environ.pop("CLAPCA_ROWLOOP", None)
    else:
        os.environ["CLAPCA_ROWLOOP"] = val


def main():
    argv = sys.argv[1:]
    prof_out = None
    if "--profile" in argv:
        i = argv.index("--profile")
        prof_out = argv[i + 1]
        del argv[i:i + 2]
    runs = int(argv[0]) if len(argv) > 0 else 7
    side = int(argv[1]) if len(argv) > 1 else 2048
    gens = int(argv[2]) if len(argv) > 2 else 50
    clap_b200.init(0)
    dev = torch.device("cuda:0")
    seed = synth.synth_torch(torch, side, side, 0, side, dev)
    torch.cuda.synchronize()
    grid = clap_b200.Grid(side, side, side)
    rule = ca3d_rule(CORAL)
    ker = {a: [] for a, _ in ARMS}
    tot = {a: [] for a, _ in ARMS}
    hashes = {}
    print(f"ca3d {side}^3 x {gens} ca_coral, {runs} timed runs per arm after one warm-up run each, arms alternated", flush=True)
    print("before:", card(), flush=True)
    t0 = time.perf_counter()
    for i in range(1 + runs):
        for name, val in (ARMS if i % 2 == 0 else ARMS[::-1]):
            set_arm(val)
            grid.upload(seed.data_ptr())
            grid.run3d(rule, gens)
            st = grid.stats()
            if i > 0:
                ker[name].append(st["kernel_ms"])
                tot[name].append(st["total_ms"])
            hashes[name] = hash_planes(grid.device_ptr(), side * side, side)
    os.environ.pop("CLAPCA_ROWLOOP", None)
    print("after: ", card(), flush=True)
    for name, _ in ARMS:
        print(f"{name:9s} sweep kernel ms: {spread(ker[name])}", flush=True)
        print(f"{name:9s} step ms:         {spread(tot[name])}", flush=True)
    g, n = statistics.median(ker["generic"]), statistics.median(ker["interior"])
    gap = g - n
    noise = max(max(v) - min(v) for v in ker.values())
    print(f"sweep kernel: interior / generic = {n / g:.4f} ({100 * (1 - n / g):.2f} % less time), "
          f"gap {gap:.3f} ms vs largest spread {noise:.3f} ms", flush=True)
    same = bool((hashes["generic"] == hashes["interior"]).all())
    print(f"plane fingerprints equal between the arms: {same} ({side} planes); wall {time.perf_counter() - t0:.1f} s")
    if prof_out:
        from torch.profiler import ProfilerActivity, profile
        with open(prof_out, "w") as f:
            f.write(f"torch.profiler kernel times, one run per arm: ca3d {side}^3 x {gens} ca_coral\n{card()}\n")
            for name, val in ARMS:
                set_arm(val)
                grid.upload(seed.data_ptr())
                torch.cuda.synchronize()
                with profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as prof:
                    grid.run3d(rule, gens)
                    torch.cuda.synchronize()
                f.write(f"\n== {name} (CLAPCA_ROWLOOP={val or 'unset'}) ==\n")
                f.write(prof.key_averages().table(sort_by="cuda_time_total", row_limit=12, max_name_column_width=100))
                f.write("\n")
        set_arm(None)
        print(f"profile written to {prof_out}", flush=True)
    grid.close()
    if not same:
        sys.exit(1)


if __name__ == "__main__":
    main()
