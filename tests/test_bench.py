"""bench.py --dump-outputs: the outputs of the last timed step, written exactly, within 64 MiB and the same from run to
run (CPU); and on the GPU, what a bench run writes equals what the library's own calls return for the same inputs."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

import bench

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_dump_outputs_are_exact_bounded_and_repeatable(tmp_path):
    rng = np.random.default_rng(1)
    cells = rng.integers(0, 256, 30_000_000).astype(np.uint8)
    indices = rng.integers(-32768, 32768, 1000).astype(np.int16)
    hashes = np.array([2 ** 64 - 1, (1 << 63) | 5, 7], np.uint64)
    arrays = {"cells": cells, "indices": indices, "hashes": bench.u64_halves(hashes), "population": np.array([2 ** 40 + 3])}
    for run in ("a", "b"):
        bench.dump_outputs(str(tmp_path / run), arrays)
    got = {}
    for name in arrays:
        a, b = np.load(tmp_path / "a" / f"{name}.npy"), np.load(tmp_path / "b" / f"{name}.npy")
        assert a.dtype in (np.float32, np.float64) and np.array_equal(a, b), name
        got[name] = a
    assert sum(a.nbytes for a in got.values()) <= bench.DUMP_BYTES
    keep = bench.dump_index(cells.size, bench.DUMP_BYTES // 8 // len(arrays))
    assert 0 < len(keep) < cells.size and got["cells"].dtype == np.float32
    assert np.array_equal(got["cells"], cells[keep])
    assert got["indices"].dtype == np.float32 and np.array_equal(got["indices"], indices)
    h = got["hashes"].astype(np.uint64)
    assert np.array_equal((h[:, 0] << np.uint64(32)) | h[:, 1], hashes)
    assert got["population"].dtype == np.float64 and got["population"].tolist() == [2 ** 40 + 3]


def _bench_dump(workload, out):
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--steps", "2", "--warmup", "1",
                        "--workload", workload, "--no-cpu", "--no-e2e", "--dump-outputs", str(out)],
                       capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-3000:]
    assert json.loads(r.stdout.strip().splitlines()[-1])["steps"] == 2
    return {p.stem: np.load(p) for p in out.glob("*.npy")}


@pytest.mark.gpu
@pytest.mark.parametrize("workload", ["ca3d_128", "ca2d_256", "noise_64", "terrain_1024", "terrain_mesh_1024"])
def test_bench_dump_holds_the_library_results(gpu, tmp_path, workload):
    from clap_b200 import synth
    from clap_b200.ca import Rand48
    got = _bench_dump(workload, tmp_path / "dump")
    cap = bench.DUMP_BYTES // 8 // len(got)

    def sample(a):
        a = a.reshape(-1)
        return a[bench.dump_index(a.size, cap)]

    if workload == "ca3d_128":
        vol = synth.synth_numpy(np, 128, 128, 0, 128)
        pop = gpu.ca3d_run(vol, 7, 10)
        assert got["population"].tolist() == [pop]
        assert np.array_equal(got["volume"], vol)
        assert np.array_equal(got["plane_hashes"], bench.u64_halves(synth.plane_hashes_numpy(np, vol)))
    elif workload == "ca2d_256":
        grid = gpu.ca2d_generate(gpu.CA_TEST, 256, 5, Rand48(1234))
        assert np.array_equal(got["grid"], grid)
        assert np.array_equal(got["row_hashes"], bench.u64_halves(synth.plane_hashes_numpy(np, grid[:, None, :])))
    elif workload == "noise_64":
        assert np.array_equal(got["rgba"], gpu.noise_grad3d_bake_rgba8(64, 4, 2.0, 0.5, 64.0, 0xC14D).reshape(-1))
    else:
        maze = gpu.ca2d_generate(gpu.CA_TEST, 128, 4, Rand48(7))
        hmap = gpu.terrain_heightmap(12345, 1024, 0.0, maze, 1.0, 4)
        if workload == "terrain_1024":
            assert np.array_equal(got["heightmap"], sample(hmap))
            assert np.array_equal(got["map0"], sample(gpu.terrain_map0(12345, 1024)))
        else:
            vx, norm, tx, idx = gpu.terrain_mesh(hmap, 0.0, 0.0, 0.0, 256.0)
            for name, want in (("vertices", vx), ("normals", norm), ("uv", tx), ("indices", idx)):
                assert np.array_equal(got[name], sample(want)), name
