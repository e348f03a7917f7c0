"""Outputs of the oracle-vs-reference tests of tests/test_oracle_golden.py on exactly their seeded inputs, so that those
tests compare the oracle with stored outputs where the reference library is not built:

    python tests/golden/make_golden_vs_ref.py           ->  tests/golden/oracle_vs_ref.npz   from oracle/_ref (the reference)
    python tests/golden/make_golden_vs_ref.py --port    ->  the same file from oracle/liboracle_port.so

The committed file holds the port's outputs (--port).  Wherever oracle/_ref is built, the same tests also compare the port
with the reference directly, and running this script without --port replaces the file with the reference's own outputs.
The inputs below must stay identical to the tests'.
"""
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
import oracle_lib  # noqa: E402


def main():
    use_port = "--port" in sys.argv[1:]
    port = oracle_lib.port()
    ref = None if use_port else oracle_lib.ref()
    if ref is None and not use_port:
        raise SystemExit("oracle/_ref/libclapref.so missing: make -C oracle ref REF=<reference sources>, or pass --port")
    out = {}

    rng = np.random.default_rng(3)                                  # test_oracle_vs_reference_ca3d_random
    for nca in range(9):
        d0, d1, d2 = (int(v) for v in rng.integers(3, 24, 3))
        vol = (rng.integers(0, 7, (d2, d1, d0)) * (rng.random((d2, d1, d0)) < 0.4)).astype(np.uint8)
        vol[rng.random(vol.shape) < 0.01] = 255
        if ref is not None:
            pop = ref.ca3d_run(vol, nca, 4)
        else:
            pop = port.ca3d_run(vol, *port.ca3d_rule(nca), 4)
        out[f"ca3d_{nca}"], out[f"ca3d_{nca}_pop"] = vol, np.int64(pop)

    rng = np.random.default_rng(4)                                  # test_oracle_vs_reference_ca2d_random
    for neigh in range(4):
        for decay in (0, 1):
            side = int(rng.integers(5, 60))
            born, surv = int(rng.integers(0, 512)), int(rng.integers(0, 512))
            nr = int(rng.integers(1, 30))
            arr = (rng.integers(0, nr + 1, (side, side)) * (rng.random((side, side)) < 0.5)).astype(np.uint8)
            if ref is not None:
                out[f"ca2d_{neigh}_{decay}"] = ref.ca2d_step(arr, born, surv, nr, decay, neigh, steps=4)
            else:
                out[f"ca2d_{neigh}_{decay}"] = port.ca2d_run(arr, born, surv, nr, decay, neigh, 4)

    rng = np.random.default_rng(6)                                  # test_oracle_vs_reference_fields
    pts = (rng.random((2000, 3)) * 300 - 100).astype(np.float32)
    impl = ref if ref is not None else port
    out["fbm3"] = impl.fbm3(pts, 5, 1.9, 0.6, 13, 7)
    out["bake_12"] = impl.noise_bake(12, 2, 2.0, 0.5, 7.0, 1)
    out["map0_777_96"] = m = impl.terrain_map0(777, 96)
    if ref is not None:
        out["maze_12"] = maze = ref.ca2d_generate(3 << 2, 3 << 7, 4, 1, 1, 12, 4, 9)
        out["heightmap_777_96"] = ref.terrain_heightmap(777, m, 1.5, maze)
    else:
        out["maze_12"] = maze = port.ca2d_run(port.ca2d_seed(12, 4, 9), 3 << 2, 3 << 7, 4, 1, 1, 4)
        out["heightmap_777_96"] = port.terrain_heightmap(m, 1.5, maze)

    rng = np.random.default_rng(8)                                  # test_terrain_mesh_port_vs_reference_normals
    for nr in (1, 2, 3, 50, 131):
        hmap = (rng.random((nr, nr)) * 9 - 4).astype(np.float32)
        out[f"normals_{nr}"] = ref.terrain_normals(hmap) if ref is not None else port.terrain_mesh(hmap, 0.0, 0.0, 0.0, 1.0)[1]

    rng = np.random.default_rng(10)                                 # test_terrain_height_port_vs_reference
    for nr, side in ((50, 77), (131, 1000), (9, 3)):
        hmap = (rng.random((nr, nr)) * 9 - 4).astype(np.float32)
        pts = (rng.random((300, 2)) * side * 1.2 - side * 0.1).astype(np.float32) + np.float32([-3.0, 8.0])
        out[f"heights_{nr}"] = impl.terrain_height(hmap, -3.0, 8.0, side, pts)

    np.savez_compressed(os.path.join(HERE, "oracle_vs_ref.npz"), **out)
    print("wrote oracle_vs_ref.npz from the", "port" if ref is None else "reference", f"({len(out)} arrays)")


if __name__ == "__main__":
    main()
