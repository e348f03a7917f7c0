"""CPU: the oracle restatement (oracle/port) against the golden vectors produced by the reference itself
(tests/golden/make_golden.py) and, when oracle/_ref is built, against the reference library directly."""
import os

import numpy as np
import pytest

import oracle_lib

G = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
CA_TEST = dict(born=3 << 2, surv=3 << 7, nr_states=4, decay=1, neigh=oracle_lib.NEIGH_M1)


@pytest.fixture(scope="module")
def g2():
    return np.load(os.path.join(G, "ca2d.npz"))


@pytest.fixture(scope="module")
def g3():
    return np.load(os.path.join(G, "ca3d.npz"))


def test_rand48_matches_libc(oracle):
    import ctypes
    libc = ctypes.CDLL(None)
    libc.lrand48.restype = ctypes.c_long
    for seed in (0, 1, 1234, -5, (1 << 35) + 3):
        libc.srand48(ctypes.c_long(seed))
        st = oracle.srand48(seed)
        assert [oracle.lrand48(st) for _ in range(2000)] == [libc.lrand48() for _ in range(2000)]


def test_ca2d_cfg1_golden(oracle, g2):
    """BASELINE config 1: ca_test 256x256, 5 generations, srand48(1234)."""
    seed = oracle.ca2d_seed(256, 4, 1234)
    assert np.array_equal(seed, g2["cfg1_seed"])
    final = oracle.ca2d_run(seed.copy(), steps=5, **CA_TEST)
    assert np.array_equal(final, g2["cfg1_final"])
    # histogram quoted in SURVEY.md 8(c)
    assert np.bincount(final.ravel()).tolist() == [28243, 99, 4638, 9159, 23397]


def test_ca2d_all_neighbourhoods_golden(oracle, g2):
    for i, (neigh, born, surv, nr, decay, side) in enumerate(g2["cases"].tolist()):
        start = g2[f"case{i}_start"]
        got = oracle.ca2d_run(start.copy(), born, surv, nr, decay, neigh, 6)
        assert np.array_equal(got, g2[f"case{i}_final6"]), (i, neigh)
        part = oracle.ca2d_run(start.copy(), born, surv, nr, decay, neigh, 3, side=side - 7)
        assert np.array_equal(part, g2[f"case{i}_partial3"]), (i, neigh)


def test_ca3d_make_and_test0_shape_golden(oracle, g3):
    seed = oracle.ca3d_make(16, 8, 4, 42)
    assert np.array_equal(seed, g3["make_16_8_4"])
    assert 255 in seed          # the prune quirk (SURVEY.md F5) is part of the contract
    s, b, n = oracle.ca3d_rule(7)
    pop = oracle.ca3d_run(seed, s, b, n, 4)
    assert pop == int(g3["make_16_8_4_coral4_pop"]) and pop != 0     # core/test.c:633 asserts != 0
    assert np.array_equal(seed, g3["make_16_8_4_coral4"])


def test_ca3d_all_rules_golden(oracle, g3):
    pops = g3["pops_37_23_32"].tolist()
    k = 0
    for nca in range(9):
        s, b, n = oracle.ca3d_rule(nca)
        for tag in "AB":
            vol = g3[f"seed{tag}_37_23_32"].copy()
            pop = oracle.ca3d_run(vol, s, b, n, 5)
            assert pop == pops[k], (nca, tag)
            assert np.array_equal(vol, g3[f"rule{nca}_seed{tag}_5gen"]), (nca, tag)
            k += 1


@pytest.mark.slow
def test_ca3d_cfg2_fingerprint(oracle, g3):
    """BASELINE config 2: 128^3, 10 generations of ca_coral on the ca3d_make seed (population 272840)."""
    oracle.ca3d_make(16, 8, 4, 42)
    vol = oracle.ca3d_make(128, 128, 128, 42)
    assert oracle.fnv(vol) == int(g3["cfg2_seed_hash"])
    s, b, n = oracle.ca3d_rule(7)
    pop = oracle.ca3d_run(vol, s, b, n, 10)
    assert pop == int(g3["cfg2_pop"]) == 272840
    assert oracle.fnv(vol) == int(g3["cfg2_final_hash"])
    assert np.bincount(vol.ravel(), minlength=256).tolist() == g3["cfg2_final_hist"].tolist()


def test_noise_golden(oracle):
    g = np.load(os.path.join(G, "noise.npz"))
    assert np.float32(oracle.lib.ora_hash31(1, 2, 3, 7)) == g["hash31_1_2_3_7"]
    assert np.array_equal(oracle.noise_bake(16, 4, 2.0, 0.5, 5.0, 0xC14D), g["bake_16_p5"])
    assert np.array_equal(oracle.noise_bake(24, 3, 2.3, 0.45, 37.0, 99), g["bake_24_p37_o3"])
    vals = oracle.fbm3(g["fbm_points"], 4, 2.0, 0.5, 37, 0xC14D)
    assert np.array_equal(vals.view(np.uint32), g["fbm_values"].view(np.uint32))     # 0 ulp
    first = oracle.noise_bake(64, 4, 2.0, 0.5, 64.0, 0xC14D, z0=0, z1=1).reshape(-1)[:64]
    assert np.array_equal(first, g["bake_64_default_first"])
    assert first[:4].tolist() == [122, 5, 93, 0]                                     # SURVEY.md 8(c)


def test_terrain_golden(oracle):
    g = np.load(os.path.join(G, "terrain.npz"))
    for seed in (12345, -99, (1 << 40) + 17):
        m = oracle.terrain_map0(seed, 64)
        assert np.array_equal(m.view(np.uint32), g[f"map0_64_seed{seed}"].view(np.uint32))
    map0 = oracle.terrain_map0(12345, 128)
    f = oracle.terrain_field(map0, 0.0, 1.0, 4)
    assert np.array_equal(f.view(np.uint32), g["field_128"].view(np.uint32))
    f = oracle.terrain_field(map0, 3.0, 2.5, 3)
    assert np.array_equal(f.view(np.uint32), g["field_128_y3_amp2_o3"].view(np.uint32))
    maze = oracle.ca2d_run(oracle.ca2d_seed(16, 4, 7), steps=4, **CA_TEST)
    assert np.array_equal(maze, g["maze_16"])
    h = oracle.terrain_heightmap(map0, 0.0, maze)
    assert np.array_equal(h.view(np.uint32), g["heightmap_128"].view(np.uint32))
    m1024 = oracle.terrain_map0(12345, 1024)
    assert m1024.reshape(-1)[7] == g["survey_map0_7"]
    assert abs(float(m1024.reshape(-1)[7]) - (-0.625764012)) < 1e-8


# ---- the oracle against the reference's outputs on seeded inputs (golden/oracle_vs_ref.npz, make_golden_vs_ref.py) and,
# ---- where oracle/_ref is built, against the reference library directly

@pytest.fixture(scope="module")
def gvr():
    return np.load(os.path.join(G, "oracle_vs_ref.npz"))


def test_oracle_vs_reference_ca3d_random(oracle, gvr):
    reference = oracle_lib.ref()
    rng = np.random.default_rng(3)
    for nca in range(9):
        d0, d1, d2 = (int(v) for v in rng.integers(3, 24, 3))
        vol = (rng.integers(0, 7, (d2, d1, d0)) * (rng.random((d2, d1, d0)) < 0.4)).astype(np.uint8)
        vol[rng.random(vol.shape) < 0.01] = 255
        a, b = vol.copy(), vol.copy()
        s, bm, n = oracle.ca3d_rule(nca)
        pop = oracle.ca3d_run(a, s, bm, n, 4)
        assert pop == int(gvr[f"ca3d_{nca}_pop"]) and np.array_equal(a, gvr[f"ca3d_{nca}"]), nca
        if reference is not None:
            assert pop == reference.ca3d_run(b, nca, 4)
            assert np.array_equal(a, b), nca


def test_oracle_vs_reference_ca2d_random(oracle, gvr):
    reference = oracle_lib.ref()
    rng = np.random.default_rng(4)
    for neigh in range(4):
        for decay in (0, 1):
            side = int(rng.integers(5, 60))
            born, surv = int(rng.integers(0, 512)), int(rng.integers(0, 512))
            nr = int(rng.integers(1, 30))
            arr = (rng.integers(0, nr + 1, (side, side)) * (rng.random((side, side)) < 0.5)).astype(np.uint8)
            a = oracle.ca2d_run(arr.copy(), born, surv, nr, decay, neigh, 4)
            assert np.array_equal(a, gvr[f"ca2d_{neigh}_{decay}"]), (neigh, decay)
            if reference is not None:
                b = reference.ca2d_step(arr.copy(), born, surv, nr, decay, neigh, steps=4)
                assert np.array_equal(a, b), (neigh, decay)


def test_oracle_vs_reference_fields(oracle, gvr):
    reference = oracle_lib.ref()
    rng = np.random.default_rng(6)
    pts = (rng.random((2000, 3)) * 300 - 100).astype(np.float32)
    a = oracle.fbm3(pts, 5, 1.9, 0.6, 13, 7)
    assert np.array_equal(a.view(np.uint32), gvr["fbm3"].view(np.uint32))
    assert np.array_equal(oracle.noise_bake(12, 2, 2.0, 0.5, 7.0, 1), gvr["bake_12"])
    m = oracle.terrain_map0(777, 96)
    assert np.array_equal(m.view(np.uint32), gvr["map0_777_96"].view(np.uint32))
    maze = oracle.ca2d_run(oracle.ca2d_seed(12, 4, 9), 3 << 2, 3 << 7, 4, 1, oracle_lib.NEIGH_M1, 4)
    assert np.array_equal(maze, gvr["maze_12"])
    h = oracle.terrain_heightmap(m, 1.5, maze)
    assert np.array_equal(h.view(np.uint32), gvr["heightmap_777_96"].view(np.uint32))
    if reference is not None:
        b = reference.fbm3(pts, 5, 1.9, 0.6, 13, 7)
        assert np.array_equal(a.view(np.uint32), b.view(np.uint32))
        assert np.array_equal(oracle.noise_bake(12, 2, 2.0, 0.5, 7.0, 1), reference.noise_bake(12, 2, 2.0, 0.5, 7.0, 1))
        rm = reference.terrain_map0(777, 96)
        assert np.array_equal(m.view(np.uint32), rm.view(np.uint32))
        rmaze = reference.ca2d_generate(3 << 2, 3 << 7, 4, 1, 1, 12, 4, 9)
        assert np.array_equal(maze, rmaze)
        b = reference.terrain_heightmap(777, rm, 1.5, rmaze)
        assert np.array_equal(h.view(np.uint32), b.view(np.uint32))


def test_terrain_mesh_normals_golden(oracle):
    """Mesh stage (core/terrain.c:93-110,479-516): the port's normals against the reference's calc_normal() outputs
    committed in golden/terrain_mesh.npz, and the trivially restated vertex / uv / index formulas at a few spots."""
    t = np.load(os.path.join(G, "terrain.npz"))
    m = np.load(os.path.join(G, "terrain_mesh.npz"))
    vx, norm, tx, idx = oracle.terrain_mesh(t["heightmap_128"], 10.0, -2.0, 5.0, 300.0)
    assert np.array_equal(norm.view(np.uint32), m["normals_128"].view(np.uint32))
    _, norm2, _, _ = oracle.terrain_mesh(m["rough_37"], 0.0, 0.0, 0.0, 1.0)
    assert np.array_equal(norm2.view(np.uint32), m["normals_rough_37"].view(np.uint32))
    nr = 128
    i, j = 5, 77
    it = i * nr + j
    f = np.float32
    assert vx[it, 0] == f(10.0) + f(j) / (f(nr) - f(1)) * f(300.0)
    assert vx[it, 1] == f(-2.0) + t["heightmap_128"][j, i]
    assert vx[it, 2] == f(5.0) + f(i) / (f(nr) - f(1)) * f(300.0)
    assert tx[it, 0] == f(j) * f(32) / (f(nr) - f(1)) and tx[it, 1] == f(i) * f(32) / (f(nr) - f(1))
    q = (i * (nr - 1) + j) * 6
    assert idx[q:q + 6].tolist() == [it, it + nr, it + 1, it + 1, it + nr, it + nr + 1]
    assert np.allclose(np.linalg.norm(norm.astype(np.float64), axis=1), 1.0, atol=1e-6)


def test_terrain_mesh_port_vs_reference_normals(oracle, gvr):
    reference = oracle_lib.ref()
    rng = np.random.default_rng(8)
    for nr in (1, 2, 3, 50, 131):
        hmap = (rng.random((nr, nr)) * 9 - 4).astype(np.float32)
        _, norm, _, _ = oracle.terrain_mesh(hmap, 0.0, 0.0, 0.0, 1.0)
        assert np.array_equal(norm.view(np.uint32), gvr[f"normals_{nr}"].view(np.uint32)), nr
        if reference is not None:
            assert np.array_equal(norm.view(np.uint32), reference.terrain_normals(hmap).view(np.uint32)), nr


def test_terrain_height_and_instantiators_golden(oracle):
    """terrain_height() (core/terrain.c:336-379) against the reference's values in golden/terrain_mesh.npz, and the
    instantiator loop (:555-570) on a small hand-checkable maze."""
    t = np.load(os.path.join(G, "terrain.npz"))
    m = np.load(os.path.join(G, "terrain_mesh.npz"))
    h = oracle.terrain_height(t["heightmap_128"], 10.0, 5.0, 300, m["height_pts"])
    assert np.array_equal(h.view(np.uint32), m["heights_128_x10_z5_side300"].view(np.uint32))
    assert (h == 0).sum() > 10 and (h != 0).sum() > 200            # points outside the square read 0
    maze = np.zeros((16, 16), np.uint8)
    maze[3, 5] = 20         # xyarray_get(maze, i=5, j=3)
    maze[9, 5] = 21
    maze[0, 7] = 20
    maze[2, 2] = 19
    rec = oracle.terrain_instantiators(maze, (20, 21), t["heightmap_128"], 10.0, 5.0, 300.0)
    assert rec["kind"].tolist() == [0, 1, 0]                        # i outer, j inner: (5,3) (5,9) (7,0)
    f = np.float32
    assert rec["dx"][0] == f(10.0) + f(5.5) * f(8) * f(300.0) / f(127) and rec["dz"][0] == f(5.0) + f(3.5) * f(8) * f(300.0) / f(127)
    want = oracle.terrain_height(t["heightmap_128"], 10.0, 5.0, 300, np.stack([rec["dx"], rec["dz"]], 1))
    assert np.array_equal(rec["dy"].view(np.uint32), want.view(np.uint32)) and (rec["dy"] != 0).all()


def test_terrain_height_port_vs_reference(oracle, gvr):
    reference = oracle_lib.ref()
    rng = np.random.default_rng(10)
    for nr, side in ((50, 77), (131, 1000), (9, 3)):
        hmap = (rng.random((nr, nr)) * 9 - 4).astype(np.float32)
        pts = (rng.random((300, 2)) * side * 1.2 - side * 0.1).astype(np.float32) + np.float32([-3.0, 8.0])
        a = oracle.terrain_height(hmap, -3.0, 8.0, side, pts)
        assert np.array_equal(a.view(np.uint32), gvr[f"heights_{nr}"].view(np.uint32)), nr
        if reference is not None:
            b = reference.terrain_height(hmap, -3.0, 8.0, side, pts)
            assert np.array_equal(a.view(np.uint32), b.view(np.uint32)), nr


def test_cfg4_chain_256cube_full_run_port_vs_reference_fingerprint(oracle):
    """The port on the 256^3 x 50 link of the config-4 parity chain must reproduce the fingerprint the unmodified
    reference left in golden/cfg4_chain_256.json (about ten seconds of CPU)."""
    import json
    with open(os.path.join(G, "cfg4_chain_256.json")) as f:
        cfg = json.load(f)
    rng = np.random.default_rng(2048)
    vol = (rng.integers(1, 6, (256, 256, 256)) * (rng.random((256, 256, 256)) < 0.25)).astype(np.uint8)
    assert "%016x" % oracle.fnv(vol) == cfg["seed_fnv1a64"] and int(np.count_nonzero(vol)) == cfg["seed_population"]
    c = cfg["ca_coral"]
    s, b, n = oracle.ca3d_rule(c["nca"])
    assert oracle.ca3d_run(vol, s, b, n, c["generations"]) == c["population"]
    assert "%016x" % oracle.fnv(vol) == c["fnv1a64"]


def test_blue_noise_port_against_numpy_fft():
    """blue_noise2d_tex (core/noise.c:96-169).  kissfft is not vendored, so the port's transform is pinned to the DFT
    contract kissfft documents (forward exp(-2 pi i kn/N), unnormalised inverse) through numpy.fft -- an independent
    implementation -- with everything else (draw order, weights, gain, joint normalisation) restated line by line."""
    ora = oracle_lib.port()
    seed = 20260101
    st0 = ((seed & 0xFFFFFFFF) << 16) | 0x330E              # srand48(seed)
    got, st1 = ora.blue_noise2d(st0)
    # the same in numpy, double precision
    a, c, m = 0x5DEECE66D, 0xB, (1 << 48) - 1
    x = st0
    d = np.empty(3 * 64 * 64)
    for i in range(d.size):
        x = (a * x + c) & m
        d[i] = x / float(1 << 48)
    assert x == st1
    w = np.array([0.299, 0.587, 0.114])
    white = (((d * 4.0 - 1.0) / 3.0).reshape(64, 64, 3) * w).astype(np.float32).astype(np.float64)
    f = np.arange(64)
    f = np.where(f <= 32, f, f - 64)
    gain = (np.sqrt(f[:, None] ** 2 + f[None, :] ** 2).astype(np.float32) / np.float32(np.sqrt(np.float32(2048.0)))).astype(np.float64)
    chans = [np.real(np.fft.ifft2(np.fft.fft2(white[:, :, k]) * gain)) for k in range(3)]
    rgb = np.stack(chans, axis=-1)
    want = (rgb - rgb.min()) / (rgb.max() - rgb.min())
    assert np.all(got[:, :, 3] == 1.0)
    assert np.abs(got[:, :, :3] - want).max() < 2e-5
    assert got[:, :, :3].min() == 0.0 and got[:, :, :3].max() == 1.0


def test_ca3d_make_small_volumes_against_the_reference_fingerprints(oracle):
    """ca3d_make() on 240 small volumes, where ca3d_prune()'s order-dependent corner is common (an empty cell with six
    occupied neighbours turns 255 and counts for the cells after it): the port must reproduce the fingerprints the
    UNMODIFIED reference produced (tests/golden/make_golden_ca3d_make.py), and the reference itself, where it is built."""
    import json
    with open(os.path.join(G, "ca3d_make_small.json")) as f:
        g = json.load(f)
    assert g["cells_255_inside"] > 100
    ref = oracle_lib.ref()
    for d0, d1, d2 in g["shapes"]:
        want = g["fnv1a64"]["%dx%dx%d" % (d0, d1, d2)]
        for seed, h in zip(g["seeds"], want):
            vol = oracle.ca3d_make(d0, d1, d2, seed)
            assert "%016x" % oracle.fnv(vol) == h, (d0, d1, d2, seed)
            if ref is not None and seed % 8 == 0:
                assert np.array_equal(ref.ca3d_make(d0, d1, d2, seed), vol)
