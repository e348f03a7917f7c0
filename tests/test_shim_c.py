"""GPU (-m gpu): a C program written like the reference's own tests (core/test.c:616-670, ca3d_test0 and
ca2d_test0) compiled against include/clap/*.h and linked to the host shim, so the drop-in boundary is
exercised from C exactly as a reference caller would use it."""
import os
import subprocess

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

C_SRC = r'''
#include <stdio.h>
#include <stdlib.h>
#include <stdint.h>
#include "ca2d.h"
#include "ca3d.h"
#include "xyarray.h"
#include "noise_bake.h"
#include "terrain_field.h"

_Static_assert(CA_RANGE(2, 4) == 12, "CA_RANGE() macro is broken");

static uint64_t fnv(const unsigned char *p, size_t n)
{
    uint64_t h = 0xcbf29ce484222325ULL;
    for (size_t i = 0; i < n; i++) { h ^= p[i]; h *= 0x100000001b3ULL; }
    return h;
}

int main(void)
{
    /* ca3d_test0 */
    srand48(42);
    for (int i = 0; i < CA3D_MAX; i++) {
        struct xyzarray *xyz = ca3d_make(16, 8, 4);
        int pop = ca3d_run(xyz, ca_coral, 4);
        if (!xyzarray_count(xyz) || pop != xyzarray_count(xyz)) return 1;
        if (i == 0) printf("ca3d %d %016llx\n", pop, (unsigned long long)fnv(xyz->arr, 16 * 8 * 4));
        free(xyz);
    }
    /* ca2d_test0 */
    const struct cell_automaton ca_test = {
        .name = "test", .born_mask = 3 << 2, .surv_mask = 3 << 7, .nr_states = 4, .decay = true,
        .neigh_2d = ca2d_neigh_m1,
    };
    srand48(1234);
    unsigned char *map = ca2d_generate(&ca_test, 256, 5);
    int count = 0;
    for (int y = 0; y < 256; y++)
        for (int x = 0; x < 256; x++)
            count += xyarray_get(map, x, y);
    if (!count) return 2;
    printf("ca2d %d %016llx\n", count, (unsigned long long)fnv(map, 256 * 256));
    printf("next %ld\n", lrand48());          /* the stream continues where 256 * 256 draws leave it */
    /* the instantiator pass of terrain.c:473-477 */
    const struct cell_automaton tree = { .name = "cool tree", .born_mask = 0x1e, .surv_mask = 0xff,
                                         .nr_states = 20, .neigh_2d = ca2d_neigh_mv };
    ca2d_step(&tree, map, 256);
    printf("tree %016llx\n", (unsigned long long)fnv(map, 256 * 256));
    xyarray_free(map);
    unsigned char *tex = clap_noise_grad3d_bake_rgba8(16, 4, 2.0f, 0.5f, 5.0f, 0xc14d);
    if (!tex) return 3;
    printf("noise %016llx\n", (unsigned long long)fnv(tex, 16 * 16 * 16 * 4));
    free(tex);
    float *m0 = clap_terrain_map0(12345, 64);
    printf("map0 %016llx\n", (unsigned long long)fnv((unsigned char *)m0, 64 * 64 * 4));
    /* the mesh stage of terrain.c:479-516, fed with the lattice as a stand-in height field */
    float *vx, *norm, *tx;
    unsigned short *idx;
    clap_terrain_mesh(m0, 64, 1.0f, 2.0f, 3.0f, 50.0f, &vx, &norm, &tx, &idx);
    printf("mesh %016llx %016llx %016llx %016llx\n", (unsigned long long)fnv((unsigned char *)vx, 64 * 64 * 12),
           (unsigned long long)fnv((unsigned char *)norm, 64 * 64 * 12),
           (unsigned long long)fnv((unsigned char *)tx, 64 * 64 * 8),
           (unsigned long long)fnv((unsigned char *)idx, 63 * 63 * 12));
    free(vx); free(norm); free(tx); free(idx);
    free(m0);
    /* the film-grain pixels of blue_noise2d_tex (noise.c:96-169) out of the process-wide drand48 stream */
    srand48(77);
    float *grain = clap_blue_noise2d_rgba32f(64);
    if (!grain) return 4;
    double gsum = 0.0;
    for (int i = 0; i < 64 * 64 * 4; i++) gsum += grain[i];
    printf("grain %.6f %.8f %.8f\n", gsum, (double)grain[4 * 1000], (double)grain[4 * 4095 + 2]);
    printf("gnext %ld\n", lrand48());         /* ... which continues 3 * 64 * 64 draws later */
    free(grain);
    return 0;
}
'''


def test_reference_style_c_program(oracle, tmp_path):
    lib_dir = os.path.join(ROOT, "clap_b200", "lib")
    if not all(os.path.exists(os.path.join(lib_dir, n)) for n in ("libclapca_cuda.so", "libclapca_host.so")):
        subprocess.run(["make", "-C", os.path.join(ROOT, "clap_b200", "csrc"), "-j8"], check=True, capture_output=True)
    exe = str(tmp_path / "clapca_shim_test")
    lib = os.path.join(ROOT, "clap_b200", "lib")
    subprocess.run(["gcc", "-std=gnu11", "-O1", "-x", "c", "-", "-I", os.path.join(ROOT, "include", "clap"),
                    "-L", lib, "-lclapca_host", "-lclapca_cuda", f"-Wl,-rpath,{lib}", "-o", exe],
                   input=C_SRC.encode(), check=True)
    r = subprocess.run([exe], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stdout + r.stderr
    out = dict(line.split(None, 1) for line in r.stdout.strip().splitlines())

    vol = oracle.ca3d_make(16, 8, 4, 42)
    s, b, n = oracle.ca3d_rule(7)
    pop = oracle.ca3d_run(vol, s, b, n, 4)
    assert out["ca3d"].split() == [str(pop), "%016x" % oracle.fnv(vol)]

    import oracle_lib
    cave = oracle.ca2d_run(oracle.ca2d_seed(256, 4, 1234), 3 << 2, 3 << 7, 4, 1, oracle_lib.NEIGH_M1, 5)
    assert out["ca2d"].split() == [str(int(cave.sum())), "%016x" % oracle.fnv(cave)]
    st = oracle.srand48(1234)
    for _ in range(256 * 256):
        oracle.lrand48(st)
    assert int(out["next"]) == oracle.lrand48(st)
    oracle.ca2d_run(cave, 0x1e, 0xff, 20, 0, oracle_lib.NEIGH_MV, 1)
    assert out["tree"] == "%016x" % oracle.fnv(cave)
    g = np.load(os.path.join(ROOT, "tests", "golden", "noise.npz"))
    assert out["noise"] == "%016x" % oracle.fnv(g["bake_16_p5"])
    t = np.load(os.path.join(ROOT, "tests", "golden", "terrain.npz"))
    assert out["map0"] == "%016x" % oracle.fnv(t["map0_64_seed12345"])
    want = oracle.terrain_mesh(t["map0_64_seed12345"], 1.0, 2.0, 3.0, 50.0)
    assert out["mesh"].split() == ["%016x" % oracle.fnv(a) for a in want]
    gpix, gst = oracle.blue_noise2d(((77 & 0xFFFFFFFF) << 16) | 0x330E)
    gsum, g1, g2 = (float(v) for v in out["grain"].split())
    assert abs(gsum - float(gpix.astype(np.float64).sum())) < 0.05
    assert abs(g1 - float(gpix.reshape(-1, 4)[1000, 0])) < 2e-5 and abs(g2 - float(gpix.reshape(-1, 4)[4095, 2])) < 2e-5
    from ctypes import c_uint64
    assert int(out["gnext"]) == oracle.lrand48(c_uint64(gst))
