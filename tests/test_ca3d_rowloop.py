"""The two row loops of the ca3d sweep (ca3d_bitplane.cuh, Sweep3::run_rows): the interior rows of an item take a
row step without edge tests, the first and last rows the general step; CLAPCA_ROWLOOP=generic sends every row through
the general step.  Both must give the oracle's volume wherever the interior and the tail meet or are empty: planes of
1..8 rows, prefetch distances around the plane height, row-segmented items, tile mode and one warp per sweep.

CPU: the kernel source on the host warp emulator (tests/emu/emu_ca3d_rowloop.cpp) against the oracle.
GPU: the 2048-row coral volume at a reduced depth under both loops, compared byte for byte."""
import os
import subprocess

import numpy as np
import pytest

EMU = os.path.join(os.path.dirname(os.path.abspath(__file__)), "emu")


@pytest.fixture(scope="module")
def emu_exe():
    """emu_ca3d with the row-loop knobs CLAPCA_PREFETCH_ROWS / CLAPCA_ROWLOOP read from the environment"""
    subprocess.run(["make", "-C", EMU, "-j4", "build/emu_ca3d_rowloop"], check=True, capture_output=True)
    return os.path.join(EMU, "build", "emu_ca3d_rowloop")


def _run(exe, args, env):
    env = dict({"CLAPCA_PREFETCH_ROWS": "0"}, **env)
    full = {k: v for k, v in os.environ.items() if k != "CLAPCA_ROWLOOP"}
    full.update(env)
    r = subprocess.run([exe] + [str(a) for a in args], capture_output=True, text=True, timeout=600, env=full)
    assert r.returncode == 0 and r.stdout.startswith("OK"), f"{args} {env}: {r.stdout} {r.stderr}"
    loop = "generic" if env.get("CLAPCA_ROWLOOP") == "generic" else "interior"
    assert f"row loop {loop}, prefetch_rows {env['CLAPCA_PREFETCH_ROWS']}" in r.stderr, r.stderr


# emu_ca3d arguments after H (see the header of tests/emu/emu_ca3d.cpp): the volume, rule, planes, seed, workers and the item kind
MODES = {
    #               W   Z  G rule P WPL kind seed warps ranks block seg flagrows genbatch pubworkers team tilegens
    "tiles":       (45, 7, 5, 7, 3, 1, 1, 3, 16, 1, 0, 0, 2, 0, 0, 4, 2),
    "wide_tiles":  (45, 14, 7, 7, 3, 2, 1, 3, 360, 1, 0, 0, 2, 0, 0, 18, 3),
    "time_key":    (45, 7, 5, 7, 3, 1, 1, 3, 4, 1, 0, 0, 2, -1),
    "segments":    (45, 7, 4, 7, 3, 1, 1, 3, 3, 1, 0, 2, 1),
    "publisher":   (45, 7, 5, 10, 4, 2, 1, 9, 4, 1, 0, 0, 1, -1, 2),
}


@pytest.mark.parametrize("mode", sorted(MODES))
@pytest.mark.parametrize("h", range(1, 9))
def test_short_planes_both_row_loops(emu_exe, mode, h):
    """H = 1..8 rows: the interior is empty or a few rows long and meets the fill and the tail; the prefetch distance
    runs from 0 (no prefetch) to beyond the plane.  Every run is compared with the oracle by the emulator."""
    args = MODES[mode]
    argv = (args[0], h) + args[1:]
    for pf in sorted({0, max(1, h - 3), max(1, h - 1), h + 1}):
        for loop in ("interior", "generic"):
            env = {"CLAPCA_PREFETCH_ROWS": str(pf)}
            if loop == "generic":
                env["CLAPCA_ROWLOOP"] = "generic"
            _run(emu_exe, argv, env)


@pytest.mark.parametrize("args", [
    #  W   H   Z   G  rule P WPL kind seed warps ranks block seg flagrows genbatch pubworkers team tilegens
    (64, 40, 6, 5, 10, 4, 2, 1, 9, 7, 1, 0, 7, 3),                        # 40 rows in segments of 7: ragged last one
    (45, 37, 12, 6, 7, 3, 1, 1, 3, 48, 2, 2, 0, 2, 0, 0, 4, 2),           # 2 ranks: ghost planes feed interior rows
    (33, 12, 8, 4, 8, 8, 4, 2, 5, 8, 1, 0, 0, 2, 0, 0, 4, 2),             # 8 planes, 4 words per lane
])
def test_segments_ranks_and_wide_variants_both_row_loops(emu_exe, args):
    for env in ({}, {"CLAPCA_ROWLOOP": "generic"}, {"CLAPCA_PREFETCH_ROWS": "6"}):
        _run(emu_exe, args, env)


@pytest.mark.gpu
def test_coral_2048_rows_both_row_loops_equal(gpu, monkeypatch):
    """The bench's row width and plane height (2048 x 2048, the wide kernel's interior loop over 2043 rows of every
    item) at a depth of 48 planes and 12 generations: the two loops leave the same volume, byte for byte."""
    from clap_b200 import synth
    seed = synth.synth_numpy(np, 2048, 2048, 0, 48)
    out = {}
    for loop in ("interior", "generic"):
        if loop == "generic":
            monkeypatch.setenv("CLAPCA_ROWLOOP", "generic")
        else:
            monkeypatch.delenv("CLAPCA_ROWLOOP", raising=False)
        grid = gpu.Grid(2048, 2048, 48)
        try:
            grid.upload(seed)
            pop = grid.run3d(7, 12)
            st = grid.stats()
            vol = np.empty_like(seed)
            grid.download(vol)
        finally:
            grid.close()
        assert st["engine"] == "bitplane" and st["planes"] == 3
        out[loop] = (pop, vol)
    assert out["interior"][0] == out["generic"][0]
    assert np.array_equal(out["interior"][1], out["generic"][1]), int((out["interior"][1] != out["generic"][1]).sum())
    assert not np.array_equal(out["interior"][1], seed)
