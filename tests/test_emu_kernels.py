"""CPU: the real bit-plane kernel source, compiled with -DCLAPCA_EMU and run on the host warp emulator
(tests/emu/), must reproduce the oracle bit for bit -- this covers the row-scan algebra, the rule tables,
the sliding windows, the pack/unpack layout and the flag-based dataflow between concurrent sweeps."""
import os
import subprocess

import pytest

EMU = os.path.join(os.path.dirname(os.path.abspath(__file__)), "emu")


@pytest.fixture(scope="module")
def emu_bin():
    subprocess.run(["make", "-C", EMU, "-j4"], check=True, capture_output=True)
    return os.path.join(EMU, "build")


def _run(exe, *args, env=None):
    r = subprocess.run([exe] + [str(a) for a in args], capture_output=True, text=True, timeout=600,
                       env=dict(os.environ, **env) if env else None)
    assert r.returncode == 0, f"{args}: {r.stdout} {r.stderr}"
    assert r.stdout.startswith("OK")


def test_bitslice_building_blocks(emu_bin):
    """adders, the 3D count tree (both forms), compile-time / run-time rule tables of all nine cas[] rules, and the
    in-row scan (D form, E form, split into its common and rare part) against plain integer arithmetic, cell by cell"""
    r = subprocess.run([os.path.join(emu_bin, "emu_bitslice")], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0 and r.stdout.startswith("OK"), r.stdout + r.stderr


@pytest.mark.parametrize("nca", range(11))
def test_ca3d_every_rule(emu_bin, nca):
    exe = os.path.join(emu_bin, "emu_ca3d")
    planes = 4 if nca in (2, 4) else 3
    #        W   H  Z  G  rule P       WPL seedkind seed warps
    _run(exe, 45, 7, 6, 3, nca, planes, 1, 0, nca, 5)
    _run(exe, 33, 5, 4, 4, nca, 8, 1, 2, nca, 3)          # ca3d_make seed: contains 255s
    _run(exe, 64, 4, 3, 2, nca, 4, 2, 1, nca, 7)


@pytest.mark.parametrize("nca", [11, 12])
def test_ca3d_chain_rules_long_dependency_runs(emu_bin, nca):
    """Rules whose table flips between every K and K+1: whole rows are one in-row dependency chain, so the scan's
    rare paths (runs of >= 8 dependent cells inside a word, lanes that never break the chain) do all the work."""
    exe = os.path.join(emu_bin, "emu_ca3d")
    _run(exe, 45, 7, 6, 3, nca, 3, 1, 0, 4, 5)
    _run(exe, 300, 5, 4, 3, nca, 3, 1, 3, 5, 3)           # binary seed: no cell ever has a state >= 2 to break the chain
    _run(exe, 1030, 3, 3, 2, nca, 3, 2, 3, 6, 3)
    _run(exe, 2048, 2, 2, 2, nca, 4, 2, 3, 7, 4)
    _run(exe, 97, 4, 5, 4, nca, 3, 4, 1, 8, 4)
    _run(exe, 500, 4, 5, 4, nca, 3, 4, 3, 8, 4)


@pytest.mark.parametrize("shape", [
    (1, 1, 1, 3), (5, 1, 1, 3), (1, 5, 1, 3), (1, 1, 5, 3), (32, 3, 3, 2), (31, 3, 3, 2), (33, 2, 2, 5),
    (40, 6, 5, 0), (16, 8, 4, 4),
])
def test_ca3d_edge_shapes(emu_bin, shape):
    w, h, z, g = shape
    _run(os.path.join(emu_bin, "emu_ca3d"), w, h, z, g, 7, 3, 1, 1, 5, 2)


def test_ca3d_wide_rows_and_words_per_lane(emu_bin):
    exe = os.path.join(emu_bin, "emu_ca3d")
    _run(exe, 97, 4, 5, 5, 7, 3, 4, 1, 7, 4)
    _run(exe, 1024, 3, 3, 2, 0, 3, 1, 1, 8, 3)
    _run(exe, 1030, 2, 3, 2, 0, 3, 2, 1, 8, 3)
    _run(exe, 2048, 2, 2, 2, 7, 3, 2, 0, 9, 4)


@pytest.mark.parametrize("nca,planes,wpl", [(nca, planes, wpl) for nca in range(11) for planes in (3, 4, 8)
                                             for wpl in (1, 2, 4) if not (planes == 3 and nca in (2, 4))])
def test_ca3d_every_rule_planes_and_words_per_lane(emu_bin, nca, planes, wpl):
    """The full (rule, state planes, words per lane) matrix the library instantiates, on ragged rows of each width
    class (pyroclastic and builder, nr_states 10, need at least 4 planes)."""
    width = {1: 1000, 2: 2047, 4: 3999}[wpl]
    seedkind = {3: 0, 4: 1, 8: 2}[planes]      # values 0..5, dense 0..15, the ca3d_make seed with its 255s
    _run(os.path.join(emu_bin, "emu_ca3d"), width, 3, 3, 2, nca, planes, wpl, seedkind, nca * 9 + planes + wpl, 5)


def test_ca3d_many_generations_few_and_many_workers(emu_bin):
    exe = os.path.join(emu_bin, "emu_ca3d")
    _run(exe, 24, 12, 10, 12, 10, 8, 1, 1, 3, 12)
    _run(exe, 24, 12, 10, 9, 10, 3, 1, 1, 5, 1)          # a single worker: pure claim order
    _run(exe, 24, 12, 10, 9, 7, 3, 1, 0, 5, 2)


@pytest.mark.parametrize("args", [
    #  W   H   Z   G  rule P WPL kind seed warps ranks block seg flagrows
    (45, 40, 12, 4, 7, 3, 1, 1, 3, 3, 1, 0, 8, 1),       # skewed row segments, counter raised every row
    (45, 40, 12, 4, 7, 3, 1, 1, 3, 3, 1, 0, 8, 3),
    (64, 33, 6, 9, 10, 4, 2, 1, 9, 7, 1, 0, 4, 5),
    (31, 20, 5, 3, 8, 3, 1, 2, 3, 3, 1, 0, 3, 1),
])
def test_ca3d_row_segments(emu_bin, args):
    _run(os.path.join(emu_bin, "emu_ca3d"), *args)


@pytest.mark.parametrize("args", [
    #  W   H   Z   G  rule P WPL kind seed warps ranks block seg flagrows genbatch pubworkers team tilegens
    (45, 7, 12, 4, 7, 3, 1, 1, 3, 3, 2, 0, 0, 2, 0, 0, 1, 1),        # 2 emulated GPUs, contiguous slabs, one plane per CTA
    (45, 37, 12, 6, 7, 3, 1, 1, 3, 6, 2, 2, 0, 2, 0, 0, 2, 1),       # 2 GPUs, z-blocks of 2 planes
    (45, 50, 13, 5, 3, 3, 1, 1, 3, 9, 3, 2, 0, 4, 0, 0, 3, 1),       # 3 GPUs, ragged last block
    (33, 30, 16, 5, 10, 8, 1, 1, 4, 4, 4, 1, 0, 2, 0, 0, 2, 1),      # 4 GPUs, single-plane blocks (every plane is an edge)
    (33, 64, 9, 6, 0, 3, 1, 0, 4, 8, 4, 5, 0, 2, 0, 0, 4, 1),        # more ranks than blocks need
    (20, 5, 3, 4, 7, 3, 1, 1, 4, 4, 4, 1, 0, 1, 0, 0, 2, 1),         # ranks without any plane
])
def test_ca3d_slab_decomposition_peer_ghost_planes(emu_bin, args):
    """The multi-GPU path: ranks run concurrently, the service warp of every tile that touches a z-block edge
    copies finished H rows into the neighbour's ghost plane and raises its counters, exactly as the peer stores
    over NVLink do on the real machine."""
    _run(os.path.join(emu_bin, "emu_ca3d"), *args)


@pytest.mark.parametrize("args", [
    #  W   H   Z   G  rule P WPL kind seed warps ranks block seg flagrows genbatch
    (45, 20, 12, 7, 7, 3, 1, 1, 3, 5, 1, 0, 0, 2, 3),        # batches of 3,2,2 generations, diagonal order
    (45, 20, 12, 7, 7, 3, 1, 1, 3, 1, 1, 0, 0, 4, 2),        # a single worker: the order alone must be executable
    (64, 16, 9, 10, 10, 4, 2, 1, 9, 9, 1, 0, 0, 3, 4),
    (33, 24, 10, 6, 8, 3, 1, 2, 4, 3, 1, 0, 0, 2, 50),       # batch larger than G == plain diagonal order
    (45, 20, 12, 5, 7, 3, 1, 1, 3, 4, 1, 0, 0, 8, -1),       # time-key order
])
def test_ca3d_generation_batched_diagonal_order(emu_bin, args):
    _run(os.path.join(emu_bin, "emu_ca3d"), *args)


@pytest.mark.parametrize("args", [
    #  W   H   Z   G  rule P WPL kind seed warps ranks block seg flagrows genbatch pubworkers
    (45, 20, 12, 5, 7, 3, 1, 1, 3, 4, 1, 0, 0, 1, -1, 2),        # 2 CTAs of 2 workers + 1 publisher, time-key order
    (45, 20, 12, 5, 7, 3, 1, 1, 3, 4, 1, 0, 0, 2, -1, 4),
    (24, 12, 10, 9, 10, 3, 1, 1, 5, 1, 1, 0, 0, 1, -1, 1),       # one worker and its publisher
    (64, 33, 6, 9, 10, 4, 2, 1, 9, 7, 1, 0, 4, 5, 0, 3),         # row segments: mailbox handed over mid-sweep
    (45, 20, 12, 7, 7, 3, 1, 1, 3, 5, 1, 0, 0, 2, 3, 5),         # generation-batched diagonals
])
def test_ca3d_publisher_warps(emu_bin, args):
    """Publisher mode: workers bump a shared-memory mailbox after every row, one extra warp per CTA does the
    gpu-scope fence and raises the global counters for all of them."""
    _run(os.path.join(emu_bin, "emu_ca3d"), *args)


@pytest.mark.parametrize("args", [
    #  W   H   Z   G  rule P WPL kind seed warps ranks block seg flagrows genbatch pubworkers team tilegens
    (45, 20, 12, 5, 7, 3, 1, 1, 3, 8, 1, 0, 0, 2, 0, 0, 4),              # 2 CTAs of 4 warps, groups of 4 planes
    (45, 20, 12, 5, 7, 3, 1, 1, 3, 3, 1, 0, 0, 8, 0, 0, 3, 1),           # a single CTA: the claim order alone
    (64, 33, 7, 9, 10, 4, 2, 1, 9, 12, 1, 0, 0, 4, 0, 0, 5, 1),          # ragged last group
    (24, 12, 10, 9, 10, 3, 1, 1, 5, 1, 1, 0, 0, 3, 0, 0, 1),             # teams of one warp
    (45, 20, 12, 5, 7, 3, 1, 1, 3, 24, 1, 0, 0, 8, 0, 0, 24),            # team larger than the volume
    (45, 37, 12, 6, 7, 3, 1, 1, 3, 6, 2, 2, 0, 2, 0, 0, 3),              # 2 ranks, z-blocks of 2 planes < team
    (45, 50, 13, 5, 3, 3, 1, 1, 3, 8, 3, 5, 0, 4, 0, 0, 4, 1),           # 3 ranks, blocks of 5 = groups of 4 + 1
    (33, 30, 16, 5, 10, 8, 1, 1, 4, 4, 4, 1, 0, 2, 0, 0, 2),             # 4 ranks, every plane is an edge
    (20, 5, 3, 4, 7, 3, 1, 1, 4, 4, 4, 1, 0, 1, 0, 0, 2),                # ranks without any plane
    (33, 5, 9, 4, 8, 8, 1, 2, 3, 6, 2, 4, 0, 2, 0, 0, 3),                # ca3d_make seed (255s), 2 ranks
])
def test_ca3d_plane_teams(emu_bin, args):
    """Tile mode with one generation per tile (plane groups): a CTA sweeps a group of consecutive planes, warp w
    follows warp w-1 through a shared-memory row counter raised after every row; the service warp publishes the
    gpu-scope counters and pushes the z-block edges' rows to the neighbouring ranks."""
    _run(os.path.join(emu_bin, "emu_ca3d"), *args)


@pytest.mark.parametrize("args", [
    #  W   H   Z   G  rule P WPL kind seed warps ranks block seg flagrows genbatch pubworkers team tilegens
    (45, 20, 12, 8, 7, 3, 1, 1, 3, 40, 1, 0, 0, 2, 0, 0, 4, 2),          # 10 CTAs, tiles of 2 planes x 2 generations
    (45, 20, 12, 9, 7, 3, 1, 1, 3, 256, 1, 0, 0, 2, 0, 0, 16, 4),        # 4 x 4 tiles, ragged last generation group
    (45, 20, 13, 7, 10, 4, 1, 1, 3, 128, 1, 0, 0, 2, 0, 0, 8, 2),        # 4 planes x 2 generations, ragged last plane group
    (64, 33, 7, 9, 10, 4, 2, 1, 9, 96, 1, 0, 0, 4, 0, 0, 6, 3),          # 2 x 3 is refused (Tg <= Tz): falls to 3 x 2
    (45, 20, 12, 8, 7, 3, 1, 1, 3, 8, 1, 0, 0, 2, 0, 0, 4, 2),           # too few CTAs for the forward dependency: 4 x 1
    (45, 37, 12, 6, 7, 3, 1, 1, 3, 48, 2, 2, 0, 2, 0, 0, 4, 2),          # 2 ranks, blocks of 2 planes: every tile has two edges
    (45, 50, 13, 5, 3, 3, 1, 1, 3, 64, 3, 5, 0, 4, 0, 0, 4, 2),          # 3 ranks, blocks of 5 = tiles of 2 + 2 + 1 planes
    (33, 30, 16, 5, 10, 8, 1, 1, 4, 64, 4, 1, 0, 2, 0, 0, 4, 2),         # 4 ranks, single-plane blocks: 1-plane tiles, 2 generations each
    (33, 30, 16, 9, 7, 3, 1, 1, 4, 256, 4, 4, 0, 2, 0, 0, 16, 4),        # 4 ranks, 4 x 4 tiles = one z-block each
    (45, 20, 14, 7, 7, 3, 1, 1, 3, 360, 1, 0, 0, 2, 0, 0, 18, 3),        # the wide kernel's 6 x 3 tiles, ragged in z and g
    (2048, 4, 7, 4, 7, 3, 2, 0, 9, 72, 1, 0, 0, 2, 0, 0, 18, 3),         # ... at the BASELINE config-4 row width
    (33, 30, 18, 7, 7, 3, 1, 1, 4, 360, 2, 6, 0, 2, 0, 0, 18, 3),        # ... 2 ranks, z-blocks of one tile
    (33, 5, 9, 6, 8, 8, 1, 2, 3, 60, 2, 4, 0, 2, 0, 0, 4, 2),            # ca3d_make seed (255s), 2 ranks
    (2048, 6, 8, 4, 7, 3, 2, 0, 9, 64, 2, 4, 0, 2, 0, 0, 16, 4),         # BASELINE config-4 row width, 2 ranks
])
def test_ca3d_tiles_of_planes_and_generations(emu_bin, args):
    """Tile mode proper: a CTA sweeps nz planes x ng generations; generation g+1 of a plane follows generation g a
    few rows behind through shared-memory counters, and tiles depend on their NEXT neighbour in z (co-residency,
    bp_plan.h).  Multi-rank cases push several generations of an edge plane through one ghost plane in place --
    with both halo-row paths of the service warp: ld / st batches (the default) and 1-D bulk copies."""
    _run(os.path.join(emu_bin, "emu_ca3d"), *args)
    if args[10] > 1:
        _run(os.path.join(emu_bin, "emu_ca3d"), *args, env={"CLAPCA_HALO_LDST": "0"})


@pytest.mark.parametrize("args", [
    #  W   H   Z   G  rule P WPL kind seed warps ranks block seg flagrows genbatch pubworkers team tilegens layout chunk
    (45, 20, 12, 5, 7, 3, 1, 1, 3, 4, 1, 0, 0, 8, -1, 0, 0, 0, 1, 2),        # time-key order, cells resident
    (45, 20, 12, 5, 7, 3, 1, 1, 3, 4, 1, 0, 0, 8, -1, 0, 0, 0, 2, 3),        # ... fed / drained chunk by chunk
    (24, 12, 10, 9, 10, 3, 1, 1, 5, 1, 1, 0, 0, 3, -1, 0, 0, 0, 2, 16),      # one worker: the claim order alone
    (45, 20, 12, 5, 7, 3, 1, 1, 3, 8, 1, 0, 0, 2, 0, 0, 4, 0, 1, 2),         # plane teams, cells resident
    (45, 20, 13, 5, 7, 3, 1, 1, 3, 8, 1, 0, 0, 2, 0, 0, 4, 0, 2, 4),         # teams, ragged last group and chunk
    (64, 33, 7, 9, 10, 4, 2, 1, 9, 12, 1, 0, 0, 4, 0, 0, 5, 1, 2, 2),        # 2 words per lane, 16-byte row path
    (48, 12, 10, 3, 2, 8, 1, 2, 5, 1, 1, 0, 0, 3, 0, 0, 1, 0, 2, 1),         # ca3d_make seed (255s), 8 planes
    (2048, 3, 5, 2, 7, 3, 2, 0, 9, 4, 1, 0, 0, 2, -1, 0, 0, 0, 2, 2),        # BASELINE config-4 row width
    (1030, 2, 3, 2, 0, 3, 2, 1, 8, 3, 1, 0, 0, 2, -1, 0, 0, 0, 2, 1),        # ragged row end inside a word
    (96, 4, 5, 5, 7, 3, 4, 1, 7, 4, 1, 0, 0, 2, 0, 0, 3, 0, 2, 2),           # 4 words per lane
    (1, 1, 1, 3, 7, 3, 1, 1, 5, 2, 1, 0, 0, 2, -1, 0, 0, 0, 2, 1),
    (45, 20, 13, 6, 7, 3, 1, 1, 3, 80, 1, 0, 0, 2, 0, 0, 4, 2, 2, 4),        # 2 x 2 tiles with pack / unpack groups around them
    (45, 20, 12, 9, 7, 3, 1, 1, 3, 320, 1, 0, 0, 2, 0, 0, 16, 4, 1, 2),      # 4 x 4 tiles, cells resident
    # sharded volumes: the pack items' service warps seed the neighbours' ghost planes ("generation -1" counters)
    (45, 37, 12, 6, 7, 3, 1, 1, 3, 48, 2, 2, 0, 2, 0, 0, 4, 2, 1, 2),        # 2 ranks, z-blocks of 2 planes, 2 x 2 tiles
    (45, 50, 13, 5, 3, 3, 1, 1, 3, 64, 3, 5, 0, 4, 0, 0, 4, 2, 1, 2),        # 3 ranks, ragged last block
    (33, 30, 16, 5, 10, 8, 1, 1, 4, 64, 4, 1, 0, 2, 0, 0, 4, 1, 1, 2),       # 4 ranks, single-plane blocks
    (33, 30, 16, 9, 7, 3, 1, 1, 4, 320, 4, 4, 0, 2, 0, 0, 16, 4, 1, 2),      # 4 ranks, 4 x 4 tiles
    (33, 30, 15, 7, 7, 3, 1, 1, 4, 300, 2, 5, 0, 2, 0, 0, 15, 3, 1, 2),      # 2 ranks, the default 5 x 3 tiles
])
def test_ca3d_layout_items_streamed(emu_bin, args):
    """Layout items: pack ("generation -1") and unpack ("generation G") run as work items of the sweep launch; a
    feeder thread plays the H2D copy stream (cells arrive chunk by chunk, then the in_ready word moves) and a
    drainer thread plays the host side of the D2H (copies a chunk out once its planes carry the epoch)."""
    _run(os.path.join(emu_bin, "emu_ca3d"), *args)


@pytest.mark.parametrize("args", [
    #  W   H   Z   G  rule P WPL kind seed warps ranks block seg flagrows genbatch pubworkers team tilegens layout chunk gskew
    (45, 20, 12, 8, 7, 3, 1, 1, 3, 40, 1, 0, 0, 2, 0, 0, 4, 2, 0, 2, 1000),      # generation groups one after the other
    (45, 20, 12, 9, 7, 3, 1, 1, 3, 256, 1, 0, 0, 2, 0, 0, 16, 4, 0, 2, 7),       # a little more skew than Tz + 1
    (45, 20, 13, 7, 10, 4, 1, 1, 3, 12, 1, 0, 0, 2, 0, 0, 8, 2, 0, 2, 1000),     # 3 CTAs only: the window rule still holds
    (33, 30, 15, 7, 7, 3, 1, 1, 4, 45, 1, 0, 0, 2, 0, 0, 15, 3, 0, 2, 2048),     # the default 5 x 3 tiles
    (45, 20, 13, 6, 7, 3, 1, 1, 3, 80, 1, 0, 0, 2, 0, 0, 4, 2, 2, 4, 1000),      # with pack / unpack groups (streamed)
    (45, 37, 12, 6, 7, 3, 1, 1, 3, 48, 2, 2, 0, 2, 0, 0, 4, 2, 0, 2, 1000),      # 2 ranks
])
def test_ca3d_tile_order_generation_group_skew(emu_bin, args):
    """The key distance between the generation groups of the tile order (bp_plan.h, bp3_make_items_tile): any value
    above Tz is a valid claim order; large values run the groups one after the other."""
    _run(os.path.join(emu_bin, "emu_ca3d"), *args)


# ---- 2D bit-plane engine (ca2d_bitplane.cuh): one CTA per generation, CTA-wide scan -----------------------

@pytest.mark.parametrize("args", [
    #  W    H   G  born   surv  nr decay moore P WPL warps kind seed ctas flagrows
    (40, 40, 3, 0xc, 0x180, 4, 1, 1, 3, 1, 1, 0, 1, 2, 2),            # ca_test (core/terrain.c:391-398)
    (40, 70, 5, 0x1e0, 0x1f0, 1, 1, 1, 1, 1, 1, 0, 2, 3, 2),          # binary cave rule, 1 bit per cell
    (33, 100, 4, 0xc, 0x180, 4, 1, 1, 3, 1, 2, 1, 3, 2, 1),
    (20, 130, 6, 0x6, 0x1c, 2, 1, 0, 3, 2, 1, 1, 4, 3, 2),            # von Neumann
    (17, 300, 3, 0x1e, 0xff, 20, 0, 1, 8, 2, 3, 0, 5, 2, 3),          # ca_instors[0] without decay, 8 planes
    (50, 64, 7, 0x1e0, 0x1f0, 1, 1, 1, 1, 4, 1, 0, 6, 4, 4),
    (1, 1, 3, 0x1, 0x0, 1, 1, 1, 1, 1, 1, 0, 7, 2, 2),
    (5, 1, 3, 0x3, 0x0, 1, 1, 1, 1, 1, 1, 0, 7, 2, 2),
    (1, 37, 3, 0x3, 0x2, 1, 1, 0, 1, 1, 1, 0, 7, 2, 2),
    (64, 257, 9, 0xc, 0x180, 4, 1, 1, 4, 1, 9, 1, 8, 5, 2),
    (12, 40, 4, 0xc, 0x180, 0, 1, 1, 3, 1, 1, 1, 8, 2, 2),            # nr_states == 0: births are no-ops
    (12, 40, 4, 0xc, 0x180, 256 + 3, 1, 1, 3, 1, 1, 1, 8, 2, 2),      # nr_states wraps through uint8
    (12, 40, 4, 0xc, 0x180, 256, 1, 1, 1, 1, 2, 1, 8, 2, 2),          # one state plane and nothing is ever born
    (40, 1500, 4, 0x1e0, 0x1f0, 1, 1, 1, 1, 1, 16, 0, 8, 3, 2),       # 16 warps per row: the packed carry masks are full
    (40, 2000, 3, 0x1e0, 0x1f0, 1, 1, 1, 1, 2, 16, 0, 9, 3, 2),
    (30, 1000, 3, 0xaa, 0x155, 1, 1, 1, 1, 2, 16, 0, 9, 3, 2),        # non-monotone rule across 16 warps
    (30, 1000, 3, 0xaa, 0x155, 1, 1, 1, 1, 1, 16, 0, 9, 3, 5),        # ... row marks every 5 rows
])
def test_ca2d_bitplane_rules_and_shapes(emu_bin, args):
    _run(os.path.join(emu_bin, "emu_ca2d"), *args)


@pytest.mark.parametrize("args", [
    #  W    H   G  born   surv  nr decay moore P WPL warps kind seed ctas flagrows forcedyn
    (40, 70, 5, 0x1e0, 0x1f0, 1, 1, 1, 1, 1, 1, 0, 2, 3, 2, 1),       # cave rule through the run-time tables + Kogge-Stone scan
    (33, 2100, 4, 0x1e0, 0x1f0, 1, 1, 1, 1, 2, 2, 0, 2, 3, 1, 1),
    (40, 40, 3, 0xc, 0x180, 4, 1, 1, 3, 1, 1, 0, 1, 2, 2, 1),         # ca_test through the run-time tables
    (33, 300, 6, 0x1e0, 0x1f0, 5, 1, 1, 3, 4, 1, 1, 3, 2, 2, 0),      # cave masks, multi-state, dense values: carry-chain path with decay
    (21, 5000, 4, 0x1e0, 0x1f0, 1, 1, 1, 1, 2, 3, 0, 9, 4, 2, 0),     # carry chain across three warps, long runs of propagating cells
    (9, 700, 5, 0x1e0, 0x1f0, 1, 1, 0, 1, 1, 1, 0, 5, 2, 2, 0),       # cave masks with the von Neumann count
    (19, 3000, 3, 0xc, 0x180, 4, 1, 1, 3, 2, 2, 1, 4, 3, 2, 0),       # ca_test compile-time tables across two warps
])
def test_ca2d_rule_instantiations_agree(emu_bin, args):
    """The compile-time rules (one LOP3 per table; the monotone cave rule resolves the in-row chain with an integer
    add) and the run-time rule (mux trees, Kogge-Stone scan) are different code: each against the oracle."""
    _run(os.path.join(emu_bin, "emu_ca2d"), *args)


@pytest.mark.parametrize("args", [
    (5, 2100, 4, 0x1e0, 0x1f0, 1, 1, 1, 1, 2, 2, 0, 2, 3, 1),         # rows span two warps, 2 words per lane
    (4, 3000, 3, 0x6, 0x1c, 2, 1, 0, 3, 1, 3, 1, 3, 2, 2),            # three warps, von Neumann
    (7, 2050, 3, 0xc, 0x180, 4, 1, 1, 3, 1, 3, 0, 4, 1, 3),           # a single CTA runs every generation in turn
    (5, 4200, 2, 0x1e0, 0x1f0, 1, 1, 1, 1, 4, 2, 0, 5, 2, 2),
    (9, 1025, 5, 0x1fe, 0x0, 3, 1, 1, 3, 1, 2, 1, 9, 3, 2),           # one cell beyond a warp's span
    (2, 32800, 2, 0x1e0, 0x1f0, 1, 1, 1, 1, 4, 16, 0, 10, 2, 2),      # 16 warps x 4 words (the widest row variant)
    (3, 16400, 2, 0x1e, 0xff, 20, 0, 1, 8, 2, 16, 1, 11, 2, 2),       # 8 planes: 16 warps x 2 words
])
def test_ca2d_bitplane_rows_across_warps(emu_bin, args):
    _run(os.path.join(emu_bin, "emu_ca2d"), *args)


# ---- 2D diagonal engine (ca2d_skew.cuh): rows = diagonals 2x + y, warps chained by mailboxes, no CTA barrier -----

@pytest.mark.parametrize("args", [
    #  W     H    G  born   surv  nr decay moore WPL seed ctas forcedyn density
    (40, 70, 3, 0x1e0, 0x1f0, 1, 1, 1, 1, 1),                          # binary cave rule (alive bit folded into the count)
    (40, 70, 5, 0x1e0, 0x1f0, 1, 1, 1, 2, 2),
    (33, 100, 4, 0xc, 0x180, 1, 1, 1, 1, 3),                           # ca_test's masks on a binary grid
    (20, 130, 6, 0x6, 0x1c, 1, 1, 0, 1, 4),                            # von Neumann
    (1, 1, 3, 0x1, 0x0, 1, 1, 1, 1, 7),
    (5, 1, 3, 0x3, 0x0, 1, 1, 1, 1, 7),
    (1, 37, 3, 0x3, 0x2, 1, 1, 0, 1, 7),
    (64, 257, 9, 0x8, 0xc, 1, 1, 1, 2, 8, 5, 0, 3),                    # Life, more generations than CTAs
    (12, 40, 4, 0xc, 0x180, 256, 1, 1, 1, 8, 2),                       # nr_states wraps to 0: nothing is ever born
    (96, 80, 4, 0x1e, 0xff, 1, 0, 1, 1, 5, 2, 0, 2),                   # no decay: survivors keep their value
    (40, 70, 5, 0x1e0, 0x1f0, 1, 1, 1, 1, 2, 3, 1),                    # cave rule through the run-time tables
    (33, 100, 4, 0xc, 0x180, 1, 1, 1, 2, 3, 2, 1),
])
def test_ca2d_diagonal_rules_and_shapes(emu_bin, args):
    _run(os.path.join(emu_bin, "emu_ca2d_skew"), *args)


@pytest.mark.parametrize("args", [
    (2100, 5, 4, 0x1e0, 0x1f0, 1, 1, 1, 1, 2),                         # three warps, the band is narrower than a warp
    (3000, 4, 3, 0x6, 0x1c, 1, 1, 0, 1, 3, 2),                         # von Neumann across warps
    (2050, 7, 3, 0xc, 0x180, 1, 1, 1, 1, 4, 1),                        # a single CTA runs every generation in turn
    (4200, 5, 2, 0x1e0, 0x1f0, 1, 1, 1, 2, 5, 2),
    (1025, 9, 5, 0x1fe, 0x0, 1, 1, 1, 1, 9, 3),                        # one cell beyond a warp's span
    (1500, 40, 4, 0xaa, 0x155, 1, 1, 1, 1, 9, 3, 0, 3),                # non-monotone rule
    (2500, 3000, 2, 0x1e0, 0x1f0, 1, 1, 1, 1, 9, 2, 0, 4),             # groups without masks (H > 2048), posts over a long window
    (3333, 2222, 7, 0x1e0, 0x1f0, 1, 0, 1, 1, 5, 3),
    (5000, 2600, 5, 0x1e0, 0x1f0, 1, 1, 1, 1, 6, 5, 0, 4),             # generations queue behind each other, 5 warps
    (7000, 1500, 4, 0xc, 0x180, 1, 1, 1, 2, 4, 4, 1, 3),               # two words per lane, run-time tables
    (16384, 100, 2, 0x1e0, 0x1f0, 1, 1, 1, 1, 11, 2),                  # BASELINE config 3's width: 16 warps x 1 word
    (16384, 4200, 2, 0x1e0, 0x1f0, 1, 1, 1, 2, 12, 2, 0, 4),           # ... 8 warps x 2 words, steady groups
])
def test_ca2d_diagonal_across_warps(emu_bin, args):
    """The chain of warps: bit 31 of a warp's last word reaches the next warp through the tagged mailbox ring, the
    ring's back-pressure, warps that start and finish with the band of valid cells, the publisher's minimum over the
    warps' step counters."""
    _run(os.path.join(emu_bin, "emu_ca2d_skew"), *args)
