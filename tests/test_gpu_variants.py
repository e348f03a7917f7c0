"""Every compiled variant of the bit-plane CA engines and every host dispatch edge, against the oracle.

The library compiles, per rule object, one 3D kernel for each (state planes P, words per lane WPL) and one 2D kernel
for each (P, WPL, Moore / von Neumann), and picks one of them from the input: P from the largest value that can
occur, WPL and the warps per CTA from the row length, the kernel kind (one warp per sweep, team, wide team) from
(P, WPL).  The host-side selection is mirrored here in plain Python.  A CPU test checks that the case tables below
reach every compiled variant (parsed from the instantiation files and the Makefile), so a new instantiation without
a case fails on a machine without a GPU.  The GPU tests run each case on a thin volume or strip the oracle finishes
in milliseconds and compare bit for bit; they also assert the engine and plane count the run reports, so that a case
cannot silently test a different variant than its id names."""
import os
import re

import numpy as np
import pytest

import oracle_lib

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
AUTO, WAVEFRONT, BITPLANE, DIAGONAL = 0, 1, 2, 3
ENGINE_NAMES = {WAVEFRONT: "wavefront", BITPLANE: "bitplane", DIAGONAL: "diagonal"}
ERR_UNSUPPORTED = 5
gpu_mark = pytest.mark.gpu


# ---- mirrors of the host-side selection (bp_plan.h, bp2_launch.h, sk2_launch.h, ca3d_bitplane.cuh, clapca_api.cu) --

TEAM_WARPS, WIDE_TEAM = 15, 18          # CLAPCA_TEAM_WARPS, BP3_WIDE_TEAM
MAX_FUSED_GENERATIONS = 4096            # kMaxFusedGenerations


def bp_planes_for(maxv):
    return 3 if maxv < 8 else 4 if maxv < 16 else 8


def bp_wpl_for(d0):
    return 1 if d0 <= 1024 else 2 if d0 <= 2048 else 4 if d0 <= 4096 else 0


def bp2_planes_for(maxv):
    return 1 if maxv < 2 else bp_planes_for(maxv)


def bp2_shape_for(n, P):
    """(WPL, warps) of the 2D row engine for rows of n cells, None = too wide"""
    rw = (n + 31) // 32
    for cap in (8, 16):
        for wpl in ((1, 2) if P >= 8 else (1, 2, 4)):
            nw = (rw + 32 * wpl - 1) // (32 * wpl)
            if nw <= cap:
                return wpl, max(nw, 1)
    return None


def sk2_shape_for(w):
    """(WPL, warps) of the 2D diagonal engine for w columns, None = too wide"""
    if w < 1 or w > 16384:
        return None
    wpl = 1 if w <= 4096 else 2
    warps = (w + 31 * 32 * wpl - 1) // (31 * 32 * wpl)
    return (wpl, warps) if warps * wpl <= 18 else None


def bp3_team_cap(P, wpl):
    return TEAM_WARPS if P <= 4 and wpl <= 2 else 7


def bp3_team_cap_wide(P, wpl):
    return WIDE_TEAM if P == 3 and wpl <= 2 else 0


def team_config(P, wpl, env=None):
    """compute warps per CTA of a single-GPU resident run (0 = one warp per sweep); env = $CLAPCA_TEAM"""
    cap = bp3_team_cap(P, wpl)
    t = cap if cap >= 12 else 0
    if bp3_team_cap_wide(P, wpl) > cap:
        t = cap = bp3_team_cap_wide(P, wpl)
    if env is not None:
        t = int(env)
        cap = max(cap, bp3_team_cap_wide(P, wpl))
    return 0 if t <= 0 else min(t, cap)


def kernel_kind(P, wpl, team):
    """the kernel bp3_inst.cu launches for a team size: ca3d_sweep_kernel, ca3d_team_kernel or ca3d_team_wide_kernel"""
    if team <= 0:
        return "sweep"
    return "wide" if P == 3 and wpl <= 2 and team > bp3_team_cap(P, wpl) else "team"


def bp2_rule_object(born, surv, nr, decay):
    """the rule object of bp2_rule_for(): the host passes surv = 0x1ff when there is no decay"""
    surv = surv & 0x1FF if decay else 0x1FF
    if not nr & 0xFF:
        return "dyn"
    if (born & 0x1FF, surv) == (0x1E0, 0x1F0):
        return "cave"
    if (born & 0x1FF, surv) == (0x00C, 0x180):
        return "test"
    return "dyn"


# ---- case tables --------------------------------------------------------------------------------------------------

def _b(*ns):
    return sum(1 << n for n in ns)


# 3D rule objects: cas[0..8] (bp3_inst.cu) and the run-time-mask object 9, here with masks outside cas[] and a
# nr_states per plane count whose births write the largest value the planes hold (7, 15) or need 8 planes (199)
DYN3_MASKS = (_b(2, 5, 6, 7, 8, 13, 26), _b(5, 6, 10, 17))      # (surv, born)
DYN3_NR = {3: 8, 4: 16, 8: 200}
WIDTH3 = {1: 1000, 2: 2047, 4: 3999}        # ragged row widths: one per words-per-lane variant


def rule3(rule, P):
    """(surv, born, nr_states) of 3D rule object `rule` in a case of P planes"""
    if rule == 9:
        return DYN3_MASKS + (DYN3_NR[P],)
    from clap_b200.rules import CA3D_RULES
    r = CA3D_RULES[rule]
    return r.surv_mask, r.born_mask, r.nr_states


def bornval(nr):
    return (nr - 1) & 0xFF


def reachable3(rule, P):
    """P >= the planes the rule's births alone need (the resident run packs with at least those)"""
    return bp_planes_for(bornval(rule3(rule, P)[2])) <= P


CASES3 = [(rule, P, wpl, WIDTH3[wpl]) for rule in range(10) for P in (3, 4, 8) for wpl in (1, 2, 4)
          if reachable3(rule, P)]
TEAM_ENVS = (None, "0", "7")        # the default kind; one warp per sweep; the team kernel the slab path runs at cap 7


def _params3():
    out = []
    for rule, P, wpl, d0 in CASES3:
        for env in TEAM_ENVS:
            kind = kernel_kind(P, wpl, team_config(P, wpl, env))
            tag = "default" if env is None else env
            out.append(pytest.param(rule, P, wpl, d0, env, id=f"rule{rule}-P{P}-WPL{wpl}-d{d0}-TEAM{tag}-{kind}"))
    return out


# 2D rule objects (bp2_inst.cu, BP2_RULE 0..2); the Dyn masks have a bit at n = 8 to use the n = K + 1 table
RULES2 = {"dyn": (_b(3, 6, 8), _b(2, 3, 8)), "cave": (0x1E0, 0x1F0), "test": (0x00C, 0x180)}
NR2 = {1: 1, 3: 5, 4: 12, 8: 200}               # nr_states per plane count (the value a born cell takes)
VMAX2 = {1: 1, 3: 7, 4: 15, 8: 255}              # largest seed value per plane count
# the neighbourhoods the Dyn object is run with: decay on and off, and vnv / mv without decay (alive-bit counts)
DYN_NEIGH = {True: ((oracle_lib.NEIGH_M1, 1), (oracle_lib.NEIGH_M1, 0), (oracle_lib.NEIGH_MV, 0)),
             False: ((oracle_lib.NEIGH_VN1, 1), (oracle_lib.NEIGH_VN1, 0), (oracle_lib.NEIGH_VNV, 0))}
NEIGH_NAMES = {oracle_lib.NEIGH_VN1: "vn1", oracle_lib.NEIGH_M1: "m1", oracle_lib.NEIGH_VNV: "vnv",
               oracle_lib.NEIGH_MV: "mv"}
# row lengths (cells per engine row = the array's height) per words-per-lane variant
LEN2 = {(1, False): (1000, 4000), (2, False): (12000,), (4, False): (20000, 32768, 40000, 65536),
        (1, True): (1000, 4000), (2, True): (16384, 32768)}          # key: (WPL, P == 8)
WIDTHS2 = (16, 24, 33, 48)


def _cases2():
    cases = []
    k = 0
    turn = {}
    for obj in RULES2:
        for P in (1, 3, 4, 8):
            for moore in (True, False):
                for wpl in ((1, 2) if P == 8 else (1, 2, 4)):
                    lens = LEN2[(wpl, P == 8)]
                    # the WPL-4 lengths and the P = 8 WPL-2 lengths rotate over the cases (every one is reached
                    # several times); the short ones run everywhere
                    if len(lens) > 1 and wpl > 1:
                        t = turn[(wpl, P == 8)] = turn.get((wpl, P == 8), -1) + 1
                        lens = (lens[t % len(lens)],)
                    for n in lens:
                        born, surv = RULES2[obj]
                        neigh, decay = (oracle_lib.NEIGH_M1 if moore else oracle_lib.NEIGH_VN1), 1
                        if obj == "dyn":
                            neigh, decay = DYN_NEIGH[moore][k % 3]
                        w, gens = WIDTHS2[k % 4], 3 + k % 3
                        k += 1
                        cases.append((obj, P, moore, wpl, n, born, surv, NR2[P], decay, neigh, w, gens))
    return cases


CASES2 = _cases2()


def _params2():
    out = []
    for c in CASES2:
        obj, P, moore, wpl, n, born, surv, nr, decay, neigh, w, gens = c
        shape = bp2_shape_for(n, P)
        tag = f"{obj}-P{P}-WPL{shape[0]}-warps{shape[1]}-{'moore' if moore else 'vn'}-n{n}-{NEIGH_NAMES[neigh]}"
        out.append(pytest.param(c, id=tag + ("-decay" if decay else "")))
    return out


# ---- CPU: the tables reach every compiled variant; the mirrors agree with the sources -----------------------------

def _read(*parts):
    with open(os.path.join(ROOT, *parts)) as f:
        return f.read()


def _cases_in(src, macro):
    body = re.sub(r"#define[^\n]*(\\\n[^\n]*)*", "", src)          # the macro's own definition is not a case
    return {tuple(int(v) for v in m) for m in re.findall(macro + r"\((\d+),\s*(\d+)\)", body)}


def _make_list(name):
    return [int(v) for v in re.search(r"^" + name + r"\s*:=\s*([\d ]+)$", _read("clap_b200", "csrc", "Makefile"),
                                      re.M).group(1).split()]


def test_case_tables_reach_every_compiled_variant():
    bp3 = _cases_in(_read("clap_b200", "csrc", "bp3_inst.cu"), "BP3_CASE")
    bp2 = _cases_in(_read("clap_b200", "csrc", "bp2_inst.cu"), "BP2_CASE")
    rules3, rules2 = _make_list("RULES"), _make_list("RULES2")
    assert len(bp3) == 9 and len(bp2) == 11 and rules3 == list(range(10)) and rules2 == [0, 1, 2]

    # 3D: every (rule, P, WPL) except those whose births need more planes than P -- the dispatch never picks them
    compiled3 = {(r, P, w) for r in rules3 for P, w in bp3}
    reached3 = set()
    for rule, P, wpl, d0 in CASES3:
        assert bp_wpl_for(d0) == wpl and d0 % 32, (rule, P, d0)
        reached3.add((rule, P, wpl))
    unreachable = {(r, P, w) for r, P, w in compiled3 if not reachable3(r, P)}
    assert unreachable == {(r, 3, w) for r in (2, 4) for w in (1, 2, 4)}       # pyroclastic, builder: nr_states 10
    assert reached3 == compiled3 - unreachable
    # every kernel kind the default dispatch picks for some variant is exercised, and the slab path's team of 7
    kinds = {(P, w, kernel_kind(P, w, team_config(P, w, e))) for _, P, w, _ in CASES3 for e in TEAM_ENVS}
    assert {k for _, _, k in kinds} == {"sweep", "team", "wide"}
    assert all((P, w, "team") in kinds and (P, w, "sweep") in kinds for P, w in bp3)

    # 2D: every (rule object, P, WPL, neighbourhood)
    names2 = {0: "dyn", 1: "cave", 2: "test"}
    compiled2 = {(names2[r], P, w, m) for r in rules2 for P, w in bp2 for m in (True, False)}
    reached2 = set()
    warps_at = {}
    for obj, P, moore, wpl, n, born, surv, nr, decay, neigh, w, gens in CASES2:
        assert bp2_rule_object(born, surv, nr, decay) == obj
        assert bp2_planes_for(max(VMAX2[P], nr & 0xFF)) == P
        assert moore == (neigh in (oracle_lib.NEIGH_M1, oracle_lib.NEIGH_MV))
        assert not (decay and neigh in (oracle_lib.NEIGH_VNV, oracle_lib.NEIGH_MV))
        assert 16 <= w <= 48 and 3 <= gens <= 5
        got = bp2_shape_for(n, P)
        assert got[0] == wpl, (obj, P, n)
        reached2.add((obj, P, wpl, moore))
        warps_at.setdefault((P == 8, wpl), set()).add(got[1])
    assert reached2 == compiled2
    # the largest warp count of each cap: 8 and 16 warps at WPL 4, and 8 and 16 at P = 8 / WPL 2
    assert {8, 16} <= warps_at[(False, 4)] and {8, 16} <= warps_at[(True, 2)]
    assert {1, 4} <= warps_at[(False, 1)] and 6 in warps_at[(False, 2)]
    assert 5 in warps_at[(False, 4)] and 10 in warps_at[(False, 4)]


def test_selection_mirrors_match_the_sources():
    """The mirrors against the limits the library states in its refusal messages and constants."""
    api = _read("clap_b200", "csrc", "clapca_api.cu")
    bp3h = _read("clap_b200", "csrc", "ca3d_bitplane.cuh")
    assert int(re.search(r"#define CLAPCA_TEAM_WARPS (\d+)", bp3h).group(1)) == TEAM_WARPS
    assert int(re.search(r"BP3_WIDE_TEAM = (\d+)", bp3h).group(1)) == WIDE_TEAM
    assert int(re.search(r"kMaxFusedGenerations = (\d+);", _read("clap_b200", "csrc", "api_internal.h")).group(1)) \
        == MAX_FUSED_GENERATIONS
    assert int(re.search(r"SK2_MAX_WARPS = (\d+)", _read("clap_b200", "csrc", "ca2d_skew.cuh")).group(1)) == 18

    lim3 = int(re.search(r"bit-plane engine handles rows of at most (\d+) cells", api).group(1))
    assert bp_wpl_for(lim3) == 4 and bp_wpl_for(lim3 + 1) == 0
    m = re.search(r"rows of at \"\s*\"most (\d+) cells \((\d+) with values >= (\d+)\)", api)
    lim2, lim2_8, v8 = (int(v) for v in m.groups())
    assert bp2_planes_for(v8) == 8 and bp2_planes_for(v8 - 1) < 8
    for P in (1, 3, 4):
        assert bp2_shape_for(lim2, P) == (4, 16) and bp2_shape_for(lim2 + 1, P) is None
    assert bp2_shape_for(lim2_8, 8) == (2, 16) and bp2_shape_for(lim2_8 + 1, 8) is None
    limd = int(re.search(r"at \"\s*\"most (\d+) columns", api).group(1))
    assert sk2_shape_for(limd) == (2, 9) and sk2_shape_for(limd + 1) is None
    # the breakpoints of the issue's dispatch table
    assert [bp2_shape_for(n, 3) for n in (1000, 4000, 12000, 16384, 20000, 32768, 40000, 65536)] == \
        [(1, 1), (1, 4), (2, 6), (2, 8), (4, 5), (4, 8), (4, 10), (4, 16)]
    assert [bp2_shape_for(n, 8) for n in (8193, 16384, 16385, 32768)] == [(2, 5), (2, 8), (2, 9), (2, 16)]
    assert [bp2_shape_for(n, 3) for n in (32769, 65536)] == [(4, 9), (4, 16)]


# ---- GPU: helpers -------------------------------------------------------------------------------------------------

def synth(rng, shape, p_alive, vmax):
    return (rng.integers(1, vmax + 1, shape) * (rng.random(shape) < p_alive)).astype(np.uint8)


def seed3(rng, shape, P):
    """values 1..5 (3 planes), 1..15 with some 15s (4 planes), or 1..5 with a few 255s (8 planes)"""
    vol = synth(rng, shape, 0.35, 15 if P == 4 else 5)
    if P == 4:
        vol.reshape(-1)[rng.integers(0, vol.size, 8)] = 15
    if P == 8:
        vol[rng.random(shape) < 0.003] = 255
        vol.reshape(-1)[rng.integers(0, vol.size, 4)] = 255
    return vol


def run3_grid(gpu, vol, rule, steps, engine):
    """(population, result, stats) of a device-resident grid run"""
    d2, d1, d0 = vol.shape
    grid = gpu.Grid(d0, d1, d2)
    try:
        grid.upload(vol)
        pop = grid.run3d(rule, steps, engine=engine)
        st = grid.stats()
        out = np.empty_like(vol)
        grid.download(out)
    finally:
        grid.close()
    return pop, out, st


def run2_grid(gpu, arr, ca, steps, engine):
    """(result, stats) of a device-resident 2D run over the whole grid"""
    h, w = arr.shape
    grid = gpu.Grid(w, h, 1)
    try:
        grid.upload(arr)
        grid.run2d(ca, steps, side=max(w, h), engine=engine)
        st = grid.stats()
        out = np.empty_like(arr)
        grid.download(out)
    finally:
        grid.close()
    return out, st


def ca3(gpu, surv, born, nr):
    return gpu.CellAutomaton("t", born_mask=born, surv_mask=surv, nr_states=nr)


# ---- GPU: 3D matrix -----------------------------------------------------------------------------------------------

@gpu_mark
@pytest.mark.parametrize("rule,P,wpl,d0,team", _params3())
def test_ca3d_variant_vs_oracle(gpu, oracle, monkeypatch, rule, P, wpl, d0, team):
    if team is None:
        monkeypatch.delenv("CLAPCA_TEAM", raising=False)
    else:
        monkeypatch.setenv("CLAPCA_TEAM", team)
    surv, born, nr = rule3(rule, P)
    rng = np.random.default_rng(rule * 100 + P * 10 + wpl)
    vol = seed3(rng, (5, 6, d0), P)
    assert bp_planes_for(max(int(vol.max()), bornval(nr))) == P
    want = vol.copy()
    wpop = oracle.ca3d_run(want, surv, born, nr, 5)
    pop, got, st = run3_grid(gpu, vol, rule if rule < 9 else ca3(gpu, surv, born, nr), 5, BITPLANE)
    assert st["engine"] == "bitplane" and st["planes"] == P
    assert pop == wpop and np.array_equal(got, want), int((got != want).sum())


# ---- GPU: 2D matrix -----------------------------------------------------------------------------------------------

@gpu_mark
@pytest.mark.parametrize("case", _params2())
def test_ca2d_variant_vs_oracle(gpu, oracle, monkeypatch, case):
    obj, P, moore, wpl, n, born, surv, nr, decay, neigh, w, gens = case
    monkeypatch.setenv("CLAPCA_2D_SKEW", "0")        # a binary grid could otherwise go to the diagonal engine
    rng = np.random.default_rng(n + 7 * w + P)
    arr = synth(rng, (n, w), 0.45, VMAX2[P])
    arr.reshape(-1)[rng.integers(0, arr.size, 4)] = VMAX2[P]
    want = oracle.ca2d_run(arr.copy(), born, surv, nr, decay, neigh, gens, side=max(n, w))
    got, st = run2_grid(gpu, arr, gpu.CellAutomaton("t", born, surv, nr, bool(decay), neigh), gens, BITPLANE)
    assert st["engine"] == "bitplane" and st["planes"] == P
    assert np.array_equal(got, want), int((got != want).sum())


# ---- GPU: dispatch edges ------------------------------------------------------------------------------------------

@gpu_mark
@pytest.mark.parametrize("d0,engine", [(4096, "bitplane"), (4097, "wavefront")])
def test_ca3d_row_width_limit(gpu, oracle, d0, engine):
    rng = np.random.default_rng(d0)
    vol = seed3(rng, (3, 4, d0), 8)
    want = vol.copy()
    s, b, n = oracle.ca3d_rule(7)
    wpop = oracle.ca3d_run(want, s, b, n, 4)
    pop, got, st = run3_grid(gpu, vol, 7, 4, AUTO)
    assert st["engine"] == engine
    assert pop == wpop and np.array_equal(got, want)
    if engine == "wavefront":
        with pytest.raises(gpu.ClapcaError) as ei:
            run3_grid(gpu, vol, 7, 4, BITPLANE)
        assert ei.value.status == ERR_UNSUPPORTED


@gpu_mark
def test_ca3d_generations_beyond_one_launch(gpu, oracle):
    """More than kMaxFusedGenerations generations are cut into several sweep launches."""
    rng = np.random.default_rng(4096)
    vol = synth(rng, (4, 5, 40), 0.3, 5)
    rule = ca3(gpu, _b(4, 5, 6), _b(4, 6), 3)           # keeps a 40 x 5 x 4 volume alive for thousands of generations
    launches = {}
    for steps in (MAX_FUSED_GENERATIONS, MAX_FUSED_GENERATIONS + 1, 9000):
        want = vol.copy()
        wpop = oracle.ca3d_run(want, rule.surv_mask, rule.born_mask, rule.nr_states, steps)
        pop, got, st = run3_grid(gpu, vol, rule, steps, BITPLANE)
        assert st["engine"] == "bitplane"
        assert pop == wpop and np.array_equal(got, want), steps
        launches[steps] = st["launches"]
    assert launches[MAX_FUSED_GENERATIONS + 1] == launches[MAX_FUSED_GENERATIONS] + 1
    assert launches[9000] == launches[MAX_FUSED_GENERATIONS] + 2
    # streamed with page-locked buffers: the one-launch pipeline holds at most kMaxFusedGenerations, longer runs
    # take the sequential upload / run / download path and still give the oracle's volume
    import torch
    keep_in = torch.empty(vol.shape, dtype=torch.uint8, pin_memory=True)
    keep_out = torch.empty(vol.shape, dtype=torch.uint8, pin_memory=True)
    host_in, host_out = keep_in.numpy(), keep_out.numpy()
    grid = gpu.Grid(40, 5, 4)
    try:
        for steps, streamed in ((MAX_FUSED_GENERATIONS, True), (MAX_FUSED_GENERATIONS + 1, False)):
            host_in[...] = vol
            host_out[...] = 0xEE
            want = vol.copy()
            wpop = oracle.ca3d_run(want, rule.surv_mask, rule.born_mask, rule.nr_states, steps)
            assert grid.run3d_streamed(rule, steps, host_in, host_out, max_value=5) == wpop
            assert grid.stats()["streamed"] == streamed
            assert np.array_equal(host_out, want), steps
    finally:
        grid.close()


@gpu_mark
@pytest.mark.parametrize("n,vmax", [(65536, 4), (65537, 4), (32768, 16), (32769, 16)])
def test_ca2d_row_length_limit(gpu, oracle, monkeypatch, n, vmax):
    """AUTO takes the row engine up to its limit and the wavefront beyond it; BITPLANE refuses beyond it."""
    monkeypatch.setenv("CLAPCA_2D_SKEW", "0")
    rng = np.random.default_rng(n + vmax)
    arr = synth(rng, (n, 16), 0.5, 4)
    if vmax == 16:
        arr[n // 2, 7] = 16
    want = oracle.ca2d_run(arr.copy(), 0xC, 0x180, 4, 1, oracle_lib.NEIGH_M1, 3, side=n)
    fits = bp2_shape_for(n, bp2_planes_for(vmax)) is not None
    got, st = run2_grid(gpu, arr, gpu.CA_TEST, 3, AUTO)
    assert st["engine"] == ("bitplane" if fits else "wavefront")
    assert np.array_equal(got, want)
    if fits:
        assert st["planes"] == bp2_planes_for(vmax)
    else:
        with pytest.raises(gpu.ClapcaError) as ei:
            run2_grid(gpu, arr, gpu.CA_TEST, 3, BITPLANE)
        assert ei.value.status == ERR_UNSUPPORTED


@gpu_mark
@pytest.mark.parametrize("w", [16384, 16385])
def test_ca2d_diagonal_width_limit(gpu, oracle, monkeypatch, w):
    rng = np.random.default_rng(w)
    arr = synth(rng, (16, w), 0.47, 1)
    ca = gpu.CellAutomaton("cave", 0x1E0, 0x1F0, 1, True, oracle_lib.NEIGH_M1)
    want = oracle.ca2d_run(arr.copy(), 0x1E0, 0x1F0, 1, 1, oracle_lib.NEIGH_M1, 3, side=w)
    if w <= 16384:
        got, st = run2_grid(gpu, arr, ca, 3, DIAGONAL)
        assert st["engine"] == "diagonal"
        assert np.array_equal(got, want)
    else:
        with pytest.raises(gpu.ClapcaError) as ei:
            run2_grid(gpu, arr, ca, 3, DIAGONAL)
        assert ei.value.status == ERR_UNSUPPORTED
    monkeypatch.setenv("CLAPCA_2D_SKEW", "1")          # asks for the diagonal engine wherever it applies
    got, st = run2_grid(gpu, arr, ca, 3, AUTO)
    assert st["engine"] == ("diagonal" if w <= 16384 else "bitplane")
    assert np.array_equal(got, want)


@gpu_mark
@pytest.mark.parametrize("d0", [50, 2000])
@pytest.mark.parametrize("nr", [0, 1, 2, 256, 257, 300])
def test_ca3d_nr_states_edges(gpu, oracle, d0, nr):
    """born cells take (nr_states - 1) & 0xff: 255 (8 planes), 0 (a birth that writes nothing), 1, 43"""
    surv, born = _b(3, 4, 5, 6, 9), _b(4, 5, 7)
    rng = np.random.default_rng(d0 + nr)
    vol = synth(rng, (5, 9, d0), 0.4, 5)
    want = vol.copy()
    wpop = oracle.ca3d_run(want, surv, born, nr, 5)
    for engine in (BITPLANE, WAVEFRONT):
        pop, got, st = run3_grid(gpu, vol, ca3(gpu, surv, born, nr), 5, engine)
        if engine == BITPLANE:
            assert st["planes"] == bp_planes_for(max(5, bornval(nr)))
        assert pop == wpop and np.array_equal(got, want), (engine, int((got != want).sum()))


@gpu_mark
def test_ca3d_mask_bits_above_the_largest_count(gpu, oracle):
    """Bits 27..31 of the 3D masks name counts a cell never has: they change nothing, on either engine."""
    rng = np.random.default_rng(27)
    for d0, (surv, born, nr) in ((300, rule3(7, 3)), (2000, rule3(3, 3)), (1500, (0, _b(4), 6))):
        vol = seed3(rng, (5, 6, d0), 8)
        want = vol.copy()
        wpop = oracle.ca3d_run(want, surv, born, nr, 4)
        for hi in (0xF8000000, 0x80000000, 0x08000000):
            for s, b in ((surv | hi, born), (surv, born | hi), (surv | hi, born | hi)):
                assert oracle.ca3d_run(chk := vol.copy(), s, b, nr, 4) == wpop and np.array_equal(chk, want)
                for engine in (BITPLANE, WAVEFRONT):
                    pop, got, _ = run3_grid(gpu, vol, ca3(gpu, s, b, nr), 4, engine)
                    assert pop == wpop and np.array_equal(got, want), (d0, hex(s), hex(b), engine)
    # a born mask of high bits only: nothing is ever born, whatever nr_states says
    vol = seed3(rng, (4, 6, 100), 3)
    want = vol.copy()
    wpop = oracle.ca3d_run(want, rule3(7, 3)[0], 0, 200, 4)
    for engine in (BITPLANE, WAVEFRONT):
        pop, got, _ = run3_grid(gpu, vol, ca3(gpu, rule3(7, 3)[0], 0x40000000, 200), 4, engine)
        assert pop == wpop and np.array_equal(got, want), engine


@gpu_mark
def test_ca2d_mask_bits_above_the_largest_count(gpu, oracle, monkeypatch):
    """Bits 9..31 of the 2D masks name counts a cell never has: they change nothing, on any engine."""
    rng = np.random.default_rng(9)
    cases = [  # born, surv, nr, decay, neigh, engines, vmax
        (0x1E0, 0x1F0, 1, 1, oracle_lib.NEIGH_M1, (BITPLANE, DIAGONAL, WAVEFRONT), 1),      # cave: its own objects
        (0x00C, 0x180, 4, 1, oracle_lib.NEIGH_M1, (BITPLANE, WAVEFRONT), 4),                # ca_test
        (0x148, 0x10C, 1, 1, oracle_lib.NEIGH_VN1, (BITPLANE, DIAGONAL, WAVEFRONT), 1),
        (0x01E, 0x0FF, 20, 0, oracle_lib.NEIGH_MV, (BITPLANE, WAVEFRONT), 20),
    ]
    for born, surv, nr, decay, neigh, engines, vmax in cases:
        arr = synth(rng, (300, 40), 0.45, vmax)
        want = oracle.ca2d_run(arr.copy(), born, surv, nr, decay, neigh, 4, side=300)
        for hi in (0xFFFFFE00, 0x200, 0x80000000):
            for b, s in ((born | hi, surv), (born, surv | hi), (born | hi, surv | hi)):
                assert np.array_equal(oracle.ca2d_run(arr.copy(), b, s, nr, decay, neigh, 4, side=300), want)
                for engine in engines:
                    monkeypatch.setenv("CLAPCA_2D_SKEW", "0")
                    got, st = run2_grid(gpu, arr, gpu.CellAutomaton("t", b, s, nr, bool(decay), neigh), 4, engine)
                    assert st["engine"] == ENGINE_NAMES[engine]
                    assert np.array_equal(got, want), (hex(b), hex(s), engine)
    # a born mask of high bits only: nothing is ever born (the row engine still sizes its planes for nr_states)
    arr = synth(rng, (200, 30), 0.45, 3)
    want = oracle.ca2d_run(arr.copy(), 0, 0x180, 20, 1, oracle_lib.NEIGH_M1, 4, side=200)
    for engine in (BITPLANE, WAVEFRONT):
        got, _ = run2_grid(gpu, arr, gpu.CellAutomaton("t", 0x1000, 0x180, 20, True, oracle_lib.NEIGH_M1), 4, engine)
        assert np.array_equal(got, want), engine


# ---- GPU: the streamed and the sharded path at the widest 8-plane variant -----------------------------------------

@gpu_mark
def test_ca3d_streamed_8_planes_4_words_per_lane(gpu, oracle, monkeypatch):
    import torch
    monkeypatch.setenv("CLAPCA_IO_CHUNK_PLANES", "2")
    rng = np.random.default_rng(3990)
    vol = seed3(rng, (7, 6, 3990), 8)
    keep_in = torch.empty(vol.shape, dtype=torch.uint8, pin_memory=True)
    keep_out = torch.empty(vol.shape, dtype=torch.uint8, pin_memory=True)
    host_in, host_out = keep_in.numpy(), keep_out.numpy()
    host_in[...] = vol
    host_out[...] = 0xEE
    want = vol.copy()
    s, b, n = oracle.ca3d_rule(7)
    wpop = oracle.ca3d_run(want, s, b, n, 5)
    grid = gpu.Grid(3990, 6, 7)
    try:
        assert grid.run3d_streamed(7, 5, host_in, host_out, max_value=255) == wpop
        st = grid.stats()
        assert st["streamed"] and st["planes"] == 8
        assert np.array_equal(host_out, want)
    finally:
        grid.close()


@gpu_mark
def test_local_ranks_8_planes_4_words_per_lane(gpu, oracle):
    """Two ranks of a volume 3000 cells wide with 255s: the team kernel at P = 8 / WPL 4, which every sharded
    ca3d_make volume of that width runs."""
    from clap_b200.slab import LocalRanks
    rng = np.random.default_rng(3000)
    full = seed3(rng, (12, 6, 3000), 8)
    want = full.copy()
    s, b, n = oracle.ca3d_rule(7)
    wpop = oracle.ca3d_run(want, s, b, n, 5)
    single = full.copy()
    assert gpu.ca3d_run(single, 7, 5, engine=BITPLANE) == wpop and np.array_equal(single, want)
    lr = LocalRanks(3000, 6, 12, 2, 5, 255, 3)
    try:
        lr.upload(full)
        assert lr.run(7, 5) == wpop
        got = lr.download()
        assert np.array_equal(got, want), int((got != want).sum())
    finally:
        lr.close()
