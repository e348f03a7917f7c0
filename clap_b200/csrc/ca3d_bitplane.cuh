/*
 * ca3d_bitplane.cuh -- bit-plane engine for ca3d_run() (core/ca3d.c:124-142).
 *
 * The reference updates the volume IN PLACE in z/y/x order, so a cell sees
 * the new generation of the 13 neighbours that precede it in the sweep and the
 * old generation of the other 13.  This engine reproduces that order exactly,
 * for all generations at once:
 *
 * Layout.  The uint8 volume is re-laid as bit planes.  For every grid row
 * (y,z) there is one "row record" of NP = 2 + P plane-rows, each RWP 32-bit
 * words (bit i of word w = cell x = 32 w + i):
 *     [ H0 | H1 | S0 ... S(P-1) ]
 * S_p is bit p of the cell state (P = bits needed for the largest value that
 * can ever occur), H1:H0 is the horizontal alive 3-sum a(x-1)+a(x)+a(x+1) of
 * the row, published so consumers never recompute it.  Padding bits of S are
 * always 0.
 *
 * Row step.  For row (y,z) of generation g every input except the new alive
 * bit of cell x-1 is known before the row starts:
 *     K = V(z-1,new)[y] + V(z+1,old)[y] + H(y-1,new) + H(y+1,old) + a_old(x+1)
 * with V = H(y-1)+H(y)+H(y+1) of one plane.  f0/f1 = new alive bit for
 * n = K / K+1 come from the rule tables, and the in-row chain is resolved by
 * the GF(2) affine scan of bitslice.cuh.  One warp updates a whole row.
 *
 * Sweeps and dataflow.  A "sweep" (z,g) = rows y = 0..H-1 of plane z at
 * generation g, run by one persistent warp.  Row y of sweep (z,g) needs rows
 * <= y+1 of (z-1,g) [new plane below], of (z+1,g-1) [old plane above] and of
 * (z,g-1) [own old state]; each sweep publishes a progress counter
 * prog[g][z] = rows completed (store after __threadfence), consumers poll it.
 * Sweeps are claimed from a ticket counter in an order that extends the
 * dependency order (key 2z+4g), so with all warps co-resident (cooperative
 * launch) the earliest unfinished sweep can always advance: no deadlock.  The
 * same in-place argument as the reference's makes single buffering safe: a row
 * is only overwritten after every reader of its previous version has passed it.
 *
 * HBM traffic depends on how far apart consecutive generations of a plane run.
 * With one generation per work item the volume streams through HBM once per
 * generation (measured, round 1: 540 GB for 2048^3 x 50).  In TILE mode (below)
 * a CTA sweeps a tile of nz planes x ng generations: generation g+1 of a row
 * runs ~6 row steps after generation g, reads it from L2 and overwrites it
 * there, so HBM sees one read and one write of the volume per ng generations.
 */
#ifndef CLAPCA_CA3D_BITPLANE_CUH
#define CLAPCA_CA3D_BITPLANE_CUH

#include "bitslice.cuh"
#include "bp3_types.h"

/* -DCLAPCA_DEBUG_HANG: the watchdog paths say what they were waiting for (debug builds only) */
#if defined(CLAPCA_DEBUG_HANG) && !defined(CLAPCA_EMU)
#include <cstdio>
#define CLAPCA_HANG_PRINT(...) printf(__VA_ARGS__)
#else
#define CLAPCA_HANG_PRINT(...) ((void)0)
#endif

namespace clapca {

struct Bp3Params {
    uint32_t *rows;         /* local row records, [(z*H + y) * NP + plane] * RWP */
    const Bp3Plane *planes; /* [Z] */
    int W, H, Z, G;         /* cells per row, rows per plane, LOCAL planes, generations */
    int RWP;                /* words per plane-row = 32 * WPL */
    int *prog;              /* [G][Z] rows completed by local sweep (z,g) */
    const int4 *order;      /* work items in claim order: (local z, g, first row, end row); tile mode: see tile_loop */
    int nsweeps;            /* number of work items */
    int flag_rows;          /* progress counters are raised every flag_rows rows (and at segment ends) */
    int prefetch_rows;      /* > 0: prefetch.L2 the own record this many rows ahead (HBM -> L2 latency) */
    int rowloop_generic;    /* != 0: every row takes the general row step, none the interior one (CLAPCA_ROWLOOP=generic:
                               A/B runs and parity checks of the two row loops) */
    unsigned *ticket;       /* next sweep to claim */
    int *err;               /* != 0: watchdog fired, everybody bails out */
    unsigned long long *diag;   /* optional: cycles [0] waiting on gpu-scope counters, [1] service warps busy, [2] in work items,
                                   [3] waiting on tile-mates */
    uint32_t surv, born;    /* rule masks (run-time rule only) */
    uint32_t bornval;       /* (nr_states - 1) & 0xff */
    long long spin_limit;   /* watchdog budget in clock ticks per wait */
    int max_ctas_per_sm;    /* host side only: > 0 caps the resident CTAs per SM of the launch */
    int max_ctas;           /* host side only: > 0 caps the CTAs of the launch (several ranks sharing one device) */
    int pub_workers;        /* > 0: every CTA = pub_workers worker warps + ONE publisher warp (see PubSlot) */
    int team;               /* > 0: tile mode -- a CTA of `team` compute warps + ONE service warp sweeps a tile (see below) */
    int halo_ldst;          /* != 0: the service warp moves halo rows with ld / st instead of TMA bulk copies */
    const uint32_t *zeros;  /* >= 2 * RWP zero words: the "row" every plane outside the volume consists of */
    /*
     * Layout items (optional, see "Layout items" below): the conversion between the reference's uint8 cells and
     * the row records runs INSIDE the sweep launch, so a volume can stream host -> device -> host through it.
     */
    int layout_items;       /* != 0: items with g == -1 pack a plane, items with g == G unpack it; prog has a row -1 */
    uint8_t *io_cells;      /* reference-layout cells of the local planes, (z*H + y)*W + x */
    const int *in_ready;    /* chunks of io_chunk planes that have landed in io_cells (raised by the copy stream) */
    int *out_done;          /* [Z] = io_epoch once the plane's final cells are back in io_cells (host-mapped memory) */
    int io_chunk;           /* planes per H2D chunk */
    int io_epoch;           /* run number written into out_done */
    unsigned long long *population;     /* += non-zero cells of every unpacked plane */
};

/*
 * Layout items.  With layout_items set the claim order holds two more item kinds around the G sweep
 * generations of every plane: "generation -1" PACKS the plane (uint8 cells -> row record, publishing
 * prog[-1][z] so that sweep (z,0) and (z-1,0) wait for it exactly as they wait for a previous generation),
 * and "generation G" UNPACKS it (row record -> uint8 cells + population) as soon as sweep (z,G-1) is done.
 * A pack item first waits until the copy engine has delivered the plane's chunk (in_ready, raised by a
 * stream-ordered 4-byte copy after each chunk's H2D copy); an unpack item stores the run's epoch into
 * out_done[z] -- host-mapped memory -- after a system-scope fence, and the host thread inside the C-ABI call
 * issues a chunk's D2H copy as soon as all of its planes carry the epoch.  Upload, all
 * generations and download of a volume then overlap inside ONE launch: the sweep follows the H2D front a
 * few planes behind and the D2H follows the last generation.  Cells whose value does not fit the P state
 * planes of the launched variant raise err = 4 (the host picks P from the caller's bound and verifies here).
 */

/*
 * Tile mode.  With one warp per sweep and gpu-scope counters, a consumer trails its producer by flag_rows + ~3 rows
 * (the counter period plus the MEMBAR.GPU / poll latency); that hop bounds how many sweeps the dependency DAG lets
 * run at once, and it keeps consecutive generations of a plane so far apart that every generation streams the
 * volume through HBM.  In tile mode a work item is a TILE of nz consecutive planes x ng consecutive generations,
 * swept by the warps of ONE CTA: compute warp w = i + nz * j takes plane z0 + i at generation g0 + j.  Its three
 * producers -- (i-1, j) the new plane below, (i+1, j-1) the old plane above, (i, j-1) its own old state -- are
 * warps of the same CTA wherever they exist, followed through shared-memory row counters raised after EVERY row
 * (CTA-scope release: MEMBAR.CTA + STS, tens of cycles): inside a tile the hop is the 3 rows the data dependency
 * and the one-row software prefetch ask for, plane to plane and generation to generation.  The row data itself
 * travels through L2 (st.cg / ld.cg by warps of the same SM, ordered by the CTA-scope release / acquire pair), so
 * generation g0+j+1 of a row finds generation g0+j in L2 and overwrites it there.
 *
 * The compute warps never execute a gpu-scope fence and never touch another GPU.  ONE extra "service" warp per CTA
 * does both for all of them: it watches the shared-memory counters and
 *   - publishes them to the gpu-scope table prog[g][z] (one fence.acq_rel.gpu per pass, cumulativity makes the rows
 *     visible before the counter) for the tile's consumers in other CTAs, and
 *   - for a z-block's edge planes (multi-GPU) copies the finished H rows into the neighbouring GPU's ghost plane
 *     with plain peer stores over NVLink, then one fence.acq_rel.sys per pass, then the peer's counter.  A ghost
 *     plane is an ordinary source for its consumer (same record stride, a counter per generation); nothing in the
 *     row loop knows about GPUs.
 * Tiles with ng > 1 depend on the NEXT tile in z of the same generation group (its plane z0+nz at generation
 * g0+j-1 feeds our last plane at g0+j) while that tile depends on ours: the two must be co-resident.  The claim
 * order (bp_plan.h, bp3_make_items_tile) keeps them a few tickets apart and bounds ng so that every rank always
 * has more CTAs than items inside that window.
 */
enum { BP3_MAX_TEAM = 24 };

/*
 * Publisher mode (one warp per sweep, no tiles).  Raising a progress counter needs a gpu-scope release, and
 * MEMBAR.GPU on a two-die B200 costs a few microseconds -- the time of two row steps.  In publisher mode the workers
 * never fence at gpu scope: after the stores of a row they bump `done` in a shared-memory mailbox (CTA-scope release:
 * cheap), and one extra warp per CTA loops { read all mailboxes; ONE fence.acq_rel.gpu; store the counters that
 * moved }.  Release cumulativity (worker stores -> CTA-scope release/acquire -> gpu-scope fence -> counter)
 * makes the rows visible before the counter, exactly like bar.sync + thread 0 fencing in a grid barrier.
 */
struct PubSlot {
    unsigned long long flag;    /* global counter of the sweep the worker is on (int *) */
    int done;                   /* rows completed (worker-written) */
    int pub;                    /* rows published (publisher-written; worker resets it between items) */
};
enum { BP3_MAX_PUB_WORKERS = 23 };

/* tile mode: the shared-memory row counters a compute warp follows / raises (nullptr: that producer is outside the tile) */
struct TileWire {
    const int *dn, *up, *own;
    int *done;
};

/* ---- rules ---------------------------------------------------------------- */

/* compile-time rule: the nine entries of cas[] (core/ca3d.c:110-122) */
template <uint32_t SURV, uint32_t BORN, uint32_t NR>
struct Rule3Const {
    static constexpr uint32_t kBornVal = (NR - 1u) & 0xffu;
    CA_MDEV uint32_t bornval(const Bp3Params &) { return kBornVal; }
    /* tables at n = K and n = K + 1 */
    CA_MDEV void eval(const Bp3Params &, const uint32_t k[5],
                            uint32_t &s0, uint32_t &s1, uint32_t &b0, uint32_t &b1)
    {
        s0 = bs_tab5<SURV>(k);
        s1 = bs_tab5<(SURV >> 1)>(k);
        if (kBornVal) {
            b0 = bs_tab5<BORN>(k);
            b1 = bs_tab5<(BORN >> 1)>(k);
        } else {
            b0 = b1 = 0u;
        }
    }
};

/* run-time rule (arbitrary masks through the C ABI) */
struct Rule3Dyn {
    CA_MDEV uint32_t bornval(const Bp3Params &p) { return p.bornval; }
    CA_MDEV void eval(const Bp3Params &p, const uint32_t k[5],
                            uint32_t &s0, uint32_t &s1, uint32_t &b0, uint32_t &b1)
    {
        s0 = bs_tab_dyn(p.surv, k, 5);
        s1 = bs_tab_dyn(p.surv >> 1, k, 5);
        if (p.bornval) {
            b0 = bs_tab_dyn(p.born, k, 5);
            b1 = bs_tab_dyn(p.born >> 1, k, 5);
        } else {
            b0 = b1 = 0u;
        }
    }
};

/* ---- vector access to a lane's WPL consecutive words ------------------------ */

template <int WPL> struct LaneVec;
template <> struct LaneVec<1> {
    CA_MDEV void ld(const uint32_t *p, uint32_t v[1]) { v[0] = dp_ld_cg(p); }
    CA_MDEV void st(uint32_t *p, const uint32_t v[1]) { dp_st_cg(p, v[0]); }
};
template <> struct LaneVec<2> {
    CA_MDEV void ld(const uint32_t *p, uint32_t v[2])
    {
        uint2 t = dp_ld_cg(reinterpret_cast<const uint2 *>(p));
        v[0] = t.x; v[1] = t.y;
    }
    CA_MDEV void st(uint32_t *p, const uint32_t v[2])
    {
        dp_st_cg(reinterpret_cast<uint2 *>(p), make_uint2(v[0], v[1]));
    }
};
template <> struct LaneVec<4> {
    CA_MDEV void ld(const uint32_t *p, uint32_t v[4])
    {
        uint4 t = dp_ld_cg(reinterpret_cast<const uint4 *>(p));
        v[0] = t.x; v[1] = t.y; v[2] = t.z; v[3] = t.w;
    }
    CA_MDEV void st(uint32_t *p, const uint32_t v[4])
    {
        dp_st_cg(reinterpret_cast<uint4 *>(p), make_uint4(v[0], v[1], v[2], v[3]));
    }
};

/* horizontal 3-sum a(x-1)+a(x)+a(x+1) of a lane-distributed row -> 2 bit planes */
template <int WPL>
CA_DEV void bp_hsum(const uint32_t a[WPL], uint32_t h0[WPL], uint32_t h1[WPL])
{
    const uint32_t prev = dp_shfl_up0(a[WPL - 1]);      /* last word of the lane on the left (0 outside the row)  */
    const uint32_t next = dp_shfl_down0(a[0]);          /* first word of the lane on the right */
#pragma unroll
    for (int j = 0; j < WPL; j++) {
        uint32_t left  = j ? a[j - 1] : prev;
        uint32_t right = (j + 1 < WPL) ? a[j + 1] : next;
        uint32_t l = dp_funnel_l(left, a[j], 1);    /* bit i = a(x-1) */
        uint32_t r = dp_funnel_r(a[j], right, 1);   /* bit i = a(x+1) */
        h0[j] = bs_xor3(l, a[j], r);
        h1[j] = bs_maj3(l, a[j], r);
    }
}

/* valid-cell mask of word w of a row of W cells */
CA_DEV uint32_t bp_valid_mask(int w, int W)
{
    int rem = W - 32 * w;
    return rem >= 32 ? ~0u : (rem <= 0 ? 0u : ((1u << rem) - 1u));
}

/* ---- the persistent sweep kernel -------------------------------------------- */

/*
 * Register budget and instruction count decide the speed of this kernel (ncu, round 1: it is issue-bound,
 * not HBM-bound), so the row loop is written for a short instruction stream:
 *   - all sliding windows live in register arrays whose slot is (row - y0) % 3 and the loop body is
 *     instantiated three times (step<0>, step<1>, step<2>): no register rotation moves;
 *   - every source is walked with a running, lane-adjusted pointer (one 64-bit add per row, plane offsets
 *     are compile-time immediates because the record stride NP * 32 * WPL is a template constant);
 *   - the producers' counters are cached as ONE number (`have` = min over the producers); the fast path of
 *     a dependency check is one compare, the slow path polls with ld.acquire in lanes 0..2 and reduces
 *     with redux.min;
 *   - there is ONE row loop: ghost planes of a neighbouring GPU look like local planes (same record stride,
 *     a progress counter per generation), so the loop carries no multi-GPU code at all.
 */
template <int P, int WPL, class Rule>
struct Sweep3 {
    static constexpr int NP = P + 2;
    static constexpr int RWP = 32 * WPL;            /* words per plane-row */
    static constexpr int RECW = NP * RWP;           /* words per row record */

    struct St {
        /* slot of row r = (r - y0 + 3) % 3 */
        uint32_t tt[3][3][WPL];                     /* T(r) = H(plane below, new)(r) + H(plane above, old)(r), rows y-1, y, y+1 */
        uint32_t hd[2][WPL], hu[2][WPL];            /* the side planes' H rows loaded last (row y+1 when a step starts) */
        uint32_t so[3][P][WPL];                     /* own state rows y, y+1, y+2 */
        uint32_t ho[2][WPL];                        /* H of own old row y+1 */
        uint32_t hn[2][WPL];                        /* H of own new row y-1 */
        uint32_t vmask[WPL];
        const uint32_t *dn, *up;                    /* lane-adjusted, at the next row to load (a plane outside the volume: the zero row) */
        int dn_step, up_step;                       /* words from row to row: RECW, or 0 on the zero row -- no null checks in the loop */
        uint32_t *rec;                              /* lane-adjusted own record of the current row */
        const uint32_t *pf;                         /* lanes < NP*WPL: one 128-byte line of the record prefetch_rows ahead
                                                       (ONE cp.async.bulk.prefetch.L2 of the record by lane 0 was measured
                                                       instead: 99.1 ms against 93.7 ms -- a one-lane branch around a
                                                       uniform-datapath instruction in a loop that is bound by issue) */
        PubSlot *slot;                              /* publisher mode: this worker's mailbox (else nullptr) */
        const int *sprod;                           /* tile mode: lanes 0..2 = shared-memory row counter of producer dn / up / own */
        int *sown;                                  /* tile mode: own shared-memory row counter */
        int have_s;                                 /* min over the rows the tile-mates have published through sprod */
        const int *flagp;                           /* the gpu-scope producer counter this lane polls (lanes 0..2) */
        bool flag_sys;                              /* ... is written by another GPU: poll at system scope */
        int have;                                   /* min over the producers' published row counts */
        int have_min;                               /* min(have_s, have): the fast path of a dependency check is ONE compare */
        int next_raise;                             /* next row count at which the own counter is raised */
    };

    /* rows < need of every producer are complete and visible.  false = watchdog fired / abort requested */
    template <bool TILE>
    CA_MDEV bool wait_rows(const Bp3Params &p, St &st, int need)
    {
        if (st.have_min >= need)
            return true;
        if (TILE && st.have_s < need && !wait_tile(p, st, need))
            return false;
        if (st.have < need && !wait_flags(p, st, need))
            return false;
        st.have_min = (TILE && st.have_s < st.have) ? st.have_s : st.have;
        return true;
    }

    /*
     * Producers outside the tile (or every producer, one warp per sweep): lanes 0..2 poll the gpu- / system-scope
     * counter of producer dn / up / own with ld.acquire, redux.min gives the row count all of them have reached.
     */
    CA_MDEV bool wait_flags(const Bp3Params &p, St &st, int need)
    {
        long long t0 = 0;
        for (unsigned spins = 0;; spins++) {
            int v = 0x7fffffff;
            if (st.flagp)
                v = st.flag_sys ? dp_ld_acquire_sys(st.flagp) : dp_ld_acquire(st.flagp);
            st.have = dp_reduce_min(v);
            if (st.have >= need)
                break;
            if (spins == 0) t0 = dp_clock();
            dp_nanosleep(32);
            if ((spins & 127u) == 127u) {
                bool bad = dp_ld_flag(p.err) != 0 || (dp_clock() - t0) > p.spin_limit;
                if (!dp_all(!bad)) {
                    CLAPCA_HANG_PRINT("wait_rows: cta %d warp %d lane %d need %d have %d have_s %d flagp %p v %d err %d\n",
                                      dp_block(), dp_warp_in_block(), dp_lane(), need, st.have, st.have_s, (const void *)st.flagp, v, dp_ld_flag(p.err));
                    if (dp_lane() == 0)
                        dp_set_error(p.err, 1);
                    return false;
                }
            }
        }
        if (t0 && p.diag && dp_lane() == 0)
            dp_atomic_add64(p.diag + 0, (unsigned long long)(dp_clock() - t0));
        dp_syncwarp();          /* the polling lanes acquired; the warp barrier extends it to every lane */
        return true;
    }

    /*
     * Tile mode: rows of the producers that are warps of this CTA.  Lanes 0..2 read the shared-memory counter of
     * producer dn / up / own (the others contribute "no limit"), redux.min gives the row count all of them have
     * reached, and every lane acquires for itself.
     */
    CA_MDEV bool wait_tile(const Bp3Params &p, St &st, int need)
    {
        long long t0 = 0;
        for (unsigned spins = 0;; spins++) {
            const int v = st.sprod ? dp_ld_volatile(st.sprod) : 0x7fffffff;
            const int m = dp_reduce_min(v);
            if (m >= need) {
                st.have_s = m;
                break;
            }
            if (spins == 0) t0 = dp_clock();
            if ((spins & 1023u) == 1023u) {
                bool bad = dp_ld_flag(p.err) != 0 || (dp_clock() - t0) > p.spin_limit;
                if (!dp_all(!bad)) {
                    CLAPCA_HANG_PRINT("wait_tile: cta %d warp %d lane %d need %d m %d v %d err %d\n",
                                      dp_block(), dp_warp_in_block(), dp_lane(), need, m, v, dp_ld_flag(p.err));
                    if (dp_lane() == 0)
                        dp_set_error(p.err, 3);
                    return false;
                }
            }
            dp_team_pause();
        }
        if (t0 && p.diag && dp_lane() == 0)
            dp_atomic_add64(p.diag + 3, (unsigned long long)(dp_clock() - t0));
        dp_fence_cta();
        return true;
    }

    CA_MDEV void zero2(uint32_t h[2][WPL])
    {
#pragma unroll
        for (int j = 0; j < WPL; j++) h[0][j] = h[1][j] = 0u;
    }

    /* next H row of the plane below / above into h; advances the running pointer */
    CA_MDEV void load_side(const uint32_t *&src, int step, uint32_t h[2][WPL])
    {
        LaneVec<WPL>::ld(src, h[0]);
        LaneVec<WPL>::ld(src + RWP, h[1]);
        src += step;
    }

    /* own record at st.rec + D rows: state planes, and optionally the H planes */
    template <int D>
    CA_MDEV void load_own_s(const St &st, uint32_t s[P][WPL])
    {
#pragma unroll
        for (int q = 0; q < P; q++)
            LaneVec<WPL>::ld(st.rec + D * RECW + (2 + q) * RWP, s[q]);
    }
    template <int D>
    CA_MDEV void load_own_h(const St &st, uint32_t h[2][WPL])
    {
        LaneVec<WPL>::ld(st.rec + D * RECW, h[0]);
        LaneVec<WPL>::ld(st.rec + D * RECW + RWP, h[1]);
    }
    /* T = Hdn + Hup of the side rows loaded last */
    CA_MDEV void pair_sum(const St &st, uint32_t t[3][WPL])
    {
#pragma unroll
        for (int j = 0; j < WPL; j++) {
            uint32_t d_[2] = { st.hd[0][j], st.hd[1][j] }, u_[2] = { st.hu[0][j], st.hu[1][j] }, t_[3];
            bs_add2x2(d_, u_, t_);
            t[0][j] = t_[0]; t[1][j] = t_[1]; t[2][j] = t_[2];
        }
    }
    CA_MDEV void zero_s(uint32_t s[P][WPL])
    {
#pragma unroll
        for (int q = 0; q < P; q++)
#pragma unroll
            for (int j = 0; j < WPL; j++) s[q][j] = 0u;
    }

    /*
     * One row step.  M = (y - y0) % 3 selects the register slots: rows y-1 / y / y+1 of the side planes
     * sit in slots (M+2)%3 / M / (M+1)%3, own state rows y / y+1 in slots M / (M+1)%3; row y+2 is
     * prefetched into slot (M+2)%3 once row y-1 has been consumed.
     * TILE: tile mode (shared-memory row counter after every row) or one warp per sweep -- fixed per call site.
     * INT: an interior row, y + 2 <= y1, y + 2 < H and y + prefetch_rows < H (run_rows): no edge test, no zero arm.
     */
    template <int M, bool TILE, bool INT>
    CA_MDEV bool step(const Bp3Params &p, St &st, int y, int y1, int *myprog)
    {
        constexpr int A = (M + 2) % 3, B = M, C = (M + 1) % 3;
        const int lane = dp_lane();
        const int H = p.H;
        const uint32_t bornval = Rule::bornval(p);
        uint32_t k[WPL][5], ao[WPL], ge2[WPL];

        /* ---- neighbour count K (everything but the in-row predecessor) ---- */
#pragma unroll
        for (int j = 0; j < WPL; j++) {
            uint32_t a = st.so[B][0][j], hi = 0u;
#pragma unroll
            for (int q = 1; q < P; q++) hi |= st.so[B][q][j];
            ao[j] = a | hi;
            ge2[j] = hi;
        }
        const uint32_t nxt = dp_shfl_down0(ao[0]);
#pragma unroll
        for (int j = 0; j < WPL; j++) {
            /* row y+1 of the side planes arrived during the previous step: its pair sum takes the slot row y-2 left */
            uint32_t d_[2] = { st.hd[0][j], st.hd[1][j] }, u_[2] = { st.hu[0][j], st.hu[1][j] }, t_[3];
            bs_add2x2(d_, u_, t_);
            st.tt[C][0][j] = t_[0]; st.tt[C][1][j] = t_[1]; st.tt[C][2][j] = t_[2];
            uint32_t a_[3] = { st.tt[A][0][j], st.tt[A][1][j], st.tt[A][2][j] };
            uint32_t b_[3] = { st.tt[B][0][j], st.tt[B][1][j], st.tt[B][2][j] };
            uint32_t n_[2] = { st.hn[0][j], st.hn[1][j] }, o_[2] = { st.ho[0][j], st.ho[1][j] };
            uint32_t right = (j + 1 < WPL) ? ao[j + 1] : nxt;
            uint32_t r = dp_funnel_r(ao[j], right, 1);      /* old alive bit of x+1 */
            bs_count3d_t(a_, b_, t_, n_, o_, r, k[j]);
        }

        /* ---- prefetch row y+2 while the rule / scan / update below run ---- */
        if (st.pf) {                /* a lane test, not a branch: the prefetch and the add are predicated */
            if (INT || y + p.prefetch_rows < H)
                dp_prefetch_l2(st.pf);
            st.pf += RECW;
        }
        if (y + 2 <= y1) {          /* row y1 is still needed (as "row y+1" of the last step), y1+1 is not */
            /*
             * Always true on an interior row, where it is the one test left: without this branch around the wait
             * and the loads ptxas schedules the interior step with ~20 more instructions per row (it
             * rematerialises the valid-cell mask and the counter address; tools/sass_hist.py).
             */
            if (INT || y + 2 < H) {
                if (!wait_rows<TILE>(p, st, (INT || y + 3 < H) ? y + 3 : H))
                    return false;
                load_own_h<2>(st, st.ho);
                load_own_s<2>(st, st.so[A]);
                load_side(st.dn, st.dn_step, st.hd);
                load_side(st.up, st.up_step, st.hu);
            } else {
                zero2(st.ho); zero2(st.hd); zero2(st.hu);
                zero_s(st.so[A]);
            }
        }

        /* ---- rule tables, in-row scan ---- */
        uint32_t s0[WPL], s1[WPL], E[WPL], Cc[WPL];
        uint32_t el = 0u, cl = 0u;          /* lane map in bit 31 (el: the chain breaks inside the lane): identity so far */
#pragma unroll
        for (int j = 0; j < WPL; j++) {
            uint32_t b0, b1;
            Rule::eval(p, k[j], s0[j], s1[j], b0, b1);
            /* new alive bit if the predecessor's new alive bit is 0 / 1 (padding cells are dead: only births need the mask) */
            const uint32_t nv = ~ao[j] & st.vmask[j];
            const uint32_t f0 = (ao[j] & (s0[j] | ge2[j])) | (b0 & nv);
            const uint32_t f1 = (ao[j] & (s1[j] | ge2[j])) | (b1 & nv);
            E[j] = ~(f0 ^ f1);
            Cc[j] = f0;
            bs_scan_word_e_lo(E[j], Cc[j]);
        }
        {
            uint32_t open8 = 0u;            /* runs of 8 dependent cells: the scan needs its last two steps */
#pragma unroll
            for (int j = 0; j < WPL; j++) open8 |= ~E[j];
            if (dp_any((open8 & 0xffffff00u) != 0u)) {
#pragma unroll
                for (int j = 0; j < WPL; j++) bs_scan_word_e_hi(E[j], Cc[j]);
            }
        }
#pragma unroll
        for (int j = 0; j < WPL; j++) {
            /* compose into the lane map: carry-out = c ^ (d & carry-in), carried in bit 31 of whole words */
            cl = Cc[j] ^ (~E[j] & cl);
            el |= E[j];
        }
        uint32_t cin = bs_scan_warp_e((int)el < 0, (int)cl < 0);

        /* ---- apply: new alive bits, state planes ---- */
        uint32_t an[WPL];
#pragma unroll
        for (int j = 0; j < WPL; j++) {
            uint32_t cm = 0u - cin;
            an[j] = Cc[j] ^ (~E[j] & cm);
            uint32_t pred = an[j] * 2u + cin;                /* new alive bit of x-1 */
            cin = an[j] >> 31;
            uint32_t sv = bs_mux(pred, s1[j], s0[j]);
            uint32_t dec = ao[j] & ~sv;                      /* alive, not surviving: state - 1 */
            uint32_t brn = an[j] & ~ao[j];                   /* dead, born: state = nr_states - 1 */
            uint32_t borrow = dec;
#pragma unroll
            for (int q = 0; q < P; q++) {
                uint32_t t = st.so[B][q][j];
                st.so[B][q][j] = t ^ borrow;
                borrow &= ~t;
                if ((bornval >> q) & 1u) st.so[B][q][j] |= brn;
            }
        }
        bp_hsum<WPL>(an, st.hn[0], st.hn[1]);

        /* ---- publish row y ---- */
        LaneVec<WPL>::st(st.rec, st.hn[0]);
        LaneVec<WPL>::st(st.rec + RWP, st.hn[1]);
#pragma unroll
        for (int q = 0; q < P; q++)
            LaneVec<WPL>::st(st.rec + (2 + q) * RWP, st.so[B][q]);
        st.rec += RECW;
        if (TILE) {
            /*
             * Tile mode: warp barrier (orders every lane's row stores before lane 0), CTA-scope release by lane 0,
             * row counter in shared memory -- after EVERY row.  The service warp carries it to gpu / system scope.
             * Lane 0's fence and store are predicated, not branched around: the warp never diverges, so the next
             * step's shuffles and votes need no convergence check.
             */
            dp_syncwarp();
            dp_release_cta_if(lane == 0, st.sown, y + 1);
            return true;
        }
        /*
         * One warp per sweep: warp barrier, then ONE release store of the counter (MEMBAR.GPU + store), or the
         * publisher's mailbox.  Raised every flag_rows rows, and after the item's last row (never an interior row).
         */
        const bool at_mark = (y + 1 == st.next_raise);
        if (at_mark)
            st.next_raise += p.flag_rows;
        if (at_mark || (!INT && y + 1 == y1)) {
            dp_syncwarp();
            if (lane == 0) {
                if (st.slot) {
                    dp_fence_cta();
                    dp_st_volatile(&st.slot->done, y + 1);
                } else {
                    dp_st_release(myprog, y + 1);
                }
            }
        }
        return true;
    }

    /* one work item: rows [y0, y1) of plane z at generation g; TILE: tw is the tile's wiring, else nullptr.  false = aborted */
    template <bool TILE>
    CA_MDEV bool run_rows(const Bp3Params &p, int z, int g, int y0, int y1, PubSlot *slot, const TileWire *tw)
    {
        const int lane = dp_lane();
        const int H = p.H, Z = p.Z;
        const Bp3Plane pl = p.planes[z];
        int *myprog = p.prog + (size_t)g * Z + z;
        St st;

        /* ---- sources ---- */
        const int first = y0 > 0 ? y0 - 1 : 0;      /* first row loaded from the side planes */
        st.dn = pl.dn_rows ? pl.dn_rows + (size_t)first * RECW + lane * WPL : p.zeros + lane * WPL;
        st.up = pl.up_rows ? pl.up_rows + (size_t)first * RECW + lane * WPL : p.zeros + lane * WPL;
        st.dn_step = pl.dn_rows ? RECW : 0;
        st.up_step = pl.up_rows ? RECW : 0;
        st.rec = p.rows + ((size_t)z * H + y0) * RECW + lane * WPL;
        st.pf = (p.prefetch_rows > 0 && lane < NP * WPL)
              ? p.rows + ((size_t)z * H + y0 + p.prefetch_rows) * RECW + lane * 32 : nullptr;

        /* ---- producers: tile-mates through shared memory, everybody else through gpu-scope counters ---- */
        {
            const int *sdn = tw ? tw->dn : nullptr, *sup = tw ? tw->up : nullptr, *sow = tw ? tw->own : nullptr;
            const int *fdn = (pl.dn_rows && !sdn) ? pl.dn_flag + (size_t)g * pl.dn_gstride : nullptr;
            /* layout items: "generation -1" is the pack item of a plane, counted in row -1 of the table */
            const bool prev = g > 0 || p.layout_items;
            const int *fup = (prev && pl.up_rows && !sup) ? pl.up_flag + ((long long)g - 1) * (long long)pl.up_gstride : nullptr;
            const int *fown = (prev && !sow) ? p.prog + ((long long)g - 1) * Z + z : nullptr;
            st.flagp = lane == 0 ? fdn : (lane == 1 ? fup : (lane == 2 ? fown : nullptr));
            st.flag_sys = (lane == 0 && (pl.ghost_mask & 1u)) || (lane == 1 && (pl.ghost_mask & 2u));
            st.have = (fdn || fup || fown) ? 0 : 0x7fffffff;
            st.sprod = lane == 0 ? sdn : (lane == 1 ? sup : (lane == 2 ? sow : nullptr));
            st.have_s = (sdn || sup || sow) ? 0 : 0x7fffffff;
        }
        st.have_min = st.have_s < st.have ? st.have_s : st.have;
        st.sown = TILE ? tw->done : nullptr;
        st.next_raise = (y0 / p.flag_rows + 1) * p.flag_rows;
        /* diagnostics go straight to the counters (the item's time as - start + end): no clock lives in a register
           across the row loop, whose register budget is exhausted */
        if (p.diag && lane == 0)
            dp_atomic_add64(p.diag + 2, 0ull - (unsigned long long)dp_clock());
#pragma unroll
        for (int j = 0; j < WPL; j++) st.vmask[j] = bp_valid_mask(lane * WPL + j, p.W);

        /* rows < y0 of this sweep belong to earlier segments (skewed-segment order only) */
        if (y0 > 0) {
            long long t0 = dp_clock();
            for (unsigned spins = 1;; spins++) {
                int v = dp_reduce_min(lane == 0 ? dp_ld_acquire(myprog) : 0x7fffffff);
                if (v >= y0)
                    break;
                dp_nanosleep(32);
                if ((spins & 127u) == 0u) {
                    bool bad = dp_ld_flag(p.err) != 0 || (dp_clock() - t0) > p.spin_limit;
                    if (!dp_all(!bad)) {
                        if (lane == 0)
                            dp_set_error(p.err, 1);
                        return false;
                    }
                }
            }
            dp_syncwarp();
        }
        /*
         * Publisher mode: hand the mailbox over to this sweep.  The previous item ended with pub == done, so
         * the publisher is idle on this slot; it reads pub, then done, then flag -- written here in the
         * opposite order -- so it can never pair an old row count with the new counter address.
         */
        st.slot = slot;
        if (slot && lane == 0) {
            dp_st_volatile64(&slot->flag, (unsigned long long)(size_t)myprog);
            dp_fence_cta();
            dp_st_volatile(&slot->done, y0);
            dp_fence_cta();
            dp_st_volatile(&slot->pub, y0);
        }
        if (!wait_rows<TILE>(p, st, y0 + 2 < H ? y0 + 2 : H))
            return false;

        /* ---- fill the windows: pair sums of rows y0-1 (slot 2) and y0 (slot 0); row y0+1 waits in hd / hu ---- */
        if (y0 > 0) {
            load_side(st.dn, st.dn_step, st.hd);
            load_side(st.up, st.up_step, st.hu);
            pair_sum(st, st.tt[2]);
            load_own_h<-1>(st, st.hn);              /* row y0-1 of this plane is already generation g */
        } else {
#pragma unroll
            for (int j = 0; j < WPL; j++) st.tt[2][0][j] = st.tt[2][1][j] = st.tt[2][2][j] = 0u;
            zero2(st.hn);
        }
        load_side(st.dn, st.dn_step, st.hd);
        load_side(st.up, st.up_step, st.hu);
        pair_sum(st, st.tt[0]);
        load_own_s<0>(st, st.so[0]);
        if (y0 + 1 < H) {
            load_side(st.dn, st.dn_step, st.hd);
            load_side(st.up, st.up_step, st.hu);
            load_own_h<1>(st, st.ho);
            load_own_s<1>(st, st.so[1]);
        } else {
            zero2(st.hd); zero2(st.hu); zero2(st.ho);
            zero_s(st.so[1]);
        }
        zero_s(st.so[2]);
#pragma unroll
        for (int j = 0; j < WPL; j++) st.tt[1][0][j] = st.tt[1][1][j] = st.tt[1][2][j] = 0u;

        /*
         * Rows [y0, yi) are interior: every edge test of the general step has a result known here, so they take
         * the step without them.  The rest (at most two of the interior rows, then the last rows of the item or
         * of the plane) take the general step; the slots continue at M = 0 because yi - y0 rows is rounded to 3.
         */
        int yi = y1 - 1;                                /* y + 2 <= y1 */
        if (yi > H - 2) yi = H - 2;                     /* y + 2 < H: row y + 2 exists, the wait is for y + 3 <= H rows */
        if (yi > H - p.prefetch_rows) yi = H - p.prefetch_rows;     /* the prefetched line is inside the plane */
        if (p.rowloop_generic) yi = y0;
        int y = y0;
        for (; y + 3 <= yi; y += 3) {
            if (!step<0, TILE, true>(p, st, y, y1, myprog)) return false;
            if (!step<1, TILE, true>(p, st, y + 1, y1, myprog)) return false;
            if (!step<2, TILE, true>(p, st, y + 2, y1, myprog)) return false;
        }
        for (; y < y1; y += 3) {
            if (!step<0, TILE, false>(p, st, y, y1, myprog)) return false;
            if (y + 1 < y1 && !step<1, TILE, false>(p, st, y + 1, y1, myprog)) return false;
            if (y + 2 < y1 && !step<2, TILE, false>(p, st, y + 2, y1, myprog)) return false;
        }
        /* publisher mode: the mailbox is reused by the next item only once the last rows are out */
        if (slot) {
            if (lane == 0)
                while (dp_ld_volatile(&slot->pub) < y1)
                    dp_nanosleep(20);
            dp_syncwarp();
        }
        if (p.diag && lane == 0)
            dp_atomic_add64(p.diag + 2, (unsigned long long)dp_clock());
        return true;
    }

    /* ---- layout items: one warp converts one plane -------------------------------------------------------- */

    /* poll *flag (written by the copy stream or by other SMs) until it reaches `need`; false = watchdog / abort */
    CA_MDEV bool wait_word(const Bp3Params &p, const int *flag, int need, bool sys, int code)
    {
        const int lane = dp_lane();
        long long t0 = 0;
        for (unsigned spins = 0;; spins++) {
            int v = 0x7fffffff;
            if (lane == 0)
                v = sys ? dp_ld_flag_sys(flag) : dp_ld_acquire(flag);
            if (dp_reduce_min(v) >= need)
                break;
            if (spins == 0) t0 = dp_clock();
            dp_nanosleep(200);
            if ((spins & 127u) == 127u) {
                /* the copy engine may take its time: 16 x the budget of a dataflow wait */
                bool bad = dp_ld_flag(p.err) != 0 || (dp_clock() - t0) > 16 * p.spin_limit;
                if (!dp_all(!bad)) {
                    if (lane == 0)
                        dp_set_error(p.err, code);
                    return false;
                }
            }
        }
        if (sys)
            dp_fence_sys();
        dp_syncwarp();
        return true;
    }

    /* uint8 cells of plane z -> row records; publishes prog[-1][z] */
    CA_MDEV bool pack_plane(const Bp3Params &p, int z)
    {
        const int lane = dp_lane();
        const int H = p.H, W = p.W;
        if (p.in_ready && !wait_word(p, p.in_ready, z / p.io_chunk + 1, true, 5))
            return false;
        int *myprog = p.prog - p.Z + z;
        const uint8_t *src = p.io_cells + (size_t)z * H * W;
        uint32_t *rec = p.rows + (size_t)z * H * RECW + lane * WPL;
        const bool vec = (W & 15) == 0;
        constexpr uint32_t kOver = (P >= 8) ? 0u : (((0xffu << P) & 0xffu) * 0x01010101u);
        uint32_t over = 0u;
        for (int y = 0; y < H; y++, src += W, rec += RECW) {
            uint32_t s[P][WPL], a[WPL], h0[WPL], h1[WPL];
#pragma unroll
            for (int j = 0; j < WPL; j++) {
                const int x0 = 32 * (lane * WPL + j);
#pragma unroll
                for (int q = 0; q < P; q++) s[q][j] = 0u;
                if (vec && x0 + 32 <= W) {
                    const uint4 lo = dp_ld_cg(reinterpret_cast<const uint4 *>(src + x0));
                    const uint4 hi = dp_ld_cg(reinterpret_cast<const uint4 *>(src + x0 + 16));
                    const uint32_t r[8] = { lo.x, lo.y, lo.z, lo.w, hi.x, hi.y, hi.z, hi.w };
#pragma unroll
                    for (int k = 0; k < 8; k++) {
                        over |= r[k];
#pragma unroll
                        for (int q = 0; q < P; q++)
                            s[q][j] |= ((((r[k] >> q) & 0x01010101u) * 0x01020408u) >> 24) << (4 * k);
                    }
                } else {
                    for (int i = 0; i < 32 && x0 + i < W; i++) {
                        const uint32_t v = dp_ld_cg(src + x0 + i);
                        over |= v;
#pragma unroll
                        for (int q = 0; q < P; q++) s[q][j] |= ((v >> q) & 1u) << i;
                    }
                }
                a[j] = 0u;
#pragma unroll
                for (int q = 0; q < P; q++) a[j] |= s[q][j];
            }
            bp_hsum<WPL>(a, h0, h1);
            LaneVec<WPL>::st(rec, h0);
            LaneVec<WPL>::st(rec + RWP, h1);
#pragma unroll
            for (int q = 0; q < P; q++)
                LaneVec<WPL>::st(rec + (2 + q) * RWP, s[q]);
            if (((y + 1) & 31) == 0 || y + 1 == H) {
                dp_syncwarp();
                if (lane == 0)
                    dp_st_release(myprog, y + 1);
            }
        }
        if (!dp_all((over & kOver) == 0u)) {
            if (lane == 0)
                dp_set_error(p.err, 4);
            return false;
        }
        return true;
    }

    /* row records of plane z after the last generation -> uint8 cells, population, out_done[z] */
    CA_MDEV bool unpack_plane(const Bp3Params &p, int z)
    {
        const int lane = dp_lane();
        const int H = p.H, W = p.W;
        if (p.G > 0 && !wait_word(p, p.prog + (size_t)(p.G - 1) * p.Z + z, H, false, 6))
            return false;
        if (p.G <= 0 && !wait_word(p, p.prog - p.Z + z, H, false, 6))
            return false;
        uint8_t *dst = p.io_cells + (size_t)z * H * W;
        const uint32_t *rec = p.rows + (size_t)z * H * RECW + lane * WPL;
        const bool vec = (W & 15) == 0;
        unsigned pop = 0u;
        for (int y = 0; y < H; y++, dst += W, rec += RECW) {
            uint32_t s[P][WPL];
#pragma unroll
            for (int q = 0; q < P; q++)
                LaneVec<WPL>::ld(rec + (2 + q) * RWP, s[q]);
#pragma unroll
            for (int j = 0; j < WPL; j++) {
                const int x0 = 32 * (lane * WPL + j);
                uint32_t alive = 0u;
#pragma unroll
                for (int q = 0; q < P; q++) alive |= s[q][j];
                pop += (unsigned)dp_popc(alive);
                if (vec && x0 + 32 <= W) {
                    uint32_t r[8];
#pragma unroll
                    for (int k = 0; k < 8; k++) {
                        uint32_t v = 0u;
#pragma unroll
                        for (int q = 0; q < P; q++)
                            v |= ((((s[q][j] >> (4 * k)) & 0xfu) * 0x00204081u) & 0x01010101u) << q;
                        r[k] = v;
                    }
                    dp_st_cg(reinterpret_cast<uint4 *>(dst + x0), make_uint4(r[0], r[1], r[2], r[3]));
                    dp_st_cg(reinterpret_cast<uint4 *>(dst + x0 + 16), make_uint4(r[4], r[5], r[6], r[7]));
                } else {
                    for (int i = 0; i < 32 && x0 + i < W; i++) {
                        uint32_t v = 0u;
#pragma unroll
                        for (int q = 0; q < P; q++) v |= ((s[q][j] >> i) & 1u) << q;
                        dst[x0 + i] = (uint8_t)v;
                    }
                }
            }
        }
        for (int o = 16; o; o >>= 1)
            pop += dp_shfl_down(pop, o);
        dp_syncwarp();
        if (lane == 0) {
            if (p.population)
                dp_atomic_add64(p.population, (unsigned long long)pop);
            if (p.out_done) {
                dp_fence_sys();             /* the cells must be visible to the copy engine before the word moves */
                dp_st_flag_sys(p.out_done + z, p.io_epoch);
            }
        }
        return true;
    }

    /* dispatch on the item kind: g == -1 pack, g == G unpack (layout items), else a sweep segment */
    CA_MDEV bool run_item(const Bp3Params &p, int z, int g, int y0, int y1, PubSlot *slot)
    {
        if (p.layout_items) {
            if (g < 0)
                return pack_plane(p, z);
            if (g >= p.G)
                return unpack_plane(p, z);
        }
        return run_rows<false>(p, z, g, y0, y1, slot, nullptr);
    }

    /* the worker loop: claim items in dependency order until the list is exhausted */
    CA_MDEV void work_loop(const Bp3Params &p, PubSlot *slot)
    {
        const int lane = dp_lane();
        for (;;) {
            unsigned t = 0;
            if (lane == 0) {
                t = dp_atomic_inc(p.ticket);
                if (dp_ld_flag(p.err) != 0)
                    t = 0xffffffffu;
            }
            t = dp_shfl(t, 0);
            if (t >= (unsigned)p.nsweeps)
                break;
            int4 it = p.order[t];
            if (!run_item(p, it.x, it.y, it.z, it.w, slot))
                break;
        }
    }

    /* publisher warp: lane i serves the mailbox of worker warp i; one gpu-scope fence per pass for all of them */
    CA_MDEV void publish_loop(PubSlot *slots, int *nexit, int nw)
    {
        const int lane = dp_lane();
        PubSlot *my = slots + (lane < nw ? lane : 0);
        for (;;) {
            int pb = 0, d = 0;
            if (lane < nw) {
                pb = dp_ld_volatile(&my->pub);
                dp_fence_cta();
                d = dp_ld_volatile(&my->done);
            }
            const bool need = d > pb;
            if (dp_any(need)) {
                unsigned long long f = 0;
                if (need) {
                    dp_fence_cta();
                    f = dp_ld_volatile64(&my->flag);
                }
                dp_fence_release();                     /* fence.acq_rel.gpu: the ONE expensive instruction */
                if (need) {
                    dp_st_flag((int *)(size_t)f, d);
                    dp_st_volatile(&my->pub, d);
                }
            } else {
                if (dp_all(dp_ld_volatile(nexit) >= nw))        /* warp-uniform: the lanes read at different times */
                    break;
                dp_nanosleep(40);
            }
        }
    }

    /* shared memory of a tile's CTA */
    struct alignas(16) TileShared {
        uint32_t stage[16][2 * RWP];        /* staging slots of the halo rows on their way to a peer (H0 | H1 of one row each) */
        unsigned long long bar;             /* mbarrier: bytes of the bulk loads into the slots */
        int cnt[BP3_MAX_TEAM + 1];          /* row counters of the compute warps, then the claimed ticket */
    };

    /*
     * The same copy by the TMA engine: 1-D bulk copies local row record -> staging slot (completion counted on an
     * mbarrier) and staging slot -> peer ghost plane over NVLink (bulk group), 16 rows per batch, issued by ONE lane:
     * the service warp spends a handful of instructions per row and holds no row data in registers.  `phase` is the
     * mbarrier phase parity, carried by the caller.  The copies are complete (bulk_done) before the peer's counter moves.
     */
    CA_MDEV void bulk_copy_h_rows(TileShared &ts, uint32_t *dst, const uint32_t *src, int r0, int r1, uint32_t &phase,
                                  const Bp3Params &p)
    {
        constexpr uint32_t ROWB = 2 * RWP * 4;
        const int lane = dp_lane();
        for (int r = r0; r < r1; r += 16) {
            const int n = r1 - r < 16 ? r1 - r : 16;
            if (lane == 0) {
                dp_bulk_wait_read();                /* the previous batch has left the slots */
                dp_mbar_expect_tx(&ts.bar, (uint32_t)n * ROWB);
                for (int i = 0; i < n; i++)
                    dp_bulk_g2s(ts.stage[i], src + (size_t)(r + i) * RECW, ROWB, &ts.bar);
                long long t0 = 0;
                for (unsigned spins = 1; !dp_mbar_try_wait(&ts.bar, phase); spins++) {
                    if (spins == 1) t0 = dp_clock();
                    if ((spins & 4095u) == 0u && (dp_ld_flag(p.err) != 0 || (dp_clock() - t0) > p.spin_limit)) {
                        dp_set_error(p.err, 9);
                        break;
                    }
                }
                for (int i = 0; i < n; i++)
                    dp_bulk_s2g(dst + (size_t)(r + i) * RECW, ts.stage[i], ROWB);
                dp_bulk_commit();
            }
            phase ^= 1u;
        }
        dp_syncwarp();
    }

    /*
     * H rows [r0, r1) of one plane from the local row records to a peer's ghost plane (both with the record stride):
     * H0 | H1 of a row are 2 * RWP contiguous words = 32 * WPL uint2, so the warp moves a row with WPL coalesced 8-byte
     * accesses per lane.  The loads of a batch of rows are ALL issued before the first store: a row-by-row copy pays
     * one L2 round trip per row (~0.5 us) and cannot follow eight streams that each finish a row every ~1.3 us
     * (measured on 2 x B200: 4 x 4 tiles with 16-plane blocks ran 2x slower than one GPU until the copies were batched).
     */
    CA_MDEV void copy_h_rows(uint32_t *dst, const uint32_t *src, int r0, int r1)
    {
        constexpr int BATCH = 16 / WPL;
        constexpr int RS = RECW / 2;                /* record stride in uint2 */
        const int lane = dp_lane();
        const uint2 *a = reinterpret_cast<const uint2 *>(src + (size_t)r0 * RECW) + lane;
        uint2 *b = reinterpret_cast<uint2 *>(dst + (size_t)r0 * RECW) + lane;
        int n = r1 - r0;
        for (; n >= BATCH; n -= BATCH, a += BATCH * RS, b += BATCH * RS) {
            uint2 v[BATCH][WPL];
#pragma unroll
            for (int i = 0; i < BATCH; i++)
#pragma unroll
                for (int k = 0; k < WPL; k++)
                    v[i][k] = dp_ld_cg(a + i * RS + 32 * k);
#pragma unroll
            for (int i = 0; i < BATCH; i++)
#pragma unroll
                for (int k = 0; k < WPL; k++)
                    dp_st_cg(b + i * RS + 32 * k, v[i][k]);
        }
        for (; n > 0; n--, a += RS, b += RS) {      /* the tail of a pass, row by row */
            uint2 v[WPL];
#pragma unroll
            for (int k = 0; k < WPL; k++)
                v[k] = dp_ld_cg(a + 32 * k);
#pragma unroll
            for (int k = 0; k < WPL; k++)
                dp_st_cg(b + 32 * k, v[k]);
        }
    }

    /*
     * Tile mode, the service warp of one tile (nz planes from local plane l0, ng generations from g0).
     * Lane w < nz * ng serves compute warp w: it carries the warp's shared-memory row counter to prog[g][z].
     * Lanes 0 .. 2 ng - 1 additionally own one push stream each: lane j < ng the H rows of warp (0, j) for the ghost
     * plane ABOVE the previous z-block (push_dn), lane ng + j those of warp (nz-1, j) for the ghost plane BELOW the
     * next z-block (push_up) -- where the tile touches a z-block edge whose other side is another GPU.  Every pass:
     * read the counters, fence.acq_rel.gpu, store the gpu-scope counters that moved; copy the new rows of every
     * stream (the whole warp copies one H row = 2 * RWP words with coalesced 8-byte peer stores), fence.acq_rel.sys,
     * store the peers' counters.  A row is copied out of the local record before anybody can overwrite it: generation
     * g+1 of an edge row needs the neighbouring GPU's generation-g (or g+1) rows, which need this push (see DESIGN.md).
     */
    CA_MDEV void service_loop(const Bp3Params &p, int l0, int g0, int nz, int ng, TileShared &ts, uint32_t &phase)
    {
        const int lane = dp_lane();
        const int H = p.H, Z = p.Z;
        const int n = nz * ng;
        int *myflag = lane < n ? p.prog + (size_t)(g0 + lane / nz) * Z + (l0 + lane % nz) : nullptr;
        int pub = 0, pushed = 0, pw = 0;
        const uint32_t *psrc = nullptr;
        uint32_t *pdst = nullptr;
        int *pflag = nullptr;
        if (lane < 2 * ng) {
            const bool up = lane >= ng;
            const int j = up ? lane - ng : lane;
            const int zl = up ? l0 + nz - 1 : l0;
            const Bp3Plane pl = p.planes[zl];
            pdst = up ? pl.push_up_rows : pl.push_dn_rows;
            pflag = (up ? pl.push_up_flag : pl.push_dn_flag);
            if (pdst) {
                pflag += g0 + j;
                psrc = p.rows + (size_t)zl * H * RECW;
                pw = (up ? nz - 1 : 0) + nz * j;
            }
        }
        const bool streams = dp_any(pdst != nullptr);
        const int *done = ts.cnt;
        long long t_idle = dp_clock(), t_busy = 0;
        unsigned idle_since = 0;
        for (unsigned spins = 0;; spins++) {
            const long long t_pass = p.diag ? dp_clock() : 0;
            const int d = lane < n ? dp_ld_volatile(done + lane) : H;
            dp_fence_cta();
            bool any = false;
            const bool moved = lane < n && d > pub;
            if (dp_any(moved)) {
                dp_fence_release();                     /* fence.acq_rel.gpu: rows before counters */
                if (moved) {
                    dp_st_flag(myflag, d);
                    pub = d;
                }
                any = true;
            }
            if (streams) {
                const int avail = (int)dp_shfl((uint32_t)d, pw);
                const bool pm = pdst && avail > pushed;
                const uint32_t mask = dp_ballot(pm);
                if (mask) {
                    if (!p.halo_ldst)
                        dp_fence_proxy_async();         /* the rows were written through the generic proxy; the bulk loads read them through the async proxy */
                    for (uint32_t m = mask; m; m &= m - 1u) {
                        const int s = dp_ffs(m) - 1;
                        const uint32_t *src = (const uint32_t *)(size_t)dp_shfl64((unsigned long long)(size_t)psrc, s);
                        uint32_t *dst = (uint32_t *)(size_t)dp_shfl64((unsigned long long)(size_t)pdst, s);
                        const int r0 = (int)dp_shfl((uint32_t)pushed, s), r1 = (int)dp_shfl((uint32_t)avail, s);
                        if (p.halo_ldst)
                            copy_h_rows(dst, src, r0, r1);
                        else
                            bulk_copy_h_rows(ts, dst, src, r0, r1, phase, p);
                    }
                    if (!p.halo_ldst && lane == 0) {
                        dp_bulk_wait();                 /* every bulk store of this pass is complete ... */
                        dp_fence_proxy_async();         /* ... and ordered before the generic-proxy counter store */
                    }
                    dp_fence_sys();                     /* fence.acq_rel.sys: peer rows before the peer's counter */
                    if (pm) {
                        dp_st_flag_sys(pflag, avail);
                        pushed = avail;
                    }
                    any = true;
                }
            }
            const bool fin = (lane >= n || pub >= H) && (!pdst || pushed >= H);
            if (dp_all(fin))
                break;
            if (any) {
                if (p.diag) t_busy += dp_clock() - t_pass;
                idle_since = spins;
            } else {
                dp_nanosleep(64);
                if ((spins & 255u) == 255u) {
                    /* a compute warp that bailed out never completes its rows */
                    if (spins - idle_since < 512u) t_idle = dp_clock();
                    bool bad = dp_ld_flag(p.err) != 0 || (dp_clock() - t_idle) > 4 * p.spin_limit;
                    if (!dp_all(!bad)) {
                        CLAPCA_HANG_PRINT("service: cta %d lane %d l0 %d g0 %d nz %d ng %d d %d pub %d pushed %d pdst %p err %d\n",
                                          dp_block(), lane, l0, g0, nz, ng, d, pub, pushed, (void *)pdst, dp_ld_flag(p.err));
                        if (lane == 0)
                            dp_set_error(p.err, 7);
                        break;
                    }
                }
            }
        }
        if (p.diag && lane == 0)
            dp_atomic_add64(p.diag + 1, (unsigned long long)t_busy);
    }

    /*
     * Layout items of a sharded volume: the first plane of a z-block is the "old plane above" of generation 0 for the
     * last plane of the previous block -- on another GPU.  While a compute warp packs that plane (and raises
     * prog[-1][z] every 32 rows) the service warp copies the finished H rows into the neighbour's ghost plane and raises
     * its "generation -1" counter: the halo seed of a resident run (api_slab.cu) moved into the launch.
     */
    CA_MDEV void seed_push(const Bp3Params &p, int zl, TileShared &ts, uint32_t &phase)
    {
        const int lane = dp_lane();
        const int H = p.H;
        const Bp3Plane pl = p.planes[zl];
        if (!pl.push_dn_rows)
            return;
        const int *myprog = p.prog - p.Z + zl;
        const uint32_t *src = p.rows + (size_t)zl * H * RECW;
        int pushed = 0;
        while (pushed < H) {
            if (!wait_word(p, myprog, pushed + 1, false, 8))
                return;
            const int avail = (int)dp_shfl((uint32_t)(lane == 0 ? dp_ld_acquire(myprog) : 0), 0);
            if (p.halo_ldst) {
                copy_h_rows(pl.push_dn_rows, src, pushed, avail);
            } else {
                dp_fence_proxy_async();
                bulk_copy_h_rows(ts, pl.push_dn_rows, src, pushed, avail, phase, p);
                if (lane == 0) {
                    dp_bulk_wait();
                    dp_fence_proxy_async();
                }
            }
            dp_fence_sys();
            if (lane == 0)
                dp_st_flag_sys(pl.push_dn_flag - 1, avail);
            pushed = avail;
        }
    }

    /*
     * Tile mode: the CTA claims one tile at a time.  Item = (first local plane, first generation, nz | ng << 8, H);
     * compute warp w = i + nz * j sweeps plane i of the tile at generation j, warps beyond nz * ng sit the item out,
     * warp `team` (the last one) is the service warp.  Layout items (g == -1 / g == G): warp w < nz packs / unpacks
     * plane w of the group and publishes its own counter.
     */
    CA_MDEV void tile_loop(const Bp3Params &p)
    {
        CA_SHARED(TileShared, tsp, 1);
        TileShared &ts = tsp[0];
        int *sm = ts.cnt;                           /* row counters of the compute warps, then the claimed ticket */
        const int w = dp_warp_in_block();
        const int T = p.team;
        uint32_t phase = 0u;                        /* service warp: parity of the staging mbarrier's current phase */
        if (dp_thread() == 0)
            dp_mbar_init(&ts.bar, 1);
        for (;;) {
            if (dp_thread() == 0) {
                unsigned t = dp_atomic_inc(p.ticket);
                if (dp_ld_flag(p.err) != 0)
                    t = 0xffffffffu;
                sm[BP3_MAX_TEAM] = (int)t;
            }
            if (dp_thread() < BP3_MAX_TEAM)
                sm[dp_thread()] = 0;
            dp_syncblock();
            const unsigned t = (unsigned)dp_ld_volatile(&sm[BP3_MAX_TEAM]);
            if (t >= (unsigned)p.nsweeps)
                break;
            const int4 it = p.order[t];
            const int nz = it.z & 0xff, ng = (it.z >> 8) & 0xff;
            if (p.layout_items && (it.y < 0 || it.y >= p.G)) {
                if (w < nz) {
                    if (it.y < 0)
                        pack_plane(p, it.x + w);
                    else
                        unpack_plane(p, it.x + w);
                } else if (w == T && it.y < 0) {
                    seed_push(p, it.x, ts, phase);  /* a packed z-block edge is the neighbour's "old plane above" of generation 0 */
                }
            } else if (w < nz * ng) {
                const int i = w % nz, j = w / nz;
                TileWire tw;
                tw.dn = i > 0 ? sm + (w - 1) : nullptr;
                tw.up = (j > 0 && i + 1 < nz) ? sm + (w - nz + 1) : nullptr;
                tw.own = j > 0 ? sm + (w - nz) : nullptr;
                tw.done = sm + w;
                run_rows<true>(p, it.x + i, it.y + j, 0, p.H, nullptr, &tw);
            } else if (w == T) {
                service_loop(p, it.x, it.y, nz, ng, ts, phase);
            }
            dp_syncblock();                         /* the counters are cleared for the next item */
        }
    }

    CA_MDEV void kernel_body(const Bp3Params &p)
    {
        if (p.pub_workers <= 0) {
            work_loop(p, nullptr);
            return;
        }
        CA_SHARED(PubSlot, slots, BP3_MAX_PUB_WORKERS + 1);     /* last entry: exit counter */
        int *nexit = &slots[BP3_MAX_PUB_WORKERS].done;
        const int nw = dp_block_threads() / 32 - 1;
        const int w = dp_warp_in_block();
        if (dp_thread() <= BP3_MAX_PUB_WORKERS) {
            slots[dp_thread()].flag = 0ull;
            slots[dp_thread()].done = 0;
            slots[dp_thread()].pub = 0;
        }
        dp_syncblock();
        if (w < nw) {
            work_loop(p, slots + w);
            dp_syncwarp();
            if (dp_lane() == 0)
                dp_atomic_add_cta(nexit, 1);
        } else {
            publish_loop(slots, nexit, nw);
        }
    }
};

/*
 * Self-publishing mode: 128-thread CTAs, 5 (2 words per lane) / 6 (1 word per lane) of them per SM.
 * Publisher mode: one CTA of up to 640 / 768 threads per SM (19 / 23 workers + the publisher).  The register
 * cap is the same either way: 65536 / 640 = 102, 65536 / 768 = 85.
 */
template <int P, int WPL>
struct Bp3Bounds {
    static constexpr int kMaxThreads = (P == 3 && WPL == 2) ? 640 : ((P <= 4 && WPL == 1) ? 768 : 160);
};

/*
 * Tile mode is a kernel of its own (one CTA per SM).  The register file is split over the SM's four sub-partitions, so
 * what a thread may use follows from the warps per SUB-PARTITION: 16 warps (15 compute + the service warp) are 4 per
 * sub-partition = 128 registers per thread; a 17th warp would put 5 on one of them and cap every thread at 96 (ptxas
 * then spills in the row loop as soon as the service path grows).  15 compute warps = tiles of 5 planes x 3 generations.
 * The widest variants (8 state planes, 4 words per lane) run 7 compute warps + the service warp.
 */
#ifndef CLAPCA_TEAM_WARPS
#define CLAPCA_TEAM_WARPS 15
#endif
template <int P, int WPL>
struct Bp3TeamBounds {
    static constexpr int kTeam = (P <= 4 && WPL <= 2) ? CLAPCA_TEAM_WARPS : 7;
    static constexpr int kMaxThreads = 32 * (kTeam + 1);
};

/* largest team (compute warps per CTA) of a variant */
inline int bp3_team_cap(int P, int WPL)
{
    return (P <= 4 && WPL <= 2) ? CLAPCA_TEAM_WARPS : 7;
}

/*
 * The wide build of the tile kernel: 18 compute warps + the service warp = 19 warps, 5 on three of the four
 * sub-partitions, which caps a thread at 96 registers (ptxas: 4 bytes of spill in the 3-plane variants).  More warps
 * hide more of the fixed-latency stalls of an ALU-bound loop: 6 x 3 tiles sweep 2048^3 x 50 in 89.3 ms against 91.8 ms
 * for 5 x 3 tiles at 116 registers, and sharded volumes gain as well (N = 2 / 4 / 8: 53.6 -> 49.0, 31.2 -> 28.2,
 * 17.8 -> 16.9 ms with z-blocks of 48 planes).  The 3-plane variants take the wide kernel, everything else the default
 * one (profiles/r02_knobs_18_compute_warps_96_regs.txt, r02_knobs_multi_wide_n{2,4,8}.txt).
 */
enum { BP3_WIDE_TEAM = 18 };
inline int bp3_team_cap_wide(int P, int WPL)
{
    return (P == 3 && WPL <= 2) ? (int)BP3_WIDE_TEAM : 0;
}

template <int P, int WPL, class Rule>
CA_GLOBAL void __launch_bounds__(Bp3Bounds<P, WPL>::kMaxThreads, 1) ca3d_sweep_kernel(Bp3Params p)
{
    Sweep3<P, WPL, Rule>::kernel_body(p);
}

template <int P, int WPL, class Rule>
CA_GLOBAL void __launch_bounds__(Bp3TeamBounds<P, WPL>::kMaxThreads, 1) ca3d_team_kernel(Bp3Params p)
{
    Sweep3<P, WPL, Rule>::tile_loop(p);
}

template <int P, int WPL, class Rule>
CA_GLOBAL void __launch_bounds__(32 * (BP3_WIDE_TEAM + 1), 1) ca3d_team_wide_kernel(Bp3Params p)
{
    Sweep3<P, WPL, Rule>::tile_loop(p);
}

} // namespace clapca
#endif
