/*
 * emu_ca3d_rowloop.cpp -- emu_ca3d (same arguments, same oracle check) with the library's row-loop knobs taken from the
 * environment, as the library's sweep_knobs() does: CLAPCA_PREFETCH_ROWS (default 0) and CLAPCA_ROWLOOP=generic
 * (every row through the general row step).  TEST ONLY: built and executed by tests/test_ca3d_rowloop.py.
 *
 * emu_ca3d.cpp is compiled unchanged.  It clears each rank's launch parameters with memset(&p, 0, sizeof p) before it
 * fills them in.  An overload for Bp3Params pointers is the one place that sees the parameters before the launch: it
 * clears them, applies the two knobs and reports them on stderr (the test checks they arrived); every other memset
 * goes to the C library as before.
 */
#include <stdio.h>
#include <string.h>
#include <stdlib.h>
#include <algorithm>
#include <chrono>
#include <thread>
#include <vector>
#include "emu_runtime.h"
#include "../../clap_b200/csrc/ca3d_bitplane.cuh"
#include "../../clap_b200/csrc/ca3d_layout.cuh"
#include "../../clap_b200/csrc/bp_plan.h"
extern "C" {
#include "../../oracle/port/oracle_port.h"
}

static void *rowloop_memset(clapca::Bp3Params *p, int c, size_t n)
{
    memset(p, c, n);
    const char *pf = getenv("CLAPCA_PREFETCH_ROWS"), *loop = getenv("CLAPCA_ROWLOOP");
    p->prefetch_rows = pf ? std::max(0, atoi(pf)) : 0;
    p->rowloop_generic = loop && strcmp(loop, "generic") == 0;
    fprintf(stderr, "row loop %s, prefetch_rows %d\n", p->rowloop_generic ? "generic" : "interior", p->prefetch_rows);
    return p;
}
template <class T>
static void *rowloop_memset(T *p, int c, size_t n)
{
    return memset(p, c, n);
}

#define memset rowloop_memset
#include "emu_ca3d.cpp"
#undef memset
