/*
 * clapca_api.cu -- the C ABI of libclapca_cuda (include/clapca.h): device
 * context, device-resident grids, ca3d / ca2d engine selection and kernel
 * launches (multi-GPU slabs: api_slab.cu, noise / terrain fields: api_fields.cu).
 * Everything here runs on the GPU or fails; there is no host fallback.
 */
#include <cooperative_groups.h>

#include <unordered_set>
#include <map>
#include <tuple>
#include "api_internal.h"
#include "bp2_launch.h"
#include "sk2_launch.h"
#include "ca2d_layout.cuh"
#include "ca2d_skew_layout.cuh"
#include "ca3d_layout.cuh"
#include "ca_wavefront.cuh"

using namespace clapca;
using namespace clapca::api;

namespace {
thread_local std::string g_err;
}

namespace clapca {
namespace api {

Ctx g_ctx;

int fail(int code, const char *fmt, ...)
{
    char buf[512];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof(buf), fmt, ap);
    va_end(ap);
    g_err = buf;
    return code;
}

bool diag_enabled()
{
    const char *e = getenv("CLAPCA_DIAG");
    return e && atoi(e) != 0;
}

/* CLAPCA_DIAG=1: where the persistent warps of the last sweep launch spent their cycles */
void diag_report(const char *what, const unsigned *d_ticket, cudaStream_t stream, int rank)
{
    if (!diag_enabled())
        return;
    unsigned long long d[4] = { 0, 0, 0, 0 };
    if (cudaMemcpyAsync(d, d_ticket + 4, sizeof(d), cudaMemcpyDeviceToHost, stream) != cudaSuccess ||
        cudaStreamSynchronize(stream) != cudaSuccess)
        return;
    fprintf(stderr, "clapca diag [%s rank %d]: in items %.3e cycles, waiting on counters %.1f %%, on ghost tags %.1f %%, "
            "on team-mates %.1f %%\n", what, rank, (double)d[2], d[2] ? 100.0 * d[0] / d[2] : 0.0,
            d[2] ? 100.0 * d[1] / d[2] : 0.0, d[2] ? 100.0 * d[3] / d[2] : 0.0);
}

int need_init()
{
    if (g_ctx.device < 0)
        return fail(CLAPCA_ERR_STATE, "clapca_init() has not been called");
    return CLAPCA_OK;
}

int grid_blocks_for(size_t work_items, int threads, int per_sm_cap)
{
    size_t b = (work_items + threads - 1) / threads;
    size_t cap = (size_t)g_ctx.sms * per_sm_cap;        /* grid-stride: a multiple of the SM count */
    if (b > cap) b = cap;
    if (b < 1) b = 1;
    return (int)b;
}

/* the nine cas[] entries: core/ca3d.c:110-122 (surv, born, nr_states) */
#define B(n) (1u << (n))
#define RANGE(s, e) (((1u << ((e) - (s))) - 1u) << (s))
const uint32_t kCas[9][3] = {
    { B(4), B(4), 5 },
    { B(6) | B(7) | B(8), B(6) | B(7) | B(8), 3 },
    { B(4) | B(5) | B(6) | B(7), B(6) | B(7) | B(8), 10 },
    { RANGE(9, 26), B(5) | B(6) | B(7) | B(12) | B(13) | B(15), 5 },
    { B(2) | B(6) | B(9), B(4) | B(6) | B(8) | B(9), 10 },
    { B(1) | B(4) | B(8) | B(11) | RANGE(13, 26), RANGE(13, 26), 5 },
    { RANGE(0, 3) | RANGE(7, 9) | RANGE(11, 13) | B(18) | B(21) | B(22) | B(24) | B(26),
      B(4) | B(13) | B(17) | RANGE(20, 24) | B(26), 4 },
    { RANGE(5, 8), RANGE(6, 7) | B(9) | B(12), 4 },
    { RANGE(0, 6), B(1) | B(3), 2 },
};

} // namespace api
} // namespace clapca

namespace clapca {
cudaError_t bp3_launch(int rule, int P, int WPL, const Bp3Params &p, int sms, cudaStream_t stream,
                       Bp3LaunchInfo *info)
{
    typedef cudaError_t (*fn_t)(int, int, const Bp3Params &, int, cudaStream_t, Bp3LaunchInfo *);
    static const fn_t tab[BP3_NRULES] = {
        bp3_launch_rule0, bp3_launch_rule1, bp3_launch_rule2, bp3_launch_rule3, bp3_launch_rule4,
        bp3_launch_rule5, bp3_launch_rule6, bp3_launch_rule7, bp3_launch_rule8, bp3_launch_rule9,
    };
    if (rule < 0 || rule >= BP3_NRULES)
        return cudaErrorInvalidValue;
    return tab[rule](P, WPL, p, sms, stream, info);
}
cudaError_t bp2_launch(int P, int WPL, bool moore, int warps, const Bp2Params &p, int sms, cudaStream_t stream,
                       Bp2LaunchInfo *info)
{
    switch (bp2_rule_for(p.born, p.surv, p.nrval)) {
    case BP2_RULE_CAVE: return bp2_launch_rule1(P, WPL, moore, warps, p, sms, stream, info);
    case BP2_RULE_TEST: return bp2_launch_rule2(P, WPL, moore, warps, p, sms, stream, info);
    default: return bp2_launch_rule0(P, WPL, moore, warps, p, sms, stream, info);
    }
}
cudaError_t sk2_launch(int WPL, bool moore, int warps, const Sk2Params &p, int sms, cudaStream_t stream,
                       Bp2LaunchInfo *info)
{
    switch (bp2_rule_for(p.born, p.surv, p.nrval)) {
    case BP2_RULE_CAVE: return sk2_launch_rule1(WPL, moore, warps, p, sms, stream, info);
    case BP2_RULE_TEST: return sk2_launch_rule2(WPL, moore, warps, p, sms, stream, info);
    default: return sk2_launch_rule0(WPL, moore, warps, p, sms, stream, info);
    }
}
int bp3_max_workers(int rule, int P, int WPL, int sms, int team, int max_ctas)
{
    Bp3Params p;
    memset(&p, 0, sizeof(p));
    p.nsweeps = -1;                     /* query only: the launcher returns before launching */
    p.team = team;
    p.max_ctas = max_ctas;
    Bp3LaunchInfo info = { 0, 0, 0, 0 };
    if (bp3_launch(rule, P, WPL, p, sms, nullptr, &info) != cudaSuccess)
        return sms * 8;
    return info.workers;
}
} // namespace clapca

struct clapca_grid {
    int64_t d0, d1, d2;
    size_t n;
    uint8_t *cells = nullptr;
    /* bit-plane engine scratch, grown on demand */
    uint32_t *rows = nullptr;
    size_t rows_bytes = 0;
    int *prog = nullptr;
    size_t prog_count = 0;
    int4 *order = nullptr;          /* work items in claim order */
    size_t order_bytes = 0;
    int n_items = 0;
    int order_Z = -1, order_H = -1, order_G = -1, order_L = -1;
    Bp3Plane *planes = nullptr;     /* per-plane source descriptors */
    size_t planes_bytes = 0;
    const void *planes_rows = nullptr;
    const void *planes_prog = nullptr;
    int planes_NP = -1, planes_RWP = -1;
    unsigned *ticket = nullptr;     /* [0] ticket, [1] err (as int) */
    /* streamed runs (layout items of the sweep kernel): chunk-arrival word and per-plane done flags */
    int *d_in_ready = nullptr;      /* device: chunks landed, written by 4-byte copies on the H2D stream */
    int *h_io = nullptr;            /* pinned + mapped: [0, d2) done flags, then the chunk ordinals 1, 2, ... */
    size_t h_io_count = 0;
    int io_epoch = 0;
    cudaEvent_t ev_io = nullptr;
    cudaStream_t stream = nullptr;
    cudaEvent_t ev[4] = { nullptr, nullptr, nullptr, nullptr };
    clapca_run_stats stats;
};

/* host buffers of a streamed run */
struct StreamIO {
    const uint8_t *host_in;
    uint8_t *host_out;
    unsigned max_value;
};

extern "C" {
#pragma GCC visibility push(default)

int clapca_device_count(void)
{
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) {
        cudaGetLastError();
        return 0;
    }
    return n;
}

const char *clapca_last_error(void) { return g_err.c_str(); }

int clapca_init(int device)
{
    if (g_ctx.device == device)
        return CLAPCA_OK;
    if (g_ctx.device >= 0)
        clapca_shutdown();
    int n = 0;
    CU(cudaGetDeviceCount(&n));
    if (device < 0 || device >= n)
        return fail(CLAPCA_ERR_ARG, "device %d out of range (have %d)", device, n);
    CU(cudaSetDevice(device));
    cudaDeviceProp prop;
    CU(cudaGetDeviceProperties(&prop, device));
    if (prop.major < 10)
        return fail(CLAPCA_ERR_CUDA, "device %d is sm_%d%d; this library carries sm_100a code only",
                    device, prop.major, prop.minor);
    g_ctx.sms = prop.multiProcessorCount;
    g_ctx.mem = prop.totalGlobalMem;
    CU(cudaDeviceGetAttribute(&g_ctx.coop, cudaDevAttrCooperativeLaunch, device));
    if (!g_ctx.coop)
        return fail(CLAPCA_ERR_CUDA, "device %d does not support cooperative launch", device);
    CU(cudaStreamCreateWithFlags(&g_ctx.stream, cudaStreamNonBlocking));
    CU(cudaStreamCreateWithFlags(&g_ctx.stream_in, cudaStreamNonBlocking));
    CU(cudaStreamCreateWithFlags(&g_ctx.stream_out, cudaStreamNonBlocking));
    CU(cudaMalloc(&g_ctx.d_count, sizeof(unsigned long long)));
    CU(cudaMalloc(&g_ctx.d_max, sizeof(unsigned)));
    CU(cudaMalloc(&g_ctx.d_zeros, 1024));
    CU(cudaMemset(g_ctx.d_zeros, 0, 1024));
    g_ctx.device = device;
    return CLAPCA_OK;
}

void clapca_shutdown(void)
{
    if (g_ctx.device < 0)
        return;
    cudaSetDevice(g_ctx.device);
    cudaDeviceSynchronize();
    if (g_ctx.d_count) cudaFree(g_ctx.d_count);
    if (g_ctx.d_max) cudaFree(g_ctx.d_max);
    if (g_ctx.d_zeros) cudaFree(g_ctx.d_zeros);
    if (g_ctx.oneshot_grid) clapca_grid_destroy((clapca_grid *)g_ctx.oneshot_grid);
    if (g_ctx.d_smooth) cudaFree(g_ctx.d_smooth);
    for (int i = 0; i < 5; i++)
        if (g_ctx.scratch[i]) cudaFree(g_ctx.scratch[i]);
    if (g_ctx.stream) cudaStreamDestroy(g_ctx.stream);
    if (g_ctx.stream_in) cudaStreamDestroy(g_ctx.stream_in);
    if (g_ctx.stream_out) cudaStreamDestroy(g_ctx.stream_out);
    g_ctx = Ctx();
}

int clapca_sm_count(void) { return g_ctx.sms; }
size_t clapca_device_mem_bytes(void) { return g_ctx.mem; }

int clapca_ca3d_rule(int nca, uint32_t *surv, uint32_t *born, uint32_t *nr_states)
{
    /* core/ca3d.c:126 computes nca % array_size(cas) in size_t: a negative index wraps through 2^64 (-1 -> rule 6) */
    const int i = (int)((size_t)(long)nca % 9u);
    if (surv) *surv = kCas[i][0];
    if (born) *born = kCas[i][1];
    if (nr_states) *nr_states = kCas[i][2];
    return CLAPCA_OK;
}

/* ---- grids ---------------------------------------------------------------- */

int clapca_grid_create(clapca_grid **out, int64_t d0, int64_t d1, int64_t d2)
{
    if (int rc = need_init()) return rc;
    if (!out || d0 < 1 || d1 < 1 || d2 < 1)
        return fail(CLAPCA_ERR_ARG, "grid_create: bad dims %lld x %lld x %lld", (long long)d0, (long long)d1,
                    (long long)d2);
    clapca_grid *g = new (std::nothrow) clapca_grid();
    if (!g)
        return fail(CLAPCA_ERR_NOMEM, "grid_create: host allocation failed");
    g->d0 = d0; g->d1 = d1; g->d2 = d2;
    g->n = (size_t)d0 * (size_t)d1 * (size_t)d2;
    memset(&g->stats, 0, sizeof(g->stats));
    g->stream = g_ctx.stream;
    cudaError_t e = cudaMalloc(&g->cells, g->n);
    if (e == cudaSuccess) e = cudaMalloc(&g->ticket, kTicketWords * sizeof(unsigned));
    for (int i = 0; i < 4 && e == cudaSuccess; i++)
        e = cudaEventCreate(&g->ev[i]);
    if (e != cudaSuccess) {
        clapca_grid_destroy(g);
        return fail(e == cudaErrorMemoryAllocation ? CLAPCA_ERR_NOMEM : CLAPCA_ERR_CUDA,
                    "grid_create: %s", cudaGetErrorString(e));
    }
    *out = g;
    return CLAPCA_OK;
}

int clapca_grid_destroy(clapca_grid *g)
{
    if (!g)
        return CLAPCA_OK;
    if (g->cells) cudaFree(g->cells);
    if (g->rows) cudaFree(g->rows);
    if (g->prog) cudaFree(g->prog);
    if (g->order) cudaFree(g->order);
    if (g->planes) cudaFree(g->planes);
    if (g->ticket) cudaFree(g->ticket);
    if (g->d_in_ready) cudaFree(g->d_in_ready);
    if (g->h_io) cudaFreeHost(g->h_io);
    if (g->ev_io) cudaEventDestroy(g->ev_io);
    for (int i = 0; i < 4; i++)
        if (g->ev[i]) cudaEventDestroy(g->ev[i]);
    delete g;
    return CLAPCA_OK;
}

/*
 * One-shot calls (host array in, host array out) run on a grid of their own.  Creating and destroying it costs several
 * cudaMalloc / cudaFree per call -- tens of milliseconds once the context has seen large allocations, more than the
 * 16384^2 x 100 run it serves (measured: 17 .. 107 ms for clapca_ca2d_generate from run to run) -- and a caller that
 * steps a grid in a loop (the reference's instantiator placement: ca2d_step per generation) pays it every time.  The
 * grid of the last one-shot call is therefore kept for the next one of the same shape, up to 1 GiB of cells.
 */
static int oneshot_acquire(clapca_grid **out, int64_t d0, int64_t d1, int64_t d2)
{
    clapca_grid *c = (clapca_grid *)g_ctx.oneshot_grid;
    if (c && c->d0 == d0 && c->d1 == d1 && c->d2 == d2) {
        g_ctx.oneshot_grid = nullptr;
        *out = c;
        return CLAPCA_OK;
    }
    return clapca_grid_create(out, d0, d1, d2);
}

static void oneshot_release(clapca_grid *g)
{
    if (!g)
        return;
    if (g->n > ((size_t)1 << 30)) {
        clapca_grid_destroy(g);
        return;
    }
    if (g_ctx.oneshot_grid)
        clapca_grid_destroy((clapca_grid *)g_ctx.oneshot_grid);
    g_ctx.oneshot_grid = g;
}

int clapca_grid_upload(clapca_grid *g, const uint8_t *host)
{
    if (!g || !host) return fail(CLAPCA_ERR_ARG, "grid_upload: NULL argument");
    CU(cudaMemcpyAsync(g->cells, host, g->n, cudaMemcpyDefault, g->stream));
    CU(cudaStreamSynchronize(g->stream));
    return CLAPCA_OK;
}

int clapca_grid_download(clapca_grid *g, uint8_t *host)
{
    if (!g || !host) return fail(CLAPCA_ERR_ARG, "grid_download: NULL argument");
    CU(cudaMemcpyAsync(host, g->cells, g->n, cudaMemcpyDefault, g->stream));
    CU(cudaStreamSynchronize(g->stream));
    return CLAPCA_OK;
}

void *clapca_grid_device_ptr(clapca_grid *g) { return g ? g->cells : nullptr; }
void *clapca_grid_stream(clapca_grid *g) { return g ? (void *)g->stream : nullptr; }

int clapca_grid_last_stats(clapca_grid *g, clapca_run_stats *st)
{
    if (!g || !st) return fail(CLAPCA_ERR_ARG, "grid_last_stats: NULL argument");
    *st = g->stats;
    return CLAPCA_OK;
}

static int count_on_stream(const uint8_t *cells, size_t n, cudaStream_t s, int64_t *population)
{
    CU(cudaMemsetAsync(g_ctx.d_count, 0, sizeof(unsigned long long), s));
    count_nonzero_kernel<<<grid_blocks_for((n + 15) / 16, 256), 256, 0, s>>>(cells, n, g_ctx.d_count);
    CU(cudaGetLastError());
    unsigned long long c = 0;
    CU(cudaMemcpyAsync(&c, g_ctx.d_count, sizeof(c), cudaMemcpyDeviceToHost, s));
    CU(cudaStreamSynchronize(s));
    *population = (int64_t)c;
    return CLAPCA_OK;
}

/*
 * Fingerprint of every plane of a uint8 volume in device memory (see clapca.h): the planes of a sharded run are
 * compared with those of a single-GPU run -- and with the oracle's -- without moving the cells.
 */
int clapca_hash_planes(const void *d_cells, size_t plane_bytes, size_t nplanes, uint64_t *hashes)
{
    if (int rc = need_init()) return rc;
    if (!d_cells || !hashes || plane_bytes == 0) return fail(CLAPCA_ERR_ARG, "hash_planes: bad arguments");
    if (nplanes == 0) return CLAPCA_OK;
    unsigned long long *d_h = nullptr;
    CU(cudaMalloc(&d_h, nplanes * sizeof(unsigned long long)));
    cudaError_t e = cudaMemsetAsync(d_h, 0, nplanes * sizeof(unsigned long long), g_ctx.stream);
    if (e == cudaSuccess) {
        const size_t words = (plane_bytes + 7) / 8;
        const unsigned bx = (unsigned)std::min<size_t>((words + 255) / 256, 64);
        dim3 grid(bx, (unsigned)std::min<size_t>(nplanes, 65535));
        plane_hash_kernel<<<grid, 256, 0, g_ctx.stream>>>((const uint8_t *)d_cells, plane_bytes, nplanes, d_h);
        e = cudaGetLastError();
    }
    if (e == cudaSuccess) e = cudaMemcpyAsync(hashes, d_h, nplanes * sizeof(unsigned long long), cudaMemcpyDeviceToHost, g_ctx.stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(g_ctx.stream);
    cudaFree(d_h);
    if (e != cudaSuccess) return fail(CLAPCA_ERR_CUDA, "hash_planes: %s", cudaGetErrorString(e));
    return CLAPCA_OK;
}

int clapca_grid_count(clapca_grid *g, int64_t *population)
{
    if (!g || !population) return fail(CLAPCA_ERR_ARG, "grid_count: NULL argument");
    return count_on_stream(g->cells, g->n, g->stream, population);
}

/* ---- ca3d ------------------------------------------------------------------- */

static int run3d_wavefront(clapca_grid *g, uint32_t surv, uint32_t born, uint32_t nr_states, int steps)
{
    Wf3Params p;
    p.a = g->cells;
    p.d0 = g->d0; p.d1 = g->d1; p.d2 = g->d2;
    p.surv = surv; p.born = born; p.bornval = (nr_states - 1u) & 0xffu;
    p.G = steps;
    int per_sm = 0;
    CU(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, ca3d_wavefront_kernel, 256, 0));
    if (per_sm < 1) return fail(CLAPCA_ERR_CUDA, "ca3d_wavefront_kernel does not fit on an SM");
    size_t pairs = (size_t)g->d1 * g->d2;
    int blocks = (int)std::min<size_t>((pairs + 255) / 256, (size_t)per_sm * g_ctx.sms);
    if (blocks < 1) blocks = 1;
    void *args[] = { &p };
    CU(cudaEventRecord(g->ev[1], g->stream));
    CU(cudaLaunchCooperativeKernel((void *)ca3d_wavefront_kernel, dim3(blocks), dim3(256), args, 0, g->stream));
    CU(cudaEventRecord(g->ev[2], g->stream));
    g->stats.launches = 1;
    g->stats.engine = CLAPCA_ENGINE_WAVEFRONT;
    g->stats.planes = 0;
    g->stats.workers = blocks * 256;
    return CLAPCA_OK;
}

#pragma GCC visibility pop
} /* extern "C" */

/* ---- helpers shared with api_slab.cu / api_fields.cu (api_internal.h) ---- */

int clapca::api::ensure_bytes(void **ptr, size_t *have, size_t want)
{
    if (*have >= want)
        return CLAPCA_OK;
    if (*ptr) cudaFree(*ptr);
    *ptr = nullptr;
    *have = 0;
    CU(cudaMalloc(ptr, want));
    *have = want;
    return CLAPCA_OK;
}

int clapca::api::timed_sync(cudaEvent_t a, cudaEvent_t b, float *ms)
{
    CU(cudaStreamSynchronize(g_ctx.stream));
    if (ms) CU(cudaEventElapsedTime(ms, a, b));
    return CLAPCA_OK;
}

cudaError_t clapca::api::launch_ca3d_pack(const Bp3Layout &L, cudaStream_t stream)
{
    /* one warp per 32 words of a row; grid-stride over a multiple of the SM count */
    const int blocks = grid_blocks_for((size_t)L.Z * L.H * L.RWP, 256, 8);
    if (L.P <= 3)      ca3d_pack_rows_kernel<3><<<blocks, 256, 0, stream>>>(L);
    else if (L.P == 4) ca3d_pack_rows_kernel<4><<<blocks, 256, 0, stream>>>(L);
    else               ca3d_pack_rows_kernel<8><<<blocks, 256, 0, stream>>>(L);
    return cudaGetLastError();
}

cudaError_t clapca::api::launch_ca3d_unpack(const Bp3Layout &L, cudaStream_t stream)
{
    const int blocks = grid_blocks_for((size_t)L.Z * L.H * L.RWP, 256, 8);
    if (L.P <= 3)      ca3d_unpack_rows_kernel<3><<<blocks, 256, 0, stream>>>(L);
    else if (L.P == 4) ca3d_unpack_rows_kernel<4><<<blocks, 256, 0, stream>>>(L);
    else               ca3d_unpack_rows_kernel<8><<<blocks, 256, 0, stream>>>(L);
    return cudaGetLastError();
}

/* force the (lazy) load of the layout kernels for P state planes: see slab_prepare() */
cudaError_t clapca::api::preload_ca3d_layout(int P)
{
    cudaFuncAttributes fa;
    cudaError_t e;
    if (P <= 3) {
        e = cudaFuncGetAttributes(&fa, ca3d_pack_rows_kernel<3>);
        if (e == cudaSuccess) e = cudaFuncGetAttributes(&fa, ca3d_unpack_rows_kernel<3>);
    } else if (P == 4) {
        e = cudaFuncGetAttributes(&fa, ca3d_pack_rows_kernel<4>);
        if (e == cudaSuccess) e = cudaFuncGetAttributes(&fa, ca3d_unpack_rows_kernel<4>);
    } else {
        e = cudaFuncGetAttributes(&fa, ca3d_pack_rows_kernel<8>);
        if (e == cudaSuccess) e = cudaFuncGetAttributes(&fa, ca3d_unpack_rows_kernel<8>);
    }
    if (e == cudaSuccess) e = cudaFuncGetAttributes(&fa, max_u8_kernel);
    if (e == cudaSuccess) e = cudaFuncGetAttributes(&fa, halo_seed_kernel);
    return e;
}

cudaError_t clapca::api::launch_max_u8(const uint8_t *cells, size_t n, unsigned *d_max, cudaStream_t stream)
{
    max_u8_kernel<<<grid_blocks_for((n + 15) / 16, 256), 256, 0, stream>>>(cells, n, d_max);
    return cudaGetLastError();
}

cudaError_t clapca::api::launch_halo_seed(uint32_t *dst, const uint32_t *src, int H, int RWP, int NP, cudaStream_t stream)
{
    halo_seed_kernel<<<grid_blocks_for((size_t)H * 2 * RWP, 256, 4), 256, 0, stream>>>(dst, src, H, RWP, NP);
    return cudaGetLastError();
}

/* progress counters are raised every kFlagRows rows: one fence per kFlagRows row steps */
static const int kFlagRows = 8;


/*
 * Tile mode (ca3d_bitplane.cuh): compute warps per CTA = planes x generations of a work item; 0 = one warp per sweep.
 * Default: 15 compute warps + the service warp (16 warps = 4 per SM sub-partition = 128 registers per thread) for the
 * variants whose register budget allows it.  Round 1 measured plane groups of 16 x 1 on B200 at 2048^3, coral
 * (profiles/r01_team_mode_lowpar.txt): 50 generations 123.3 -> 121.0 ms against one warp per sweep, and 35.2 -> 16.4 ms
 * in the low-parallelism regime a rank of an 8-GPU run sees.
 */
int clapca::api::team_config(int P, int WPL, bool single_gpu)
{
    int cap = bp3_team_cap(P, WPL);
    int t = cap >= 12 ? cap : 0;
    /* single-GPU runs of the 3-plane variants: the wide (19-warp, 96-register) kernel -- see bp3_team_cap_wide() */
    if (single_gpu && bp3_team_cap_wide(P, WPL) > cap)
        t = cap = bp3_team_cap_wide(P, WPL);
    if (const char *e = getenv("CLAPCA_TEAM")) {
        t = atoi(e);
        cap = std::max(cap, bp3_team_cap_wide(P, WPL));
    }
    if (t <= 0) return 0;
    return std::min(t, cap);
}

/*
 * Generations per tile.  Tiles of several generations keep those generations of a row within ~20 row steps of each
 * other: generation g+1 reads generation g from L2 and overwrites it there, and HBM sees 1 / ng of the per-generation
 * streaming of plane groups (measured with 4 x 4 tiles: 540 -> 138 GB per 2048^3 x 50 run).  The planner lowers it when the launch has too few CTAs for the forward dependency (bp_plan.h).
 */
int clapca::api::tile_gens_config(int team)
{
    /* the largest divisor g of the team with g <= team / g: 15 -> 3 (5 x 3), 16 -> 4 (4 x 4), 12 -> 3 (4 x 3) */
    int tg = 1;
    for (int g = 2; g * g <= team; g++)
        if (team % g == 0) tg = g;
    if (team < 12) tg = 1;
    if (const char *e = getenv("CLAPCA_TILE_GENS")) { int v = atoi(e); if (v > 0) tg = v; }
    return tg;
}

void clapca::api::sweep_knobs(Bp3Params &p, int team, bool single_gpu)
{
    p.flag_rows = kFlagRows;
    /* the generation groups of a single-GPU run are far apart in time (order_config): a tile's first generation reads
       its rows from HBM, 6 rows ahead covers that latency (98.3 -> 94.5 ms at 2048^3 x 50; 16 rows ahead: 108 ms) */
    p.prefetch_rows = (single_gpu && team > 0) ? 6 : 0;
    if (const char *e = getenv("CLAPCA_FLAG_ROWS")) { int v = atoi(e); if (v > 0) p.flag_rows = v; }
    if (const char *e = getenv("CLAPCA_PREFETCH_ROWS")) p.prefetch_rows = std::max(0, atoi(e));
    if (const char *e = getenv("CLAPCA_CTAS_PER_SM")) p.max_ctas_per_sm = std::max(0, atoi(e));
    if (const char *e = getenv("CLAPCA_MAX_CTAS")) p.max_ctas = std::max(0, atoi(e));
    if (const char *e = getenv("CLAPCA_PUB_WORKERS")) p.pub_workers = std::max(0, atoi(e));
    /* CLAPCA_ROWLOOP=generic: every row takes the general row step (same volumes; A/B of the interior row loop) */
    if (const char *e = getenv("CLAPCA_ROWLOOP")) p.rowloop_generic = strcmp(e, "generic") == 0;
    p.team = team;
    /*
     * Halo rows: batched ld / st of the service warp by default.  The TMA variant (1-D bulk copies record -> shared
     * staging -> peer ghost plane, CLAPCA_HALO_LDST=0) was measured on 2 and 8 x B200 with the final kernel and loses:
     * 61.5 vs 58.1 ms at N = 2, 20.3 vs 17.8 ms at N = 8 (profiles/r02_knobs_multi_n8_final.txt) -- a batch of bulk
     * copies is a load round trip, an mbarrier wait, a store round trip and a wait_group in series before the peer's
     * counter may move, where 32 lanes keep 16 rows of loads in flight and the stores drain behind one fence.
     */
    p.halo_ldst = 1;
    if (const char *e = getenv("CLAPCA_HALO_LDST")) p.halo_ldst = atoi(e) != 0;
}

static const int kGenBatch = 16;

OrderCfg clapca::api::order_config(int Z, int H, int G, int max_workers, int team)
{
    OrderCfg oc = { 0, 0, kGenBatch, team, team, 1, 0, 0 };
    if (team > 0) {
        oc.mode = 3;
        oc.tile_g = tile_gens_config(team);     /* wanted; make_items() settles the shape for the plane list at hand */
        oc.ctas = std::max(1, max_workers / team);
        /*
         * Key distance between generation groups on one GPU (bp_plan.h, bp3_make_items_tile; slabs set their own).
         * A tile follows its z-predecessor (3 tz + flag_rows) rows behind, so one generation group keeps at most
         * H / (3 tz + flag_rows) CTAs busy; `active` groups in flight keep all of them busy, and no more groups than
         * that should be: every active group puts one more ticket between a tile and its forward partner (the tile's
         * late warps wait for the partner, its early warps for them at the end-of-item barrier).  Measured at
         * 2048^3 x 50, 148 CTAs of 5 x 3 tiles (profiles/r02_knobs_tile_skew_ca3d_2048.txt): distance tz + 1 (all 17
         * groups interleaved) 98.0 ms, Z / 4 .. Z / 2 94.4-94.9 ms, 2100 (one group at a time, 89 CTAs busy) 119 ms.
         */
        {
            const int tz = std::max(1, team / std::max(1, oc.tile_g));
            const int active = 1 + (oc.ctas * (3 * tz + kFlagRows) + H - 1) / std::max(H, 1);
            oc.tile_skew = std::max(tz + 1, Z / active);
        }
        if (const char *e = getenv("CLAPCA_TILE_SKEW")) oc.tile_skew = std::max(0, atoi(e));
        return oc;
    }
    if (const char *e = getenv("CLAPCA_ORDER")) { int v = atoi(e); if (v >= 0 && v <= 2) oc.mode = v; }
    if (oc.mode == 1) {
        oc.seg_rows = bp3_segment_rows(Z, H, G, max_workers);
        if (const char *e = getenv("CLAPCA_SEG_ROWS")) { int v = atoi(e); if (v > 0) oc.seg_rows = std::min(v, H); }
    }
    if (oc.mode == 2) {
        if (const char *e = getenv("CLAPCA_GEN_BATCH")) { int v = atoi(e); if (v > 0) oc.gen_batch = v; }
    }
    return oc;
}

void clapca::api::make_items(const OrderCfg &oc, const std::vector<Bp3Plane> &planes, int Zg, int H, int G,
                       std::vector<WorkItem> &items, bool layout_items)
{
    if (oc.mode == 3) bp3_make_items_tile(planes, H, G, oc.tile_z, oc.tile_g, items, layout_items, nullptr, oc.tile_skew);
    else if (oc.mode == 1) bp3_make_items(planes, Zg, H, G, oc.seg_rows, items);
    else if (oc.mode == 2) bp3_make_items_batched(planes, Zg, H, G, oc.gen_batch, items);
    else bp3_make_items_timekey(planes, H, G, items, layout_items);
}

/* planes per H2D chunk of a streamed run: ~32 MiB; CLAPCA_IO_CHUNK_MB / CLAPCA_IO_CHUNK_PLANES override */
int clapca::api::io_chunk_planes(size_t plane_bytes, int Z)
{
    size_t mb = 32;
    if (const char *e = getenv("CLAPCA_IO_CHUNK_MB")) { int v = atoi(e); if (v > 0) mb = (size_t)v; }
    size_t c = (mb << 20) / std::max<size_t>(plane_bytes, 1);
    if (const char *e = getenv("CLAPCA_IO_CHUNK_PLANES")) { int v = atoi(e); if (v > 0) c = (size_t)v; }
    if (c < 1) c = 1;
    if (c > (size_t)Z) c = (size_t)Z;
    while (((size_t)Z + c - 1) / c > 4096) c *= 2;         /* bounded number of copies */
    return (int)c;
}

extern "C" {
#pragma GCC visibility push(default)

/* CLAPCA_FUSED_LAYOUT=1: device-resident runs also convert the layout inside the sweep launch (layout items) */
static bool fused_layout_default()
{
    const char *e = getenv("CLAPCA_FUSED_LAYOUT");
    return e && atoi(e) != 0;
}

static inline void cpu_relax()
{
#if defined(__x86_64__) || defined(__i386__)
    __builtin_ia32_pause();
#endif
}

#pragma GCC visibility pop
} /* extern "C" */

/*
 * Host side of a streamed run (the sweep launch with layout items is already in flight on sp.s_kernel).  H2D: every
 * chunk of planes, then its ordinal into the device word the pack items poll (stream order = arrival order).  D2H:
 * this thread follows the unpack items' per-plane flags in host-mapped memory and releases a chunk's copy as soon as
 * all its planes carry the run's epoch.  *stuck = the launch ended without finishing a chunk.
 */
int clapca::api::stream_volume(const StreamPlan &sp, bool *stuck)
{
    const int nchunks = (sp.Z + sp.chunk - 1) / sp.chunk;
    for (int c = 0; c < nchunks; c++) {
        const size_t off = (size_t)c * sp.chunk * sp.plane_bytes;
        const size_t len = (size_t)std::min(sp.chunk, sp.Z - c * sp.chunk) * sp.plane_bytes;
        CU(cudaMemcpyAsync(sp.d_cells + off, sp.host_in + off, len, cudaMemcpyHostToDevice, sp.s_in));
        CU(cudaMemcpyAsync(sp.d_in_ready, sp.h_io + sp.Z + c, sizeof(int), cudaMemcpyHostToDevice, sp.s_in));
    }
    volatile const int *flag = sp.h_io;
    bool kernel_done = false;
    unsigned spins = 0;
    *stuck = false;
    for (int c = 0; c < nchunks && !*stuck;) {
        const int z0 = c * sp.chunk, z1 = std::min(sp.Z, z0 + sp.chunk);
        bool ready = true;
        for (int z = z0; z < z1; z++)
            if (flag[z] != sp.epoch) { ready = false; break; }
        if (ready) {
            const size_t off = (size_t)z0 * sp.plane_bytes;
            CU(cudaMemcpyAsync(sp.host_out + off, sp.d_cells + off, (size_t)(z1 - z0) * sp.plane_bytes,
                               cudaMemcpyDeviceToHost, sp.s_out));
            c++;
            continue;
        }
        if (kernel_done) { *stuck = true; break; }      /* the launch ended without finishing this chunk */
        if ((++spins & 255u) == 0u) {
            cudaError_t e = cudaStreamQuery(sp.s_kernel);
            if (e == cudaSuccess) kernel_done = true;   /* one more look at the flags, then give up */
            else if (e != cudaErrorNotReady) return fail(CLAPCA_ERR_CUDA, "streamed run: %s", cudaGetErrorString(e));
        }
        cpu_relax();
    }
    CU(cudaStreamSynchronize(sp.s_in));
    CU(cudaStreamSynchronize(sp.s_out));
    return CLAPCA_OK;
}

extern "C" {
#pragma GCC visibility push(default)

/*
 * The bit-plane engine on a device-resident grid.  io == nullptr: the cells are in g->cells and the result
 * goes back there.  io != nullptr ("streamed"): the cells are in pinned HOST memory; upload, every generation
 * and download run as one pipeline inside a single sweep launch (layout items, ca3d_bitplane.cuh): chunks of
 * planes are copied in on one copy stream, each followed by a 4-byte copy that tells the kernel's pack items
 * the chunk has landed, and the calling thread issues a chunk's D2H copy on a second copy stream as soon as
 * the kernel's unpack items have flagged all of its planes in host-mapped memory.
 */
static int run3d_bitplane(clapca_grid *g, uint32_t surv, uint32_t born, uint32_t nr_states, int steps,
                          int64_t *population, const StreamIO *io)
{
    const int W = (int)g->d0, H = (int)g->d1, Z = (int)g->d2;
    const int WPL = bp_wpl_for(W);
    const uint32_t bornval = (nr_states - 1u) & 0xffu;

    CU(cudaEventRecord(g->ev[0], g->stream));
    /*
     * The largest value that can ever occur decides the number of state planes.  Streamed runs take the caller's
     * bound (the pack items verify it: err = 4).  Resident runs with separate layout kernels pack SPECULATIVELY with
     * the planes the rule alone needs (a running automaton holds values below nr_states) and let the pack kernel
     * report cells that do not fit; only then -- seeds with other values, e.g. the 255s ca3d_prune() leaves
     * (core/ca3d.c:41-59) -- the volume is scanned for its maximum and packed again.  The scan would cost every run
     * a pass over the volume (1.4 ms at 2048^3), the wasted pack only the rare one.
     */
    const bool fused_cfg = io != nullptr || fused_layout_default();
    const bool speculate = !fused_cfg;
    unsigned maxv = 0;
    if (io) {
        maxv = io->max_value;
    } else if (!speculate) {
        CU(cudaMemsetAsync(g_ctx.d_max, 0, sizeof(unsigned), g->stream));
        max_u8_kernel<<<grid_blocks_for((g->n + 15) / 16, 256), 256, 0, g->stream>>>(g->cells, g->n, g_ctx.d_max);
        CU(cudaGetLastError());
        CU(cudaMemcpyAsync(&maxv, g_ctx.d_max, sizeof(maxv), cudaMemcpyDeviceToHost, g->stream));
        CU(cudaStreamSynchronize(g->stream));
    }
    if (born && bornval > maxv) maxv = bornval;
    if (speculate && !born && bornval > maxv) maxv = bornval;      /* the same guess for a rule that gives no birth */
    int P = bp_planes_for(maxv);
    int packed = 0;                     /* kernels spent on the layout before the sweep */
    if (speculate) {
        const int RWPs = 32 * WPL;
        size_t bytes = (size_t)Z * H * (P + 2) * RWPs * sizeof(uint32_t);
        void *rp = g->rows;
        if (int rc = ensure_bytes(&rp, &g->rows_bytes, bytes)) { g->rows = nullptr; return rc; }
        g->rows = (uint32_t *)rp;
        unsigned over = 0;
        if (P < 8) {
            CU(cudaMemsetAsync(g_ctx.d_max, 0, sizeof(unsigned), g->stream));
            Bp3Layout Ls = { g->cells, g->rows, W, H, Z, P, RWPs, g_ctx.d_count, g_ctx.d_max };
            CU(launch_ca3d_pack(Ls, g->stream));
            CU(cudaMemcpyAsync(&over, g_ctx.d_max, sizeof(over), cudaMemcpyDeviceToHost, g->stream));
            CU(cudaStreamSynchronize(g->stream));
            packed = 1;
        }
        if (over || P >= 8) {
            if (over) {
                CU(cudaMemsetAsync(g_ctx.d_max, 0, sizeof(unsigned), g->stream));
                max_u8_kernel<<<grid_blocks_for((g->n + 15) / 16, 256), 256, 0, g->stream>>>(g->cells, g->n, g_ctx.d_max);
                CU(cudaGetLastError());
                unsigned m2 = 0;
                CU(cudaMemcpyAsync(&m2, g_ctx.d_max, sizeof(m2), cudaMemcpyDeviceToHost, g->stream));
                CU(cudaStreamSynchronize(g->stream));
                maxv = std::max(maxv, m2);
                P = bp_planes_for(maxv);
                packed++;
            }
            bytes = (size_t)Z * H * (P + 2) * RWPs * sizeof(uint32_t);
            rp = g->rows;
            if (int rc = ensure_bytes(&rp, &g->rows_bytes, bytes)) { g->rows = nullptr; return rc; }
            g->rows = (uint32_t *)rp;
            Bp3Layout Ls = { g->cells, g->rows, W, H, Z, P, RWPs, g_ctx.d_count, nullptr };
            CU(launch_ca3d_pack(Ls, g->stream));
            packed++;
        }
    }
    const int NP = P + 2, RWP = 32 * WPL;

    int rule = BP3_RULE_DYN;
    for (int i = 0; i < 9; i++)
        if (kCas[i][0] == surv && kCas[i][1] == born && kCas[i][2] == nr_states) { rule = i; break; }

    size_t rows_bytes = (size_t)Z * H * NP * RWP * sizeof(uint32_t);
    {
        void *p = g->rows;
        if (int rc = ensure_bytes(&p, &g->rows_bytes, rows_bytes)) { g->rows = nullptr; return rc; }
        g->rows = (uint32_t *)p;
    }

    int team = team_config(P, WPL, io == nullptr);
    /* CLAPCA_STREAM_TEAM: team size of streamed runs only (the output lags the input by (team + 1) planes per generation) */
    if (io)
        if (const char *e = getenv("CLAPCA_STREAM_TEAM")) team = std::max(0, std::min(atoi(e), bp3_team_cap(P, WPL)));
    /* layout items need whole-plane items and all generations in one launch */
    bool fused = fused_cfg;
    if (fused && steps > kMaxFusedGenerations) {
        if (io) return fail(CLAPCA_ERR_UNSUPPORTED, "streamed run: at most %d generations", kMaxFusedGenerations);
        fused = false;
    }

    unsigned long long *d_pop = g_ctx.d_count;
    Bp3Layout L = { g->cells, g->rows, W, H, Z, P, RWP, d_pop };
    const size_t plane_bytes = (size_t)W * H;
    const int chunk = io_chunk_planes(plane_bytes, Z);
    const int nchunks = (Z + chunk - 1) / chunk;

    if (io) {
        if (!g->d_in_ready) CU(cudaMalloc(&g->d_in_ready, 64));
        if (!g->ev_io) CU(cudaEventCreateWithFlags(&g->ev_io, cudaEventDisableTiming));
        const size_t want = (size_t)Z + nchunks;
        if (g->h_io_count < want) {
            if (g->h_io) cudaFreeHost(g->h_io);
            g->h_io = nullptr;
            g->h_io_count = 0;
            CU(cudaHostAlloc((void **)&g->h_io, want * sizeof(int), cudaHostAllocMapped | cudaHostAllocPortable));
            memset(g->h_io, 0, want * sizeof(int));
            g->h_io_count = want;
            g->io_epoch = 0;
        }
        for (int c = 0; c < nchunks; c++) g->h_io[Z + c] = c + 1;
        g->io_epoch++;
    }

    if (!fused && !speculate) {
        CU(launch_ca3d_pack(L, g->stream));
        packed = 2;                     /* max scan + pack */
    }
    CU(cudaEventRecord(g->ev[1], g->stream));

    int launches = 0, workers = 0;
    for (int done = 0; done < steps;) {
        const int G = std::min(steps - done, kMaxFusedGenerations);
        {
            /* [G + 1][Z]: row 0 is "generation -1" (the pack items of a fused run), p.prog points at row 1 */
            size_t have = g->prog_count * sizeof(int);
            void *p = g->prog;
            if (int rc = ensure_bytes(&p, &have, (size_t)(G + 1) * Z * sizeof(int))) { g->prog = nullptr; return rc; }
            g->prog = (int *)p;
            g->prog_count = have / sizeof(int);
        }
        int *prog = g->prog + Z;
        /* per-plane source descriptors: on one GPU every neighbour plane is local (one z-block, no ghosts) */
        std::vector<Bp3Plane> planes;
        {
            SlabGeom geo = { Z, 1, 0, Z };
            SlabPtrs ptr = { g->rows, prog, nullptr, nullptr, nullptr };
            HaloLayout hl = slab_halo_layout(geo, H, RWP, NP, 1);
            bp3_build_planes(geo, ptr, hl, H, RWP, NP, planes);
        }
        if (g->planes_rows != g->rows || g->planes_prog != prog || g->planes_NP != NP || g->planes_RWP != RWP ||
            g->planes_bytes < planes.size() * sizeof(Bp3Plane)) {
            void *p = g->planes;
            if (int rc = ensure_bytes(&p, &g->planes_bytes, planes.size() * sizeof(Bp3Plane))) {
                g->planes = nullptr;
                return rc;
            }
            g->planes = (Bp3Plane *)p;
            CU(cudaMemcpyAsync(g->planes, planes.data(), planes.size() * sizeof(Bp3Plane), cudaMemcpyHostToDevice,
                               g->stream));
            CU(cudaStreamSynchronize(g->stream));
            g->planes_rows = g->rows; g->planes_prog = prog; g->planes_NP = NP; g->planes_RWP = RWP;
        }
        /*
         * Claim order (bp_plan.h).  Default: time-key order.  Measured on B200 at 2048^3 x 50
         * (profiles/r01_knobs_order_ca3d_2048.txt): the generation-batched diagonals (CLAPCA_ORDER=2) cut DRAM
         * traffic from 493 GB to 127-221 GB per run but not the run time (122 ms either way at batch 16, slower
         * for smaller batches and for smaller volumes) -- the kernel is bound by the ALU pipe (LOP3), not by HBM.
         * CLAPCA_ORDER=1 selects the skewed row segments; CLAPCA_GEN_BATCH / CLAPCA_SEG_ROWS tune them.
         */
        Bp3Params knobs;
        memset(&knobs, 0, sizeof(knobs));
        sweep_knobs(knobs, team, true);
        OrderCfg oc = order_config(Z, H, G, bp3_max_workers(rule, P, WPL, g_ctx.sms, team, knobs.max_ctas), team);
        /* layout items: the unpack items of a plane sit one group distance behind its last generation -- a streamed
           run wants its output to follow its input closely (DESIGN 4a), so the groups stay interleaved there */
        if (fused && oc.mode == 3 && !getenv("CLAPCA_TILE_SKEW")) {
            oc.tile_skew = 0;
            knobs.prefetch_rows = 0;
        }
        if (fused && oc.mode != 0 && oc.mode != 3) {
            if (io) oc.mode = 0;                    /* layout items exist for whole-plane orders only */
            else return fail(CLAPCA_ERR_UNSUPPORTED, "CLAPCA_FUSED_LAYOUT needs the time-key or the tile order");
        }
        if (oc.mode == 3)
            oc.tile_g = bp3_tile_shape(planes, H, G, team, oc.tile_g, oc.ctas, fused, &oc.tile_z, oc.tile_skew);
        const int okey = oc.key() + (fused ? 50000000 : 0);
        if (g->order_Z != Z || g->order_H != H || g->order_G != G || g->order_L != okey) {
            std::vector<WorkItem> items;
            make_items(oc, planes, Z, H, G, items, fused);
            static_assert(sizeof(WorkItem) == sizeof(int4), "WorkItem must alias int4");
            void *p = g->order;
            if (int rc = ensure_bytes(&p, &g->order_bytes, items.size() * sizeof(int4))) { g->order = nullptr; return rc; }
            g->order = (int4 *)p;
            CU(cudaMemcpyAsync(g->order, items.data(), items.size() * sizeof(int4), cudaMemcpyHostToDevice,
                               g->stream));
            CU(cudaStreamSynchronize(g->stream));       /* `items` is a stack vector */
            g->n_items = (int)items.size();
            g->order_Z = Z; g->order_H = H; g->order_G = G; g->order_L = okey;
        }
        CU(cudaMemsetAsync(g->prog, 0, (size_t)(G + 1) * Z * sizeof(int), g->stream));
        CU(cudaMemsetAsync(g->ticket, 0, kTicketWords * sizeof(unsigned), g->stream));

        Bp3Params p;
        memset(&p, 0, sizeof(p));
        p.rows = g->rows;
        p.planes = g->planes;
        p.W = W; p.H = H; p.Z = Z; p.G = G; p.RWP = RWP;
        p.prog = prog;
        p.order = g->order;
        p.nsweeps = g->n_items;
        p.zeros = g_ctx.d_zeros;
        sweep_knobs(p, team, !fused);
        p.ticket = g->ticket;
        p.err = (int *)(g->ticket + 1);
        p.diag = diag_enabled() ? (unsigned long long *)(g->ticket + 4) : nullptr;
        p.surv = surv; p.born = born; p.bornval = bornval;
        p.spin_limit = 4000000000LL;        /* ~2 s of SM clock in a single wait */
        if (fused) {
            p.layout_items = 1;
            p.io_cells = g->cells;
            p.io_chunk = chunk;
            p.population = d_pop;
            CU(cudaMemsetAsync(d_pop, 0, sizeof(unsigned long long), g->stream));
        }
        if (io) {
            int *h_io_dev = nullptr;
            CU(cudaHostGetDevicePointer((void **)&h_io_dev, g->h_io, 0));
            p.in_ready = g->d_in_ready;
            p.out_done = h_io_dev;
            p.io_epoch = g->io_epoch;
            CU(cudaMemsetAsync(g->d_in_ready, 0, sizeof(int), g->stream));
            CU(cudaEventRecord(g->ev_io, g->stream));
            CU(cudaStreamWaitEvent(g_ctx.stream_in, g->ev_io, 0));
        }
        Bp3LaunchInfo info;
        CU(bp3_launch(rule, P, WPL, p, g_ctx.sms, g->stream, &info));
        launches++;
        workers = info.workers;
        done += G;
    }
    CU(cudaEventRecord(g->ev[2], g->stream));

    if (io) {
        bool stuck = false;
        StreamPlan sp = { g->cells, io->host_in, io->host_out, plane_bytes, Z, chunk, g->d_in_ready, g->h_io, g->io_epoch,
                          g->stream, g_ctx.stream_in, g_ctx.stream_out };
        if (int rc = stream_volume(sp, &stuck)) return rc;
        CU(cudaEventRecord(g->ev[3], g->stream));
        unsigned long long pop = 0;
        int err = 0;
        CU(cudaMemcpyAsync(&pop, d_pop, sizeof(pop), cudaMemcpyDeviceToHost, g->stream));
        CU(cudaMemcpyAsync(&err, g->ticket + 1, sizeof(err), cudaMemcpyDeviceToHost, g->stream));
        CU(cudaStreamSynchronize(g->stream));
        diag_report("grid (streamed)", g->ticket, g->stream, 0);
        if (err == 4)
            return fail(CLAPCA_ERR_ARG, "streamed run: a cell value exceeds max_value = %u", io->max_value);
        if (err || stuck)
            return fail(CLAPCA_ERR_TIMEOUT, "ca3d bit-plane engine (streamed): dataflow watchdog fired (err=%d)", err);
        if (population) *population = (int64_t)pop;
        g->stats.launches = launches;
        g->stats.engine = CLAPCA_ENGINE_BITPLANE;
        g->stats.planes = P;
        g->stats.workers = workers;
        return CLAPCA_OK;
    }
    diag_report("grid", g->ticket, g->stream, 0);

    if (!fused) {
        CU(cudaMemsetAsync(d_pop, 0, sizeof(unsigned long long), g->stream));
        CU(launch_ca3d_unpack(L, g->stream));
    }
    CU(cudaEventRecord(g->ev[3], g->stream));

    unsigned long long pop = 0;
    int err = 0;
    CU(cudaMemcpyAsync(&pop, d_pop, sizeof(pop), cudaMemcpyDeviceToHost, g->stream));
    CU(cudaMemcpyAsync(&err, g->ticket + 1, sizeof(err), cudaMemcpyDeviceToHost, g->stream));
    CU(cudaStreamSynchronize(g->stream));
    if (err)
        return fail(CLAPCA_ERR_TIMEOUT, "ca3d bit-plane engine: dataflow watchdog fired (err=%d)", err);
    if (population) *population = (int64_t)pop;
    g->stats.launches = launches + (fused ? 1 : packed + 1);    /* + layout kernels before the sweep (+ unpack) */
    g->stats.engine = CLAPCA_ENGINE_BITPLANE;
    g->stats.planes = P;
    g->stats.workers = workers;
    return CLAPCA_OK;
}

/* shapes / step counts the bit-plane engine takes */
static bool bp3_supported(const clapca_grid *g, int steps)
{
    return g->d0 <= 4096 && g->d1 < (1 << 30) && g->d2 < (1 << 30) &&
           (double)g->d2 * (double)std::min(steps, kMaxFusedGenerations) < 2.0e9;
}

int clapca_grid_run3d(clapca_grid *g, uint32_t surv, uint32_t born, uint32_t nr_states, int steps, int engine,
                      int64_t *population)
{
    if (int rc = need_init()) return rc;
    if (!g) return fail(CLAPCA_ERR_ARG, "grid_run3d: NULL grid");
    if (steps < 0) return fail(CLAPCA_ERR_ARG, "grid_run3d: negative step count");
    memset(&g->stats, 0, sizeof(g->stats));
    if (steps == 0) {
        int64_t pop = 0;
        if (int rc = count_on_stream(g->cells, g->n, g->stream, &pop)) return rc;
        if (population) *population = pop;
        return CLAPCA_OK;
    }
    const bool bp_ok = bp3_supported(g, steps);
    if (engine == CLAPCA_ENGINE_AUTO)
        engine = bp_ok ? CLAPCA_ENGINE_BITPLANE : CLAPCA_ENGINE_WAVEFRONT;
    if (engine == CLAPCA_ENGINE_BITPLANE) {
        if (!bp_ok)
            return fail(CLAPCA_ERR_UNSUPPORTED, "bit-plane engine handles rows of at most 4096 cells (d0 = %lld)",
                        (long long)g->d0);
        if (int rc = run3d_bitplane(g, surv, born, nr_states, steps, population, nullptr)) return rc;
        float ms = 0;
        CU(cudaEventElapsedTime(&ms, g->ev[0], g->ev[3]));
        g->stats.total_ms = ms;
        CU(cudaEventElapsedTime(&ms, g->ev[1], g->ev[2]));
        g->stats.kernel_ms = ms;
        return CLAPCA_OK;
    }
    if (engine != CLAPCA_ENGINE_WAVEFRONT)
        return fail(CLAPCA_ERR_ARG, "grid_run3d: unknown engine %d", engine);
    if (int rc = run3d_wavefront(g, surv, born, nr_states, steps)) return rc;
    int64_t pop = 0;
    if (int rc = count_on_stream(g->cells, g->n, g->stream, &pop)) return rc;
    if (population) *population = pop;
    float ms = 0;
    CU(cudaEventElapsedTime(&ms, g->ev[1], g->ev[2]));
    g->stats.kernel_ms = g->stats.total_ms = ms;
    return CLAPCA_OK;
}

static bool is_pinned_host(const void *p)
{
    cudaPointerAttributes a;
    if (cudaPointerGetAttributes(&a, p) != cudaSuccess) {
        cudaGetLastError();
        return false;
    }
    return a.type == cudaMemoryTypeHost;
}

int clapca_grid_run3d_streamed(clapca_grid *g, const uint8_t *host_in, uint8_t *host_out, unsigned max_value,
                               uint32_t surv, uint32_t born, uint32_t nr_states, int steps, int64_t *population)
{
    if (int rc = need_init()) return rc;
    if (!g || !host_in || !host_out) return fail(CLAPCA_ERR_ARG, "grid_run3d_streamed: NULL argument");
    if (steps < 0) return fail(CLAPCA_ERR_ARG, "grid_run3d_streamed: negative step count");
    if (max_value > 255u) return fail(CLAPCA_ERR_ARG, "grid_run3d_streamed: max_value %u > 255", max_value);
    const char *e = getenv("CLAPCA_STREAMED");
    const bool pipelined = steps > 0 && steps <= kMaxFusedGenerations && bp3_supported(g, steps) &&
                           !(e && atoi(e) == 0) && is_pinned_host(host_in) && is_pinned_host(host_out);
    if (!pipelined) {
        /* pageable buffers / shapes outside the bit-plane engine: the same three steps one after the other */
        if (int rc = clapca_grid_upload(g, host_in)) return rc;
        if (int rc = clapca_grid_run3d(g, surv, born, nr_states, steps, CLAPCA_ENGINE_AUTO, population)) return rc;
        return clapca_grid_download(g, host_out);
    }
    memset(&g->stats, 0, sizeof(g->stats));
    StreamIO io = { host_in, host_out, max_value };
    if (int rc = run3d_bitplane(g, surv, born, nr_states, steps, population, &io)) return rc;
    float ms = 0;
    CU(cudaEventElapsedTime(&ms, g->ev[1], g->ev[2]));
    g->stats.kernel_ms = g->stats.total_ms = ms;
    g->stats.streamed = 1;
    return CLAPCA_OK;
}

int clapca_ca3d_run(uint8_t *arr, const int64_t dim[3], uint32_t surv, uint32_t born, uint32_t nr_states,
                    int steps, int engine, int64_t *population)
{
    if (int rc = need_init()) return rc;
    if (!arr || !dim) return fail(CLAPCA_ERR_ARG, "ca3d_run: NULL argument");
    clapca_grid *g = nullptr;
    int rc = oneshot_acquire(&g, dim[0], dim[1], dim[2]);
    if (rc) return rc;
    rc = clapca_grid_upload(g, arr);
    if (!rc) rc = clapca_grid_run3d(g, surv, born, nr_states, steps, engine, population);
    if (!rc && steps > 0) rc = clapca_grid_download(g, arr);
    oneshot_release(g);
    return rc;
}

/* ---- ca2d ------------------------------------------------------------------- */

/* the bit engines count alive bits and sweep the whole grid */
static bool alive_bit_full_sweep(const clapca_grid *g, int64_t side, int decay, int neigh)
{
    if (side < g->d0 || side < g->d1)
        return false;                       /* partial sweeps: cell-wavefront engine */
    if ((neigh == CLAPCA_NEIGH_VNV || neigh == CLAPCA_NEIGH_MV) && decay)
        return false;                       /* value-comparing counts that matter: cell-wavefront engine */
    return true;
}

/* rows are cut into at most 16 warps x 32 lanes x 4 words: 65536 cells (32768 with 8 state planes) */
static bool bp2_supported(const clapca_grid *g, int64_t side, int decay, int neigh, int P)
{
    int wpl, warps;
    return alive_bit_full_sweep(g, side, decay, neigh) && g->d0 < (1 << 30) && bp2_shape_for(g->d1, P, &wpl, &warps);
}

/* the diagonal engine: one state plane, at most 16384 columns (cells per diagonal), any number of rows an int holds */
static bool sk2_supported(const clapca_grid *g, int64_t side, int decay, int neigh, int P)
{
    int wpl, warps;
    return P == 1 && alive_bit_full_sweep(g, side, decay, neigh) && sk2_shape_for(g->d0, &wpl, &warps) && g->d1 <= (1LL << 28);
}

/* largest cell value of the grid (device reduction) */
static int grid_max_value(clapca_grid *g, unsigned *maxv)
{
    CU(cudaMemsetAsync(g_ctx.d_max, 0, sizeof(unsigned), g->stream));
    CU(launch_max_u8(g->cells, g->n, g_ctx.d_max, g->stream));
    CU(cudaMemcpyAsync(maxv, g_ctx.d_max, sizeof(*maxv), cudaMemcpyDeviceToHost, g->stream));
    CU(cudaStreamSynchronize(g->stream));
    return CLAPCA_OK;
}

/*
 * One-plane grids on the diagonal engine (ca2d_skew.cuh): no in-row chain, no CTA barrier in the sweep.  First measured
 * against the row engine on B200 at BASELINE config 3 (profiles/r02_ca2d_diagonal_ab.txt): bit-identical grids, 13.1 ms
 * against 8.9 ms.  Which engine is faster depends on the shape (and on the kernel version), so nothing is assumed:
 * CLAPCA_ENGINE_DIAGONAL or CLAPCA_2D_SKEW=1 / 0 force an engine, and otherwise the first large run of a shape class
 * MEASURES both (run2d_tune below) and later runs of the class take the faster one.
 */
enum { SK2_CHOICE_UNKNOWN = 0, SK2_CHOICE_ROW = 1, SK2_CHOICE_DIAGONAL = 2 };
static const long long kTune2MinCells = 1LL << 22;
static const int kTune2MinSteps = 16;
static std::map<std::tuple<int64_t, int64_t, int, uint32_t, uint32_t>, int> g_tune2;

static int sk2_choice(const clapca_grid *g, uint32_t born, uint32_t surv, int neigh, int steps)
{
    if (const char *e = getenv("CLAPCA_2D_SKEW"))
        return atoi(e) != 0 ? SK2_CHOICE_DIAGONAL : SK2_CHOICE_ROW;
    if (g->d0 * g->d1 < kTune2MinCells || steps < kTune2MinSteps)
        return SK2_CHOICE_ROW;
    if (const char *e = getenv("CLAPCA_2D_TUNE"))
        if (atoi(e) == 0)
            return SK2_CHOICE_ROW;
    auto it = g_tune2.find(std::make_tuple(g->d0, g->d1, neigh, born & 0x1ffu, surv & 0x1ffu));
    return it == g_tune2.end() ? SK2_CHOICE_UNKNOWN : it->second;
}

static int run2d_skew(clapca_grid *g, uint32_t born, uint32_t surv, uint32_t nr_states, int decay, int neigh, int steps)
{
    const int W = (int)g->d0, H = (int)g->d1;
    const uint32_t nrval = nr_states & 0xffu;
    const bool moore = (neigh == CLAPCA_NEIGH_M1 || neigh == CLAPCA_NEIGH_MV);
    int WPL = 0, warps = 0;
    if (!sk2_shape_for(W, &WPL, &warps))
        return fail(CLAPCA_ERR_UNSUPPORTED, "2D diagonal engine: %d cells per diagonal are too many", W);
    if (const char *e = getenv("CLAPCA_2D_SKEW_WPL")) {     /* tuning: words per lane */
        const int v = atoi(e);
        if ((v == 1 || v == 2) && sk2_warps_for(W, v) * v <= SK2_MAX_WARPS) { WPL = v; warps = sk2_warps_for(W, v); }
    }
    const int T = sk2_diagonals(W, H), TR = sk2_rows_alloc(W, H);
    const size_t rows_bytes = (size_t)TR * SK2_RS * sizeof(uint32_t);
    {
        void *p = g->rows;
        if (int rc = ensure_bytes(&p, &g->rows_bytes, rows_bytes)) { g->rows = nullptr; return rc; }
        g->rows = (uint32_t *)p;
    }
    unsigned long long *d_pop = g_ctx.d_count;
    Sk2Layout L = { g->cells, g->rows, W, H, d_pop };
    const size_t cols = (size_t)(W + 31) / 32;
    const size_t pack_tiles = cols * ((T + SK2_TILE_T - 1) / SK2_TILE_T), unpack_tiles = cols * ((H + SK2_TILE_T - 1) / SK2_TILE_T);

    CU(cudaEventRecord(g->ev[0], g->stream));
    CU(cudaMemsetAsync(g->rows, 0, rows_bytes, g->stream));         /* everything outside the band of cells stays zero */
    ca2d_skew_pack_kernel<<<grid_blocks_for(pack_tiles * 256, 256, 8), 256, 0, g->stream>>>(L);
    CU(cudaGetLastError());
    CU(cudaEventRecord(g->ev[1], g->stream));

    int launches = 0, ctas = 0;
    for (int done = 0; done < steps;) {
        const int G = std::min(steps - done, 1 << 20);
        {
            size_t have = g->prog_count * sizeof(int);
            void *p = g->prog;
            if (int rc = ensure_bytes(&p, &have, (size_t)G * sizeof(int))) { g->prog = nullptr; return rc; }
            g->prog = (int *)p;
            g->prog_count = have / sizeof(int);
            g->planes_prog = nullptr;       /* the 3D plane descriptors cached on this grid are stale now */
        }
        CU(cudaMemsetAsync(g->prog, 0, (size_t)G * sizeof(int), g->stream));
        CU(cudaMemsetAsync(g->ticket, 0, kTicketWords * sizeof(unsigned), g->stream));
        Sk2Params p;
        memset(&p, 0, sizeof(p));
        p.rows = g->rows;
        p.W = W; p.H = H; p.G = G; p.T = T;
        p.prog = g->prog;
        p.ticket = g->ticket;
        p.err = (int *)(g->ticket + 1);
        p.born = born & 0x1ffu;
        /* a cell that neither survives nor decays keeps its value: same as surviving (core/ca2d.c:72-75) */
        p.surv = decay ? (surv & 0x1ffu) : 0x1ffu;
        p.nrval = nrval;
        p.spin_limit = 4000000000LL;
        Bp2LaunchInfo info;
        CU(sk2_launch(WPL, moore, warps, p, g_ctx.sms, g->stream, &info));
        launches++;
        ctas = info.blocks;
        done += G;
    }
    CU(cudaEventRecord(g->ev[2], g->stream));
    CU(cudaMemsetAsync(d_pop, 0, sizeof(unsigned long long), g->stream));
    ca2d_skew_unpack_kernel<<<grid_blocks_for(unpack_tiles * 256, 256, 8), 256, 0, g->stream>>>(L);
    CU(cudaGetLastError());
    CU(cudaEventRecord(g->ev[3], g->stream));
    int err = 0;
    CU(cudaMemcpyAsync(&err, g->ticket + 1, sizeof(err), cudaMemcpyDeviceToHost, g->stream));
    CU(cudaStreamSynchronize(g->stream));
    if (err)
        return fail(CLAPCA_ERR_TIMEOUT, "ca2d diagonal engine: dataflow watchdog fired (err=%d)", err);
    float ms = 0;
    CU(cudaEventElapsedTime(&ms, g->ev[0], g->ev[3]));
    g->stats.total_ms = ms;
    CU(cudaEventElapsedTime(&ms, g->ev[1], g->ev[2]));
    g->stats.kernel_ms = ms;
    g->stats.launches = launches + 2;
    g->stats.engine = CLAPCA_ENGINE_DIAGONAL;
    g->stats.planes = 1;
    g->stats.workers = ctas * warps;
    return CLAPCA_OK;
}

static int run2d_bitplane(clapca_grid *g, uint32_t born, uint32_t surv, uint32_t nr_states, int decay, int neigh,
                          int steps, int P)
{
    const int W = (int)g->d0, H = (int)g->d1;       /* x extent = engine rows, y extent = cells per row */
    const uint32_t nrval = nr_states & 0xffu;
    const bool moore = (neigh == CLAPCA_NEIGH_M1 || neigh == CLAPCA_NEIGH_MV);

    int WPL = 0, warps = 0;
    if (!bp2_shape_for(H, P, &WPL, &warps))
        return fail(CLAPCA_ERR_UNSUPPORTED, "2D bit-plane engine: rows of %d cells with %d state planes are too wide", H, P);
    if (const char *e = getenv("CLAPCA_2D_WPL")) {          /* tuning: words per lane (more = fewer warps per row) */
        int v = atoi(e);
        const long long rw = (H + 31) / 32, nw = (rw + 32 * v - 1) / (32 * v);
        if ((v == 1 || v == 2 || v == 4) && nw <= 16 && !(P >= 8 && v == 4)) { WPL = v; warps = (int)(nw < 1 ? 1 : nw); }
    }
    const int RWS = warps * 32 * WPL;

    const size_t rows_bytes = (size_t)W * P * RWS * sizeof(uint32_t);
    {
        void *p = g->rows;
        if (int rc = ensure_bytes(&p, &g->rows_bytes, rows_bytes)) { g->rows = nullptr; return rc; }
        g->rows = (uint32_t *)p;
    }
    unsigned long long *d_pop = g_ctx.d_count;
    Bp2Layout L = { g->cells, g->rows, W, H, P, RWS, d_pop };
    const size_t tiles = (size_t)((W + 127) / 128) * ((H + 31) / 32);

    CU(cudaEventRecord(g->ev[0], g->stream));
    CU(cudaMemsetAsync(g->rows, 0, rows_bytes, g->stream));         /* padding words stay zero */
    ca2d_pack_kernel<<<grid_blocks_for(tiles * 32, 256, 8), 256, 0, g->stream>>>(L);
    CU(cudaGetLastError());
    CU(cudaEventRecord(g->ev[1], g->stream));

    int launches = 0, ctas = 0;
    for (int done = 0; done < steps;) {
        const int G = std::min(steps - done, 1 << 20);
        {
            size_t have = g->prog_count * sizeof(int);
            void *p = g->prog;
            if (int rc = ensure_bytes(&p, &have, (size_t)G * sizeof(int))) { g->prog = nullptr; return rc; }
            g->prog = (int *)p;
            g->prog_count = have / sizeof(int);
            g->planes_prog = nullptr;       /* the 3D plane descriptors cached on this grid are stale now */
        }
        CU(cudaMemsetAsync(g->prog, 0, (size_t)G * sizeof(int), g->stream));
        CU(cudaMemsetAsync(g->ticket, 0, kTicketWords * sizeof(unsigned), g->stream));
        Bp2Params p;
        memset(&p, 0, sizeof(p));
        p.rows = g->rows;
        p.N = H; p.M = W; p.G = G; p.RWS = RWS;
        p.prog = g->prog;
        p.ticket = g->ticket;
        p.err = (int *)(g->ticket + 1);
        p.born = born & 0x1ffu;
        /* a cell that neither survives nor decays keeps its value: same as surviving (core/ca2d.c:72-75) */
        p.surv = decay ? (surv & 0x1ffu) : 0x1ffu;
        p.nrval = nrval;
        p.flag_rows = 8;        /* measured on B200, 16384^2 x 100: 10.3 / 9.8 / 9.3 ms with 2 / 4 / 8 rows per counter update */
        if (const char *e = getenv("CLAPCA_2D_FLAG_ROWS")) { int v = atoi(e); if (v > 0) p.flag_rows = v; }
        p.spin_limit = 4000000000LL;
        Bp2LaunchInfo info;
        CU(bp2_launch(P, WPL, moore, warps, p, g_ctx.sms, g->stream, &info));
        launches++;
        ctas = info.blocks;
        done += G;
    }
    CU(cudaEventRecord(g->ev[2], g->stream));
    CU(cudaMemsetAsync(d_pop, 0, sizeof(unsigned long long), g->stream));
    ca2d_unpack_kernel<<<grid_blocks_for(tiles * 32, 256, 8), 256, 0, g->stream>>>(L);
    CU(cudaGetLastError());
    CU(cudaEventRecord(g->ev[3], g->stream));
    int err = 0;
    CU(cudaMemcpyAsync(&err, g->ticket + 1, sizeof(err), cudaMemcpyDeviceToHost, g->stream));
    CU(cudaStreamSynchronize(g->stream));
    if (err)
        return fail(CLAPCA_ERR_TIMEOUT, "ca2d bit-plane engine: dataflow watchdog fired (err=%d)", err);
    float ms = 0;
    CU(cudaEventElapsedTime(&ms, g->ev[0], g->ev[3]));
    g->stats.total_ms = ms;
    CU(cudaEventElapsedTime(&ms, g->ev[1], g->ev[2]));
    g->stats.kernel_ms = ms;
    g->stats.launches = launches + 2;
    g->stats.engine = CLAPCA_ENGINE_BITPLANE;
    g->stats.planes = P;
    g->stats.workers = ctas * warps;
    return CLAPCA_OK;
}

/*
 * First large run of a shape class under AUTO / BITPLANE: measure both engines on this very input, over at most
 * kTune2Gens generations.  Each engine runs twice from a scratch copy of the input (the second run is the timed one:
 * the first launch of a kernel pays its module load); then the input comes back and the ROW engine does the caller's
 * run -- the first call of a class never depends on the outcome.  The diagonal engine is chosen for later runs of
 * the class only if its grid had the same fingerprint as the row engine's and its run was faster (pack + sweep +
 * unpack, CUDA events).
 */
static const int kTune2Gens = 32;
static int run2d_tune(clapca_grid *g, uint32_t born, uint32_t surv, uint32_t nr_states, int decay, int neigh, int steps, int P)
{
    const auto key = std::make_tuple(g->d0, g->d1, neigh, born & 0x1ffu, surv & 0x1ffu);
    const int gens = std::min(steps, kTune2Gens);
    void *copy = nullptr;
    if (cudaMalloc(&copy, g->n) != cudaSuccess) {
        (void)cudaGetLastError();               /* no room for the scratch copy: no measurement, the proven engine */
        g_tune2[key] = SK2_CHOICE_ROW;
        return run2d_bitplane(g, born, surv, nr_states, decay, neigh, steps, P);
    }
    int choice = SK2_CHOICE_ROW;
    float ms_diag = 0.f, ms_row = 0.f;
    uint64_t h_diag = 0, h_row = 1;
    bool diag_ok = true, row_ok = true;
    cudaError_t e = cudaMemcpyAsync(copy, g->cells, g->n, cudaMemcpyDeviceToDevice, g->stream);
    for (int i = 0; i < 2 && e == cudaSuccess && diag_ok; i++) {
        if (i) e = cudaMemcpyAsync(g->cells, copy, g->n, cudaMemcpyDeviceToDevice, g->stream);
        if (e == cudaSuccess)
            diag_ok = run2d_skew(g, born, surv, nr_states, decay, neigh, gens) == CLAPCA_OK;
        ms_diag = g->stats.total_ms;
    }
    if (e == cudaSuccess && diag_ok)
        diag_ok = clapca_hash_planes(g->cells, g->n, 1, &h_diag) == CLAPCA_OK;
    for (int i = 0; i < 2 && e == cudaSuccess && row_ok; i++) {
        e = cudaMemcpyAsync(g->cells, copy, g->n, cudaMemcpyDeviceToDevice, g->stream);
        if (e == cudaSuccess)
            row_ok = run2d_bitplane(g, born, surv, nr_states, decay, neigh, gens, P) == CLAPCA_OK;
        ms_row = g->stats.total_ms;
    }
    if (e == cudaSuccess && row_ok && diag_ok && clapca_hash_planes(g->cells, g->n, 1, &h_row) == CLAPCA_OK &&
        h_row == h_diag && ms_diag < 0.98f * ms_row)       /* a clear win, not measurement noise */
        choice = SK2_CHOICE_DIAGONAL;
    if (e == cudaSuccess)
        e = cudaMemcpyAsync(g->cells, copy, g->n, cudaMemcpyDeviceToDevice, g->stream);
    if (e == cudaSuccess)
        e = cudaStreamSynchronize(g->stream);
    cudaFree(copy);
    if (e != cudaSuccess)
        return fail(CLAPCA_ERR_CUDA, "grid_run2d (engine measurement): %s", cudaGetErrorString(e));
    g_tune2[key] = choice;
    if (getenv("CLAPCA_VERBOSE"))
        fprintf(stderr, "clapca: 2D engines on %lld x %lld, %d generations: diagonal %.3f ms%s, row %.3f ms -> %s\n",
                (long long)g->d0, (long long)g->d1, gens, ms_diag,
                diag_ok ? (h_row == h_diag ? "" : " (DIFFERENT GRID)") : " (failed)", ms_row,
                choice == SK2_CHOICE_DIAGONAL ? "diagonal" : "row");
    return run2d_bitplane(g, born, surv, nr_states, decay, neigh, steps, P);
}

int clapca_grid_run2d(clapca_grid *g, int64_t side, uint32_t born, uint32_t surv, uint32_t nr_states, int decay,
                      int neigh, int steps, int engine)
{
    if (int rc = need_init()) return rc;
    if (!g) return fail(CLAPCA_ERR_ARG, "grid_run2d: NULL grid");
    if (g->d2 != 1) return fail(CLAPCA_ERR_ARG, "grid_run2d: grid is not 2D (d2 = %lld)", (long long)g->d2);
    if (neigh < CLAPCA_NEIGH_VN1 || neigh > CLAPCA_NEIGH_MV)
        return fail(CLAPCA_ERR_ARG, "grid_run2d: unknown neighbourhood %d", neigh);
    if (steps < 0) return fail(CLAPCA_ERR_ARG, "grid_run2d: negative step count");
    memset(&g->stats, 0, sizeof(g->stats));
    if (steps == 0 || side <= 0)
        return CLAPCA_OK;
    /*
     * The number of state planes -- and with it the widest row the bit-plane engine takes (32768 cells with 8 planes,
     * 65536 below) -- depends on the largest value that can occur: scan the data BEFORE choosing the engine, so that
     * AUTO falls back to the cell-wavefront engine instead of failing (the reference handles any size).
     */
    int P = 3;
    if (engine != CLAPCA_ENGINE_WAVEFRONT) {
        unsigned maxv = 0;
        if (int rc = grid_max_value(g, &maxv)) return rc;
        if (born && (nr_states & 0xffu) > maxv) maxv = nr_states & 0xffu;
        P = bp2_planes_for(maxv);
    }
    const bool bp_ok = engine != CLAPCA_ENGINE_WAVEFRONT && bp2_supported(g, side, decay, neigh, P);
    const bool sk_ok = engine != CLAPCA_ENGINE_WAVEFRONT && sk2_supported(g, side, decay, neigh, P);
    if (engine == CLAPCA_ENGINE_AUTO)
        engine = bp_ok ? CLAPCA_ENGINE_BITPLANE : CLAPCA_ENGINE_WAVEFRONT;
    if (engine == CLAPCA_ENGINE_DIAGONAL) {
        if (!sk_ok)
            return fail(CLAPCA_ERR_UNSUPPORTED, "2D diagonal engine: needs a full sweep (side >= extent), cell values 0 / 1, at "
                        "most 16384 columns and an alive-bit neighbourhood (vnv/mv only without decay)");
        return run2d_skew(g, born, surv, nr_states, decay, neigh, steps);
    }
    if (engine == CLAPCA_ENGINE_BITPLANE) {
        if (!bp_ok)
            return fail(CLAPCA_ERR_UNSUPPORTED, "2D bit-plane engine: needs a full sweep (side >= extent), rows of at "
                        "most 65536 cells (32768 with values >= 16) and an alive-bit neighbourhood (vnv/mv only without decay)");
        const int choice = sk_ok ? sk2_choice(g, born, surv, neigh, steps) : SK2_CHOICE_ROW;
        if (choice == SK2_CHOICE_UNKNOWN)
            return run2d_tune(g, born, surv, nr_states, decay, neigh, steps, P);
        if (choice == SK2_CHOICE_DIAGONAL)
            return run2d_skew(g, born, surv, nr_states, decay, neigh, steps);
        return run2d_bitplane(g, born, surv, nr_states, decay, neigh, steps, P);
    }
    if (engine != CLAPCA_ENGINE_WAVEFRONT)
        return fail(CLAPCA_ERR_ARG, "grid_run2d: unknown engine %d", engine);

    Wf2Params p;
    p.a = g->cells;
    p.w = g->d0; p.h = g->d1;
    p.sx = std::min<long long>(side, g->d0);
    p.sy = std::min<long long>(side, g->d1);
    p.born = born; p.surv = surv; p.nrval = nr_states & 0xffu;
    p.decay = decay ? 1 : 0; p.neigh = neigh; p.G = steps;
    int per_sm = 0;
    CU(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, ca2d_wavefront_kernel, 256, 0));
    if (per_sm < 1) return fail(CLAPCA_ERR_CUDA, "ca2d_wavefront_kernel does not fit on an SM");
    int blocks = (int)std::min<size_t>(((size_t)p.sx + 255) / 256, (size_t)per_sm * g_ctx.sms);
    if (blocks < 1) blocks = 1;
    void *args[] = { &p };
    CU(cudaEventRecord(g->ev[1], g->stream));
    CU(cudaLaunchCooperativeKernel((void *)ca2d_wavefront_kernel, dim3(blocks), dim3(256), args, 0, g->stream));
    CU(cudaEventRecord(g->ev[2], g->stream));
    CU(cudaStreamSynchronize(g->stream));
    float ms = 0;
    CU(cudaEventElapsedTime(&ms, g->ev[1], g->ev[2]));
    g->stats.kernel_ms = g->stats.total_ms = ms;
    g->stats.launches = 1;
    g->stats.engine = CLAPCA_ENGINE_WAVEFRONT;
    g->stats.workers = blocks * 256;
    return CLAPCA_OK;
}

int clapca_ca2d_run(uint8_t *arr, int64_t w, int64_t h, int64_t side, uint32_t born, uint32_t surv,
                    uint32_t nr_states, int decay, int neigh, int steps, int engine)
{
    if (int rc = need_init()) return rc;
    if (!arr) return fail(CLAPCA_ERR_ARG, "ca2d_run: NULL array");
    clapca_grid *g = nullptr;
    int rc = oneshot_acquire(&g, w, h, 1);
    if (rc) return rc;
    rc = clapca_grid_upload(g, arr);
    if (!rc) rc = clapca_grid_run2d(g, side, born, surv, nr_states, decay, neigh, steps, engine);
    if (!rc && steps > 0) rc = clapca_grid_download(g, arr);
    oneshot_release(g);
    return rc;
}

/*
 * Seeding loop of ca2d_generate() (core/ca2d.c:86-90) on the device: draw k = x*side + y of the caller's
 * lrand48() stream decides cell (x,y).  Cells outside side x side are zero, like the reference's fresh xyarray.
 */
int clapca_grid_seed2d(clapca_grid *g, int64_t side, uint32_t nr_states, uint64_t rand48_state,
                       uint64_t *rand48_state_after)
{
    if (int rc = need_init()) return rc;
    if (!g) return fail(CLAPCA_ERR_ARG, "grid_seed2d: NULL grid");
    if (g->d2 != 1 || side < 0 || side > g->d0 || side > g->d1 || side > 46340)
        return fail(CLAPCA_ERR_ARG, "grid_seed2d: side %lld does not fit the %lld x %lld grid", (long long)side,
                    (long long)g->d0, (long long)g->d1);
    rand48_state &= (1ull << 48) - 1;
    if (side != g->d0 || side != g->d1)
        CU(cudaMemsetAsync(g->cells, 0, g->n, g->stream));
    if (side > 0) {
        dim3 grid((unsigned)((side + 31) / 32), (unsigned)((side + 255) / 256));
        ca2d_seed_kernel<<<grid, 256, 0, g->stream>>>(g->cells, (int)g->d0, (int)side, nr_states,
                                                      (unsigned long long)rand48_state);
        CU(cudaGetLastError());
    }
    CU(cudaStreamSynchronize(g->stream));
    if (rand48_state_after)
        *rand48_state_after = r48_advance(rand48_state, (unsigned long long)side * (unsigned long long)side);
    return CLAPCA_OK;
}

/*
 * ca3d_make() (core/ca3d.c:144-169) into a device-resident grid.  The faces and the prune are kernels
 * (ca3d_layout.cuh); ca3d_walk() (:63-99) is a serial chain of data-dependent lrand48() draws and runs here, on the
 * host, against a SPARSE picture of the volume: before the prune a cell is occupied iff it lies on a face or the walk
 * has been there, so the walk needs a hash set of its own cells, not the 8.6 GB volume.  Quirks kept: HIST_SIZE /
 * TRIES, the history that stops growing when it is full; the undefined history[-1] read of the reference on an empty
 * history is "stay put", as in the host shim and the oracle port.
 */
int clapca_grid_make3d(clapca_grid *g, uint64_t rand48_state, uint64_t *rand48_state_after, int64_t *population)
{
    if (int rc = need_init()) return rc;
    if (!g) return fail(CLAPCA_ERR_ARG, "grid_make3d: NULL grid");
    const long long d0 = g->d0, d1 = g->d1, d2 = g->d2;
    if (d0 < 1 || d1 < 1 || d2 < 1 || d0 > 46340 || d1 > 46340 || d2 > 46340)
        return fail(CLAPCA_ERR_ARG, "grid_make3d: bad extents");
    unsigned long long st = rand48_state & ((1ull << 48) - 1ull);
    auto next = [&st]() -> long {
        st = (st * 0x5DEECE66Dull + 0xBull) & ((1ull << 48) - 1ull);
        return (long)(st >> 17);
    };
    /* min3(d0 * d1, d1 * d2, d0 * d2) in the reference's int arithmetic (extents are bounded above) */
    const long long steps = std::min(std::min(d0 * d1, d1 * d2), d0 * d2);
    auto on_face = [&](long long x, long long y, long long z) {
        return x == 0 || y == 0 || z == 0 || x == d0 - 1 || y == d1 - 1 || z == d2 - 1;
    };
    auto index = [&](long long x, long long y, long long z) { return (unsigned long long)((z * d1 + y) * d0 + x); };
    std::unordered_set<unsigned long long> seen;
    std::vector<unsigned long long> walked;
    seen.reserve((size_t)std::min<long long>(steps, 1 << 24) * 2);
    {
        enum { HISTORY = 128, ATTEMPTS = 12 };
        long long trail[HISTORY][3], at[3] = { d0 / 2, d1 / 2, d2 / 2 };
        int depth = 0;
        for (long long s = 0; s < steps; s++) {
            long long to[3] = { 0, 0, 0 };
            int k;
            if (seen.insert(index(at[0], at[1], at[2])).second)
                walked.push_back(index(at[0], at[1], at[2]));
            for (k = 0; k < ATTEMPTS; k++) {
                to[0] = at[0]; to[1] = at[1]; to[2] = at[2];
                const int axis = (int)(next() % 3);
                const int delta = (next() & 1) ? 1 : -1;
                to[axis] += delta;
                const bool valid = to[0] >= 0 && to[1] >= 0 && to[2] >= 0 && to[0] < d0 && to[1] < d1 && to[2] < d2;
                if (valid && !on_face(to[0], to[1], to[2]) && !seen.count(index(to[0], to[1], to[2])))
                    break;
            }
            if (k == ATTEMPTS) {
                if (depth > 0) {
                    depth--;
                    at[0] = trail[depth][0]; at[1] = trail[depth][1]; at[2] = trail[depth][2];
                }
                continue;
            }
            if (depth == HISTORY)
                continue;
            trail[depth][0] = to[0]; trail[depth][1] = to[1]; trail[depth][2] = to[2];
            depth++;
            at[0] = to[0]; at[1] = to[1]; at[2] = to[2];
        }
    }
    if (rand48_state_after) *rand48_state_after = st;

    CU(cudaMemsetAsync(g->cells, 0, g->n, g->stream));
    make3d_faces_kernel<<<grid_blocks_for((size_t)d1 * d2, 256, 8), 256, 0, g->stream>>>(g->cells, (int)d0, (int)d1, (int)d2);
    CU(cudaGetLastError());
    if (!walked.empty()) {
        const size_t bytes = walked.size() * sizeof(unsigned long long);
        if (int rc = ensure_bytes(&g_ctx.scratch[3], &g_ctx.scratch_bytes[3], bytes)) return rc;
        CU(cudaMemcpyAsync(g_ctx.scratch[3], walked.data(), bytes, cudaMemcpyHostToDevice, g->stream));
        make3d_scatter_kernel<<<grid_blocks_for(walked.size(), 256, 8), 256, 0, g->stream>>>(
            g->cells, (const unsigned long long *)g_ctx.scratch[3], walked.size());
        CU(cudaGetLastError());
        CU(cudaStreamSynchronize(g->stream));           /* `walked` is a local */
    }
    /* ca3d_prune(): passes until no empty cell turns occupied any more (almost always two) */
    for (int pass = 0;; pass++) {
        unsigned changed = 0;
        CU(cudaMemsetAsync(g_ctx.d_max, 0, sizeof(unsigned), g->stream));
        make3d_prune_kernel<<<grid_blocks_for(g->n, 256, 16), 256, 0, g->stream>>>(g->cells, (int)d0, (int)d1, (int)d2,
                                                                                  g_ctx.d_max);
        CU(cudaGetLastError());
        CU(cudaMemcpyAsync(&changed, g_ctx.d_max, sizeof(changed), cudaMemcpyDeviceToHost, g->stream));
        CU(cudaStreamSynchronize(g->stream));
        if (!changed)
            break;
        if (pass > 100000)
            return fail(CLAPCA_ERR_STATE, "grid_make3d: the prune did not settle");
    }
    unsigned long long pop = 0;
    CU(cudaMemsetAsync(g_ctx.d_count, 0, sizeof(unsigned long long), g->stream));
    make3d_finish_kernel<<<grid_blocks_for(g->n, 256, 16), 256, 0, g->stream>>>(g->cells, g->n, g_ctx.d_count);
    CU(cudaGetLastError());
    CU(cudaMemcpyAsync(&pop, g_ctx.d_count, sizeof(pop), cudaMemcpyDeviceToHost, g->stream));
    CU(cudaStreamSynchronize(g->stream));
    if (population) *population = (int64_t)pop;
    return CLAPCA_OK;
}

int clapca_ca2d_generate(uint8_t *arr, int64_t side, uint32_t born, uint32_t surv, uint32_t nr_states, int decay,
                         int neigh, int steps, int engine, uint64_t rand48_state, uint64_t *rand48_state_after)
{
    if (int rc = need_init()) return rc;
    if (!arr || side < 1) return fail(CLAPCA_ERR_ARG, "ca2d_generate: bad arguments");
    clapca_grid *g = nullptr;
    int rc = oneshot_acquire(&g, side, side, 1);
    if (rc) return rc;
    rc = clapca_grid_seed2d(g, side, nr_states, rand48_state, rand48_state_after);
    if (!rc && steps > 0) rc = clapca_grid_run2d(g, side, born, surv, nr_states, decay, neigh, steps, engine);
    if (!rc) rc = clapca_grid_download(g, arr);
    oneshot_release(g);
    return rc;
}


/* ---- fields ------------------------------------------------------------------- */

void *clapca_device_alloc(size_t bytes)
{
    void *p = nullptr;
    if (g_ctx.device < 0 || cudaMalloc(&p, bytes) != cudaSuccess) {
        cudaGetLastError();
        return nullptr;
    }
    return p;
}

int clapca_device_free(void *p)
{
    if (p) CU(cudaFree(p));
    return CLAPCA_OK;
}

int clapca_memcpy_h2d(void *dst, const void *src, size_t bytes)
{
    if (int rc = need_init()) return rc;
    CU(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyHostToDevice, g_ctx.stream));
    CU(cudaStreamSynchronize(g_ctx.stream));
    return CLAPCA_OK;
}

int clapca_memcpy_d2h(void *dst, const void *src, size_t bytes)
{
    if (int rc = need_init()) return rc;
    CU(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDeviceToHost, g_ctx.stream));
    CU(cudaStreamSynchronize(g_ctx.stream));
    return CLAPCA_OK;
}

#pragma GCC visibility pop
} /* extern "C" */
