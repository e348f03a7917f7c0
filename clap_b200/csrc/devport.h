/*
 * devport.h -- the handful of CUDA device primitives the CA kernels use, with a
 * second implementation for the host-side *kernel emulator* (tests/emu/).
 *
 * Product builds (nvcc, sm_100a) see only the CUDA branch.  The emulator branch
 * (-DCLAPCA_EMU, g++) runs the very same kernel source on the CPU: every warp
 * is a ring of 32 ucontext fibers, warp collectives are rendez-vous points
 * between the fibers, and persistent warps run on separate OS threads so the
 * flag-based dataflow protocol is exercised with real concurrency.  It is test
 * infrastructure for the `-m "not gpu"` suite; it is never linked into
 * libclapca_cuda and there is no CPU fallback in the product.
 */
#ifndef CLAPCA_DEVPORT_H
#define CLAPCA_DEVPORT_H

#include <stdint.h>

#ifndef CLAPCA_EMU
/* ------------------------------------------------------------------ CUDA -- */
#include <cuda_runtime.h>

#define CA_DEV      __device__ __forceinline__
#define CA_MDEV     __device__ __forceinline__ static      /* static member function */
#define CA_MEMBER   __device__ __forceinline__             /* non-static member function */
#define CA_MCOLD    __device__ __noinline__ static          /* static member function kept out of line (cold paths) */
#define CA_HOSTDEV  __host__ __device__ __forceinline__
#define CA_GLOBAL   __global__
#define CA_FULL     0xffffffffu
#define CA_SHARED(type, name, n) __shared__ type name[n]

namespace clapca {

CA_DEV int  dp_lane()            { return (int)(threadIdx.x & 31); }
CA_DEV int  dp_warp_in_block()   { return (int)(threadIdx.x >> 5); }
CA_DEV int  dp_block()           { return (int)blockIdx.x; }
CA_DEV int  dp_grid_blocks()     { return (int)gridDim.x; }
CA_DEV int  dp_block_threads()   { return (int)blockDim.x; }
CA_DEV int  dp_thread()          { return (int)threadIdx.x; }

CA_DEV uint32_t dp_shfl(uint32_t v, int src)      { return __shfl_sync(CA_FULL, v, src); }
CA_DEV uint32_t dp_shfl_up(uint32_t v, int d)     { return __shfl_up_sync(CA_FULL, v, d); }
CA_DEV uint32_t dp_shfl_down(uint32_t v, int d)   { return __shfl_down_sync(CA_FULL, v, d); }
/* neighbour lane's value, 0 where there is no such lane (the shuffle's own range predicate: no lane compare, no select) */
CA_DEV uint32_t dp_shfl_up0(uint32_t v)
{
    uint32_t r;
    asm volatile("{\n\t.reg .pred p;\n\tshfl.sync.up.b32 %0|p, %1, 1, 0, 0xffffffff;\n\t@!p mov.b32 %0, 0;\n\t}" : "=r"(r) : "r"(v));
    return r;
}
CA_DEV uint32_t dp_shfl_down0(uint32_t v)
{
    uint32_t r;
    asm volatile("{\n\t.reg .pred p;\n\tshfl.sync.down.b32 %0|p, %1, 1, 31, 0xffffffff;\n\t@!p mov.b32 %0, 0;\n\t}" : "=r"(r) : "r"(v));
    return r;
}
CA_DEV uint32_t dp_ballot(bool p)                 { return __ballot_sync(CA_FULL, p); }
CA_DEV bool     dp_all(bool p)                    { return __all_sync(CA_FULL, p); }
CA_DEV void     dp_syncwarp()                     { __syncwarp(); }
CA_DEV void     dp_syncblock()                    { __syncthreads(); }
/* named barrier over the first `nthreads` threads' worth of warps that use it (bar.sync id, nthreads) */
CA_DEV void     dp_syncblock_named(int id, int nthreads)
{
    asm volatile("bar.sync %0, %1;" :: "r"(id), "r"(nthreads) : "memory");
}

/* data written by other SMs inside the same launch: bypass the (incoherent) L1 */
CA_DEV uint32_t dp_ld_cg(const uint32_t *p)       { return __ldcg(p); }
CA_DEV uint2    dp_ld_cg(const uint2 *p)          { return __ldcg(p); }
CA_DEV uint4    dp_ld_cg(const uint4 *p)          { return __ldcg(p); }
CA_DEV uint8_t  dp_ld_cg(const uint8_t *p)        { return __ldcg(p); }
CA_DEV unsigned long long dp_ld_cg(const unsigned long long *p) { return __ldcg(p); }
/* the halves of a 64-bit value, taken HERE (volatile: not hoisted to the load that produced it) */
CA_DEV void dp_unpack64_here(unsigned long long v, uint32_t &lo, uint32_t &hi)
{
    asm volatile("mov.b64 {%0, %1}, %2;" : "=r"(lo), "=r"(hi) : "l"(v));
}
CA_DEV void     dp_st_cg(uint32_t *p, uint32_t v) { __stcg(p, v); }
CA_DEV void     dp_st_cg(uint2 *p, uint2 v)       { __stcg(p, v); }
CA_DEV void     dp_st_cg(uint4 *p, uint4 v)       { __stcg(p, v); }

/* progress flags: relaxed polling load, release store (gpu scope) */
CA_DEV int dp_ld_flag(const int *p)
{
    int v;
    asm volatile("ld.relaxed.gpu.global.s32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}
CA_DEV void dp_st_flag(int *p, int v)
{
    asm volatile("st.relaxed.gpu.global.s32 [%0], %1;" :: "l"(p), "r"(v) : "memory");
}
/* acquire load / release store (gpu scope): LDG.STRONG + CCTL, MEMBAR.GPU + STG -- no separate fence */
CA_DEV int dp_ld_acquire(const int *p)
{
    int v;
    asm volatile("ld.acquire.gpu.global.s32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}
CA_DEV void dp_st_release(int *p, int v)
{
    asm volatile("st.release.gpu.global.s32 [%0], %1;" :: "l"(p), "r"(v) : "memory");
}
CA_DEV int dp_reduce_min(int v)                   { return __reduce_min_sync(CA_FULL, v); }
/* counters written by ANOTHER GPU (peer stores over NVLink): acquire at system scope */
CA_DEV int dp_ld_acquire_sys(const int *p)
{
    int v;
    asm volatile("ld.acquire.sys.global.s32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}
CA_DEV unsigned long long dp_shfl64(unsigned long long v, int src)
{
    const uint32_t lo = __shfl_sync(CA_FULL, (uint32_t)v, src), hi = __shfl_sync(CA_FULL, (uint32_t)(v >> 32), src);
    return ((unsigned long long)hi << 32) | lo;
}
CA_DEV int dp_ffs(uint32_t v)                     { return __ffs((int)v); }
CA_DEV int dp_ld_flag_sys(const int *p)
{
    int v;
    asm volatile("ld.relaxed.sys.global.s32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}
CA_DEV void dp_st_flag_sys(int *p, int v)
{
    asm volatile("st.relaxed.sys.global.s32 [%0], %1;" :: "l"(p), "r"(v) : "memory");
}
CA_DEV void dp_fence_sys()                        { asm volatile("fence.acq_rel.sys;" ::: "memory"); }
/* fence.acq_rel.gpu (MEMBAR.ALL.GPU); __threadfence() would be the heavier fence.sc */
CA_DEV void dp_fence_release()                    { asm volatile("fence.acq_rel.gpu;" ::: "memory"); }
/* CTA-scope mailboxes in shared memory: volatile accesses ordered by fence.acq_rel.cta (MEMBAR.CTA: cheap) */
CA_DEV void dp_fence_cta()                        { asm volatile("fence.acq_rel.cta;" ::: "memory"); }
CA_DEV int  dp_ld_volatile(const int *p)          { return *(const volatile int *)p; }
CA_DEV void dp_st_volatile(int *p, int v)         { *(volatile int *)p = v; }
CA_DEV uint32_t dp_ld_volatile_u32(const uint32_t *p) { return *(const volatile uint32_t *)p; }
CA_DEV unsigned long long dp_ld_volatile64(const unsigned long long *p) { return *(const volatile unsigned long long *)p; }
CA_DEV void dp_st_volatile64(unsigned long long *p, unsigned long long v) { *(volatile unsigned long long *)p = v; }
CA_DEV void dp_atomic_add_cta(int *p, int v)      { atomicAdd(p, v); }
CA_DEV void dp_atomic_or_cta(uint32_t *p, uint32_t v) { atomicOr(p, v); }
CA_DEV bool dp_any(bool p)                        { return __any_sync(CA_FULL, p); }
CA_DEV void dp_fence_acquire()                    { asm volatile("fence.acq_rel.gpu;" ::: "memory"); }
CA_DEV void dp_nanosleep(unsigned ns)             { __nanosleep(ns); }
/* polling a shared-memory counter of a sibling warp: give the issue slots away for a moment */
CA_DEV void dp_team_pause()                       { __nanosleep(20); }
CA_DEV void dp_prefetch_l2(const void *p)         { asm volatile("prefetch.global.L2 [%0];" :: "l"(p)); }
CA_DEV long long dp_clock()                       { return clock64(); }
CA_DEV unsigned dp_atomic_inc(unsigned *p)        { return atomicAdd(p, 1u); }
CA_DEV void dp_atomic_add64(unsigned long long *p, unsigned long long v) { atomicAdd(p, v); }
CA_DEV void dp_atomic_max(int *p, int v)          { atomicMax(p, v); }
CA_DEV void dp_atomic_or_global(unsigned *p, unsigned v) { atomicOr(p, v); }
/* error words: the FIRST non-zero code sticks (later bail-outs are consequences of it) */
CA_DEV void dp_set_error(int *p, int v)           { atomicCAS(p, 0, v); }
CA_DEV int  dp_popc(uint32_t v)                   { return __popc(v); }
CA_DEV uint32_t dp_funnel_l(uint32_t lo, uint32_t hi, int s) { return __funnelshift_l(lo, hi, s); }
CA_DEV uint32_t dp_funnel_r(uint32_t lo, uint32_t hi, int s) { return __funnelshift_r(lo, hi, s); }
/* upper word of (hi:lo) << min(s, 32) */
CA_DEV uint32_t dp_funnel_l_clamp(uint32_t lo, uint32_t hi, uint32_t s) { return __funnelshift_lc(lo, hi, s); }

/*
 * 1-D bulk copies of the TMA engine (cp.async.bulk) and the mbarrier that counts their bytes.  Issued by ONE thread;
 * the copy itself runs in the async proxy, off the issuing warp.  Addresses and sizes are multiples of 16 bytes.
 */
CA_DEV uint32_t dp_smem_addr(const void *p)       { return (uint32_t)__cvta_generic_to_shared(p); }
/*
 * CTA-scope release of a shared-memory counter by the lanes with `pub`: fence.acq_rel.cta, then the volatile store, with
 * no branch, so the warp never diverges.  The whole warp executes the fence (ptxas branches around a predicated MEMBAR;
 * it is one MEMBAR per warp either way) and only the `pub` lanes store.  p points into shared memory.
 */
CA_DEV void dp_release_cta_if(bool pub, int *p, int v)
{
    asm volatile("{\n\t.reg .pred q;\n\tsetp.ne.u32 q, %2, 0;\n\tfence.acq_rel.cta;\n\t@q st.volatile.shared.s32 [%0], %1;\n\t}"
                 :: "r"(dp_smem_addr(p)), "r"(v), "r"((uint32_t)pub) : "memory");
}
CA_DEV void dp_mbar_init(unsigned long long *bar, int arrivals)
{
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" :: "r"(dp_smem_addr(bar)), "r"(arrivals) : "memory");
}
/* this thread arrives and announces `bytes` of bulk-copy traffic for the current phase */
CA_DEV void dp_mbar_expect_tx(unsigned long long *bar, uint32_t bytes)
{
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" :: "r"(dp_smem_addr(bar)), "r"(bytes) : "memory");
}
/* has the phase with this parity completed? */
CA_DEV bool dp_mbar_try_wait(unsigned long long *bar, uint32_t parity)
{
    uint32_t ok;
    asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}"
                 : "=r"(ok) : "r"(dp_smem_addr(bar)), "r"(parity) : "memory");
    return ok != 0;
}
/* global -> shared, completion counted on `bar` */
CA_DEV void dp_bulk_g2s(void *smem_dst, const void *gsrc, uint32_t bytes, unsigned long long *bar)
{
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 :: "r"(dp_smem_addr(smem_dst)), "l"(gsrc), "r"(bytes), "r"(dp_smem_addr(bar)) : "memory");
}
/* shared -> global (any global address: local HBM or a peer's over NVLink), completion through bulk groups */
CA_DEV void dp_bulk_s2g(void *gdst, const void *smem_src, uint32_t bytes)
{
    asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;"
                 :: "l"(gdst), "r"(dp_smem_addr(smem_src)), "r"(bytes) : "memory");
}
CA_DEV void dp_bulk_commit()                      { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
/* all committed shared -> global copies have READ their source (the staging slots may be reused) / are complete */
CA_DEV void dp_bulk_wait_read()                   { asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory"); }
CA_DEV void dp_bulk_wait()                        { asm volatile("cp.async.bulk.wait_group 0;" ::: "memory"); }
/* order this thread's generic-proxy accesses against its async-proxy (bulk copy) accesses */
CA_DEV void dp_fence_proxy_async()                { asm volatile("fence.proxy.async;" ::: "memory"); }

/* one LOP3 with a compile-time truth table: bit (a<<2|b<<1|c) of LUT */
template <unsigned LUT>
CA_DEV uint32_t dp_lop3(uint32_t a, uint32_t b, uint32_t c)
{
    uint32_t r;
    asm("lop3.b32 %0, %1, %2, %3, %4;" : "=r"(r) : "r"(a), "r"(b), "r"(c), "n"(LUT));
    return r;
}

} // namespace clapca

#else
/* -------------------------------------------------------------- emulator -- */
#include <string.h>
#include <stddef.h>

#define CA_DEV      static inline
#define CA_MDEV     static inline
#define CA_MEMBER   inline
#define CA_MCOLD    static
#define CA_HOSTDEV  static inline
#define CA_GLOBAL   static
#define CA_FULL     0xffffffffu
#define CA_SHARED(type, name, n) type *name = (type *)clapca::emu_block_shared((n) * sizeof(type))
#define __restrict__
#define __launch_bounds__(...)

struct uint2 { uint32_t x, y; };
struct uint4 { uint32_t x, y, z, w; };
struct int2  { int x, y; };
struct int4  { int x, y, z, w; };
static inline uint2 make_uint2(uint32_t x, uint32_t y) { uint2 r = { x, y }; return r; }
static inline uint4 make_uint4(uint32_t x, uint32_t y, uint32_t z, uint32_t w) { uint4 r = { x, y, z, w }; return r; }
static inline int2  make_int2(int x, int y) { int2 r = { x, y }; return r; }
static inline int4  make_int4(int x, int y, int z, int w) { int4 r = { x, y, z, w }; return r; }

namespace clapca {

/* provided by tests/emu/emu_runtime.cpp */
int      emu_lane();
int      emu_warp_in_block();
int      emu_block();
int      emu_grid_blocks();
int      emu_block_threads();
uint32_t emu_exchange(uint32_t v, int src_lane);     /* returns v deposited by src_lane (or own if out of range) */
uint32_t emu_ballot(bool p);
void     emu_yield();
long long emu_clock();
void     emu_syncblock();                            /* all warps of the block */
void     emu_syncblock_named(int id, int nthreads);  /* nthreads / 32 warps of the block */
void    *emu_block_shared(size_t bytes);             /* the block's shared memory (same buffer for every thread) */

CA_DEV int  dp_lane()            { return emu_lane(); }
CA_DEV int  dp_warp_in_block()   { return emu_warp_in_block(); }
CA_DEV int  dp_block()           { return emu_block(); }
CA_DEV int  dp_grid_blocks()     { return emu_grid_blocks(); }
CA_DEV int  dp_block_threads()   { return emu_block_threads(); }
CA_DEV int  dp_thread()          { return emu_warp_in_block() * 32 + emu_lane(); }

CA_DEV uint32_t dp_shfl(uint32_t v, int src)      { return emu_exchange(v, src); }
CA_DEV uint32_t dp_shfl_up(uint32_t v, int d)     { int l = emu_lane(); return emu_exchange(v, l - d >= 0 ? l - d : l); }
CA_DEV uint32_t dp_shfl_down(uint32_t v, int d)   { int l = emu_lane(); return emu_exchange(v, l + d < 32 ? l + d : l); }
CA_DEV uint32_t dp_shfl_up0(uint32_t v)           { int l = emu_lane(); uint32_t r = emu_exchange(v, l - 1 >= 0 ? l - 1 : l); return l ? r : 0u; }
CA_DEV uint32_t dp_shfl_down0(uint32_t v)         { int l = emu_lane(); uint32_t r = emu_exchange(v, l + 1 < 32 ? l + 1 : l); return l < 31 ? r : 0u; }
CA_DEV uint32_t dp_ballot(bool p)                 { return emu_ballot(p); }
CA_DEV bool     dp_all(bool p)                    { return emu_ballot(p) == CA_FULL; }
CA_DEV void     dp_syncwarp()                     { (void)emu_ballot(true); }
CA_DEV void     dp_syncblock()                    { emu_syncblock(); }
CA_DEV void     dp_syncblock_named(int id, int nthreads) { emu_syncblock_named(id, nthreads); }

template <typename T> CA_DEV T dp_ld_cg_any(const T *p)
{
    T v;
    __atomic_thread_fence(__ATOMIC_SEQ_CST);
    memcpy(&v, (const void *)p, sizeof(T));
    return v;
}
CA_DEV uint32_t dp_ld_cg(const uint32_t *p)       { return dp_ld_cg_any(p); }
CA_DEV uint2    dp_ld_cg(const uint2 *p)          { return dp_ld_cg_any(p); }
CA_DEV uint4    dp_ld_cg(const uint4 *p)          { return dp_ld_cg_any(p); }
CA_DEV uint8_t  dp_ld_cg(const uint8_t *p)        { return dp_ld_cg_any(p); }
CA_DEV unsigned long long dp_ld_cg(const unsigned long long *p) { return dp_ld_cg_any(p); }
CA_DEV void dp_unpack64_here(unsigned long long v, uint32_t &lo, uint32_t &hi) { lo = (uint32_t)v; hi = (uint32_t)(v >> 32); }
CA_DEV void     dp_st_cg(uint32_t *p, uint32_t v) { *p = v; }
CA_DEV void     dp_st_cg(uint2 *p, uint2 v)       { *p = v; }
CA_DEV void     dp_st_cg(uint4 *p, uint4 v)       { *p = v; }

CA_DEV int  dp_ld_flag(const int *p)              { return __atomic_load_n(p, __ATOMIC_ACQUIRE); }
CA_DEV void dp_st_flag(int *p, int v)             { __atomic_store_n(p, v, __ATOMIC_RELEASE); }
CA_DEV int  dp_ld_acquire(const int *p)           { return __atomic_load_n(p, __ATOMIC_ACQUIRE); }
CA_DEV void dp_st_release(int *p, int v)          { __atomic_store_n(p, v, __ATOMIC_RELEASE); }
CA_DEV int  dp_reduce_min(int v)
{
    for (int o = 16; o; o >>= 1) {
        int w = (int)emu_exchange((uint32_t)v, emu_lane() ^ o);
        v = w < v ? w : v;
    }
    return v;
}
CA_DEV int  dp_ld_acquire_sys(const int *p)       { return __atomic_load_n(p, __ATOMIC_ACQUIRE); }
CA_DEV unsigned long long dp_shfl64(unsigned long long v, int src)
{
    const uint32_t lo = emu_exchange((uint32_t)v, src), hi = emu_exchange((uint32_t)(v >> 32), src);
    return ((unsigned long long)hi << 32) | lo;
}
CA_DEV int  dp_ffs(uint32_t v)                    { return __builtin_ffs((int)v); }
CA_DEV void dp_fence_release()                    { __atomic_thread_fence(__ATOMIC_SEQ_CST); }
CA_DEV void dp_fence_cta()                        { __atomic_thread_fence(__ATOMIC_SEQ_CST); }
CA_DEV int  dp_ld_volatile(const int *p)          { return __atomic_load_n(p, __ATOMIC_ACQUIRE); }
CA_DEV void dp_st_volatile(int *p, int v)         { __atomic_store_n(p, v, __ATOMIC_RELEASE); }
CA_DEV uint32_t dp_ld_volatile_u32(const uint32_t *p) { return __atomic_load_n(p, __ATOMIC_ACQUIRE); }
CA_DEV unsigned long long dp_ld_volatile64(const unsigned long long *p) { return __atomic_load_n(p, __ATOMIC_ACQUIRE); }
CA_DEV void dp_st_volatile64(unsigned long long *p, unsigned long long v) { __atomic_store_n(p, v, __ATOMIC_RELEASE); }
CA_DEV void dp_atomic_add_cta(int *p, int v)      { __atomic_fetch_add(p, v, __ATOMIC_SEQ_CST); }
CA_DEV void dp_atomic_or_cta(uint32_t *p, uint32_t v) { __atomic_fetch_or(p, v, __ATOMIC_SEQ_CST); }
CA_DEV bool dp_any(bool p)                        { return emu_ballot(p) != 0u; }
CA_DEV void dp_fence_sys()                        { __atomic_thread_fence(__ATOMIC_SEQ_CST); }
CA_DEV int  dp_ld_flag_sys(const int *p)          { return __atomic_load_n(p, __ATOMIC_ACQUIRE); }
CA_DEV void dp_st_flag_sys(int *p, int v)         { __atomic_store_n(p, v, __ATOMIC_RELEASE); }
CA_DEV void dp_fence_acquire()                    { __atomic_thread_fence(__ATOMIC_SEQ_CST); }
CA_DEV void dp_nanosleep(unsigned)                { emu_yield(); }
CA_DEV void dp_team_pause()                       { emu_yield(); }
CA_DEV void dp_prefetch_l2(const void *)          { }
CA_DEV long long dp_clock()                       { return emu_clock(); }
CA_DEV unsigned dp_atomic_inc(unsigned *p)        { return __atomic_fetch_add(p, 1u, __ATOMIC_SEQ_CST); }
CA_DEV void dp_atomic_add64(unsigned long long *p, unsigned long long v) { __atomic_fetch_add(p, v, __ATOMIC_SEQ_CST); }
CA_DEV void dp_atomic_max(int *p, int v)
{
    int o = __atomic_load_n(p, __ATOMIC_RELAXED);
    while (o < v && !__atomic_compare_exchange_n(p, &o, v, false, __ATOMIC_SEQ_CST, __ATOMIC_RELAXED))
        ;
}
CA_DEV void dp_atomic_or_global(unsigned *p, unsigned v) { __atomic_fetch_or(p, v, __ATOMIC_SEQ_CST); }
CA_DEV void dp_set_error(int *p, int v)
{
    int o = 0;
    __atomic_compare_exchange_n(p, &o, v, false, __ATOMIC_SEQ_CST, __ATOMIC_RELAXED);
}
CA_DEV int  dp_popc(uint32_t v)                   { return __builtin_popcount(v); }
CA_DEV uint32_t dp_funnel_l(uint32_t lo, uint32_t hi, int s)
{
    return s ? (hi << s) | (lo >> (32 - s)) : hi;
}
CA_DEV uint32_t dp_funnel_r(uint32_t lo, uint32_t hi, int s)
{
    return s ? (lo >> s) | (hi << (32 - s)) : lo;
}
CA_DEV uint32_t dp_funnel_l_clamp(uint32_t lo, uint32_t hi, uint32_t s)
{
    return s >= 32 ? lo : (s ? (hi << s) | (lo >> (32 - s)) : hi);
}

CA_DEV void dp_release_cta_if(bool pub, int *p, int v)
{
    if (pub) {
        __atomic_thread_fence(__ATOMIC_SEQ_CST);
        __atomic_store_n(p, v, __ATOMIC_RELEASE);
    }
}

/*
 * bulk copies on the emulator: synchronous memcpy; the "mbarrier" word holds the phase (bit 0 of the low half) and the
 * bytes still expected (high half) -- one issuing thread, so no atomics are needed for the bookkeeping itself
 */
CA_DEV void dp_mbar_init(unsigned long long *bar, int) { __atomic_store_n(bar, 0ull, __ATOMIC_SEQ_CST); }
CA_DEV void dp_mbar_expect_tx(unsigned long long *bar, uint32_t bytes)
{
    __atomic_store_n(bar, (__atomic_load_n(bar, __ATOMIC_SEQ_CST) & 1ull) | ((unsigned long long)bytes << 32), __ATOMIC_SEQ_CST);
}
CA_DEV bool dp_mbar_try_wait(unsigned long long *bar, uint32_t parity)
{
    return (uint32_t)(__atomic_load_n(bar, __ATOMIC_SEQ_CST) & 1ull) != (parity & 1u);
}
CA_DEV void dp_bulk_g2s(void *smem_dst, const void *gsrc, uint32_t bytes, unsigned long long *bar)
{
    __atomic_thread_fence(__ATOMIC_SEQ_CST);
    memcpy(smem_dst, gsrc, bytes);
    unsigned long long v = __atomic_load_n(bar, __ATOMIC_SEQ_CST);
    unsigned long long left = (v >> 32) - bytes;
    v = left ? ((v & 1ull) | (left << 32)) : ((v & 1ull) ^ 1ull);
    __atomic_store_n(bar, v, __ATOMIC_SEQ_CST);
}
CA_DEV void dp_bulk_s2g(void *gdst, const void *smem_src, uint32_t bytes)
{
    memcpy(gdst, smem_src, bytes);
    __atomic_thread_fence(__ATOMIC_SEQ_CST);
}
CA_DEV void dp_bulk_commit()                      { }
CA_DEV void dp_bulk_wait_read()                   { }
CA_DEV void dp_bulk_wait()                        { }
CA_DEV void dp_fence_proxy_async()                { __atomic_thread_fence(__ATOMIC_SEQ_CST); }

template <unsigned LUT>
CA_DEV uint32_t dp_lop3(uint32_t a, uint32_t b, uint32_t c)
{
    uint32_t r = 0;
    for (int i = 0; i < 8; i++)
        if (LUT & (1u << i)) {
            uint32_t ta = (i & 4) ? a : ~a, tb = (i & 2) ? b : ~b, tc = (i & 1) ? c : ~c;
            r |= ta & tb & tc;
        }
    return r;
}

} // namespace clapca
#endif /* CLAPCA_EMU */

#endif /* CLAPCA_DEVPORT_H */
