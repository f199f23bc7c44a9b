// Shared device/host helpers for libeod_memory.so (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <cuda_fp16.h>
#include <stdint.h>
#include <stdio.h>

#include "../../include/eod_memory.h"

#define EOD_NUM_SMS_FALLBACK 148

void eod_set_error(const char *fmt, ...);
int eod_check_launch(const char *what);
int eod_num_sms();
int *eod_work_tickets();      // zeroed {next, done} pair for one dynamically scheduled launch (api.cu)

#define EOD_REQUIRE(cond, code, ...)      \
    do {                                  \
        if (!(cond)) {                    \
            eod_set_error(__VA_ARGS__);   \
            return (code);                \
        }                                 \
    } while (0)

static inline bool eod_aligned16(const void *p) { return (reinterpret_cast<uintptr_t>(p) & 15u) == 0; }

// cudaFuncAttributeMaxDynamicSharedMemorySize is a PER-DEVICE attribute: `done` is a per-kernel bitmask over device
// ordinals (one bit per device of the process), so a second GPU used from the same process gets the attribute too.
// Returns EOD_OK or EOD_ERR_LAUNCH (message set).  Racing threads at worst set the attribute twice.
template <typename F>
static inline int eod_ensure_dyn_smem(F func, int bytes, unsigned long long *done, const char *what)
{
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess) dev = 0;
    const unsigned long long bit = 1ull << (dev & 63);
    if (__atomic_load_n(done, __ATOMIC_ACQUIRE) & bit) return EOD_OK;
    const cudaError_t e = cudaFuncSetAttribute(func, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes);
    if (e != cudaSuccess) {
        eod_set_error("%s: cannot raise dynamic shared memory to %d bytes: %s", what, bytes, cudaGetErrorString(e));
        return EOD_ERR_LAUNCH;
    }
    __atomic_fetch_or(done, bit, __ATOMIC_RELEASE);
    return EOD_OK;
}

// ---- device helpers -------------------------------------------------------------------------------

// feature element type: fp32, or bf16 / fp16 widened exactly to fp32 before any arithmetic
enum { FEAT_F32 = 0, FEAT_BF16 = 1, FEAT_F16 = 2 };
template <int F> struct FeatElem { using T = uint16_t; };
template <> struct FeatElem<FEAT_F32> { using T = float; };
template <int F>
__device__ __forceinline__ float widen1(typename FeatElem<F>::T x)
{
    if constexpr (F == FEAT_F32) return x;
    else if constexpr (F == FEAT_BF16) return __uint_as_float((uint32_t)x << 16);
    else return __half2float(__ushort_as_half(x));
}
// the two 16-bit elements of a 32-bit word (element 0 in the low half), widened exactly
template <int F>
__device__ __forceinline__ float2 widen2(uint32_t w)
{
    if constexpr (F == FEAT_BF16) return make_float2(__uint_as_float(w << 16), __uint_as_float(w & 0xffff0000u));
    else return __half22float2(*reinterpret_cast<const __half2 *>(&w));
}

// 128-bit fp32 reduction to global memory (sm_90+): one L2 atomic transaction for four floats.
__device__ __forceinline__ void red_add_v4(float *addr, float a, float b, float c, float d)
{
    asm volatile("red.global.add.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(addr), "f"(a), "f"(b), "f"(c), "f"(d)
                 : "memory");
}

__device__ __forceinline__ void red_add_f32(float *addr, float a)
{
    asm volatile("red.global.add.f32 [%0], %1;" ::"l"(addr), "f"(a) : "memory");
}

__device__ __forceinline__ float4 ldg_stream_f4(const float *p)
{
    float4 r;
    asm volatile("ld.global.nc.L1::no_allocate.v4.f32 {%0, %1, %2, %3}, [%4];"
                 : "=f"(r.x), "=f"(r.y), "=f"(r.z), "=f"(r.w)
                 : "l"(p));
    return r;
}

__device__ __forceinline__ uint32_t smem_u32(const void *p) { return static_cast<uint32_t>(__cvta_generic_to_shared(p)); }

// Every wrapper below addresses shared memory by its 32-bit shared-window address (smem_u32).  Kernels that keep pointers
// to their barriers and tiles call the one-line pointer overloads.

// ---- mbarrier / TMA (inline PTX) --------------------------------------------------------------------
__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count)
{
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count));
}
__device__ __forceinline__ void mbar_init(uint64_t *bar, uint32_t count) { mbar_init(smem_u32(bar), count); }
__device__ __forceinline__ void mbar_fence_init()
{
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void fence_proxy_async()
{
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes)
{
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t *bar, uint32_t bytes) { mbar_expect_tx(smem_u32(bar), bytes); }
__device__ __forceinline__ void mbar_arrive(uint32_t bar)
{
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t *bar) { mbar_arrive(smem_u32(bar)); }
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity)
{
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "WAIT_LOOP:\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
        "@p bra DONE;\n\t"
        "bra WAIT_LOOP;\n\t"
        "DONE:\n\t"
        "}" ::"r"(bar),
        "r"(parity)
        : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t *bar, uint32_t parity) { mbar_wait(smem_u32(bar), parity); }
// same wait with a suspend-time hint (ns): the warp sleeps in hardware instead of re-issuing the poll; 0 = the plain loop
__device__ __forceinline__ void mbar_wait_hint(uint32_t bar, uint32_t parity, uint32_t hint_ns)
{
    if (hint_ns == 0) { mbar_wait(bar, parity); return; }
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "WAIT_LOOP_H:\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1, %2;\n\t"
        "@p bra DONE_H;\n\t"
        "bra WAIT_LOOP_H;\n\t"
        "DONE_H:\n\t"
        "}" ::"r"(bar),
        "r"(parity), "r"(hint_ns)
        : "memory");
}
// L2 policy for data read exactly once
__device__ __forceinline__ uint64_t make_evict_first_policy()
{
    uint64_t pol;
    asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(pol));
    return pol;
}
// Tiled TMA loads global -> shared, completion signalled on an mbarrier (SASS: UTMALDG).
__device__ __forceinline__ void tma_load_2d(uint32_t dst, const void *tmap, int x, int y, uint32_t bar)
{
    asm volatile("cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];" ::"r"(dst),
                 "l"(tmap), "r"(x), "r"(y), "r"(bar)
                 : "memory");
}
__device__ __forceinline__ void tma_load_2d(void *dst, const void *tmap, int x, int y, uint64_t *bar) { tma_load_2d(smem_u32(dst), tmap, x, y, smem_u32(bar)); }
__device__ __forceinline__ void tma_load_3d(uint32_t dst, const void *tmap, int x, int y, int z, uint32_t bar)
{
    asm volatile(
        "cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3, %4}], [%5];" ::"r"(dst),
        "l"(tmap), "r"(x), "r"(y), "r"(z), "r"(bar)
        : "memory");
}
__device__ __forceinline__ void tma_load_3d(void *dst, const void *tmap, int x, int y, int z, uint64_t *bar) { tma_load_3d(smem_u32(dst), tmap, x, y, z, smem_u32(bar)); }
// ... with an L2 cache policy (make_evict_first_policy)
__device__ __forceinline__ void tma_load_3d_hint(uint32_t dst, const void *tmap, int x, int y, int z, uint32_t bar, uint64_t pol)
{
    asm volatile(
        "cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint [%0], [%1, {%2, %3, %4}], [%5], %6;" ::"r"(dst),
        "l"(tmap), "r"(x), "r"(y), "r"(z), "r"(bar), "l"(pol)
        : "memory");
}
// L2 prefetch of a 3-D tile (no shared-memory destination)
__device__ __forceinline__ void tma_prefetch_3d(const void *tmap, int x, int y, int z)
{
    asm volatile("cp.async.bulk.prefetch.tensor.3d.L2.global.tile [%0, {%1, %2, %3}];" ::"l"(tmap), "r"(x), "r"(y), "r"(z) : "memory");
}
// 1-D bulk copy global -> shared (SASS: UBLKCP); bytes % 16 == 0, both addresses 16-byte aligned.
__device__ __forceinline__ void bulk_load_1d(uint32_t dst, const void *src, uint32_t bytes, uint32_t bar)
{
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(dst), "l"(src), "r"(bytes), "r"(bar)
                 : "memory");
}
__device__ __forceinline__ void named_bar_sync(int id, int nthreads)
{
    asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(nthreads) : "memory");
}

// ---- shared memory by address (inline PTX) ------------------------------------------------------------
// The compiler keeps one base register instead of re-deriving `&array[warp][...]` from %tid / %cluster_ctaid inside loops.
// Values are raw 32-bit words: callers reinterpret float bits with __uint_as_float / __float_as_uint.
__device__ __forceinline__ uint4 lds128(uint32_t a)
{
    uint4 v;
    asm volatile("ld.shared.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "r"(a));
    return v;
}
__device__ __forceinline__ uint2 lds64(uint32_t a)
{
    uint2 v;
    asm volatile("ld.shared.v2.u32 {%0, %1}, [%2];" : "=r"(v.x), "=r"(v.y) : "r"(a));
    return v;
}
__device__ __forceinline__ uint32_t lds32(uint32_t a)
{
    uint32_t v;
    asm volatile("ld.shared.u32 %0, [%1];" : "=r"(v) : "r"(a));
    return v;
}
__device__ __forceinline__ uint32_t lds8(uint32_t a)
{
    uint32_t v;
    asm volatile("ld.shared.u8 %0, [%1];" : "=r"(v) : "r"(a));
    return v;
}
__device__ __forceinline__ void sts128(uint32_t a, uint32_t x, uint32_t y, uint32_t z, uint32_t w)
{
    asm volatile("st.shared.v4.u32 [%0], {%1, %2, %3, %4};" ::"r"(a), "r"(x), "r"(y), "r"(z), "r"(w) : "memory");
}
__device__ __forceinline__ void sts64(uint32_t a, uint32_t x, uint32_t y)
{
    asm volatile("st.shared.v2.u32 [%0], {%1, %2};" ::"r"(a), "r"(x), "r"(y) : "memory");
}
__device__ __forceinline__ void sts32(uint32_t a, uint32_t x) { asm volatile("st.shared.u32 [%0], %1;" ::"r"(a), "r"(x) : "memory"); }
__device__ __forceinline__ void sts16(uint32_t a, uint32_t x) { asm volatile("st.shared.u16 [%0], %1;" ::"r"(a), "h"((unsigned short)x) : "memory"); }

// ---- tcgen05: tensor memory and the 5th-generation tensor core (inline PTX) ---------------------------
__device__ __forceinline__ void tmem_alloc(uint32_t dst_smem, uint32_t ncols)
{
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(dst_smem), "r"(ncols) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_alloc(uint32_t *dst_smem, uint32_t ncols) { tmem_alloc(smem_u32(dst_smem), ncols); }
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t ncols)
{
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
// D[tmem] (+)= A[smem desc] * B[smem desc] with fp32 accumulators, issued by ONE thread; kind::f16 or kind::tf32 operands
#define EOD_UMMA_ASM(kind)                                                                                                     \
    asm volatile("{\n\t"                                                                                                       \
                 ".reg .pred p;\n\t"                                                                                           \
                 "setp.ne.b32 p, %4, 0;\n\t"                                                                                   \
                 "tcgen05.mma.cta_group::1.kind::" kind " [%0], %1, %2, %3, p;\n\t"                                            \
                 "}" ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)                                        \
                 : "memory")
__device__ __forceinline__ void umma_f16(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) { EOD_UMMA_ASM("f16"); }
__device__ __forceinline__ void umma_tf32(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) { EOD_UMMA_ASM("tf32"); }
#undef EOD_UMMA_ASM
// mbarrier arrive once all tcgen05.mma issued so far by this thread have completed (implies fence::before_thread_sync)
__device__ __forceinline__ void umma_commit(uint32_t bar)
{
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void umma_commit(uint64_t *bar) { umma_commit(smem_u32(bar)); }
// 16 consecutive fp32 columns of this thread's TMEM lane
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, uint32_t (&v)[16])
{
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
        : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]), "=r"(v[9]), "=r"(v[10]),
          "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15])
        : "r"(taddr)
        : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }
// K-major, SWIZZLE_128B shared-memory matrix descriptor (cute/arch/mma_sm100_desc.hpp SmemDescriptor): start address >> 4 in
// bits [0,14), leading byte offset (unused for swizzled K-major; 1) in [16,30), stride byte offset = 1024 B (one 8-row
// swizzle atom) >> 4 in [32,46), version 1 in [46,48), layout type 2 (SWIZZLE_128B) in [61,64).
__device__ __forceinline__ uint64_t umma_desc_sw128(uint32_t smem_addr)
{
    return (uint64_t)((smem_addr >> 4) & 0x3fffu) | (1ull << 16) | (64ull << 32) | (1ull << 46) | (2ull << 61);
}
