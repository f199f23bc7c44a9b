// 1x1 projection + weighted fusion in ONE kernel on the 5th-generation tensor cores (SURVEY 8a row A13, 8f rank 4):
//
//     mem = Conv2d(C_mem -> C_out, 1x1, bias)(level.float())      timm.py:174   (fp32, eval, autocast off)
//     mem = mem * MAP_FEATURE_WEIGHT                               timm.py:177
//     out = res + mem | mem                                        timm.py:181-184
//
// `level` is what eod_read_pool wrote: (E, h, w, K) fp16 channels-last, i.e. an (M = E*h*w, K) K-major matrix whose
// elements are EXACT fp16 numbers (the reference rounds the pooled level to half before the conv, timm.py:168).  The
// fp32 weight is split once on the device into two fp16 terms,  W = W_hi + 2^-11 * W_lo  (W_hi = half(W),
// W_lo = half((W - W_hi) * 2^11); 22 mantissa bits), so that  x . W = x . W_hi + 2^-11 * (x . W_lo)  with every product
// exact in the fp32 accumulator: two kind::f16 UMMAs against the SAME staged A tile give fp32-GEMM accuracy
// (measured against an fp64 reference in the tests) at fp16 tensor-core rate, instead of a CUDA-core SGEMM + a
// separate elementwise pass.
//
// Tile: 128 rows (pixels) x 128 output channels; the UMMA is M=128, N=256 (columns 0..127 = W_hi block, 128..255 =
// W_lo block of the same output channels), K=16 per instruction, fp32 accumulators in 256 TMEM columns.
// One CTA (128 threads) per tile, two CTAs resident per SM (2 x 256 TMEM columns, 2 x 97 KB shared memory): while one
// CTA streams its epilogue (res in, out out: the HBM-bound part), the other runs its main loop.
//   warp 0 / lane 0 : TMA producer  - A box {64 K, 128 rows}, B box {64 K, 256 rows}, SWIZZLE_128B, 2-stage ring
//   warp 1 / lane 0 : MMA issuer    - 4 x tcgen05.mma per stage, tcgen05.commit releases the stage / publishes the tile
//   warps 0-3       : epilogue      - tcgen05.ld 32x32b (thread = one pixel row), + bias, * weight, + res, NCHW store
//                                     (for a fixed channel the 32 lanes of a warp touch 32 consecutive pixels = 128 B)
#include <cuda.h>
#include <string.h>

#include "eod_common.cuh"
#include "tmap_cache.cuh"

namespace {

constexpr int PF_BM = 128;                    // pixels per tile
constexpr int PF_BN = 128;                    // output channels per tile
constexpr int PF_BK = 64;                     // fp16 elements per 128-byte swizzle row
constexpr int PF_STAGES = 2;
constexpr int PF_A_BYTES = PF_BM * PF_BK * 2;             // 16 KB
constexpr int PF_B_BYTES = 2 * PF_BN * PF_BK * 2;         // 32 KB (hi + lo rows)
constexpr int PF_STAGE_BYTES = PF_A_BYTES + PF_B_BYTES;
constexpr int PF_TMEM_COLS = 2 * PF_BN;                   // 256 fp32 columns
constexpr int PF_SMEM_BYTES = PF_STAGES * PF_STAGE_BYTES + 1024 /* alignment slack */ + 64 /* barriers + tmem ptr */;
constexpr float PF_LO_SCALE = 2048.f, PF_LO_INV = 1.f / 2048.f;

// instruction descriptor (InstrDescriptor): D = F32 (1 << 4), A = B = F16 (0), both K-major, N >> 3 in [17,23), M >> 4 in [24,29)
constexpr uint32_t PF_IDESC = (1u << 4) | ((uint32_t)(2 * PF_BN >> 3) << 17) | ((uint32_t)(PF_BM >> 4) << 24);

// kSum: out = res + w * mem, else out = w * mem
template <bool kSum>
__global__ void __launch_bounds__(128) project_fuse_kernel(const __grid_constant__ CUtensorMap tm_a, const __grid_constant__ CUtensorMap tm_b,
                                                           const float *__restrict__ bias, const float *__restrict__ res, float *__restrict__ out,
                                                           float weight, int M, int hw, int N, int n_kblocks)
{
    extern __shared__ uint8_t pf_smem_raw[];
    uint8_t *smem = reinterpret_cast<uint8_t *>((reinterpret_cast<uintptr_t>(pf_smem_raw) + 1023) & ~uintptr_t(1023));
    uint64_t *bars = reinterpret_cast<uint64_t *>(smem + PF_STAGES * PF_STAGE_BYTES);
    uint64_t *full = bars, *empty = bars + PF_STAGES, *tmem_full = bars + 2 * PF_STAGES;
    uint32_t *tmem_slot = reinterpret_cast<uint32_t *>(bars + 2 * PF_STAGES + 1);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int n_nblocks = N / PF_BN;
    const int mb = blockIdx.x / n_nblocks, nb = blockIdx.x % n_nblocks;      // the n-blocks of one m-block are neighbours: A comes from L2 the 2nd time

    if (warp == 1 && lane == 0) {
        for (int s = 0; s < PF_STAGES; ++s) {
            mbar_init(full + s, 1);
            mbar_init(empty + s, 1);
        }
        mbar_init(tmem_full, 1);
        mbar_fence_init();
        asm volatile("prefetch.tensormap [%0];" ::"l"(&tm_a) : "memory");
        asm volatile("prefetch.tensormap [%0];" ::"l"(&tm_b) : "memory");
    }
    if (warp == 0) tmem_alloc(tmem_slot, PF_TMEM_COLS);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;

    if (warp == 0 && lane == 0) {
        // ===== TMA producer =====
        for (int kb = 0; kb < n_kblocks; ++kb) {
            const int s = kb % PF_STAGES;
            mbar_wait(empty + s, ((kb / PF_STAGES) & 1) ^ 1);
            uint8_t *a = smem + s * PF_STAGE_BYTES, *b = a + PF_A_BYTES;
            mbar_expect_tx(full + s, PF_STAGE_BYTES);
            tma_load_2d(a, &tm_a, kb * PF_BK, mb * PF_BM, full + s);
            tma_load_2d(b, &tm_b, kb * PF_BK, nb * 2 * PF_BN, full + s);
        }
    } else if (warp == 1 && lane == 0) {
        // ===== MMA issuer =====
        for (int kb = 0; kb < n_kblocks; ++kb) {
            const int s = kb % PF_STAGES;
            mbar_wait(full + s, (kb / PF_STAGES) & 1);
            tc_fence_after();
            const uint32_t a = smem_u32(smem + s * PF_STAGE_BYTES), b = a + PF_A_BYTES;
#pragma unroll
            for (int k = 0; k < PF_BK / 16; ++k)       // 16 fp16 = 32 bytes along K inside the swizzle row
                umma_f16(tmem_base, umma_desc_sw128(a + k * 32), umma_desc_sw128(b + k * 32), PF_IDESC, (kb | k) != 0);
            umma_commit(empty + s);                     // the stage may be refilled once these MMAs have read it
        }
        umma_commit(tmem_full);                         // accumulators complete
    }
    __syncwarp();

    // ===== epilogue: all four warps; warp w owns TMEM lanes [32w, 32w + 32) =====
    mbar_wait(tmem_full, 0);
    tc_fence_after();
    const int m = mb * PF_BM + warp * 32 + lane;
    const bool live = m < M;
    const int e = live ? m / hw : 0, pix = live ? m - e * hw : 0;
    const size_t base = ((size_t)e * N + (size_t)nb * PF_BN) * hw + pix;      // NCHW: + channel * hw
    const uint32_t taddr = tmem_base + ((uint32_t)(warp * 32) << 16);
    const float *bias_n = bias ? bias + nb * PF_BN : nullptr;
#pragma unroll 1
    for (int c0 = 0; c0 < PF_BN; c0 += 16) {
        uint32_t hi[16], lo[16];
        float r[16];
        tmem_ld16(taddr + c0, hi);
        tmem_ld16(taddr + PF_BN + c0, lo);
        if (kSum) {
#pragma unroll
            for (int j = 0; j < 16; ++j) r[j] = live ? __ldg(res + base + (size_t)(c0 + j) * hw) : 0.f;
        }
        tmem_ld_wait();
#pragma unroll
        for (int j = 0; j < 16; ++j) {
            float v = __fmaf_rn(__uint_as_float(lo[j]), PF_LO_INV, __uint_as_float(hi[j]));      // x.W_hi + 2^-11 x.W_lo: the GEMM result
            if (bias_n) v = __fadd_rn(v, __ldg(bias_n + c0 + j));                                 // conv bias
            v = __fmul_rn(v, weight);                                                             // timm.py:177
            if (kSum) v = __fadd_rn(r[j], v);                                                     // timm.py:182
            if (live) out[base + (size_t)(c0 + j) * hw] = v;
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 0) tmem_dealloc(tmem_base, PF_TMEM_COLS);
}

// ------------------------------------------------------------------------------------------------------------------
// v2: persistent, all levels in one launch.  One CTA per SM walks a static tile list (tile = 256 pixels of ONE episode x
// 128 output channels); 11 warps:
//   warps 0-7 : epilogue   (warp w reads TMEM lanes 32*(w%4).. of accumulator w/4, i.e. pixels (w/4)*128 + (w%4)*32 + lane).
//               Phase 1 drains the thread's 128 output channels (hi + 2^-11 lo) into REGISTERS and hands TMEM back, so
//               the next tile's MMAs run under phase 2 (+ bias, * weight, + res from the ring, NCHW stores); the two
//               epilogue warpgroups raise their register budget with setmaxnreg, the third warpgroup lowers its own
//   warp  8   : A/B producer - 3-stage ring of {A 256 rows x 64 K, B 256 rows x 64 K} (64 KB per stage)
//   warp  9   : TMEM owner + MMA issuer - per k-block 4 k-steps x 2 UMMAs (pixel rows 0-127 -> columns [0,256),
//               rows 128-255 -> columns [256,512)); both halves share the staged B tile
//   warp 10   : res producer - 2-slot ring of {256 px x 16 channels} fp32 boxes (NCHW rows are pixel-contiguous)
// Why this shape: the kernel moves (A + B) per tile from L2 into shared memory on top of the compulsory res / out
// stream; with 128-row tiles the operand refill (384 KB per 32 K outputs, 2.5 GB per frame-step at E=64) is what
// bounds it (measured: v1 0.53 ms).  256-row tiles halve the B refill per output (1.6 GB), single-launch persistence
// keeps the rings full across tiles and levels, and res arrives by TMA instead of 128 dependent loads per thread.
constexpr int P2_BM = 256, P2_STAGES = 3, P2_RCH = 16, P2_RSLOTS = 2;
constexpr int P2_A_BYTES = P2_BM * PF_BK * 2;                 // 32 KB
constexpr int P2_STAGE_BYTES = P2_A_BYTES + PF_B_BYTES;       // 64 KB
constexpr int P2_R_BYTES = P2_RCH * P2_BM * 4;                // 16 KB
constexpr int P2_BAR_BYTES = 128;                               // 12 mbarriers (96 B) + the TMEM base address (4 B), padded
constexpr int P2_BIAS_BYTES = 2 * PF_BN * 4;                    // the tile's bias values, double buffered
constexpr int P2_SMEM_BYTES = P2_STAGES * P2_STAGE_BYTES + P2_RSLOTS * P2_R_BYTES + P2_BAR_BYTES + P2_BIAS_BYTES + 1024 /* alignment slack */;
static_assert((2 * P2_STAGES + 2 * P2_RSLOTS + 2) * 8 + 4 <= P2_BAR_BYTES, "barrier block too small");
static_assert(P2_SMEM_BYTES <= 232448, "exceeds 227 KB of shared memory");
constexpr int P2_THREADS = 12 * 32;                 // 3 warpgroups: 2 x epilogue, 1 x {A/B producer, MMA, res producer, idle}
constexpr int P2_MAX_LEVELS = 3;

struct P2Params {
    CUtensorMap tm_a[P2_MAX_LEVELS];      // (K, hw, E) f16, box {64, 256, 1}, SWIZZLE_128B
    CUtensorMap tm_b[P2_MAX_LEVELS];      // (K, 2N) f16,    box {64, 256},    SWIZZLE_128B
    CUtensorMap tm_r[P2_MAX_LEVELS];      // (hw, N, E) f32, box {256, 16, 1}
    const float *bias[P2_MAX_LEVELS];
    float *out[P2_MAX_LEVELS];
    int hw[P2_MAX_LEVELS];
    int tiles_per_ep[P2_MAX_LEVELS];      // ceil(hw / 256)
    int tile_start[P2_MAX_LEVELS + 1];    // first global tile id of each level
    int n_levels, n_nblocks, N, n_kblocks, n_tiles;
    float weight;
};

struct P2Tile { int l, nb, e, p0; };

__device__ __forceinline__ P2Tile p2_decode(const P2Params &P, int t)
{
    P2Tile r;
    r.l = 0;
    while (r.l + 1 < P.n_levels && t >= P.tile_start[r.l + 1]) ++r.l;
    t -= P.tile_start[r.l];
    r.nb = t % P.n_nblocks;
    const int mt = t / P.n_nblocks;
    r.e = mt / P.tiles_per_ep[r.l];
    r.p0 = (mt - r.e * P.tiles_per_ep[r.l]) * P2_BM;
    return r;
}

template <bool kSum>
__global__ void __launch_bounds__(P2_THREADS, 1) project_fuse_persistent_kernel(const __grid_constant__ P2Params P)
{
    extern __shared__ uint8_t pf_smem_raw[];
    uint8_t *smem = reinterpret_cast<uint8_t *>((reinterpret_cast<uintptr_t>(pf_smem_raw) + 1023) & ~uintptr_t(1023));
    float *res_s = reinterpret_cast<float *>(smem + P2_STAGES * P2_STAGE_BYTES);
    uint64_t *bars = reinterpret_cast<uint64_t *>(smem + P2_STAGES * P2_STAGE_BYTES + P2_RSLOTS * P2_R_BYTES);
    uint64_t *full = bars, *empty = full + P2_STAGES, *rfull = empty + P2_STAGES, *rempty = rfull + P2_RSLOTS;
    uint64_t *tmem_full = rempty + P2_RSLOTS, *tmem_empty = tmem_full + 1;
    uint32_t *tmem_slot = reinterpret_cast<uint32_t *>(tmem_empty + 1);
    float *bias_s = reinterpret_cast<float *>(reinterpret_cast<uint8_t *>(bars) + P2_BAR_BYTES);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    if (warp == 8 && lane == 0) {
        for (int s = 0; s < P2_STAGES; ++s) { mbar_init(full + s, 1); mbar_init(empty + s, 1); }
        for (int s = 0; s < P2_RSLOTS; ++s) { mbar_init(rfull + s, 1); mbar_init(rempty + s, 8); }
        mbar_init(tmem_full, 1);
        mbar_init(tmem_empty, 8);
        mbar_fence_init();
    }
    if (warp == 9) tmem_alloc(tmem_slot, 512);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;

    if (warp >= 8) {
    asm volatile("setmaxnreg.dec.sync.aligned.u32 64;");
    if (warp == 8) {
        if (lane == 0) {
            // ===== A / B producer =====
            uint32_t it = 0;
            for (int t = blockIdx.x; t < P.n_tiles; t += gridDim.x) {
                const P2Tile T = p2_decode(P, t);
                for (int kb = 0; kb < P.n_kblocks; ++kb, ++it) {
                    const int s = it % P2_STAGES;
                    mbar_wait(empty + s, ((it / P2_STAGES) & 1) ^ 1);
                    uint8_t *a = smem + s * P2_STAGE_BYTES, *b = a + P2_A_BYTES;
                    mbar_expect_tx(full + s, P2_STAGE_BYTES);
                    tma_load_3d(a, &P.tm_a[T.l], kb * PF_BK, T.p0, T.e, full + s);
                    tma_load_2d(b, &P.tm_b[T.l], kb * PF_BK, T.nb * 2 * PF_BN, full + s);
                }
            }
        }
    } else if (warp == 9) {
        if (lane == 0) {
            // ===== MMA issuer =====
            uint32_t it = 0, tile_it = 0;
            for (int t = blockIdx.x; t < P.n_tiles; t += gridDim.x, ++tile_it) {
                mbar_wait(tmem_empty, (tile_it & 1) ^ 1);          // epilogue has drained the previous tile's accumulators
                tc_fence_after();
                for (int kb = 0; kb < P.n_kblocks; ++kb, ++it) {
                    const int s = it % P2_STAGES;
                    mbar_wait(full + s, (it / P2_STAGES) & 1);
                    tc_fence_after();
                    const uint32_t a = smem_u32(smem + s * P2_STAGE_BYTES), b = a + P2_A_BYTES;
#pragma unroll
                    for (int k = 0; k < PF_BK / 16; ++k) {
                        const uint64_t bd = umma_desc_sw128(b + k * 32);
                        umma_f16(tmem_base, umma_desc_sw128(a + k * 32), bd, PF_IDESC, (kb | k) != 0);
                        umma_f16(tmem_base + 256, umma_desc_sw128(a + 128 * 128 + k * 32), bd, PF_IDESC, (kb | k) != 0);
                    }
                    umma_commit(empty + s);
                }
                umma_commit(tmem_full);
            }
        }
    } else if (warp == 10) {
        if (kSum && lane == 0) {
            // ===== res producer =====
            uint32_t rc = 0;
            for (int t = blockIdx.x; t < P.n_tiles; t += gridDim.x) {
                const P2Tile T = p2_decode(P, t);
                // the ring holds 32 KB; what hides the DRAM latency is the L2 prefetch of the NEXT tile's res block (128 KB)
                // issued one tile ahead (and of this one, for the first tile)
                for (int ahead = (t == (int)blockIdx.x ? 0 : 1); ahead < 2; ++ahead) {
                    const int tn = t + ahead * gridDim.x;
                    if (tn >= P.n_tiles) break;
                    const P2Tile Tn = p2_decode(P, tn);
                    for (int c = 0; c < PF_BN / P2_RCH; ++c) tma_prefetch_3d(&P.tm_r[Tn.l], Tn.p0, Tn.nb * PF_BN + c * P2_RCH, Tn.e);
                }
                for (int c = 0; c < PF_BN / P2_RCH; ++c, ++rc) {
                    const int s = rc % P2_RSLOTS;
                    mbar_wait(rempty + s, ((rc / P2_RSLOTS) & 1) ^ 1);
                    mbar_expect_tx(rfull + s, P2_R_BYTES);
                    tma_load_3d(res_s + s * (P2_R_BYTES / 4), &P.tm_r[T.l], T.p0, T.nb * PF_BN + c * P2_RCH, T.e, rfull + s);
                }
            }
        }
    }
    } else {
        asm volatile("setmaxnreg.inc.sync.aligned.u32 208;");
        // ===== epilogue (warps 0-7) =====
        const int acc = warp >> 2, row = (warp & 3) * 32 + lane;           // TMEM lane = row; accumulator = pixel half
        const int px_local = acc * 128 + row;
        const uint32_t taddr = tmem_base + ((uint32_t)((warp & 3) * 32) << 16) + acc * 256;
        uint32_t rc = 0, tile_it = 0;
        for (int t = blockIdx.x; t < P.n_tiles; t += gridDim.x, ++tile_it) {
            const P2Tile T = p2_decode(P, t);
            const int hw = P.hw[T.l];
            const int pix = T.p0 + px_local;
            const bool live = pix < hw;
            float *out = P.out[T.l] + ((size_t)T.e * P.N + (size_t)T.nb * PF_BN) * hw + (live ? pix : 0);
            const float *bias_n = P.bias[T.l] ? P.bias[T.l] + T.nb * PF_BN : nullptr;
            // the tile's 128 bias values go through shared memory (a dependent L1 load per output element was 1/3 of the
            // epilogue's stalls); the load overlaps the wait for the accumulators.  Double buffered: a warp may be two phases
            // apart from the slowest one only across the named barrier below.
            float *bias_t = bias_s + (tile_it & 1) * PF_BN;
            if (bias_n && threadIdx.x < PF_BN) bias_t[threadIdx.x] = __ldg(bias_n + threadIdx.x);
            named_bar_sync(1, 256);
            // phase 1: TMEM -> registers (the GEMM result x.W_hi + 2^-11 x.W_lo of this pixel's 128 channels)
            float v[PF_BN];
            mbar_wait(tmem_full, tile_it & 1);
            tc_fence_after();
#pragma unroll
            for (int c = 0; c < PF_BN / 16; ++c) {
                uint32_t hi[16], lo[16];
                tmem_ld16(taddr + c * 16, hi);
                tmem_ld16(taddr + PF_BN + c * 16, lo);
                tmem_ld_wait();
#pragma unroll
                for (int j = 0; j < 16; ++j) v[c * 16 + j] = __fmaf_rn(__uint_as_float(lo[j]), PF_LO_INV, __uint_as_float(hi[j]));
            }
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(tmem_empty);             // the MMA warp may start the next tile
            // phase 2: + bias, * weight, + res, store
#pragma unroll
            for (int c = 0; c < PF_BN / P2_RCH; ++c, ++rc) {
                float r[P2_RCH];
                if (kSum) {
                    const int s = rc % P2_RSLOTS;
                    mbar_wait(rfull + s, (rc / P2_RSLOTS) & 1);
                    const float *rs = res_s + s * (P2_R_BYTES / 4) + px_local;
#pragma unroll
                    for (int j = 0; j < P2_RCH; ++j) r[j] = rs[j * P2_BM];
                }
#pragma unroll
                for (int j = 0; j < P2_RCH; ++j) {
                    float x = v[c * P2_RCH + j];
                    if (bias_n) x = __fadd_rn(x, bias_t[c * P2_RCH + j]);              // conv bias
                    x = __fmul_rn(x, P.weight);                                          // timm.py:177
                    if (kSum) x = __fadd_rn(r[j], x);                                    // timm.py:182
                    if (live) out[(size_t)(c * P2_RCH + j) * hw] = x;
                }
                if (kSum) {
                    // release the slot only after the adds above have CONSUMED r[]: an in-order issue of those FADDs means the
                    // shared-memory reads have returned; arriving right behind the LDS instructions let the refill overtake them
                    __syncwarp();
                    if (lane == 0) mbar_arrive(rempty + (rc % P2_RSLOTS));
                }
            }
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 9) tmem_dealloc(tmem_base, 512);
}

// W (N,K) f32 -> (2N,K) f16: per block of 128 output channels, 128 rows of W_hi then 128 rows of W_lo
__global__ void __launch_bounds__(256) split_weights_kernel(const float *__restrict__ w, int N, int K, __half *__restrict__ out)
{
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= (int64_t)N * K) return;
    const int n = (int)(i / K), k = (int)(i - (int64_t)n * K);
    const float x = __ldg(w + i);
    const __half hi = __float2half_rn(x);
    const __half lo = __float2half_rn(__fmul_rn(__fsub_rn(x, __half2float(hi)), PF_LO_SCALE));
    const int64_t row_hi = (int64_t)(n / PF_BN) * (2 * PF_BN) + (n % PF_BN);
    out[row_hi * K + k] = hi;
    out[(row_hi + PF_BN) * K + k] = lo;
}

// (rows, K) fp16 row-major -> 2-D map with a {64, box_rows} SWIZZLE_128B box; rows beyond `rows` read as zero
int pf_make_tmap(const void *ptr, int64_t rows, int K, int box_rows, CUtensorMap *tm)
{
    const cuuint64_t gdim[2] = {(cuuint64_t)K, (cuuint64_t)rows};
    const cuuint64_t gstr[1] = {(cuuint64_t)K * 2};
    const cuuint32_t box[2] = {PF_BK, (cuuint32_t)box_rows};
    return eod_encode_tmap("eod_project_fuse", tm, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 2, ptr, gdim, gstr, box, CU_TENSOR_MAP_L2_PROMOTION_L2_256B);
}

// level (E, hw, K) f16 -> 3-D map, box {64, 256, 1}: rows beyond hw of an episode read as zero (never the next episode)
int p2_make_tmap_a(const void *ptr, int E, int hw, int K, CUtensorMap *tm)
{
    const cuuint64_t gdim[3] = {(cuuint64_t)K, (cuuint64_t)hw, (cuuint64_t)E};
    const cuuint64_t gstr[2] = {(cuuint64_t)K * 2, (cuuint64_t)hw * K * 2};
    const cuuint32_t box[3] = {PF_BK, P2_BM, 1};
    return eod_encode_tmap("eod_project_fuse", tm, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 3, ptr, gdim, gstr, box, CU_TENSOR_MAP_L2_PROMOTION_L2_256B);
}

// res (E, N, hw) f32 -> 3-D map, box {256 px, 16 channels, 1}
int p2_make_tmap_r(const float *ptr, int E, int hw, int N, CUtensorMap *tm)
{
    const cuuint64_t gdim[3] = {(cuuint64_t)hw, (cuuint64_t)N, (cuuint64_t)E};
    const cuuint64_t gstr[2] = {(cuuint64_t)hw * 4, (cuuint64_t)hw * N * 4};
    const cuuint32_t box[3] = {P2_BM, P2_RCH, 1};
    return eod_encode_tmap("eod_project_fuse", tm, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 3, ptr, gdim, gstr, box, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                           CU_TENSOR_MAP_SWIZZLE_NONE);
}

// the single-level, one-tile-per-CTA kernel: any hw (no TMA on res), also the comparator for the persistent one
int pf_launch_v1(const void *level, const void *w_split, const float *bias, const float *res, float weight, int mode, int n_episodes, int hw,
                 int K, int N, float *out, cudaStream_t st)
{
    const int M = n_episodes * hw;
    CUtensorMap tm_a, tm_b;
    int rc = pf_make_tmap(level, M, K, PF_BM, &tm_a);
    if (rc) return rc;
    rc = pf_make_tmap(w_split, 2 * (int64_t)N, K, 2 * PF_BN, &tm_b);
    if (rc) return rc;
    static unsigned long long attr_done[2] = {0ull, 0ull};
    if (int rc_attr = eod_ensure_dyn_smem(project_fuse_kernel<true>, PF_SMEM_BYTES, &attr_done[0], "eod_project_fuse")) return rc_attr;
    if (int rc_attr = eod_ensure_dyn_smem(project_fuse_kernel<false>, PF_SMEM_BYTES, &attr_done[1], "eod_project_fuse")) return rc_attr;
    const unsigned grid = (unsigned)((M + PF_BM - 1) / PF_BM) * (unsigned)(N / PF_BN);
    if (mode == EOD_FUSE_SUM)
        project_fuse_kernel<true><<<grid, 128, PF_SMEM_BYTES, st>>>(tm_a, tm_b, bias, res, out, weight, M, hw, N, K / PF_BK);
    else
        project_fuse_kernel<false><<<grid, 128, PF_SMEM_BYTES, st>>>(tm_a, tm_b, bias, res, out, weight, M, hw, N, K / PF_BK);
    return eod_check_launch("eod_project_fuse");
}

}  // namespace

extern "C" int eod_project_split_weights(const float *weight, int N, int K, void *w_split, eod_stream_t stream)
{
    EOD_REQUIRE(weight && w_split, EOD_ERR_BADARG, "eod_project_split_weights: null pointer");
    EOD_REQUIRE(N > 0 && K > 0, EOD_ERR_BADARG, "eod_project_split_weights: bad sizes");
    EOD_REQUIRE(N % PF_BN == 0 && K % PF_BK == 0, EOD_ERR_UNSUPPORTED, "eod_project_split_weights: N %% 128 == 0 and K %% 64 == 0 required");
    const int64_t n = (int64_t)N * K;
    split_weights_kernel<<<(unsigned)((n + 255) / 256), 256, 0, (cudaStream_t)stream>>>(weight, N, K, reinterpret_cast<__half *>(w_split));
    return eod_check_launch("eod_project_split_weights");
}

extern "C" int eod_project_fuse_levels(int n_levels, const void *const *level, const void *const *w_split, const float *const *bias,
                                       const float *const *res, float *const *out, const int *hw, float weight, int mode, int n_episodes,
                                       int K, int N, int variant, eod_stream_t stream)
{
    EOD_REQUIRE(level && w_split && out && hw, EOD_ERR_BADARG, "eod_project_fuse_levels: null pointer");
    EOD_REQUIRE(n_levels >= 1 && n_levels <= P2_MAX_LEVELS, EOD_ERR_BADARG, "eod_project_fuse_levels: 1..3 levels");
    EOD_REQUIRE(mode == EOD_FUSE_SUM || mode == EOD_FUSE_MEM_ONLY, EOD_ERR_BADARG, "eod_project_fuse_levels: mode must be sum or mem_only");
    EOD_REQUIRE(mode != EOD_FUSE_SUM || res, EOD_ERR_BADARG, "eod_project_fuse_levels: res is required for sum");
    EOD_REQUIRE(n_episodes > 0 && n_episodes <= 65535, EOD_ERR_BADARG, "eod_project_fuse_levels: bad sizes");
    EOD_REQUIRE(N > 0 && K > 0 && N % PF_BN == 0 && K % PF_BK == 0, EOD_ERR_UNSUPPORTED, "eod_project_fuse_levels: N %% 128 == 0 and K %% 64 == 0 required");
    EOD_REQUIRE(variant >= 0 && variant <= 2, EOD_ERR_BADARG, "eod_project_fuse_levels: variant 0 (auto) | 1 (tile per CTA) | 2 (persistent)");
    bool tma_res_ok = true;
    for (int l = 0; l < n_levels; ++l) {
        EOD_REQUIRE(level[l] && w_split[l] && out[l] && (mode != EOD_FUSE_SUM || res[l]), EOD_ERR_BADARG, "eod_project_fuse_levels: null pointer (level %d)", l);
        EOD_REQUIRE(hw[l] > 0 && (int64_t)n_episodes * hw[l] < (1ll << 31) - P2_BM, EOD_ERR_BADARG, "eod_project_fuse_levels: bad hw (level %d)", l);
        EOD_REQUIRE(eod_aligned16(level[l]) && eod_aligned16(w_split[l]), EOD_ERR_ALIGN, "eod_project_fuse_levels: level and w_split must be 16-byte aligned");
        if (mode == EOD_FUSE_SUM && (hw[l] % 4 != 0 || !eod_aligned16(res[l]))) tma_res_ok = false;     // TMA row pitch must be a multiple of 16 bytes
    }
    cudaStream_t st = (cudaStream_t)stream;
    EOD_REQUIRE(variant != 2 || tma_res_ok, EOD_ERR_UNSUPPORTED, "eod_project_fuse_levels: persistent variant needs hw %% 4 == 0 and 16-byte aligned res");
    if (variant == 1 || !tma_res_ok) {
        for (int l = 0; l < n_levels; ++l) {
            const int rc = pf_launch_v1(level[l], w_split[l], bias ? bias[l] : nullptr, res ? res[l] : nullptr, weight, mode, n_episodes, hw[l], K, N, out[l], st);
            if (rc) return rc;
        }
        return EOD_OK;
    }
    P2Params P;
    memset(&P, 0, sizeof(P));
    P.n_levels = n_levels; P.n_nblocks = N / PF_BN; P.N = N; P.n_kblocks = K / PF_BK; P.weight = weight;
    int tiles = 0;
    for (int l = 0; l < n_levels; ++l) {
        int rc = p2_make_tmap_a(level[l], n_episodes, hw[l], K, &P.tm_a[l]);
        if (rc) return rc;
        rc = pf_make_tmap(w_split[l], 2 * (int64_t)N, K, 2 * PF_BN, &P.tm_b[l]);
        if (rc) return rc;
        if (mode == EOD_FUSE_SUM) {
            rc = p2_make_tmap_r(res[l], n_episodes, hw[l], N, &P.tm_r[l]);
            if (rc) return rc;
        }
        P.bias[l] = bias ? bias[l] : nullptr;
        P.out[l] = out[l];
        P.hw[l] = hw[l];
        P.tiles_per_ep[l] = (hw[l] + P2_BM - 1) / P2_BM;
        P.tile_start[l] = tiles;
        tiles += n_episodes * P.tiles_per_ep[l] * P.n_nblocks;
    }
    for (int l = n_levels; l <= P2_MAX_LEVELS; ++l) P.tile_start[l] = tiles;
    P.n_tiles = tiles;
    static unsigned long long attr_done[2] = {0ull, 0ull};
    if (int rc_attr = eod_ensure_dyn_smem(project_fuse_persistent_kernel<true>, P2_SMEM_BYTES, &attr_done[0], "eod_project_fuse_levels")) return rc_attr;
    if (int rc_attr = eod_ensure_dyn_smem(project_fuse_persistent_kernel<false>, P2_SMEM_BYTES, &attr_done[1], "eod_project_fuse_levels")) return rc_attr;
    const int grid = tiles < eod_num_sms() ? tiles : eod_num_sms();
    if (mode == EOD_FUSE_SUM) project_fuse_persistent_kernel<true><<<grid, P2_THREADS, P2_SMEM_BYTES, st>>>(P);
    else project_fuse_persistent_kernel<false><<<grid, P2_THREADS, P2_SMEM_BYTES, st>>>(P);
    return eod_check_launch("eod_project_fuse_levels");
}

extern "C" int eod_project_fuse(const void *level, const void *w_split, const float *bias, const float *res, float weight, int mode,
                                int n_episodes, int hw, int K, int N, float *out, eod_stream_t stream)
{
    EOD_REQUIRE(level && w_split && out, EOD_ERR_BADARG, "eod_project_fuse: null pointer");
    return eod_project_fuse_levels(1, &level, &w_split, bias ? &bias : nullptr, res ? &res : nullptr, &out, &hw, weight, mode, n_episodes, K, N, 0, stream);
}
