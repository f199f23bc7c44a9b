// Row GEMM with fp32 accuracy on the 5th-generation tensor cores (3xTF32): Y[dst(i), j] = scale * (sum_l A(i,l) * B(j,l) + bias[j]).
//
// The path's small dense contractions that are NOT the fp16-valued read levels of csrc/project_fuse.cu: the 'replace' update of the
// SMNet height-max write (state[winner cells] = linlayer(feature[winner pixels]): SMNet/__pycache__/model.cpython-310.pyc, listing
// smnet_encode_model_py310.txt src lines 126-128), the 1x1 forward projection of the dense backbone-feature write (A7''), the
// projection of per-ROI memory features, and the training path of the fusion (forward and both gradients).  They used to run on the
// library's fp32 GEMM; this kernel keeps them in-tree.
//
// tcgen05.mma kind::tf32 multiplies 10-bit-mantissa operands.  Every fp32 operand x is split on the fly into two tf32 numbers,
// big = tf32(x) and small = tf32(x - big) (round to nearest; x - big is exact in fp32), and the product is accumulated as
// small*big + big*small + big*big in the fp32 accumulator in TMEM: the dropped terms are below 2^-21 of |a*b| and of either sign,
// the same order as the rounding of an fp32 FMA chain (measured against fp64 in tests/test_gpu_parity.py).
//
// One CTA per 128-row tile of A x up to 256 columns; 128 threads:
//   all threads : gather their A row (any row / element stride, optional per-row offsets: winner pixels of a CHW feature tensor) and
//                 B rows of the 32-wide K chunk, split, and store both halves into shared memory in the canonical K-major
//                 SWIZZLE_128B layout (what a TMA box {32 fp32, rows} would produce) - two stages, so chunk k+1 is loaded while the
//                 tensor core works on chunk k;
//   thread 0    : 4 k-steps x 3 tcgen05.mma (M=128, N, K=8) per chunk, tcgen05.commit frees the stage;
//   all threads : epilogue - tcgen05.ld of the thread's row, + bias, * scale, row store (optionally scattered: dst row ids).
// Rows beyond *m_count (device-side count: the number of winners is only known on the device) are skipped.
#include "eod_common.cuh"

namespace {

constexpr int LN_BM = 128;                 // rows per tile = TMEM lanes
constexpr int LN_BK = 32;                  // fp32 elements per 128-byte swizzle row
constexpr int LN_MAXN = 256;
constexpr int LN_A_BYTES = LN_BM * 128;    // one half (big or small) of the A chunk
constexpr int LN_B_BYTES = LN_MAXN * 128;
constexpr int LN_STAGE_BYTES = 2 * LN_A_BYTES + 2 * LN_B_BYTES;     // 96 KB
constexpr int LN_SMEM_BYTES = 2 * LN_STAGE_BYTES + 1024 + 64;

// instruction descriptor: D = F32 (1 << 4), A = B = TF32 (2 << 7, 2 << 10), both K-major, N >> 3 in [17,23), M >> 4 in [24,29)
__device__ __forceinline__ uint32_t ln_idesc(int n) { return (1u << 4) | (2u << 7) | (2u << 10) | ((uint32_t)(n >> 3) << 17) | ((uint32_t)(LN_BM >> 4) << 24); }

// nearest tf32 (10-bit mantissa, low 13 bits zero).  Rounding - not truncation - keeps the split's residual symmetric: with truncated
// halves the error of every product has the sign of the product and grows linearly in K (measured 4.5e-6 of scale at K=512).
__device__ __forceinline__ float tf32_big(float x)
{
    uint32_t r;
    asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(r) : "f"(x));
    return __uint_as_float(r);
}

// second half of the split; a non-finite x has no remainder (inf - inf would turn an infinite product into NaN)
__device__ __forceinline__ float tf32_small(float x, float big)
{
    const float d = __fsub_rn(x, big);
    return (__float_as_uint(big) & 0x7f800000u) == 0x7f800000u ? 0.f : tf32_big(d);
}

// one 16-byte chunk (4 consecutive k) of row `r` of a chunk tile -> its swizzled place in the big / small halves
__device__ __forceinline__ void ln_store4(uint32_t big_base, uint32_t small_base, int r, int c, float4 x)
{
    const uint32_t off = (uint32_t)((r >> 3) * 1024 + (r & 7) * 128 + ((c ^ (r & 7)) << 4));
    float4 b, s;
    b.x = tf32_big(x.x); b.y = tf32_big(x.y); b.z = tf32_big(x.z); b.w = tf32_big(x.w);
    s.x = tf32_small(x.x, b.x); s.y = tf32_small(x.y, b.y); s.z = tf32_small(x.z, b.z); s.w = tf32_small(x.w, b.w);
    // f32 stores, not sts128: moving the halves into .b32 registers makes ptxas spill in linear_rows_kernel
    asm volatile("st.shared.v4.f32 [%0], {%1, %2, %3, %4};" ::"r"(big_base + off), "f"(b.x), "f"(b.y), "f"(b.z), "f"(b.w) : "memory");
    asm volatile("st.shared.v4.f32 [%0], {%1, %2, %3, %4};" ::"r"(small_base + off), "f"(s.x), "f"(s.y), "f"(s.z), "f"(s.w) : "memory");
}

// the 32-wide K chunk starting at k0 of one operand row (base pointer of the row, element stride ks; valid = row exists)
__device__ __forceinline__ void ln_load_row(const float *row, int64_t ks, bool vec, bool valid, int k0, int K, uint32_t big_base, uint32_t small_base, int r)
{
#pragma unroll
    for (int c = 0; c < LN_BK / 4; ++c) {
        const int k = k0 + 4 * c;
        float4 x = make_float4(0.f, 0.f, 0.f, 0.f);
        if (valid && k < K) {
            if (vec) {
                x = __ldg(reinterpret_cast<const float4 *>(row + k));          // K % 4 == 0 on this path
            } else {
                x.x = __ldg(row + (int64_t)k * ks);
                if (k + 1 < K) x.y = __ldg(row + (int64_t)(k + 1) * ks);
                if (k + 2 < K) x.z = __ldg(row + (int64_t)(k + 2) * ks);
                if (k + 3 < K) x.w = __ldg(row + (int64_t)(k + 3) * ks);
            }
        }
        ln_store4(big_base, small_base, r, c, x);
    }
}

struct LinearParams {
    const float *A; int64_t a_rs, a_ks; const int64_t *a_off;
    const float *B; int64_t b_rs, b_ks;
    const float *bias; float scale;
    int M, N, K; const int32_t *m_count;
    float *Y; int64_t y_rs; const int64_t *y_dst;
};

__global__ void __launch_bounds__(128) linear_rows_kernel(const LinearParams P)
{
    extern __shared__ uint8_t ln_smem_raw[];
    const uint32_t smem = (smem_u32(ln_smem_raw) + 1023u) & ~1023u;
    uint8_t *gen = ln_smem_raw + (smem - smem_u32(ln_smem_raw));
    uint64_t *bars = reinterpret_cast<uint64_t *>(gen + 2 * LN_STAGE_BYTES);       // [0,1]: MMAs of a stage done; [2]: accumulator complete
    uint32_t *tmem_slot = reinterpret_cast<uint32_t *>(bars + 3);

    const int tid = threadIdx.x, warp = tid >> 5;
    const int M = P.m_count ? min(P.M, __ldg(P.m_count)) : P.M;
    const int m0 = blockIdx.x * LN_BM;
    if (m0 >= M) return;                                    // uniform for the CTA: nothing was allocated yet
    const int N = P.N, K = P.K;
    const uint32_t tmem_cols = N <= 32 ? 32u : (N <= 64 ? 64u : (N <= 128 ? 128u : 256u));

    if (tid == 0) {
        mbar_init(bars + 0, 1);
        mbar_init(bars + 1, 1);
        mbar_init(bars + 2, 1);
        mbar_fence_init();
    }
    if (warp == 0) tmem_alloc(tmem_slot, tmem_cols);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;

    // this thread's operand rows
    const int m = m0 + tid;
    const bool a_valid = m < M;
    const float *a_row = P.A + (a_valid ? (P.a_off ? __ldg(P.a_off + m) : (int64_t)m * P.a_rs) : 0);
    const bool a_vec = P.a_ks == 1 && (K & 3) == 0 && ((reinterpret_cast<uintptr_t>(a_row) & 15u) == 0);
    const bool b_vec = P.b_ks == 1 && (K & 3) == 0 && (P.b_rs & 3) == 0 && ((reinterpret_cast<uintptr_t>(P.B) & 15u) == 0);
    const uint32_t idesc = ln_idesc(N);
    const int n_kb = (K + LN_BK - 1) / LN_BK;

    for (int kb = 0; kb < n_kb; ++kb) {
        const int s = kb & 1;
        if (kb >= 2) mbar_wait(bars + s, ((kb >> 1) - 1) & 1);            // the MMAs that read this stage two chunks ago have completed
        const uint32_t a_big = smem + s * LN_STAGE_BYTES, a_small = a_big + LN_A_BYTES, b_big = a_small + LN_A_BYTES, b_small = b_big + LN_B_BYTES;
        ln_load_row(a_row, P.a_ks, a_vec, a_valid, kb * LN_BK, K, a_big, a_small, tid);
        for (int j = tid; j < N; j += LN_BM) ln_load_row(P.B + (int64_t)j * P.b_rs, P.b_ks, b_vec, true, kb * LN_BK, K, b_big, b_small, j);
        fence_proxy_async();                                 // generic-proxy stores -> visible to the tensor core's async-proxy reads
        __syncthreads();
        if (tid == 0) {
            tc_fence_after();
#pragma unroll
            for (int k = 0; k < LN_BK / 8; ++k) {            // 8 tf32 = 32 bytes along K inside the swizzle row
                const uint64_t ab = umma_desc_sw128(a_big + k * 32), as = umma_desc_sw128(a_small + k * 32);
                const uint64_t bb = umma_desc_sw128(b_big + k * 32), bs = umma_desc_sw128(b_small + k * 32);
                umma_tf32(tmem_base, as, bb, idesc, (kb | k) != 0);       // small terms first, the dominant one last
                umma_tf32(tmem_base, ab, bs, idesc, 1u);
                umma_tf32(tmem_base, ab, bb, idesc, 1u);
            }
            umma_commit(bars + s);
            if (kb == n_kb - 1) umma_commit(bars + 2);
        }
    }

    // ===== epilogue: warp w owns TMEM lanes [32w, 32w + 32) = rows m0 + 32w + lane =====
    mbar_wait(bars + 2, 0);
    tc_fence_after();
    const uint32_t taddr = tmem_base + ((uint32_t)(warp * 32) << 16);
    float *y_row = a_valid ? P.Y + (P.y_dst ? __ldg(P.y_dst + m) : (int64_t)m) * P.y_rs : nullptr;
    const bool y_vec = (P.y_rs & 3) == 0 && ((reinterpret_cast<uintptr_t>(P.Y) & 15u) == 0);
#pragma unroll 1
    for (int c0 = 0; c0 < N; c0 += 16) {
        uint32_t acc[16];
        tmem_ld16(taddr + c0, acc);
        tmem_ld_wait();
        if (a_valid) {
            float v[16];
#pragma unroll
            for (int j = 0; j < 16; ++j) {
                float x = __uint_as_float(acc[j]);
                if (P.bias) x = __fadd_rn(x, __ldg(P.bias + c0 + j));
                v[j] = __fmul_rn(x, P.scale);
            }
            if (y_vec) {
#pragma unroll
                for (int j = 0; j < 4; ++j) reinterpret_cast<float4 *>(y_row + c0)[j] = make_float4(v[4 * j], v[4 * j + 1], v[4 * j + 2], v[4 * j + 3]);
            } else {
#pragma unroll
                for (int j = 0; j < 16; ++j) y_row[c0 + j] = v[j];
            }
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 0) tmem_dealloc(tmem_base, tmem_cols);
}

// winners of eod_write_max -> compact (source element offset, destination row) list for the 'replace' update
__global__ void __launch_bounds__(256) winner_list_kernel(const int32_t *__restrict__ arg_pix, int64_t n_cells, int64_t total, int HW, int C, int layout,
                                                          int64_t *__restrict__ src_off, int64_t *__restrict__ dst_row, int32_t *__restrict__ count, int cap)
{
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const int p = i < total ? __ldg(arg_pix + i) : -1;
    const unsigned lane = threadIdx.x & 31;
    const unsigned won = __ballot_sync(0xffffffffu, p >= 0);
    if (!won) return;
    int base = 0;
    if (lane == 0) base = atomicAdd(count, __popc(won));
    base = __shfl_sync(0xffffffffu, base, 0);
    if (p >= 0) {
        const int slot = base + __popc(won & ((1u << lane) - 1u));
        if (slot < cap) {
            const int64_t e = i / n_cells;
            src_off[slot] = layout == EOD_LAYOUT_HWC ? (e * HW + p) * (int64_t)C : e * (int64_t)C * HW + p;
            dst_row[slot] = i;
        }
    }
}

}  // namespace

extern "C" int eod_linear_rows(const float *A, int64_t a_row_stride, int64_t a_k_stride, const int64_t *a_off, const float *B, int64_t b_row_stride,
                               int64_t b_k_stride, const float *bias, float scale, int M, const int32_t *m_count, int N, int K, float *Y,
                               int64_t y_row_stride, const int64_t *y_dst, eod_stream_t stream)
{
    EOD_REQUIRE(A && B && Y, EOD_ERR_BADARG, "eod_linear_rows: null pointer");
    EOD_REQUIRE(M >= 0 && K > 0, EOD_ERR_BADARG, "eod_linear_rows: bad sizes");
    EOD_REQUIRE(N >= 16 && N % 16 == 0, EOD_ERR_UNSUPPORTED, "eod_linear_rows: N must be a multiple of 16 (got %d)", N);
    EOD_REQUIRE(y_row_stride >= N, EOD_ERR_BADARG, "eod_linear_rows: y_row_stride < N");
    if (M == 0) return EOD_OK;
    static unsigned long long attr_done = 0ull;
    if (int rc = eod_ensure_dyn_smem(linear_rows_kernel, LN_SMEM_BYTES, &attr_done, "eod_linear_rows")) return rc;
    const int tiles = (M + LN_BM - 1) / LN_BM;
    for (int n0 = 0; n0 < N; n0 += LN_MAXN) {                 // column blocks of up to 256 (one TMEM allocation each)
        const int nb = N - n0 < LN_MAXN ? N - n0 : LN_MAXN;
        LinearParams P{A, a_row_stride, a_k_stride, a_off, B + (int64_t)n0 * b_row_stride, b_row_stride, b_k_stride, bias ? bias + n0 : nullptr, scale,
                       M, nb, K, m_count, Y + n0, y_row_stride, y_dst};
        linear_rows_kernel<<<tiles, 128, LN_SMEM_BYTES, (cudaStream_t)stream>>>(P);
        if (int rc = eod_check_launch("eod_linear_rows")) return rc;
    }
    return EOD_OK;
}

extern "C" int eod_max_winner_list(const int32_t *arg_pix, int n_episodes, int64_t n_cells, int H, int W, int C, int layout, int64_t *src_off,
                                   int64_t *dst_row, int32_t *count, int capacity, eod_stream_t stream)
{
    EOD_REQUIRE(arg_pix && src_off && dst_row && count, EOD_ERR_BADARG, "eod_max_winner_list: null pointer");
    EOD_REQUIRE(n_episodes > 0 && n_cells > 0 && H > 0 && W > 0 && C > 0 && capacity > 0, EOD_ERR_BADARG, "eod_max_winner_list: bad sizes");
    EOD_REQUIRE(layout == EOD_LAYOUT_CHW || layout == EOD_LAYOUT_HWC, EOD_ERR_BADARG, "eod_max_winner_list: bad layout");
    cudaStream_t st = (cudaStream_t)stream;
    const cudaError_t err = cudaMemsetAsync(count, 0, sizeof(int32_t), st);
    EOD_REQUIRE(err == cudaSuccess, EOD_ERR_LAUNCH, "eod_max_winner_list: memset failed: %s", cudaGetErrorString(err));
    const int64_t total = (int64_t)n_episodes * n_cells;
    const int64_t blocks = (total + 255) / 256;
    EOD_REQUIRE(blocks < (1ll << 31), EOD_ERR_BADARG, "eod_max_winner_list: grid too large");
    winner_list_kernel<<<(unsigned)blocks, 256, 0, st>>>(arg_pix, n_cells, total, H * W, C, layout, src_off, dst_row, count, capacity);
    return eod_check_launch("eod_max_winner_list");
}
