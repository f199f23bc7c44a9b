// Memory write, mean mode (SURVEY 8a rows A6-A8).
//
//   pre-pass   eod_frame_count      n_c  = #sampled pixels per cell (+ visibility bit)      [index plane only]
//   main pass  eod_write_mean       sums[c] += (sum over the cell's sampled pixels of f_p) / n_c
//   post-pass  eod_finalize_counts  counts[c] += 1 for every visible cell ; scratch := 0
//
// The main pass streams the per-pixel feature tensor exactly once (N*C*4 bytes per frame - the term that
// bounds the whole path) and is written for HBM bandwidth:
//   * CHW features (the reference's (1,C,480,640) layout): a persistent CTA per SM, 6 consumer warps + 1 producer
//     warp.  Unit of work = (32-pixel tile, 256-channel block) = one 32 KB 3-D TMA box (128B-swizzled; at C=128 the whole
//     tile, 16 KB, with 12 consumer warps) plus bulk copies of the tile's cell ids / sample mask (/ reciprocal divisors in
//     pixel_divisors mode); the producer CLAIMS chunks of tile groups from a global ticket (eod_work_tickets), the stage a
//     unit lands in belongs to one consumer warp (the full/empty mbarrier pair of the stage is the only synchronisation; the
//     unit's {tile, channel block} travels in the stage's aux area).  All pixels of the tile that fall into one cell form a
//     group (MATCH.ANY; runs in the deterministic variant): lane l sums channels l, l+32, ..., l+224 over the group's pixels
//     with conflict-free LDS.128, scales by 1/n_cell (looked up in frame_cnt) and the group leaves the SM as eight warp-wide
//     red.global.add.f32 (128 contiguous bytes of the cell row each) - one L2 reduction per (tile, cell, channel) instead of
//     one per pixel.  DESIGN.md 3.1.
//   * bf16 / fp16 CHW features (EOD_LAYOUT_CHW_BF16 / _F16: a 16-bit backbone's NCHW output) take the same ring with 64-pixel
//     units - a box row is again 128 bytes, so the unit, the swizzle and the ring are unchanged - and are widened exactly before the
//     fp32 arithmetic above (DESIGN.md 3.1c).
//   * an LDG-staged variant of the same algorithm (padded smem tile, runs) handles shapes the TMA path does
//     not (HW % 32 != 0; 16-bit: HW % 64 != 0) and is the bring-up comparator (variant = EOD_WRITE_LDG).
//   * HWC features (fp32 / bf16 / fp16): a warp owns a strip of 32 pixels, lanes own float4 channel groups; the strip's pixels
//     are grouped by cell the same way, a group's rows are requested in batches before they are added, and the group is
//     flushed straight from registers (red.global.add.v4.f32).
//   * deterministic variant (eod_write_mean_det_layout): fp32 CHW through the TMA ring, fp32 / bf16 / fp16 channels-last through the
//     HWC kernel; both store raster-ordered run sums that the same segmented reduce adds in a fixed order.
#include <cuda.h>
#include <stdio.h>
#include <stdlib.h>

#include "det.cuh"
#include "eod_common.cuh"
#include "tmap_cache.cuh"

namespace {

// ------------------------------------------------------------------------------------------------------
// pre-pass / post-pass: one thread per pixel, warp-level run aggregation of the cell id
// ------------------------------------------------------------------------------------------------------
constexpr int kCountSpan = 4;

__global__ void __launch_bounds__(256) frame_count_kernel(const int32_t *__restrict__ idx, const uint8_t *__restrict__ samp,
                                                          const int32_t *__restrict__ active, int HW, int64_t n_cells,
                                                          uint32_t *__restrict__ frame_cnt, int32_t *__restrict__ slot_of_cell,
                                                          int32_t *__restrict__ slot_cell, int32_t *__restrict__ n_slots, int S)
{
    const int e = blockIdx.y;
    if (active && __ldg(active + e) <= 0) return;      // episode without a kept detection: no write, no visibility (custom_rcnn.py:686)
    const unsigned lane = threadIdx.x & 31;
    // kCountSpan consecutive 256-pixel spans per CTA, all loads issued first: a quarter of the CTAs (the launch was bound by block
    // scheduling: 77 k CTAs of a dozen instructions at E=64) and four independent loads in flight per thread
    int cellv[kCountSpan];
    bool sv[kCountSpan], validv[kCountSpan];
#pragma unroll
    for (int it = 0; it < kCountSpan; ++it) {
        const int p = (blockIdx.x * kCountSpan + it) * (int)blockDim.x + (int)threadIdx.x;
        validv[it] = p < HW;
        const size_t g = (size_t)e * HW + (validv[it] ? p : 0);
        cellv[it] = validv[it] ? __ldg(idx + g) : -1;
        sv[it] = validv[it] && (samp ? __ldg(samp + g) != 0 : true);
    }
#pragma unroll
    for (int it = 0; it < kCountSpan; ++it) {
        const int cell = cellv[it];
        const bool valid = validv[it];
        const int prev = __shfl_up_sync(0xffffffffu, cell, 1);
        const bool head = valid && (lane == 0 || prev != cell);
        const unsigned heads = __ballot_sync(0xffffffffu, head);
        const unsigned samps = __ballot_sync(0xffffffffu, sv[it]);
        const unsigned valids = __ballot_sync(0xffffffffu, valid);
        if (head) {
            const unsigned above = heads & ~((2u << lane) - 1u);               // heads strictly after this lane
            const unsigned end = above ? (unsigned)(__ffs(above) - 1) : 32u;   // run = [lane, end)
            const unsigned run = ((end >= 32u) ? 0xffffffffu : ((1u << end) - 1u)) & ~((1u << lane) - 1u) & valids;
            const unsigned n = __popc(samps & run);
            uint32_t *dst = frame_cnt + (size_t)e * n_cells + cell;
            if (n) {
                const uint32_t old = atomicAdd(dst, n);
                if (slot_of_cell && (old & 0x7fffffffu) == 0u) {               // first samples of this cell in this frame: claim a slot
                    const int sl = atomicAdd(n_slots + e, 1);
                    if (sl < S) {
                        slot_of_cell[(size_t)e * n_cells + cell] = sl + 1;
                        slot_cell[(size_t)e * S + sl] = cell;
                    }
                }
            } else atomicOr(dst, 0x80000000u);
        }
    }
}

__global__ void __launch_bounds__(256) finalize_counts_kernel(const int32_t *__restrict__ idx, int HW, int64_t n_cells,
                                                              uint32_t *__restrict__ frame_cnt, float *__restrict__ counts,
                                                              uint8_t *__restrict__ touched, const float *__restrict__ sums,
                                                              __half *__restrict__ norm16, int C)
{
    const int e = blockIdx.y;
    const int p = blockIdx.x * blockDim.x + threadIdx.x;
    const unsigned lane = threadIdx.x & 31;
    const bool valid = p < HW;
    const int cell = valid ? __ldg(idx + (size_t)e * HW + p) : -1;
    const int prev = __shfl_up_sync(0xffffffffu, cell, 1);
    bool win = false;
    float n_new = 0.f;
    if (valid && (lane == 0 || prev != cell)) {
        const size_t c = (size_t)e * n_cells + cell;
        const uint32_t old = atomicExch(frame_cnt + c, 0u);   // exactly one run head per cell sees old != 0
        if (old) {
            n_new = counts[c] + 1.0f;                        // custom_rcnn.py:699-701,743
            counts[c] = n_new;
            if (touched && (old & 0x7fffffffu)) touched[c] = 1;
            win = true;
        }
    }
    if (!norm16) return;
    // Refresh the normalised fp16 row (custom_rcnn.py:764-774 + :1036) of every visible cell: its count just
    // changed, so its normalised value did.  The warp serves its winners cooperatively (lanes over channels).
    unsigned todo = __ballot_sync(0xffffffffu, win);
    while (todo) {
        const int src = __ffs(todo) - 1;
        todo &= todo - 1;
        const int wc = __shfl_sync(0xffffffffu, cell, src);
        const float wn = __shfl_sync(0xffffffffu, n_new, src);
        const size_t row = ((size_t)e * n_cells + wc) * C;
        const float4 *src_row = reinterpret_cast<const float4 *>(sums + row);
        uint2 *dst_row = reinterpret_cast<uint2 *>(norm16 + row);
        for (int k = lane; k < C / 4; k += 32) {
            float4 v = src_row[k];
            if (wn > 1.0f) { v.x = __fdiv_rn(v.x, wn); v.y = __fdiv_rn(v.y, wn); v.z = __fdiv_rn(v.z, wn); v.w = __fdiv_rn(v.w, wn); }
            __half2 a = __floats2half2_rn(v.x, v.y), b = __floats2half2_rn(v.z, v.w);
            uint2 raw;
            raw.x = *reinterpret_cast<uint32_t *>(&a);
            raw.y = *reinterpret_cast<uint32_t *>(&b);
            dst_row[k] = raw;
        }
    }
}

// Same post-pass driven by the CELL plane instead of the pixel plane: a warp scans 32 consecutive cells of
// frame_cnt (coalesced, no atomics - every cell has exactly one owner), bumps the counts of the non-zero ones and
// refreshes their fp16 rows.  Cheaper than the pixel-driven pass whenever the grid is not much larger than the
// image (E*cells*4 bytes streamed instead of E*HW*4 plus one atomic per run of pixels).
__global__ void __launch_bounds__(256) finalize_cells_kernel(int64_t n_rows, int64_t n_cells, uint32_t *__restrict__ frame_cnt,
                                                             float *__restrict__ counts, uint8_t *__restrict__ touched,
                                                             const float *__restrict__ sums, __half *__restrict__ norm16, int C)
{
    // Visible cells are rare (a few hundred of 250 000 per episode) and clustered (a frustum footprint): a block scans
    // 2048 cells per trip, 16 bytes per lane (8 KB of frame_cnt in flight per block), collects the visible ones in shared
    // memory, and then refreshes their fp16 rows with all 8 warps, two rows and up to 8 independent 16-byte loads per lane
    // in flight - a warp that owns the footprint no longer walks its rows one dependent load at a time.
    constexpr int kCellsPerTrip = 2048;
    __shared__ int s_row[kCellsPerTrip];
    __shared__ float s_new[kCellsPerTrip];
    __shared__ int s_cnt;
    const unsigned lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int64_t n_vec = n_rows >> 2;                              // the host guarantees n_rows % 4 == 0 and 16-byte alignment
    const uint4 *cnt4 = reinterpret_cast<const uint4 *>(frame_cnt);
    for (int64_t vb = (int64_t)blockIdx.x * (kCellsPerTrip / 4); vb < n_vec; vb += (int64_t)gridDim.x * (kCellsPerTrip / 4)) {
        if (threadIdx.x == 0) s_cnt = 0;
        __syncthreads();
        uint4 q[2];
#pragma unroll
        for (int u = 0; u < 2; ++u) {
            const int64_t vi = vb + warp * 64 + u * 32 + lane;
            q[u] = vi < n_vec ? __ldcs(cnt4 + vi) : make_uint4(0u, 0u, 0u, 0u);
        }
#pragma unroll
        for (int u = 0; u < 2; ++u) {
            if ((q[u].x | q[u].y | q[u].z | q[u].w) == 0u) continue;
            const int local = (warp * 64 + u * 32 + lane) * 4;
            const int64_t row0 = vb * 4 + local;
            const uint32_t v[4] = {q[u].x, q[u].y, q[u].z, q[u].w};
            reinterpret_cast<uint4 *>(frame_cnt)[vb + warp * 64 + u * 32 + lane] = make_uint4(0u, 0u, 0u, 0u);
#pragma unroll
            for (int b = 0; b < 4; ++b)
                if (v[b]) {
                    const float n_new = counts[row0 + b] + 1.0f;     // custom_rcnn.py:699-701,743
                    counts[row0 + b] = n_new;
                    if (touched && (v[b] & 0x7fffffffu)) touched[row0 + b] = 1;
                    if (norm16) {
                        const int pos = atomicAdd(&s_cnt, 1);
                        s_row[pos] = local + b;
                        s_new[pos] = n_new;
                    }
                }
        }
        __syncthreads();
        const int n = s_cnt;
        const int c4 = C >> 2;
        for (int i0 = warp; i0 < n; i0 += 16) {                      // rows i0 and i0 + 8 together
            float4 x[2][4];
            float wn[2];
            size_t r[2];
#pragma unroll
            for (int h = 0; h < 2; ++h) {
                const int i = i0 + 8 * h;
                wn[h] = i < n ? s_new[i] : 0.f;
                r[h] = i < n ? (size_t)(vb * 4 + s_row[i]) * C : 0;
#pragma unroll
                for (int k = 0; k < 4; ++k)
                    if (i < n && (int)lane + 32 * k < c4) x[h][k] = reinterpret_cast<const float4 *>(sums + r[h])[lane + 32 * k];
            }
#pragma unroll
            for (int h = 0; h < 2; ++h) {
                if (i0 + 8 * h >= n) continue;
                uint2 *dst_row = reinterpret_cast<uint2 *>(norm16 + r[h]);
#pragma unroll
                for (int k = 0; k < 4; ++k) {
                    if ((int)lane + 32 * k >= c4) continue;
                    float4 y = x[h][k];
                    if (wn[h] > 1.0f) { y.x = __fdiv_rn(y.x, wn[h]); y.y = __fdiv_rn(y.y, wn[h]); y.z = __fdiv_rn(y.z, wn[h]); y.w = __fdiv_rn(y.w, wn[h]); }
                    __half2 a = __floats2half2_rn(y.x, y.y), b2 = __floats2half2_rn(y.z, y.w);
                    uint2 raw;
                    raw.x = *reinterpret_cast<uint32_t *>(&a);
                    raw.y = *reinterpret_cast<uint32_t *>(&b2);
                    dst_row[lane + 32 * k] = raw;
                }
                for (int k = lane + 128; k < c4; k += 32) {          // C > 512
                    float4 y = reinterpret_cast<const float4 *>(sums + r[h])[k];
                    if (wn[h] > 1.0f) { y.x = __fdiv_rn(y.x, wn[h]); y.y = __fdiv_rn(y.y, wn[h]); y.z = __fdiv_rn(y.z, wn[h]); y.w = __fdiv_rn(y.w, wn[h]); }
                    __half2 a = __floats2half2_rn(y.x, y.y), b2 = __floats2half2_rn(y.z, y.w);
                    uint2 raw;
                    raw.x = *reinterpret_cast<uint32_t *>(&a);
                    raw.y = *reinterpret_cast<uint32_t *>(&b2);
                    dst_row[k] = raw;
                }
            }
        }
        __syncthreads();
    }
}

// pix_n[p] = 1 / (number of sampled pixels of p's cell in this frame), correctly rounded: lets the main pass take
// the scale of a run from the staged tile instead of a dependent global load (and a division) per run.
__global__ void __launch_bounds__(256) expand_counts_kernel(const int32_t *__restrict__ idx, const uint32_t *__restrict__ frame_cnt,
                                                            int HW, int64_t n_cells, float *__restrict__ pix_n)
{
    const int e = blockIdx.y;
    const int p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= HW) return;
    const size_t g = (size_t)e * HW + p;
    const uint32_t n = __ldg(frame_cnt + (size_t)e * n_cells + __ldg(idx + g)) & 0x7fffffffu;
    pix_n[g] = n ? __frcp_rn((float)n) : 0.f;
}

// four pixels per thread (HW % 4 == 0, 16-byte aligned planes): 128-bit index load and divisor store, four gathers in flight
__global__ void __launch_bounds__(256) expand_counts_vec4_kernel(const int32_t *__restrict__ idx, const uint32_t *__restrict__ frame_cnt,
                                                                 int HW, int64_t n_cells, float *__restrict__ pix_n)
{
    const int e = blockIdx.y;
    const int p = (blockIdx.x * blockDim.x + threadIdx.x) * 4;
    if (p >= HW) return;
    const size_t g = (size_t)e * HW + p;
    const int4 c = __ldg(reinterpret_cast<const int4 *>(idx + g));
    const uint32_t *cnt = frame_cnt + (size_t)e * n_cells;
    const uint32_t n0 = __ldg(cnt + c.x) & 0x7fffffffu, n1 = __ldg(cnt + c.y) & 0x7fffffffu, n2 = __ldg(cnt + c.z) & 0x7fffffffu,
                   n3 = __ldg(cnt + c.w) & 0x7fffffffu;
    *reinterpret_cast<float4 *>(pix_n + g) = make_float4(n0 ? __frcp_rn((float)n0) : 0.f, n1 ? __frcp_rn((float)n1) : 0.f,
                                                         n2 ? __frcp_rn((float)n2) : 0.f, n3 ? __frcp_rn((float)n3) : 0.f);
}

// ------------------------------------------------------------------------------------------------------
// raster-order every-stride-th-observed-pixel selection (custom_rcnn.py:905-914): one CTA per episode,
// chunked block scan with a running carry.
// ------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(1024) sample_mask_kernel(const uint8_t *__restrict__ observed, int HW, int stride,
                                                           uint8_t *__restrict__ samp, int32_t *__restrict__ n_sampled)
{
    __shared__ int s_warp[32];
    __shared__ int s_carry;
    const int e = blockIdx.x;
    const uint8_t *obs = observed + (size_t)e * HW;
    uint8_t *out = samp + (size_t)e * HW;
    const unsigned lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    if (threadIdx.x == 0) s_carry = 0;
    __syncthreads();
    int sampled_total = 0;
    for (int base = 0; base < HW; base += 1024) {
        const int p = base + threadIdx.x;
        const bool o = p < HW && obs[p] != 0;
        const unsigned bal = __ballot_sync(0xffffffffu, o);
        const int within = __popc(bal & ((1u << lane) - 1u));
        if (lane == 0) s_warp[warp] = __popc(bal);
        __syncthreads();
        int pre = 0;
        for (int w = 0; w < (int)warp; ++w) pre += s_warp[w];      // 32 broadcast reads; negligible
        const int carry = s_carry;
        const int rank = carry + pre + within;
        const bool s = o && (rank % stride == 0);
        if (p < HW) out[p] = s ? 1 : 0;
        sampled_total += s ? 1 : 0;
        __syncthreads();
        if (threadIdx.x == 1023) s_carry = carry + pre + __popc(bal);
        __syncthreads();
    }
    if (n_sampled) {
        // block reduction of sampled_total
        for (int o = 16; o > 0; o >>= 1) sampled_total += __shfl_xor_sync(0xffffffffu, sampled_total, o);
        if (lane == 0) s_warp[warp] = sampled_total;
        __syncthreads();
        if (threadIdx.x == 0) {
            int t = 0;
            for (int w = 0; w < 32; ++w) t += s_warp[w];
            n_sampled[e] = t;
        }
    }
}

// Same selection, 16 pixels per thread (HW % 16 == 0, 16-byte aligned planes): 16 KB of the plane per block-wide scan step
// instead of 1 KB - the 480x640 plane takes 19 steps instead of 300.
__global__ void __launch_bounds__(1024) sample_mask_vec_kernel(const uint8_t *__restrict__ observed, int HW, int stride,
                                                               uint8_t *__restrict__ samp, int32_t *__restrict__ n_sampled)
{
    __shared__ int s_warp[2][32];
    const int e = blockIdx.x;
    const uint4 *obs = reinterpret_cast<const uint4 *>(observed + (size_t)e * HW);
    uint4 *out = reinterpret_cast<uint4 *>(samp + (size_t)e * HW);
    const unsigned lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int n_vec = HW >> 4;
    int carry = 0, sampled_total = 0, buf = 0;
    for (int base = 0; base < n_vec; base += 1024, buf ^= 1) {
        const int vi = base + threadIdx.x;
        uint4 q = vi < n_vec ? __ldg(obs + vi) : make_uint4(0u, 0u, 0u, 0u);
        uint32_t w[4] = {q.x, q.y, q.z, q.w};
        int cnt = 0;
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            // per byte: 0x01 where the byte is non-zero
            uint32_t nz = w[k] | (w[k] >> 4);
            nz |= nz >> 2;
            nz |= nz >> 1;
            w[k] = nz & 0x01010101u;
            cnt += __popc(w[k]);
        }
        int incl = cnt;                                              // inclusive warp scan of the per-thread counts
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const int up = __shfl_up_sync(0xffffffffu, incl, o);
            if ((int)lane >= o) incl += up;
        }
        if (lane == 31) s_warp[buf][warp] = incl;
        __syncthreads();                                             // double-buffered totals: one barrier per step
        int pre = 0, total = 0;
#pragma unroll 8
        for (int x = 0; x < 32; ++x) {
            const int t = s_warp[buf][x];
            pre += x < (int)warp ? t : 0;
            total += t;
        }
        int r = (carry + pre + incl - cnt) % stride;                 // rank of this thread's first observed pixel, mod stride
        carry += total;
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            uint32_t o4 = 0;
#pragma unroll
            for (int b = 0; b < 4; ++b)
                if ((w[k] >> (8 * b)) & 1u) {
                    if (r == 0) { o4 |= 1u << (8 * b); ++sampled_total; }
                    if (++r == stride) r = 0;
                }
            w[k] = o4;
        }
        if (vi < n_vec) out[vi] = make_uint4(w[0], w[1], w[2], w[3]);
    }
    if (n_sampled) {
        for (int o = 16; o > 0; o >>= 1) sampled_total += __shfl_xor_sync(0xffffffffu, sampled_total, o);
        __syncthreads();
        if (lane == 0) s_warp[0][warp] = sampled_total;
        __syncthreads();
        if (threadIdx.x == 0) {
            int t = 0;
            for (int x = 0; x < 32; ++x) t += s_warp[0][x];
            n_sampled[e] = t;
        }
    }
}

// ------------------------------------------------------------------------------------------------------
// A6: per-pixel mean of the kept objects' feature vectors (custom_rcnn.py:884-901), same fp32 add order.
// Thread = 4 consecutive pixels of one channel; K <= 128 object rows cached in shared memory per channel.
// ------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) box_to_image_kernel(const float *__restrict__ box_features, const uint8_t *__restrict__ masks,
                                                           int K, int C, int HW, float *__restrict__ image_features,
                                                           uint8_t *__restrict__ observed)
{
    extern __shared__ float s_feat[];          // (K, CH) channel slice of box_features
    constexpr int CH = 16;                     // channels per CTA (blockIdx.y selects the slice)
    const int c0 = blockIdx.y * CH;
    for (int i = threadIdx.x; i < K * CH; i += blockDim.x) {
        const int k = i / CH, c = i % CH;
        s_feat[i] = (c0 + c < C) ? box_features[(size_t)k * C + c0 + c] : 0.f;
    }
    __syncthreads();
    const int p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= HW) return;
    float acc[CH];
#pragma unroll
    for (int c = 0; c < CH; ++c) acc[c] = 0.f;
    int n = 0;
    for (int k = 0; k < K; ++k) {
        if (__ldg(masks + (size_t)k * HW + p)) {
            ++n;
#pragma unroll
            for (int c = 0; c < CH; ++c) acc[c] = __fadd_rn(acc[c], s_feat[k * CH + c]);
        }
    }
    const float fn = (float)n;
#pragma unroll
    for (int c = 0; c < CH; ++c)
        if (c0 + c < C) image_features[(size_t)(c0 + c) * HW + p] = n ? __fdiv_rn(acc[c], fn) : 0.f;
    if (blockIdx.y == 0 && observed) observed[p] = n ? 1 : 0;
}

// ------------------------------------------------------------------------------------------------------
// main pass, shared pieces
// ------------------------------------------------------------------------------------------------------

// Element (channel c, pixel p) of a 128B-swizzled tile whose rows are 32 floats (TMA SWIZZLE_128B: the
// 16-byte chunk index is XOR-ed with (row % 8)).
__device__ __forceinline__ int swz(int c, int p) { return c * TILE_PX + ((((p >> 2) ^ (c & 7)) << 2) | (p & 3)); }

// Flush the run sums of one tile: item (r, g) = run r, channels 4g..4g+3.  tile[swz(c, r)] holds run r of channel c.
template <int C>
__device__ __forceinline__ void flush_runs(const float *tile, const int *s_cells, unsigned heads, unsigned samps, int pvalid,
                                           const uint32_t *__restrict__ frame_cnt_e, float *__restrict__ sums_e, int tid)
{
    constexpr int G = C / 4;
    const int nruns = __popc(heads);
    for (int item = tid; item < nruns * G; item += C) {
        const int r = item / G, g = item - r * G;
        const int p0 = __fns(heads, 0, r + 1);                          // first pixel of run r
        const unsigned above = heads & ~((2u << p0) - 1u);
        const int p1 = above ? (__ffs(above) - 1) : pvalid;
        const unsigned run = ((p1 >= 32) ? 0xffffffffu : ((1u << p1) - 1u)) & ~((1u << p0) - 1u);
        if (!(samps & run)) continue;                                   // no sampled pixel in this run
        const int cell = s_cells[p0];
        const float n = (float)(__ldg(frame_cnt_e + cell) & 0x7fffffffu);
        const int c = 4 * g;
        const float a = tile[swz(c, r)], b = tile[swz(c + 1, r)], d = tile[swz(c + 2, r)], f = tile[swz(c + 3, r)];
        red_add_v4(sums_e + (size_t)cell * C + c, __fdiv_rn(a, n), __fdiv_rn(b, n), __fdiv_rn(d, n), __fdiv_rn(f, n));
    }
}

// Consumer thread c: accumulate runs over the tile's pixels (tile row c, swizzled), write run sums in place.
__device__ __forceinline__ void accumulate_runs(float *tile, int c, unsigned heads, unsigned samps)
{
    float acc = 0.f;
    int r = 0;
    const float4 *row = reinterpret_cast<const float4 *>(tile + c * TILE_PX);
#pragma unroll
    for (int j = 0; j < 8; ++j) {
        const float4 v = row[j ^ (c & 7)];
        const float vv[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            const int p = 4 * j + k;
            if (p > 0 && ((heads >> p) & 1u)) {        // CTA-uniform
                tile[swz(c, r)] = acc;                // slot r <= p - 1: its chunk was read already
                ++r;
                acc = 0.f;
            }
            if ((samps >> p) & 1u) acc = __fadd_rn(acc, vv[k]);
        }
    }
    tile[swz(c, r)] = acc;
}

__device__ __forceinline__ void tile_masks(const int *s_cells, const uint8_t *s_samp, bool has_samp, int pvalid, unsigned lane,
                                           unsigned &heads, unsigned &samps)
{
    const bool valid = (int)lane < pvalid;
    const int cell = valid ? s_cells[lane] : -1;
    const int prev = __shfl_up_sync(0xffffffffu, cell, 1);
    heads = __ballot_sync(0xffffffffu, valid && (lane == 0 || prev != cell));
    samps = __ballot_sync(0xffffffffu, valid && (has_samp ? s_samp[lane] != 0 : true));
}

// ------------------------------------------------------------------------------------------------------
// main pass, CHW, LDG-staged
// ------------------------------------------------------------------------------------------------------
template <int C, int F = FEAT_F32>
__global__ void __launch_bounds__(C) write_mean_chw_ldg_kernel(const typename FeatElem<F>::T *__restrict__ feat, const int32_t *__restrict__ idx,
                                                               const uint8_t *__restrict__ samp, const uint32_t *__restrict__ frame_cnt,
                                                               const int32_t *__restrict__ active, int HW, int64_t n_cells, int tiles_per_ep, int n_tiles,
                                                               float *__restrict__ sums)
{
    extern __shared__ __align__(1024) unsigned char smem_raw[];
    float *tile = reinterpret_cast<float *>(smem_raw);              // C x 32, swizzled like the TMA path
    int *s_cells = reinterpret_cast<int *>(tile + C * TILE_PX);
    uint8_t *s_samp = reinterpret_cast<uint8_t *>(s_cells + TILE_PX);
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    constexpr int NW = C / 32;

    for (int t = blockIdx.x; t < n_tiles; t += gridDim.x) {
        const int e = t / tiles_per_ep, p0 = (t - e * tiles_per_ep) * TILE_PX;
        if (active && __ldg(active + e) <= 0) continue;              // CTA-uniform: an idle slot of the batch is not even read
        const int pvalid = min(TILE_PX, HW - p0);
        const typename FeatElem<F>::T *feat_e = feat + (size_t)e * C * HW;
        // coalesced 128 B (16-bit features: 64 B) row segments: warp w loads channels w, w+NW, ...; widened on the way into the tile
#pragma unroll 4
        for (int c = warp; c < C; c += NW)
            tile[swz(c, lane)] = lane < pvalid ? widen1<F>(__ldg(feat_e + (size_t)c * HW + p0 + lane)) : 0.f;
        if (tid < TILE_PX) {
            s_cells[tid] = tid < pvalid ? __ldg(idx + (size_t)e * HW + p0 + tid) : -1;
            s_samp[tid] = (samp && tid < pvalid) ? __ldg(samp + (size_t)e * HW + p0 + tid) : 1;
        }
        __syncthreads();
        unsigned heads, samps;
        tile_masks(s_cells, s_samp, samp != nullptr, pvalid, lane, heads, samps);
        accumulate_runs(tile, tid, heads, samps);
        __syncthreads();
        flush_runs<C>(tile, s_cells, heads, samps, pvalid, frame_cnt + (size_t)e * n_cells, sums + (size_t)e * n_cells * C, tid);
        __syncthreads();
    }
}

// ------------------------------------------------------------------------------------------------------
// main pass, CHW, TMA-staged persistent kernel
//
// One CTA per SM: kStages consumer warps + 1 producer warp.  The unit of work is (32-pixel tile, block of 256
// channels) = one 32 KB TMA box (C=128: the whole 16 KB tile); unit u of the CTA lands in ring stage u % kStages and
// is consumed by warp u % kStages, i.e. every consumer warp OWNS one stage: no CTA- or group-level barrier anywhere,
// the only synchronisation is the full/empty mbarrier pair of the stage.  The ring holds 192 KB whatever the unit
// (6 x 32 KB, or 12 x 16 KB at C=128).  Per unit the warp
//   waits full[stage] -> derives the group / sample masks from the staged cell ids (MATCH.ANY, ballot) ->
//   per group (the tile's pixels of one map cell): lane l sums channels l, l+32, ..., l+32*(kJ-1) over the group's
//   pixels straight from the swizzled tile (kJ = 8 independent LDS.128 + FADD chains; 4 at C=128), scales by
//   1/n_cell and issues kJ x red.global.add.f32 (each a warp-wide 128-byte segment of the cell row) ->
//   __syncwarp, one arrive on empty[stage].
// A 256-channel unit does the per-tile work (barrier wait, group derivation, divisor look-up, chunk walk) once for
// what two 128-channel units did twice; the box height is the TMA limit, so C=512 is two units per tile.
// 16-bit features (F = FEAT_BF16 / FEAT_F16): a tile is 64 pixels, so a box row is again 128 bytes and the unit, the swizzle,
// the ring and the raster-neighbour pairs are those of fp32; lane l holds pixels l and l + 32 of the tile (chw16_unit).
// ------------------------------------------------------------------------------------------------------

template <int C, int F = FEAT_F32>
struct TmaCfg {
    static constexpr int kTilePx = F == FEAT_F32 ? TILE_PX : 2 * TILE_PX; // pixels per tile: one 128-byte box row
    static constexpr int kRowBytes = 128;
    static constexpr int kChanBlk = C < 256 ? C : 256;                    // channels per unit (TMA box height; 256 is the box limit)
    static constexpr int kBlocks = C / kChanBlk;                          // units per tile
    static constexpr int kJ = kChanBlk / 32;                              // channels (accumulator chains) per lane
    static constexpr int kUnitBytes = kChanBlk * kRowBytes;               // 32 KB (16 KB at C=128), keeps every stage 1 KB aligned (SWIZZLE_128B)
    static constexpr int kStages = (192 * 1024) / kUnitBytes;             // ring depth == consumer warps: 192 KB in flight per SM
    static constexpr int kThreads = 32 * (kStages + 1);
    // aux area per stage: cells (128 B) | samp (32 B) | pad | per-pixel 1/n (128 B) | unit descriptor {tile, channel block} (8 B);
    // 16-bit features: cells (256 B) | samp (64 B) | pad | unit descriptor (no per-pixel divisors)
    static constexpr int kAuxCells = 0, kAuxSamp = 4 * kTilePx, kAuxPixN = 256, kAuxUnit = 384, kAuxBytes = 512;
    static constexpr int kSmemBytes = kStages * (kUnitBytes + kAuxBytes) + 1024 /*align slack*/ + 256 /*barriers*/;
    static_assert(C % kChanBlk == 0 && kChanBlk % 128 == 0, "C must be 128 or a multiple of 256");
    static_assert(kSmemBytes <= 232448, "exceeds 227 KB of shared memory");
};

// One staged unit of 16-bit features: 64 pixels x kChanBlk channels, row `lane` of the box at `tile`.  Lane l looks at pixels l and
// l + 32.  Groups are formed per half (MATCH.ANY) and joined across the halves with one ballot per group of the lower half; the
// upper-half groups no lower-half group claimed are cells the lower half does not see.  Per group, lane l sums channels l, l+32, ...
// over the group's sampled pixels in raster order, 8 pixels (one LDS.128) per chunk, widened exactly, then scales by 1/n_cell and
// issues kJ red.global.add.f32 - the arithmetic of the fp32 consumer on the widened values.
template <int C, int F>
__device__ __forceinline__ void chw16_unit(uint32_t tile, uint32_t aux, int t, int cb, int tiles_per_ep, bool has_samp, unsigned lane,
                                           int64_t n_cells, const uint32_t *__restrict__ frame_cnt, float *__restrict__ sums, int no_red)
{
    using Cfg = TmaCfg<C, F>;
    constexpr int kJ = Cfg::kJ;
    const uint32_t sw = lane & 7;
    const int e = t / tiles_per_ep;
    const int cell_lo = (int)lds32(aux + Cfg::kAuxCells + 4 * lane), cell_hi = (int)lds32(aux + Cfg::kAuxCells + 128 + 4 * lane);
    const unsigned grp_lo = __match_any_sync(0xffffffffu, cell_lo), grp_hi = __match_any_sync(0xffffffffu, cell_hi);
    unsigned lead_lo = __ballot_sync(0xffffffffu, (unsigned)(__ffs(grp_lo) - 1) == lane);
    unsigned lead_hi = __ballot_sync(0xffffffffu, (unsigned)(__ffs(grp_hi) - 1) == lane);
    const unsigned samp_lo = has_samp ? __ballot_sync(0xffffffffu, lds8(aux + Cfg::kAuxSamp + lane) != 0) : 0xffffffffu;
    const unsigned samp_hi = has_samp ? __ballot_sync(0xffffffffu, lds8(aux + Cfg::kAuxSamp + 32 + lane) != 0) : 0xffffffffu;
    float *dst = sums + ((size_t)e * n_cells) * C + cb * Cfg::kChanBlk + lane;
    const uint32_t *cnt_e = frame_cnt + (size_t)e * n_cells;

    while (lead_lo | lead_hi) {                                    // warp-uniform
        int rc;
        uint64_t m;                                                // sampled pixels of the group, bit p = pixel p of the tile
        if (lead_lo) {
            const int p0 = __ffs(lead_lo) - 1;
            lead_lo &= lead_lo - 1;
            rc = __shfl_sync(0xffffffffu, cell_lo, p0);
            const unsigned hi = __ballot_sync(0xffffffffu, cell_hi == rc);
            lead_hi &= ~hi;                                        // the upper half of this cell belongs to this group
            m = ((uint64_t)(samp_hi & hi) << 32) | (samp_lo & __shfl_sync(0xffffffffu, grp_lo, p0));
        } else {
            const int p0 = __ffs(lead_hi) - 1;
            lead_hi &= lead_hi - 1;
            rc = __shfl_sync(0xffffffffu, cell_hi, p0);
            m = (uint64_t)(samp_hi & __shfl_sync(0xffffffffu, grp_hi, p0)) << 32;
        }
        if (m == 0) continue;                                      // no sampled pixel in this group
        float acc[kJ];
#pragma unroll
        for (int k = 0; k < kJ; ++k) acc[k] = 0.f;
        const int j1 = (63 - __clzll((long long)m)) >> 3;
#pragma unroll 1
        for (int j = (__ffsll((long long)m) - 1) >> 3; j <= j1; ++j) {
            const unsigned mj = (unsigned)(m >> (8 * j)) & 0xffu;
            if (mj == 0) continue;
            const uint32_t a = tile + (((uint32_t)j ^ sw) << 4);
            uint4 v[kJ];
#pragma unroll
            for (int k = 0; k < kJ; ++k) v[k] = lds128(a + k * 32 * Cfg::kRowBytes);
            if (mj == 0xffu) {                                     // whole chunk inside the group, all sampled
#pragma unroll
                for (int k = 0; k < kJ; ++k) {
                    const uint32_t w[4] = {v[k].x, v[k].y, v[k].z, v[k].w};
#pragma unroll
                    for (int q = 0; q < 4; ++q) {
                        const float2 f = widen2<F>(w[q]);
                        acc[k] = __fadd_rn(__fadd_rn(acc[k], f.x), f.y);
                    }
                }
            } else {                                               // group edge / sparsely sampled chunk (warp-uniform predicates)
#pragma unroll
                for (int i = 0; i < 8; ++i) {
                    if (mj & (1u << i)) {
#pragma unroll
                        for (int k = 0; k < kJ; ++k) {
                            const uint32_t *vk = reinterpret_cast<const uint32_t *>(&v[k]);
                            const float2 f = widen2<F>(vk[i >> 1]);
                            acc[k] = __fadd_rn(acc[k], (i & 1) ? f.y : f.x);
                        }
                    }
                }
            }
        }
        const float inv = __frcp_rn((float)(__ldg(cnt_e + rc) & 0x7fffffffu));
        float *d = dst + (size_t)rc * C;
        if (no_red) continue;                                      // diagnostics (EOD_TMA_NO_RED): everything but the reductions
#pragma unroll
        for (int k = 0; k < kJ; ++k) red_add_f32(d + 32 * k, __fmul_rn(acc[k], inv));
    }
}

// kDry: consumers only wait and release (no accumulation, no atomics) - measures the pure streaming
// ceiling of this tile shape; selected with variant EOD_WRITE_TMA_DRY (bring-up / profiling only).
// kPixN: the per-pixel reciprocal divisors 1/n_cell arrive with the tile (pix_n workspace); otherwise the
// divisor of a run is a dependent global load from frame_cnt.
// kDet: deterministic variant - the main pass of det.cuh: a run's (unscaled) channel sums are STORED to partials (DetArgs);
// runs beyond the workspace capacity fall back to the reductions of the default variant and raise *status.

// F: feature element type (FEAT_BF16 / FEAT_F16 take the 64-pixel unit and chw16_unit; neither kPixN nor kDet)
template <int C, bool kDry, bool kPixN, bool kDet, int F = FEAT_F32>
__global__ void __launch_bounds__(TmaCfg<C, F>::kThreads, 1)
write_mean_chw_tma_kernel(const __grid_constant__ CUtensorMap tmap, const int32_t *__restrict__ idx, const uint8_t *__restrict__ samp,
                          const uint32_t *__restrict__ frame_cnt, const float *__restrict__ pix_n, const int32_t *__restrict__ active, int HW,
                          int64_t n_cells, int tiles_per_ep, int n_tiles, int group, float *__restrict__ sums, const DetArgs det,
                          int *__restrict__ work, int chunk, uint32_t wait_hint, int n_stages, int no_red)
{
    using Cfg = TmaCfg<C, F>;
    static_assert(F == FEAT_F32 || (!kPixN && !kDet), "16-bit features: no per-pixel divisors, no deterministic variant");
    constexpr int kTilePx = Cfg::kTilePx;
    extern __shared__ unsigned char smem_dyn[];
    const uint32_t base = (smem_u32(smem_dyn) + 1023u) & ~1023u;          // shared-window address of stage 0
    const uint32_t aux0 = base + Cfg::kStages * Cfg::kUnitBytes;
    const uint32_t full0 = aux0 + Cfg::kStages * Cfg::kAuxBytes, empty0 = full0 + 8 * Cfg::kStages;

    const int tid = threadIdx.x;
    const int warp = tid >> 5;
    const unsigned lane = tid & 31;
    const bool has_samp = samp != nullptr;
    if (tid == 0) {
        for (int s = 0; s < Cfg::kStages; ++s) {
            mbar_init(full0 + 8 * s, 1);        // producer's arrive.expect_tx
            mbar_init(empty0 + 8 * s, 1);       // the owning warp's arrive
        }
        mbar_fence_init();
        fence_proxy_async();
    }
    __syncthreads();

    // Tiles are handed out in GROUPS of `group` raster neighbours and a group's units are issued channel-block-major: the
    // 128-byte row segments of neighbouring tiles are requested back to back, so they share one 256-byte L2 line fill (no
    // second DRAM fetch by some other CTA at some other time) and fall into the same open DRAM page.
    // Groups are CLAIMED, not pre-assigned: the producer takes the next group from a global ticket (`work[0]`; the first one is
    // the CTA's own index), so a CTA that starts late or shares its SM with the read / count kernels of the neighbouring frames
    // simply takes fewer groups instead of stretching the launch (static q -> CTA q % G measured 3.19 ms alone but 3.4-3.9 ms
    // next to the other stages).  The unit's {tile, channel block} travels to the owning consumer warp in the stage's aux area;
    // a negative tile ends the consumer.  work == nullptr keeps the static round-robin (comparator).
    const int G = (int)gridDim.x, b = (int)blockIdx.x;
    const int n_groups = n_tiles / group;                        // host guarantees n_tiles % group == 0
    const int units_per_group = group * Cfg::kBlocks;

    if (warp == Cfg::kStages) {
        // ===== producer warp: one elected lane issues all copies =====
        if (lane == 0) {
            const uint64_t pol = make_evict_first_policy();     // the feature stream is read exactly once
            const uint32_t tx = Cfg::kUnitBytes + kTilePx * 4 + (has_samp ? kTilePx : 0) + (kPixN ? kTilePx * 4 : 0);
            int stage = 0;
            uint32_t phase = 0;
            // a ticket = `chunk` consecutive groups; the next ticket is drawn one chunk ahead (the round trip of an atomic under a
            // saturated memory system is several microseconds - longer than one group lasts)
            int c = b;
            int c_next = work ? G + atomicAdd(work, 1) : c + G;
            while (c * chunk < n_groups) {
              const int c_next2 = work ? G + atomicAdd(work, 1) : c_next + G;
              const int q_end = min(n_groups, (c + 1) * chunk);
              for (int q = c * chunk; q < q_end; ++q) {
                for (int k = 0; k < units_per_group; ++k) {
                    const int cb = k / group, t = group * q + (k - cb * group);
                    const int e = t / tiles_per_ep, p0 = (t - e * tiles_per_ep) * kTilePx;
                    const uint32_t fullb = full0 + 8 * stage, aux = aux0 + stage * Cfg::kAuxBytes;
                    mbar_wait_hint(empty0 + 8 * stage, phase ^ 1, wait_hint);
                    const bool idle = active && __ldg(active + e) <= 0;
                    sts64(aux + Cfg::kAuxUnit, (uint32_t)t, (uint32_t)cb | (idle ? 0x100u : 0u));
                    if (idle) {
                        // idle slot of the batch: the stage is handed over empty, nothing is fetched
                        mbar_arrive(fullb);
                    } else {
                        mbar_expect_tx(fullb, tx);
                        tma_load_3d_hint(base + stage * Cfg::kUnitBytes, &tmap, p0, cb * Cfg::kChanBlk, e, fullb, pol);
                        bulk_load_1d(aux + Cfg::kAuxCells, idx + (size_t)e * HW + p0, kTilePx * 4, fullb);
                        if (has_samp) bulk_load_1d(aux + Cfg::kAuxSamp, samp + (size_t)e * HW + p0, kTilePx, fullb);
                        if (kPixN) bulk_load_1d(aux + Cfg::kAuxPixN, pix_n + (size_t)e * HW + p0, kTilePx * 4, fullb);
                    }
                    if (++stage == n_stages) { stage = 0; phase ^= 1; }
                }
              }
              c = c_next;
              c_next = c_next2;
            }
            for (int s = 0; s < n_stages; ++s) {                              // one end marker per consumer warp
                mbar_wait_hint(empty0 + 8 * stage, phase ^ 1, wait_hint);
                sts64(aux0 + stage * Cfg::kAuxBytes + Cfg::kAuxUnit, 0xffffffffu, 0u);
                mbar_arrive(full0 + 8 * stage);
                if (++stage == n_stages) { stage = 0; phase ^= 1; }
            }
            if (work) {
                // every CTA has drawn its last ticket before it counts itself done: the last one re-arms the pair for the next launch
                __threadfence();
                if (atomicAdd(work + 1, 1) == G - 1) {
                    work[0] = 0;
                    work[1] = 0;
                    __threadfence();
                }
            }
        }
        return;
    }

    if (warp >= n_stages) return;                                  // diagnostics: a shallower ring (EOD_TMA_STAGES)
    // ===== consumer warp `warp`: owns ring stage `warp`, lane l owns channels l, l+32, ..., l+32*(kJ-1) of the block =====
    constexpr int kJ = Cfg::kJ;
    const uint32_t tile = base + warp * Cfg::kUnitBytes + lane * Cfg::kRowBytes;  // row `lane` of the box
    const uint32_t aux = aux0 + warp * Cfg::kAuxBytes;
    const uint32_t fullb = full0 + 8 * warp, emptyb = empty0 + 8 * warp;
    const uint32_t sw = lane & 7;                                                  // rows l + 32k share the swizzle phase
    for (uint32_t phase = 0;; phase ^= 1) {
        mbar_wait_hint(fullb, phase, wait_hint);
        const int t = (int)lds32(aux + Cfg::kAuxUnit);
        if (t < 0) break;                                          // end marker: no more units for this stage
        const uint32_t cbw = lds32(aux + Cfg::kAuxUnit + 4);
        const int cb = (int)(cbw & 0xffu);
        const bool idle = (cbw & 0x100u) != 0;
        int run_pos = kDet ? __ldg(det.tile_off + t) : 0;
        if constexpr (F != FEAT_F32) {
            if (!kDry && !idle) chw16_unit<C, F>(tile, aux, t, cb, tiles_per_ep, has_samp, lane, n_cells, frame_cnt, sums, no_red);
        } else if (!kDry && !idle) {
            const int e = t / tiles_per_ep;
            // run structure of the tile: lane p looks at pixel p
            const int cell = (int)lds32(aux + Cfg::kAuxCells + 4 * lane);
            // kDet: runs of equal cell id (the deterministic reduce orders RUNS).  Default: all pixels of the tile that fall into one
            // cell form ONE group, contiguous or not (MATCH.ANY) - with noisy depth or fine cells a tile alternates between a few
            // cells (A B A A B ...) and every extra run would cost four more L2 reductions (profiles/r2: run-length sweep).
            const int prev = __shfl_up_sync(0xffffffffu, cell, 1);
            const unsigned grp = kDet ? 0u : __match_any_sync(0xffffffffu, cell);
            unsigned heads = __ballot_sync(0xffffffffu, kDet ? (lane == 0 || prev != cell) : ((unsigned)(__ffs(grp) - 1) == lane));
            const unsigned samps = has_samp ? __ballot_sync(0xffffffffu, lds8(aux + Cfg::kAuxSamp + lane) != 0) : 0xffffffffu;
            const float my_inv = kPixN ? __uint_as_float(lds32(aux + Cfg::kAuxPixN + 4 * lane)) : 0.f;
            float *dst = sums + ((size_t)e * n_cells) * C + cb * Cfg::kChanBlk + lane;
            const uint32_t *cnt_e = frame_cnt + (size_t)e * n_cells;

            while (heads) {
                const int p0 = __ffs(heads) - 1;                       // first pixel of the run / group
                heads &= heads - 1;
                unsigned m;
                if (kDet) m = det_run_mask(heads, samps, p0);
                else m = samps & __shfl_sync(0xffffffffu, grp, p0);
                if (m == 0) continue;                                  // no sampled pixel in this run / group
                float acc[kJ];
#pragma unroll
                for (int k = 0; k < kJ; ++k) acc[k] = 0.f;
                const int j1 = (31 - __clz(m)) >> 2;
#pragma unroll 1
                for (int j = (__ffs(m) - 1) >> 2; j <= j1; ++j) {
                    const unsigned mj = (m >> (4 * j)) & 15u;
                    if (mj == 0) continue;
                    const uint32_t a = tile + (((uint32_t)j ^ sw) << 4);
                    float4 v[kJ];
#pragma unroll
                    for (int k = 0; k < kJ; ++k) {
                        const uint4 u = lds128(a + k * 32 * TILE_PX * 4);
                        v[k] = make_float4(__uint_as_float(u.x), __uint_as_float(u.y), __uint_as_float(u.z), __uint_as_float(u.w));
                    }
                    if (mj == 15u) {                                   // whole chunk inside the run, all sampled
#pragma unroll
                        for (int k = 0; k < kJ; ++k) acc[k] = __fadd_rn(__fadd_rn(__fadd_rn(__fadd_rn(acc[k], v[k].x), v[k].y), v[k].z), v[k].w);
                    } else {                                           // run edge / sparsely sampled chunk (warp-uniform predicates)
                        if (mj & 1u) {
#pragma unroll
                            for (int k = 0; k < kJ; ++k) acc[k] = __fadd_rn(acc[k], v[k].x);
                        }
                        if (mj & 2u) {
#pragma unroll
                            for (int k = 0; k < kJ; ++k) acc[k] = __fadd_rn(acc[k], v[k].y);
                        }
                        if (mj & 4u) {
#pragma unroll
                            for (int k = 0; k < kJ; ++k) acc[k] = __fadd_rn(acc[k], v[k].z);
                        }
                        if (mj & 8u) {
#pragma unroll
                            for (int k = 0; k < kJ; ++k) acc[k] = __fadd_rn(acc[k], v[k].w);
                        }
                    }
                }
                const int rc = __shfl_sync(0xffffffffu, cell, p0);
                if (kDet) {
                    const int pos = run_pos++;
                    if (pos < det.cap) {
                        float *d = det.partials + ((size_t)e * det.cap + pos) * C + cb * Cfg::kChanBlk + lane;
#pragma unroll
                        for (int k = 0; k < kJ; ++k) d[32 * k] = acc[k];
                        if (cb == 0 && lane == 0) det.run_cell[(size_t)e * det.cap + pos] = rc;
                        continue;
                    }
                    if (cb == 0 && lane == 0) *det.status = 1;     // workspace too small: correct, but not reproducible
                }
                float inv = __shfl_sync(0xffffffffu, my_inv, p0);
                if (!kPixN) inv = __frcp_rn((float)(__ldg(cnt_e + rc) & 0x7fffffffu));
                float *d = dst + (size_t)rc * C;
                if (no_red) continue;                                  // diagnostics (EOD_TMA_NO_RED): everything but the reductions
#pragma unroll
                for (int k = 0; k < kJ; ++k) red_add_f32(d + 32 * k, __fmul_rn(acc[k], inv));
            }
        }
        __syncwarp();                                                  // every lane's tile reads are done: release the stage
        if (lane == 0) mbar_arrive(emptyb);
    }
}

// ------------------------------------------------------------------------------------------------------
// main pass, HWC: warp per strip of 32 pixels, lanes own float4 channel groups
// ------------------------------------------------------------------------------------------------------
// four consecutive channels of one pixel as fp32: fp32 features (16 B), or bf16 / fp16 features (8 B) widened exactly
template <int F> struct FeatRaw { uint2 q; };
template <> struct FeatRaw<FEAT_F32> { float4 q; };
template <int F>
__device__ __forceinline__ FeatRaw<F> load_feat_raw(const void *row, int k)       // k-th group of 4 channels of the pixel row
{
    FeatRaw<F> r;
    if constexpr (F == FEAT_F32) r.q = ldg_stream_f4(reinterpret_cast<const float *>(row) + 4 * k);
    else asm volatile("ld.global.nc.L1::no_allocate.v2.u32 {%0, %1}, [%2];" : "=r"(r.q.x), "=r"(r.q.y) : "l"(reinterpret_cast<const uint2 *>(row) + k));
    return r;
}
template <int F>
__device__ __forceinline__ float4 widen_feat(const FeatRaw<F> &r)
{
    if constexpr (F == FEAT_F32) return r.q;
    else if constexpr (F == FEAT_BF16)
        return make_float4(__uint_as_float(r.q.x << 16), __uint_as_float(r.q.x & 0xffff0000u), __uint_as_float(r.q.y << 16), __uint_as_float(r.q.y & 0xffff0000u));
    else {
        const float2 a = __half22float2(*reinterpret_cast<const __half2 *>(&r.q.x)), b = __half22float2(*reinterpret_cast<const __half2 *>(&r.q.y));
        return make_float4(a.x, a.y, b.x, b.y);
    }
}

// kDet: deterministic variant (HW % 32 == 0: a strip is one tile of the det pre-passes) - the strip's RUNS of equal cell id in raster
// order (det_tile_masks) take the place of the groups, and a run's unscaled sums are stored to partials[tile_off[strip] + r] like the
// CHW kDet consumer does: every layout sums a run's sampled pixels in raster order from +0.f, so the partials are the same fp32 values.
template <int C, int F, bool kDet = false>
__global__ void __launch_bounds__(256, 3) write_mean_hwc_kernel(const void *__restrict__ feat, const int32_t *__restrict__ idx,
                                                             const uint8_t *__restrict__ samp, const uint32_t *__restrict__ frame_cnt,
                                                             const int32_t *__restrict__ active, int HW, int64_t n_cells, int strips_per_ep,
                                                             int n_strips, float *__restrict__ sums, const DetArgs det)
{
    constexpr int V = C / 128;                 // float4 per lane per pixel
    const unsigned lane = threadIdx.x & 31;
    const int warps_total = gridDim.x * (blockDim.x >> 5);
    for (int s = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5); s < n_strips; s += warps_total) {
        const int e = s / strips_per_ep, p0 = (s - e * strips_per_ep) * TILE_PX;
        if (active && __ldg(active + e) <= 0) continue;              // warp-uniform: idle slot of the batch
        const int pvalid = min(TILE_PX, HW - p0);
        const size_t pix0 = (size_t)e * HW + p0;
        const int my_cell = (int)lane < pvalid ? __ldg(idx + pix0 + lane) : -1;
        const bool my_s = (int)lane < pvalid && (samp ? __ldg(samp + pix0 + lane) != 0 : true);
        const unsigned samps = __ballot_sync(0xffffffffu, my_s);
        const uint32_t *cnt_e = frame_cnt + (size_t)e * n_cells;
        float *sums_e = sums + (size_t)e * n_cells * C;
        // All sampled pixels of the strip that fall into one cell form ONE group, contiguous or not (MATCH.ANY, as in the CHW kernel: with
        // noisy depth a strip alternates between a few cells and every extra run would cost V more 128-bit reductions).  Groups are
        // served in the order of their first pixel; a group's pixels are walked in raster order, in batches of PB whose rows are all
        // requested before the first one is added (32 registers of raw data per lane: 4 fp32 pixels or 8 sixteen-bit ones at C=256 -
        // the same bytes in flight whatever the feature type).
        unsigned grp = 0u, leaders;
        if constexpr (kDet) {
            const int prev = __shfl_up_sync(0xffffffffu, my_cell, 1);
            leaders = __ballot_sync(0xffffffffu, lane == 0 || prev != my_cell);   // run heads (pvalid == 32)
        } else {
            grp = __match_any_sync(0xffffffffu, my_cell);
            leaders = __ballot_sync(0xffffffffu, (int)lane < pvalid && (unsigned)(__ffs(grp) - 1) == lane);
        }
        int run_pos = kDet ? __ldg(det.tile_off + s) : 0;
        constexpr int PB = (F == FEAT_F32 ? 8 : 16) / V > 0 ? (F == FEAT_F32 ? 8 : 16) / V : 1;
        while (leaders) {
            const int lead = __ffs(leaders) - 1;
            leaders &= leaders - 1;
            unsigned rem;
            if constexpr (kDet) rem = det_run_mask(leaders, samps, lead);       // sampled pixels of this run
            else rem = __shfl_sync(0xffffffffu, grp, lead) & samps;             // sampled pixels of this cell
            if (rem == 0u) continue;
            const int cell = __shfl_sync(0xffffffffu, my_cell, lead);
            float4 acc[V];
#pragma unroll
            for (int v = 0; v < V; ++v) acc[v] = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll 1
            while (rem) {
                FeatRaw<F> raw[PB][V];
                unsigned batch = rem;
                int nb = 0;
#pragma unroll
                for (int b = 0; b < PB; ++b) {
                    if (batch) {
                        const int p = __ffs(batch) - 1;
                        batch &= batch - 1;
                        ++nb;
                        const char *row = reinterpret_cast<const char *>(feat) + (pix0 + p) * C * (F == FEAT_F32 ? 4 : 2);
#pragma unroll
                        for (int v = 0; v < V; ++v) raw[b][v] = load_feat_raw<F>(row, v * 32 + (int)lane);
                    }
                }
                rem = batch;
#pragma unroll
                for (int b = 0; b < PB; ++b) {
                    if (b < nb) {
#pragma unroll
                        for (int v = 0; v < V; ++v) {
                            const float4 f = widen_feat<F>(raw[b][v]);
                            acc[v].x = __fadd_rn(acc[v].x, f.x); acc[v].y = __fadd_rn(acc[v].y, f.y);
                            acc[v].z = __fadd_rn(acc[v].z, f.z); acc[v].w = __fadd_rn(acc[v].w, f.w);
                        }
                    }
                }
            }
            if constexpr (kDet) {
                const int pos = run_pos++;
                if (pos < det.cap) {
                    float *d = det.partials + ((size_t)e * det.cap + pos) * C + 4 * lane;
#pragma unroll
                    for (int v = 0; v < V; ++v) *reinterpret_cast<float4 *>(d + v * 128) = acc[v];
                    if (lane == 0) det.run_cell[(size_t)e * det.cap + pos] = cell;
                    continue;
                }
                if (lane == 0) *det.status = 1;                                  // workspace too small: correct, but not reproducible
            }
            const float n = (float)(__ldg(cnt_e + cell) & 0x7fffffffu);
#pragma unroll
            for (int v = 0; v < V; ++v)
                red_add_v4(sums_e + (size_t)cell * C + v * 128 + 4 * lane, __fdiv_rn(acc[v].x, n), __fdiv_rn(acc[v].y, n), __fdiv_rn(acc[v].z, n),
                           __fdiv_rn(acc[v].w, n));
        }
    }
}

// ------------------------------------------------------------------------------------------------------
// host side
// ------------------------------------------------------------------------------------------------------
template <int C, bool kDry, bool kPixN, bool kDet = false, int F = FEAT_F32>
int launch_tma_kernel(const CUtensorMap &tmap, const int32_t *idx, const uint8_t *samp, const uint32_t *frame_cnt, const float *pix_n,
                      const int32_t *active, int E, int HW, int64_t n_cells, float *sums, cudaStream_t st, const DetArgs det = DetArgs{})
{
    using Cfg = TmaCfg<C, F>;
    static unsigned long long attr_done = 0ull;
    if (int rc_attr = eod_ensure_dyn_smem(write_mean_chw_tma_kernel<C, kDry, kPixN, kDet, F>, Cfg::kSmemBytes, &attr_done, "eod_write_mean[tma]")) return rc_attr;
    const int tiles_per_ep = HW / Cfg::kTilePx, n_tiles = tiles_per_ep * E;
    static const int group_env = [] { const char *v = getenv("EOD_TMA_TILE_GROUP"); return v ? atoi(v) : 2; }();   // tuning knob: 1 | 2 | 4 | 8
    int group = (group_env == 1 || group_env == 2 || group_env == 4 || group_env == 8) ? group_env : 2;
    while (group > 1 && n_tiles % group) group >>= 1;
    const int n_groups = n_tiles / group;
    const int grid = n_groups < eod_num_sms() ? n_groups : eod_num_sms();
    static const int static_env = [] { const char *v = getenv("EOD_TMA_STATIC_TILES"); return v ? atoi(v) : 0; }();   // comparator: pre-assigned groups
    // a captured launch takes the static partition: a ticket pair would be pinned for the graph's lifetime while eager launches keep
    // rotating through the pool.  The capture is checked BEFORE the pool is touched: its first use allocates and zero-fills it
    // (cudaMalloc + cudaMemset), which would invalidate the capture, and every draw advances the round-robin counter.
    cudaStreamCaptureStatus cap = cudaStreamCaptureStatusNone;
    const bool capturing = cudaStreamIsCapturing(st, &cap) != cudaSuccess || cap != cudaStreamCaptureStatusNone;
    int *work = (static_env || capturing) ? nullptr : eod_work_tickets();
    static const int chunk_env = [] { const char *v = getenv("EOD_TMA_CHUNK"); return v ? atoi(v) : 8; }();        // groups per ticket
    static const int hint_env = [] { const char *v = getenv("EOD_TMA_WAIT_HINT_NS"); return v ? atoi(v) : 0; }();   // suspend-time hint of the barrier waits
    static const int stages_env = [] { const char *v = getenv("EOD_TMA_STAGES"); const int n = v ? atoi(v) : Cfg::kStages; return n >= 2 && n <= Cfg::kStages ? n : Cfg::kStages; }();
    static const int nored_env = [] { const char *v = getenv("EOD_TMA_NO_RED"); return v ? atoi(v) : 0; }();   // profiling only: wrong results
    const int chunk = work ? (chunk_env > 0 ? chunk_env : 8) : 1;
    write_mean_chw_tma_kernel<C, kDry, kPixN, kDet, F><<<grid, Cfg::kThreads, Cfg::kSmemBytes, st>>>(tmap, idx, samp, frame_cnt, pix_n, active, HW, n_cells, tiles_per_ep, n_tiles, group, sums, det, work, chunk, (uint32_t)hint_env, stages_env, nored_env);
    return eod_check_launch("eod_write_mean[tma]");
}

template <int C, int F = FEAT_F32>
int make_feature_tmap(const void *feat, int E, int HW, CUtensorMap *tmap)
{
    using Cfg = TmaCfg<C, F>;
    constexpr cuuint64_t esz = F == FEAT_F32 ? 4 : 2;
    constexpr CUtensorMapDataType dtype = F == FEAT_F32 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT32
                                          : (F == FEAT_BF16 ? CU_TENSOR_MAP_DATA_TYPE_BFLOAT16 : CU_TENSOR_MAP_DATA_TYPE_FLOAT16);
    const cuuint64_t gdim[3] = {(cuuint64_t)HW, (cuuint64_t)C, (cuuint64_t)E};
    const cuuint64_t gstr[2] = {(cuuint64_t)HW * esz, (cuuint64_t)HW * C * esz};
    const cuuint32_t box[3] = {(cuuint32_t)Cfg::kTilePx, (cuuint32_t)Cfg::kChanBlk, 1};
    static const int promo_env = [] { const char *v = getenv("EOD_TMA_L2_PROMOTION"); return v ? atoi(v) : 256; }();   // tuning knob: 0 | 128 | 256
    const CUtensorMapL2promotion promo = promo_env == 0 ? CU_TENSOR_MAP_L2_PROMOTION_NONE
                                         : (promo_env == 128 ? CU_TENSOR_MAP_L2_PROMOTION_L2_128B : CU_TENSOR_MAP_L2_PROMOTION_L2_256B);
    return eod_encode_tmap("eod_write_mean", tmap, dtype, 3, feat, gdim, gstr, box, promo);
}

template <int C, bool kDry>
int launch_tma(const float *feat, const int32_t *idx, const uint8_t *samp, const uint32_t *frame_cnt, const float *pix_n, const int32_t *active,
               int E, int HW, int64_t n_cells, float *sums, cudaStream_t st)
{
    CUtensorMap tmap;
    const int rc = make_feature_tmap<C>(feat, E, HW, &tmap);
    if (rc) return rc;
    if (pix_n) return launch_tma_kernel<C, kDry, true>(tmap, idx, samp, frame_cnt, pix_n, active, E, HW, n_cells, sums, st);
    return launch_tma_kernel<C, kDry, false>(tmap, idx, samp, frame_cnt, nullptr, active, E, HW, n_cells, sums, st);
}

// 16-bit CHW features (the host has refused pix_n for them)
template <int C, int F, bool kDry>
int launch_tma16(const void *feat, const int32_t *idx, const uint8_t *samp, const uint32_t *frame_cnt, const int32_t *active, int E, int HW,
                 int64_t n_cells, float *sums, cudaStream_t st)
{
    CUtensorMap tmap;
    const int rc = make_feature_tmap<C, F>(feat, E, HW, &tmap);
    if (rc) return rc;
    return launch_tma_kernel<C, kDry, false, false, F>(tmap, idx, samp, frame_cnt, nullptr, active, E, HW, n_cells, sums, st);
}

// ------------------------------------------------------------------------------------------------------
// deterministic variant (EOD_WRITE_DET): raster-ordered run partials + per-cell segmented reduce in fixed order
//
//   det_tile_runs      runs (with samples) per 32-pixel tile                       -> tile_off (counts)
//   det_scan_tiles     exclusive scan per episode                                 -> tile_off, n_runs
//   det_cell_runs      runs per cell (only runs that fit the workspace); the first run of a cell appends the cell
//                      to the episode's compact cell list                         -> cell_runs, cell_list, n_list
//   det_scan_list      exclusive scan of the listed cells' run counts             -> list_off, cell_off[cell]
//   main pass (kDet)   partials[tile_off[tile] + r] = run sums, run_cell[...] = cell            (no atomics)
//   det_claim          run -> slot inside its cell's segment (claim order is arbitrary)         -> seg
//   det_reduce         warp per listed cell: SORT the segment by run position (registers / shared-memory bitonic),
//                      add the partials in that order, divide by n, add ONCE to sums[cell]
//                      => bitwise reproducible, and the reference's own arithmetic shape
// List order and slot order depend on scheduling; the result does not: every cell is reduced on its own, in raster order.
// ------------------------------------------------------------------------------------------------------
// does the run starting at head bit p0 contain a sampled pixel?
__device__ __forceinline__ bool det_run_sampled(unsigned heads, unsigned samps, int p0)
{
    return det_run_mask(heads & ~((2u << p0) - 1u), samps, p0) != 0;
}

__global__ void __launch_bounds__(256) det_tile_runs_kernel(const int32_t *__restrict__ idx, const uint8_t *__restrict__ samp,
                                                            const int32_t *__restrict__ active, int HW, int tiles_per_ep,
                                                            int32_t *__restrict__ tile_off, int32_t *__restrict__ n_list,
                                                            int32_t *__restrict__ chunk_rows, int32_t *__restrict__ n_long)
{
    const int e = blockIdx.y, tile = blockIdx.x * 8 + (threadIdx.x >> 5);
    const unsigned lane = threadIdx.x & 31;
    if (blockIdx.x == 0 && threadIdx.x == 0) {                     // consumed by the previous call's reduce, refilled by this one's
        n_list[e] = 0;
        chunk_rows[e] = 0;
        n_long[e] = 0;
    }
    if (tile >= tiles_per_ep) return;
    if (active && __ldg(active + e) <= 0) {                        // idle slot: no runs, its planes are not read
        if (lane == 0) tile_off[(size_t)e * tiles_per_ep + tile] = 0;
        return;
    }
    int cell;
    unsigned heads, samps;
    det_tile_masks(idx, samp, (size_t)e * HW + (size_t)tile * 32, lane, cell, heads, samps);
    const bool mine = ((heads >> lane) & 1u) && det_run_sampled(heads, samps, lane);
    const unsigned runs = __ballot_sync(0xffffffffu, mine);
    if (lane == 0) tile_off[(size_t)e * tiles_per_ep + tile] = __popc(runs);
}

// one CTA per episode: in-place exclusive scan of n values (chunks of 1024 with a running carry); total -> *total_out
__device__ void det_block_exclusive_scan(const int32_t *in, int32_t *out, int n, int32_t *total_out)
{
    __shared__ int s_warp[32];
    __shared__ int s_carry;
    const unsigned lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    if (threadIdx.x == 0) s_carry = 0;
    __syncthreads();
    for (int base = 0; base < n; base += 1024) {
        const int i = base + threadIdx.x;
        const int v = i < n ? in[i] : 0;
        int x = v;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const int y = __shfl_up_sync(0xffffffffu, x, o);
            if ((int)lane >= o) x += y;
        }
        if (lane == 31) s_warp[warp] = x;
        __syncthreads();
        if (warp == 0) {
            int w = s_warp[lane];
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const int y = __shfl_up_sync(0xffffffffu, w, o);
                if ((int)lane >= o) w += y;
            }
            s_warp[lane] = w;                              // inclusive scan of the warp totals
        }
        __syncthreads();
        const int carry = s_carry;
        const int excl = carry + (warp ? s_warp[warp - 1] : 0) + x - v;
        if (i < n) out[i] = excl;
        __syncthreads();
        if (threadIdx.x == 1023) s_carry = carry + s_warp[31];
        __syncthreads();
    }
    if (threadIdx.x == 0 && total_out) *total_out = s_carry;
}

__global__ void __launch_bounds__(1024) det_scan_tiles_kernel(int32_t *__restrict__ tile_off, int tiles_per_ep, int32_t *__restrict__ n_runs)
{
    const int e = blockIdx.x;
    det_block_exclusive_scan(tile_off + (size_t)e * tiles_per_ep, tile_off + (size_t)e * tiles_per_ep, tiles_per_ep, n_runs + e);
}

__global__ void __launch_bounds__(256) det_cell_runs_kernel(const int32_t *__restrict__ idx, const uint8_t *__restrict__ samp,
                                                            const int32_t *__restrict__ active, int HW, int tiles_per_ep, int64_t n_cells,
                                                            const int32_t *__restrict__ tile_off, int cap, int32_t *__restrict__ cell_runs,
                                                            int32_t *__restrict__ cell_list, int32_t *__restrict__ n_list)
{
    const int e = blockIdx.y, tile = blockIdx.x * 8 + (threadIdx.x >> 5);
    const unsigned lane = threadIdx.x & 31;
    if (tile >= tiles_per_ep || (active && __ldg(active + e) <= 0)) return;     // an idle slot's cell list stays empty
    int cell;
    unsigned heads, samps;
    det_tile_masks(idx, samp, (size_t)e * HW + (size_t)tile * 32, lane, cell, heads, samps);
    const bool mine = ((heads >> lane) & 1u) && det_run_sampled(heads, samps, lane);
    const unsigned runs = __ballot_sync(0xffffffffu, mine);
    if (mine) {
        const int pos = __ldg(tile_off + (size_t)e * tiles_per_ep + tile) + __popc(runs & ((1u << lane) - 1u));
        if (pos < cap && atomicAdd(cell_runs + (size_t)e * n_cells + cell, 1) == 0)      // integer count: order-independent
            cell_list[(size_t)e * cap + atomicAdd(n_list + e, 1)] = cell;                // #cells <= #runs <= cap
    }
}

// one CTA per episode: list_off = exclusive scan of the listed cells' run counts; cell_off[cell] = its segment start
__global__ void __launch_bounds__(1024) det_scan_list_kernel(const int32_t *__restrict__ cell_runs, const int32_t *__restrict__ cell_list,
                                                             const int32_t *__restrict__ n_list, int cap, int64_t n_cells,
                                                             int32_t *__restrict__ list_off, int32_t *__restrict__ cell_off)
{
    const int e = blockIdx.x;
    const int n = __ldg(n_list + e);
    const int32_t *list = cell_list + (size_t)e * cap;
    int32_t *off = list_off + (size_t)e * cap;
    for (int i = threadIdx.x; i < n; i += 1024) off[i] = cell_runs[(size_t)e * n_cells + list[i]];
    __syncthreads();
    det_block_exclusive_scan(off, off, n, nullptr);
    __syncthreads();
    for (int i = threadIdx.x; i < n; i += 1024) cell_off[(size_t)e * n_cells + list[i]] = off[i];
}

__global__ void __launch_bounds__(256) det_claim_kernel(const int32_t *__restrict__ run_cell, const int32_t *__restrict__ n_runs, int cap,
                                                        int64_t n_cells, const int32_t *__restrict__ cell_off, int32_t *__restrict__ cell_runs,
                                                        int32_t *__restrict__ seg)
{
    const int e = blockIdx.y, pos = blockIdx.x * blockDim.x + threadIdx.x;
    if (pos >= min(__ldg(n_runs + e), cap)) return;
    const int c = __ldg(run_cell + (size_t)e * cap + pos);
    const int k = atomicSub(cell_runs + (size_t)e * n_cells + c, 1) - 1;           // leaves cell_runs all-zero again
    seg[(size_t)e * cap + cell_off[(size_t)e * n_cells + c] + k] = pos;
}

// ascending bitonic sort of buf[0, n2) (n2 a power of two >= 32) by one warp
__device__ __forceinline__ void bitonic_sort_warp(int *buf, int n2, unsigned lane)
{
    for (int size = 2; size <= n2; size <<= 1)
        for (int stride = size >> 1; stride > 0; stride >>= 1) {
            for (int q = lane; q < (n2 >> 1); q += 32) {
                const int lo = 2 * q - (q & (stride - 1)), hi = lo + stride;
                const int a = buf[lo], b = buf[hi];
                const bool asc = (lo & size) == 0;
                if ((a > b) == asc) { buf[lo] = b; buf[hi] = a; }
            }
            __syncwarp();
        }
}

constexpr int DET_SORT_MAX = 2048;       // segment length a warp sorts in shared memory (bitonic); longer ones are bitmap-sorted
constexpr int DET_WARPS = 4;
constexpr int DET_DIRECT = 256;          // segments up to this length are summed by the warp that sorted them
constexpr int DET_CHUNK = 128;           // longer ones are cut into chunks of this many runs, summed by separate warps

// Long segments (a cell that takes a large part of the frame has 10^3-10^4 runs): their sorted positions, the chunk tasks
// and the per-chunk partial sums.  The chunking is relative to the segment's own sorted order, so the summation tree of a
// cell is fixed: chunk c = sorted runs [128c, 128c + 128) added in order, then the chunk sums added in order.
struct DetLong {
    int32_t *seg2;          // (E, cap)  sorted positions of long segments, at the segment's own offsets
    int32_t *task_start;    // (E, rows) start of a chunk in seg2 (episode-relative)
    int32_t *task_len;      // (E, rows)
    int32_t *long_i;        // (E, rows) index into cell_list of a long cell ...
    int32_t *long_base;     // (E, rows) ... and its first chunk row
    int32_t *chunk_rows;    // (E) rows handed out this frame
    int32_t *n_long;        // (E) long cells this frame
    float *cparts;          // (E, rows, C) chunk sums
    int rows;
};

// rows of `count` positions (kGlobal: read-only global memory, else shared), U rows in flight, added strictly in order
template <int J, bool kGlobal>
__device__ __forceinline__ void det_sum_sorted(const float *part_e, int C, const int *sorted, int count, float (&acc)[J])
{
    constexpr int U = (J <= 8) ? 8 : 4;
    int it = 0;
#pragma unroll 1
    for (; it + U <= count; it += U) {
        int pos[U];
#pragma unroll
        for (int u = 0; u < U; ++u) pos[u] = kGlobal ? __ldg(sorted + it + u) : sorted[it + u];
        float r[U][J];
#pragma unroll
        for (int u = 0; u < U; ++u) {
            const float *row = part_e + (size_t)pos[u] * C;
#pragma unroll
            for (int j = 0; j < J; ++j) r[u][j] = __ldg(row + 32 * j);
        }
#pragma unroll
        for (int u = 0; u < U; ++u)
#pragma unroll
            for (int j = 0; j < J; ++j) acc[j] = __fadd_rn(acc[j], r[u][j]);
    }
    for (; it < count; ++it) {
        const float *row = part_e + (size_t)(kGlobal ? __ldg(sorted + it) : sorted[it]) * C;
#pragma unroll
        for (int j = 0; j < J; ++j) acc[j] = __fadd_rn(acc[j], __ldg(row + 32 * j));
    }
}

// warp per listed cell: sort the segment by run position; short segments are summed and finished here, long ones are
// written out sorted and cut into chunk tasks for det_chunk_kernel / det_final_kernel
template <int C>
__global__ void __launch_bounds__(32 * DET_WARPS) det_reduce_kernel(const int32_t *__restrict__ cell_list, const int32_t *__restrict__ list_off,
                                                                    const int32_t *__restrict__ n_list, const int32_t *__restrict__ n_runs, int cap,
                                                                    int64_t n_cells, const int32_t *__restrict__ seg, const float *__restrict__ partials,
                                                                    const uint32_t *__restrict__ frame_cnt, float *__restrict__ sums, const DetLong L,
                                                                    int32_t *__restrict__ status)
{
    constexpr int J = C / 32;
    __shared__ int s_sort[DET_WARPS][DET_SORT_MAX];
    const int e = blockIdx.y;
    const unsigned lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int n = __ldg(n_list + e);
    const int total = min(__ldg(n_runs + e), cap);
    const float *part_e = partials + (size_t)e * cap * C + lane;
    int *buf = s_sort[warp];
    for (int i = blockIdx.x * DET_WARPS + warp; i < n; i += gridDim.x * DET_WARPS) {
        const int cell = __ldg(cell_list + (size_t)e * cap + i);
        const int s0 = __ldg(list_off + (size_t)e * cap + i);
        const int s1 = (i + 1 < n) ? __ldg(list_off + (size_t)e * cap + i + 1) : total;
        const int k = s1 - s0;
        const int32_t *sg = seg + (size_t)e * cap + s0;
        float acc[J];
#pragma unroll
        for (int j = 0; j < J; ++j) acc[j] = 0.f;
        bool finish_here = true;

        if (k <= DET_SORT_MAX) {
            int n2 = 32;
            while (n2 < k) n2 <<= 1;
            for (int q = lane; q < n2; q += 32) buf[q] = q < k ? sg[q] : 0x7fffffff;
            __syncwarp();
            bitonic_sort_warp(buf, n2, lane);
            if (k <= DET_DIRECT) det_sum_sorted<J, false>(part_e, C, buf, k, acc);
            else {
                int32_t *out = L.seg2 + (size_t)e * cap + s0;
                for (int q = lane; q < k; q += 32) out[q] = buf[q];
                finish_here = false;
            }
        } else {
            // bitmap sort: positions are distinct integers below `total`; 65 536 of them per pass fit the warp's 8 KB slice.
            // Every pass streams the whole segment (coalesced) and emits the range's members in ascending order.
            int32_t *out = L.seg2 + (size_t)e * cap + s0;
            int written = 0;
            for (int r0 = 0; r0 < total && written < k; r0 += DET_SORT_MAX * 32) {
                for (int q = lane; q < DET_SORT_MAX; q += 32) buf[q] = 0;
                __syncwarp();
                for (int q = lane; q < k; q += 32) {
                    const int v = sg[q] - r0;
                    if (v >= 0 && v < DET_SORT_MAX * 32) atomicOr(reinterpret_cast<unsigned *>(buf) + (v >> 5), 1u << (v & 31));
                }
                __syncwarp();
                for (int w0 = 0; w0 < DET_SORT_MAX; w0 += 32) {
                    unsigned word = (unsigned)buf[w0 + lane];
                    const int cnt = __popc(word);
                    int incl = cnt;
#pragma unroll
                    for (int o = 1; o < 32; o <<= 1) {
                        const int up = __shfl_up_sync(0xffffffffu, incl, o);
                        if ((int)lane >= o) incl += up;
                    }
                    int at = written + incl - cnt;
                    while (word) {
                        out[at++] = r0 + (w0 + (int)lane) * 32 + __ffs(word) - 1;
                        word &= word - 1;
                    }
                    written += __shfl_sync(0xffffffffu, incl, 31);
                }
                __syncwarp();
            }
            finish_here = false;
        }

        if (!finish_here) {
            // hand the sorted segment to the chunk pass
            const int nch = (k + DET_CHUNK - 1) / DET_CHUNK;
            int base = 0, j = 0;
            if (lane == 0) {
                base = atomicAdd(L.chunk_rows + e, nch);           // which rows a cell gets is arbitrary; what is summed into them is not
                j = atomicAdd(L.n_long + e, 1);
            }
            base = __shfl_sync(0xffffffffu, base, 0);
            j = __shfl_sync(0xffffffffu, j, 0);
            if (base + nch <= L.rows && j < L.rows) {
                for (int c = lane; c < nch; c += 32) {
                    L.task_start[(size_t)e * L.rows + base + c] = s0 + c * DET_CHUNK;
                    L.task_len[(size_t)e * L.rows + base + c] = min(DET_CHUNK, k - c * DET_CHUNK);
                }
                if (lane == 0) {
                    L.long_i[(size_t)e * L.rows + j] = i;
                    L.long_base[(size_t)e * L.rows + j] = base;
                }
                __syncwarp();
                continue;
            }
            // chunk rows exhausted (cannot happen with the rows sized by det_carve): same tree, walked by this warp alone
            if (lane == 0) {
                L.long_i[(size_t)e * L.rows + min(j, L.rows - 1)] = -1;
                *status = 2;
            }
            __threadfence();
            __syncwarp();
            const int *sorted = L.seg2 + (size_t)e * cap + s0;
            for (int c = 0; c < nch; ++c) {
                float ch[J];
#pragma unroll
                for (int jj = 0; jj < J; ++jj) ch[jj] = 0.f;
                det_sum_sorted<J, true>(part_e, C, sorted + c * DET_CHUNK, min(DET_CHUNK, k - c * DET_CHUNK), ch);
#pragma unroll
                for (int jj = 0; jj < J; ++jj) acc[jj] = __fadd_rn(acc[jj], ch[jj]);
            }
        }
        const float nn = (float)(__ldg(frame_cnt + (size_t)e * n_cells + cell) & 0x7fffffffu);
        float *dst = sums + ((size_t)e * n_cells + cell) * C + lane;
#pragma unroll
        for (int j = 0; j < J; ++j) dst[32 * j] = __fadd_rn(dst[32 * j], __fdiv_rn(acc[j], nn));     // custom_rcnn.py:934, :742
        __syncwarp();
    }
}

// warp per chunk task: cparts[row] = sum of the chunk's partial rows, in sorted order
template <int C>
__global__ void __launch_bounds__(256) det_chunk_kernel(const float *__restrict__ partials, int cap, const DetLong L)
{
    constexpr int J = C / 32;
    const int e = blockIdx.y;
    const unsigned lane = threadIdx.x & 31;
    const int n_rows = min(__ldg(L.chunk_rows + e), L.rows);
    const float *part_e = partials + (size_t)e * cap * C + lane;
    for (int r = blockIdx.x * 8 + (threadIdx.x >> 5); r < n_rows; r += gridDim.x * 8) {
        const int len = __ldg(L.task_len + (size_t)e * L.rows + r);
        if (len <= 0) continue;                                  // a row of a cell that fell back (stale task)
        const int start = __ldg(L.task_start + (size_t)e * L.rows + r);
        float acc[J];
#pragma unroll
        for (int j = 0; j < J; ++j) acc[j] = 0.f;
        det_sum_sorted<J, true>(part_e, C, L.seg2 + (size_t)e * cap + start, len, acc);
        float *dst = L.cparts + ((size_t)e * L.rows + r) * C + lane;
#pragma unroll
        for (int j = 0; j < J; ++j) dst[32 * j] = acc[j];
    }
}

// warp per long cell: add its chunk sums in chunk order, divide by n, add ONCE to sums[cell]
template <int C>
__global__ void __launch_bounds__(256) det_final_kernel(const int32_t *__restrict__ cell_list, const int32_t *__restrict__ list_off,
                                                        const int32_t *__restrict__ n_list, const int32_t *__restrict__ n_runs, int cap,
                                                        int64_t n_cells, const uint32_t *__restrict__ frame_cnt, float *__restrict__ sums,
                                                        const DetLong L)
{
    constexpr int J = C / 32;
    const int e = blockIdx.y;
    const unsigned lane = threadIdx.x & 31;
    const int n = __ldg(n_list + e), total = min(__ldg(n_runs + e), cap);
    const int n_long = min(__ldg(L.n_long + e), L.rows);
    for (int jl = blockIdx.x * 8 + (threadIdx.x >> 5); jl < n_long; jl += gridDim.x * 8) {
        const int i = __ldg(L.long_i + (size_t)e * L.rows + jl);
        if (i < 0) continue;                                     // finished by the sorting warp (row overflow)
        const int base = __ldg(L.long_base + (size_t)e * L.rows + jl);
        const int cell = __ldg(cell_list + (size_t)e * cap + i);
        const int s0 = __ldg(list_off + (size_t)e * cap + i);
        const int s1 = (i + 1 < n) ? __ldg(list_off + (size_t)e * cap + i + 1) : total;
        const int nch = (s1 - s0 + DET_CHUNK - 1) / DET_CHUNK;
        float acc[J];
#pragma unroll
        for (int j = 0; j < J; ++j) acc[j] = 0.f;
        const float *rows = L.cparts + ((size_t)e * L.rows + base) * C + lane;
        for (int c = 0; c < nch; ++c)
#pragma unroll
            for (int j = 0; j < J; ++j) acc[j] = __fadd_rn(acc[j], rows[(size_t)c * C + 32 * j]);
        const float nn = (float)(__ldg(frame_cnt + (size_t)e * n_cells + cell) & 0x7fffffffu);
        float *dst = sums + ((size_t)e * n_cells + cell) * C + lane;
#pragma unroll
        for (int j = 0; j < J; ++j) dst[32 * j] = __fadd_rn(dst[32 * j], __fdiv_rn(acc[j], nn));     // custom_rcnn.py:934, :742
    }
}

size_t det_align(size_t x) { return (x + 255) & ~size_t(255); }

// chunk rows per episode: every long segment (> DET_DIRECT runs) needs ceil(k / DET_CHUNK) <= k / DET_CHUNK + 1 rows and there
// are fewer than cap / DET_DIRECT of them
int det_rows(int cap) { return cap / DET_CHUNK + cap / DET_DIRECT + 8; }

// Carves the caller's workspace.  cell_runs must be all-zero between frames (the library leaves it so; the caller
// zero-fills the workspace once).  Returns the bytes needed for `cap` runs per episode.
size_t det_carve(void *ws, int E, int C, int tiles_per_ep, int64_t n_cells, int cap, DetWorkspace *out)
{
    size_t o = 0;
    auto take = [&](size_t bytes) { size_t at = o; o += det_align(bytes); return ws ? (char *)ws + at : (char *)nullptr; };
    DetWorkspace w;
    const int rows = det_rows(cap);
    w.cell_runs = (int32_t *)take((size_t)E * n_cells * 4);
    w.status = (int32_t *)take(256);
    w.n_runs = (int32_t *)take((size_t)E * 4);
    w.n_list = (int32_t *)take((size_t)E * 4);
    w.tile_off = (int32_t *)take((size_t)E * tiles_per_ep * 4);
    w.cell_off = (int32_t *)take((size_t)E * n_cells * 4);
    w.chunk_rows = (int32_t *)take((size_t)E * 4);
    w.n_long = (int32_t *)take((size_t)E * 4);
    w.run_cell = (int32_t *)take((size_t)E * cap * 4);
    w.seg = (int32_t *)take((size_t)E * cap * 4);
    w.cell_list = (int32_t *)take((size_t)E * cap * 4);
    w.list_off = (int32_t *)take((size_t)E * cap * 4);
    w.seg2 = (int32_t *)take((size_t)E * cap * 4);
    w.task_start = (int32_t *)take((size_t)E * rows * 4);
    w.task_len = (int32_t *)take((size_t)E * rows * 4);
    w.long_i = (int32_t *)take((size_t)E * rows * 4);
    w.long_base = (int32_t *)take((size_t)E * rows * 4);
    w.cparts = (float *)take((size_t)E * rows * C * 4);
    w.partials = (float *)take((size_t)E * cap * C * 4);
    w.rows = rows;
    w.cap = cap;
    if (out) *out = w;
    return o;
}

// eod_check_launch with the stage of the deterministic write in the message ("<what>[<stage>]")
int det_check_launch(const char *what, const char *stage)
{
    if (cudaPeekAtLastError() == cudaSuccess) return EOD_OK;
    char buf[128];
    snprintf(buf, sizeof buf, "%s[%s]", what, stage);
    return eod_check_launch(buf);
}

template <int C>
int launch_det_reduce(const char *what, const DetWorkspace &w, int E, int64_t n_cells, const uint32_t *frame_cnt, float *sums, cudaStream_t st)
{
    const DetLong L{w.seg2, w.task_start, w.task_len, w.long_i, w.long_base, w.chunk_rows, w.n_long, w.cparts, w.rows};
    dim3 gc((w.cap + 255) / 256, E);
    det_claim_kernel<<<gc, 256, 0, st>>>(w.run_cell, w.n_runs, w.cap, n_cells, w.cell_off, w.cell_runs, w.seg);
    // at most min(cells, cap) cells carry runs; warps beyond n_list[e] exit at once
    const int64_t max_list = n_cells < (int64_t)w.cap ? n_cells : (int64_t)w.cap;
    const int64_t want_blocks = (max_list + DET_WARPS - 1) / DET_WARPS;
    dim3 gr((unsigned)(want_blocks < 128 ? want_blocks : 128), E);          // warps stride over the episode's cell list
    det_reduce_kernel<C><<<gr, 32 * DET_WARPS, 0, st>>>(w.cell_list, w.list_off, w.n_list, w.n_runs, w.cap, n_cells, w.seg, w.partials, frame_cnt, sums,
                                                        L, w.status);
    const int chunk_blocks = (L.rows + 7) / 8;
    dim3 gk((unsigned)(chunk_blocks < 64 ? chunk_blocks : 64), E);
    det_chunk_kernel<C><<<gk, 256, 0, st>>>(w.partials, w.cap, L);
    dim3 gf(8, E);
    det_final_kernel<C><<<gf, 256, 0, st>>>(w.cell_list, w.list_off, w.n_list, w.n_runs, w.cap, n_cells, frame_cnt, sums, L);
    return det_check_launch(what, "reduce");
}

}  // namespace

int det_prepass(const char *what, const int32_t *idx, const uint8_t *samp, const int32_t *active, int E, int C, int HW, int64_t n_cells,
                void *ws, size_t ws_bytes, DetWorkspace *out, cudaStream_t st)
{
    EOD_REQUIRE(HW % TILE_PX == 0 && (!samp || (reinterpret_cast<uintptr_t>(samp) % 16 == 0)), EOD_ERR_UNSUPPORTED,
                "%s: needs HW %% 32 == 0 and a 16-byte aligned sample mask", what);
    EOD_REQUIRE(n_cells < (int64_t)INT32_MAX, EOD_ERR_BADARG, "%s: grid too large", what);
    const int tiles_per_ep = HW / TILE_PX;
    // capacity: whatever the workspace holds beyond the fixed planes (at most one run per pixel)
    const size_t fixed = det_carve(nullptr, E, C, tiles_per_ep, n_cells, 0, nullptr);
    EOD_REQUIRE(ws && eod_aligned16(ws) && ws_bytes > fixed + 4096, EOD_ERR_BADARG,
                "%s: workspace missing or too small (see eod_write_mean_det_workspace_bytes)", what);
    // per run: partial row + 5 ints; per chunk row (cap / 128 + cap / 256 of them): a partial row + 4 ints
    const size_t per_run = (size_t)C * 4 + 20 + ((size_t)C * 4 + 16) * 3 / 256 + 1;
    int64_t cap = ws_bytes > fixed + 16 * 256 ? (int64_t)((ws_bytes - fixed - 16 * 256) / ((size_t)E * per_run)) : 0;
    if (cap > HW) cap = HW;
    EOD_REQUIRE(cap >= 1, EOD_ERR_BADARG, "%s: workspace too small", what);
    DetWorkspace w;
    while (det_carve(ws, E, C, tiles_per_ep, n_cells, (int)cap, &w) > ws_bytes) --cap;
    dim3 gt((tiles_per_ep + 7) / 8, E);
    det_tile_runs_kernel<<<gt, 256, 0, st>>>(idx, samp, active, HW, tiles_per_ep, w.tile_off, w.n_list, w.chunk_rows, w.n_long);
    det_scan_tiles_kernel<<<E, 1024, 0, st>>>(w.tile_off, tiles_per_ep, w.n_runs);
    det_cell_runs_kernel<<<gt, 256, 0, st>>>(idx, samp, active, HW, tiles_per_ep, n_cells, w.tile_off, w.cap, w.cell_runs, w.cell_list, w.n_list);
    det_scan_list_kernel<<<E, 1024, 0, st>>>(w.cell_runs, w.cell_list, w.n_list, w.cap, n_cells, w.list_off, w.cell_off);
    *out = w;
    return det_check_launch(what, "prepass");
}

int det_reduce(const char *what, const DetWorkspace &w, int C, int E, int64_t n_cells, const uint32_t *frame_cnt, float *sums, cudaStream_t st)
{
    switch (C) {
    case 128: return launch_det_reduce<128>(what, w, E, n_cells, frame_cnt, sums, st);
    case 256: return launch_det_reduce<256>(what, w, E, n_cells, frame_cnt, sums, st);
    case 512: return launch_det_reduce<512>(what, w, E, n_cells, frame_cnt, sums, st);
    default:
        eod_set_error("%s: C=%d not compiled in (128, 256, 512)", what, C);
        return EOD_ERR_UNSUPPORTED;
    }
}

namespace {

template <int C, bool kDet = false>
int launch_hwc(const void *feat, int feat_type, const int32_t *idx, const uint8_t *samp, const uint32_t *frame_cnt, const int32_t *active, int E,
               int HW, int64_t n_cells, float *sums, cudaStream_t st, const DetArgs det = DetArgs{});

// layout: EOD_LAYOUT_CHW (TMA kDet consumer) or a channels-last layout (write_mean_hwc_kernel kDet); the pre-passes and the reduce do
// not depend on it.  active: idle slots get no runs and their features are not read.
template <int C>
int launch_det(const void *feat, int layout, const int32_t *idx, const uint8_t *samp, const uint32_t *frame_cnt, const int32_t *active, int E,
               int HW, int64_t n_cells, float *sums, void *ws, size_t ws_bytes, cudaStream_t st)
{
    // the tensor map is encoded before any launch: a failure must not leave the pre-passes' counts in the workspace
    CUtensorMap tmap;
    int rc = layout == EOD_LAYOUT_CHW && HW % TILE_PX == 0 ? make_feature_tmap<C>(feat, E, HW, &tmap) : EOD_OK;
    if (rc) return rc;
    DetWorkspace w;
    if ((rc = det_prepass("eod_write_mean_det", idx, samp, active, E, C, HW, n_cells, ws, ws_bytes, &w, st))) return rc;
    if (layout == EOD_LAYOUT_CHW)
        rc = launch_tma_kernel<C, false, false, true>(tmap, idx, samp, frame_cnt, nullptr, active, E, HW, n_cells, sums, st, det_args(w));
    else
        rc = launch_hwc<C, true>(feat, layout == EOD_LAYOUT_HWC_BF16 ? FEAT_BF16 : (layout == EOD_LAYOUT_HWC_F16 ? FEAT_F16 : FEAT_F32), idx, samp,
                                 frame_cnt, active, E, HW, n_cells, sums, st, det_args(w));
    if (rc) return rc;
    return det_reduce("eod_write_mean_det", w, C, E, n_cells, frame_cnt, sums, st);
}

template <int C, int F = FEAT_F32>
int launch_ldg(const void *feat, const int32_t *idx, const uint8_t *samp, const uint32_t *frame_cnt, const int32_t *active, int E, int HW,
               int64_t n_cells, float *sums, cudaStream_t st)
{
    const int smem = C * TILE_PX * 4 + TILE_PX * 4 + TILE_PX;
    static unsigned long long attr_done = 0ull;
    if (int rc_attr = eod_ensure_dyn_smem(write_mean_chw_ldg_kernel<C, F>, smem, &attr_done, "eod_write_mean[ldg]")) return rc_attr;
    const int tiles_per_ep = (HW + TILE_PX - 1) / TILE_PX, n_tiles = tiles_per_ep * E;
    const int per_sm = (C >= 512) ? 3 : (C == 256 ? 6 : 8);
    const int grid = min(n_tiles, eod_num_sms() * per_sm);
    write_mean_chw_ldg_kernel<C, F><<<grid, C, smem, st>>>(reinterpret_cast<const typename FeatElem<F>::T *>(feat), idx, samp, frame_cnt, active, HW,
                                                           n_cells, tiles_per_ep, n_tiles, sums);
    return eod_check_launch("eod_write_mean[ldg]");
}

template <int C, bool kDet>
int launch_hwc(const void *feat, int feat_type, const int32_t *idx, const uint8_t *samp, const uint32_t *frame_cnt, const int32_t *active, int E,
               int HW, int64_t n_cells, float *sums, cudaStream_t st, const DetArgs det)
{
    const int strips_per_ep = (HW + TILE_PX - 1) / TILE_PX, n_strips = strips_per_ep * E;
    const int blocks = min((n_strips + 7) / 8, eod_num_sms() * 8);
    if (feat_type == FEAT_BF16) write_mean_hwc_kernel<C, FEAT_BF16, kDet><<<blocks, 256, 0, st>>>(feat, idx, samp, frame_cnt, active, HW, n_cells, strips_per_ep, n_strips, sums, det);
    else if (feat_type == FEAT_F16) write_mean_hwc_kernel<C, FEAT_F16, kDet><<<blocks, 256, 0, st>>>(feat, idx, samp, frame_cnt, active, HW, n_cells, strips_per_ep, n_strips, sums, det);
    else write_mean_hwc_kernel<C, FEAT_F32, kDet><<<blocks, 256, 0, st>>>(feat, idx, samp, frame_cnt, active, HW, n_cells, strips_per_ep, n_strips, sums, det);
    return eod_check_launch(kDet ? "eod_write_mean_det[hwc]" : "eod_write_mean[hwc]");
}

// 16-bit CHW features: the TMA ring takes 64-pixel tiles, the LDG kernel any HW with 16-byte aligned rows (checked by the caller)
template <int C, int F>
int dispatch_chw16(const void *feat, const int32_t *idx, const uint8_t *samp, const uint32_t *frame_cnt, const int32_t *active, int E, int HW,
                   int64_t n_cells, float *sums, int variant, cudaStream_t st)
{
    const bool tma_ok = (HW % TmaCfg<C, F>::kTilePx == 0) && (!samp || (reinterpret_cast<uintptr_t>(samp) % 16 == 0));
    if (variant == EOD_WRITE_TMA || variant == EOD_WRITE_TMA_DRY)
        EOD_REQUIRE(tma_ok, EOD_ERR_UNSUPPORTED, "eod_write_mean: TMA variant of 16-bit CHW features needs HW %% 64 == 0 and a 16-byte aligned samp");
    if (variant == EOD_WRITE_TMA_DRY) return launch_tma16<C, F, true>(feat, idx, samp, frame_cnt, active, E, HW, n_cells, sums, st);
    if (variant == EOD_WRITE_LDG || !tma_ok) return launch_ldg<C, F>(feat, idx, samp, frame_cnt, active, E, HW, n_cells, sums, st);
    return launch_tma16<C, F, false>(feat, idx, samp, frame_cnt, active, E, HW, n_cells, sums, st);
}

template <int C>
int dispatch(const float *feat, int layout, const int32_t *idx, const uint8_t *samp, const uint32_t *frame_cnt, const float *pix_n,
             const int32_t *active, int E, int HW, int64_t n_cells, float *sums, int variant, cudaStream_t st)
{
    if (layout == EOD_LAYOUT_HWC) return launch_hwc<C>(feat, FEAT_F32, idx, samp, frame_cnt, active, E, HW, n_cells, sums, st);
    if (layout == EOD_LAYOUT_HWC_BF16) return launch_hwc<C>(feat, FEAT_BF16, idx, samp, frame_cnt, active, E, HW, n_cells, sums, st);
    if (layout == EOD_LAYOUT_HWC_F16) return launch_hwc<C>(feat, FEAT_F16, idx, samp, frame_cnt, active, E, HW, n_cells, sums, st);
    if (layout == EOD_LAYOUT_CHW_BF16) return dispatch_chw16<C, FEAT_BF16>(feat, idx, samp, frame_cnt, active, E, HW, n_cells, sums, variant, st);
    if (layout == EOD_LAYOUT_CHW_F16) return dispatch_chw16<C, FEAT_F16>(feat, idx, samp, frame_cnt, active, E, HW, n_cells, sums, variant, st);
    const bool tma_ok = (HW % TILE_PX == 0) && (!samp || (reinterpret_cast<uintptr_t>(samp) % 16 == 0));
    if (variant == EOD_WRITE_TMA || variant == EOD_WRITE_TMA_DRY) EOD_REQUIRE(tma_ok, EOD_ERR_UNSUPPORTED, "eod_write_mean: TMA variant needs HW %% 32 == 0");
    if (variant == EOD_WRITE_TMA_DRY) return launch_tma<C, true>(feat, idx, samp, frame_cnt, pix_n, active, E, HW, n_cells, sums, st);
    if (variant == EOD_WRITE_LDG || !tma_ok) return launch_ldg<C>(feat, idx, samp, frame_cnt, active, E, HW, n_cells, sums, st);
    return launch_tma<C, false>(feat, idx, samp, frame_cnt, pix_n, active, E, HW, n_cells, sums, st);
}

}  // namespace

extern "C" int eod_sample_mask(const uint8_t *observed, int n_episodes, int HW, int stride, uint8_t *samp, int32_t *n_sampled,
                               eod_stream_t stream)
{
    EOD_REQUIRE(observed && samp, EOD_ERR_BADARG, "eod_sample_mask: null pointer");
    EOD_REQUIRE(n_episodes > 0 && HW > 0 && stride > 0, EOD_ERR_BADARG, "eod_sample_mask: bad sizes");
    if (HW % 16 == 0 && eod_aligned16(observed) && eod_aligned16(samp))
        sample_mask_vec_kernel<<<n_episodes, 1024, 0, (cudaStream_t)stream>>>(observed, HW, stride, samp, n_sampled);
    else
        sample_mask_kernel<<<n_episodes, 1024, 0, (cudaStream_t)stream>>>(observed, HW, stride, samp, n_sampled);
    return eod_check_launch("eod_sample_mask");
}

extern "C" int eod_frame_count(const int32_t *idx, const uint8_t *samp, const int32_t *active, int n_episodes, int HW,
                               int64_t n_cells, uint32_t *frame_cnt, int32_t *slot_of_cell, int32_t *slot_cell, int32_t *n_slots,
                               int n_slots_max, eod_stream_t stream)
{
    EOD_REQUIRE(idx && frame_cnt, EOD_ERR_BADARG, "eod_frame_count: null pointer");
    EOD_REQUIRE(n_episodes > 0 && n_episodes <= 65535 && HW > 0 && n_cells > 0, EOD_ERR_BADARG, "eod_frame_count: bad sizes");
    dim3 grid((HW + 256 * kCountSpan - 1) / (256 * kCountSpan), n_episodes);
    EOD_REQUIRE(!slot_of_cell || (slot_cell && n_slots && n_slots_max > 0), EOD_ERR_BADARG, "eod_frame_count: slot_of_cell needs slot_cell, n_slots and n_slots_max");
    frame_count_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(idx, samp, active, HW, n_cells, frame_cnt, slot_of_cell, slot_cell, n_slots, n_slots_max);
    return eod_check_launch("eod_frame_count");
}

extern "C" int eod_finalize_counts(const int32_t *idx, int n_episodes, int HW, int64_t n_cells, uint32_t *frame_cnt,
                                   float *counts, uint8_t *touched, const float *sums, void *norm16, int C,
                                   eod_stream_t stream)
{
    EOD_REQUIRE(!norm16 || (sums && C > 0 && C % 4 == 0 && eod_aligned16(sums) && eod_aligned16(norm16)), EOD_ERR_BADARG,
                "eod_finalize_counts: norm16 needs sums, C %% 4 == 0 and 16-byte aligned pointers");
    EOD_REQUIRE(idx && frame_cnt && counts, EOD_ERR_BADARG, "eod_finalize_counts: null pointer");
    EOD_REQUIRE(n_episodes > 0 && n_episodes <= 65535 && HW > 0 && n_cells > 0, EOD_ERR_BADARG, "eod_finalize_counts: bad sizes");
    if (n_cells <= 4 * (int64_t)HW && ((int64_t)n_episodes * n_cells) % 4 == 0 && eod_aligned16(frame_cnt)) {
        // grid comparable to the image: stream the cell plane once, no atomics
        const int64_t n_rows = (int64_t)n_episodes * n_cells;
        int64_t blocks = (n_rows + 2047) / 2048;                         // 2048 cells per block trip
        const int64_t cap = (int64_t)eod_num_sms() * 16;
        if (blocks > cap) blocks = cap;
        finalize_cells_kernel<<<(int)blocks, 256, 0, (cudaStream_t)stream>>>(n_rows, n_cells, frame_cnt, counts, touched, sums, (__half *)norm16, C);
        return eod_check_launch("eod_finalize_counts[cells]");
    }
    dim3 grid((HW + 255) / 256, n_episodes);
    finalize_counts_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(idx, HW, n_cells, frame_cnt, counts, touched, sums, (__half *)norm16, C);
    return eod_check_launch("eod_finalize_counts");
}

extern "C" int64_t eod_write_mean_det_workspace_bytes(int n_episodes, int C, int HW, int64_t n_cells, int runs_per_episode)
{
    if (n_episodes <= 0 || C <= 0 || HW <= 0 || n_cells <= 0) return -1;
    const int cap = runs_per_episode > 0 ? (runs_per_episode < HW ? runs_per_episode : HW) : HW / 4;
    return (int64_t)det_carve(nullptr, n_episodes, C, HW / TILE_PX, n_cells, cap, nullptr) + 4096;
}

extern "C" int64_t eod_write_mean_det_status_offset(int n_episodes, int64_t n_cells)
{
    return (int64_t)det_align((size_t)n_episodes * n_cells * 4);
}

extern "C" int eod_write_mean_det_layout(const void *feat, int layout, const int32_t *idx, const uint8_t *samp, const uint32_t *frame_cnt,
                                         const int32_t *active, int n_episodes, int C, int HW, int64_t n_cells, float *sums, void *workspace,
                                         int64_t workspace_bytes, eod_stream_t stream)
{
    EOD_REQUIRE(feat && idx && frame_cnt && sums, EOD_ERR_BADARG, "eod_write_mean_det: null pointer");
    EOD_REQUIRE(n_episodes > 0 && n_episodes <= 65535 && HW > 0 && n_cells > 0 && workspace_bytes > 0, EOD_ERR_BADARG, "eod_write_mean_det: bad sizes");
    EOD_REQUIRE(layout >= EOD_LAYOUT_CHW && layout <= EOD_LAYOUT_CHW_F16, EOD_ERR_BADARG, "eod_write_mean_det: bad layout");
    EOD_REQUIRE(layout != EOD_LAYOUT_CHW_BF16 && layout != EOD_LAYOUT_CHW_F16, EOD_ERR_UNSUPPORTED,
                "eod_write_mean_det: no deterministic write for 16-bit CHW features (use EOD_LAYOUT_CHW with fp32 features)");
    EOD_REQUIRE(eod_aligned16(feat) && eod_aligned16(idx) && eod_aligned16(sums), EOD_ERR_ALIGN, "eod_write_mean_det: pointers must be 16-byte aligned");
    cudaStream_t st = (cudaStream_t)stream;
    switch (C) {
    case 128: return launch_det<128>(feat, layout, idx, samp, frame_cnt, active, n_episodes, HW, n_cells, sums, workspace, (size_t)workspace_bytes, st);
    case 256: return launch_det<256>(feat, layout, idx, samp, frame_cnt, active, n_episodes, HW, n_cells, sums, workspace, (size_t)workspace_bytes, st);
    case 512: return launch_det<512>(feat, layout, idx, samp, frame_cnt, active, n_episodes, HW, n_cells, sums, workspace, (size_t)workspace_bytes, st);
    default:
        eod_set_error("eod_write_mean_det: C=%d not compiled in (128, 256, 512)", C);
        return EOD_ERR_UNSUPPORTED;
    }
}

extern "C" int eod_write_mean_det(const float *feat, const int32_t *idx, const uint8_t *samp, const uint32_t *frame_cnt, int n_episodes, int C,
                                  int HW, int64_t n_cells, float *sums, void *workspace, int64_t workspace_bytes, eod_stream_t stream)
{
    return eod_write_mean_det_layout(feat, EOD_LAYOUT_CHW, idx, samp, frame_cnt, nullptr, n_episodes, C, HW, n_cells, sums, workspace, workspace_bytes, stream);
}

extern "C" int eod_expand_counts(const int32_t *idx, const uint32_t *frame_cnt, int n_episodes, int HW, int64_t n_cells,
                                 float *pix_inv_n, eod_stream_t stream)
{
    EOD_REQUIRE(idx && frame_cnt && pix_inv_n, EOD_ERR_BADARG, "eod_expand_counts: null pointer");
    EOD_REQUIRE(n_episodes > 0 && n_episodes <= 65535 && HW > 0 && n_cells > 0, EOD_ERR_BADARG, "eod_expand_counts: bad sizes");
    if (HW % 4 == 0 && eod_aligned16(idx) && eod_aligned16(pix_inv_n)) {
        dim3 grid4((HW / 4 + 255) / 256, n_episodes);
        expand_counts_vec4_kernel<<<grid4, 256, 0, (cudaStream_t)stream>>>(idx, frame_cnt, HW, n_cells, pix_inv_n);
        return eod_check_launch("eod_expand_counts");
    }
    dim3 grid((HW + 255) / 256, n_episodes);
    expand_counts_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(idx, frame_cnt, HW, n_cells, pix_inv_n);
    return eod_check_launch("eod_expand_counts");
}

extern "C" int eod_write_mean(const void *feat_any, int layout, const int32_t *idx, const uint8_t *samp, const uint32_t *frame_cnt,
                              int n_episodes, int C, int HW, int64_t n_cells, float *sums, int variant, const float *pix_inv_n,
                              const int32_t *active, eod_stream_t stream)
{
    const float *feat = reinterpret_cast<const float *>(feat_any);
    EOD_REQUIRE(!pix_inv_n || eod_aligned16(pix_inv_n), EOD_ERR_ALIGN, "eod_write_mean: pix_inv_n must be 16-byte aligned");
    EOD_REQUIRE(feat && idx && frame_cnt && sums, EOD_ERR_BADARG, "eod_write_mean: null pointer");
    EOD_REQUIRE(n_episodes > 0 && HW > 0 && n_cells > 0, EOD_ERR_BADARG, "eod_write_mean: bad sizes");
    EOD_REQUIRE(layout >= EOD_LAYOUT_CHW && layout <= EOD_LAYOUT_CHW_F16, EOD_ERR_BADARG, "eod_write_mean: bad layout");
    EOD_REQUIRE(variant >= EOD_WRITE_AUTO && variant <= EOD_WRITE_TMA_DRY, EOD_ERR_BADARG, "eod_write_mean: bad variant");
    EOD_REQUIRE(eod_aligned16(feat) && eod_aligned16(sums) && eod_aligned16(idx), EOD_ERR_ALIGN, "eod_write_mean: pointers must be 16-byte aligned");
    EOD_REQUIRE(layout != EOD_LAYOUT_CHW || HW % 4 == 0, EOD_ERR_ALIGN, "eod_write_mean: CHW rows must be 16-byte aligned (HW %% 4 == 0)");
    const bool chw16 = layout == EOD_LAYOUT_CHW_BF16 || layout == EOD_LAYOUT_CHW_F16;
    EOD_REQUIRE(!chw16 || HW % 8 == 0, EOD_ERR_ALIGN, "eod_write_mean: 16-bit CHW rows must be 16-byte aligned (HW %% 8 == 0)");
    EOD_REQUIRE(!chw16 || !pix_inv_n, EOD_ERR_UNSUPPORTED, "eod_write_mean: pix_inv_n is not supported with 16-bit CHW features");
    cudaStream_t st = (cudaStream_t)stream;
    switch (C) {
    case 128: return dispatch<128>(feat, layout, idx, samp, frame_cnt, pix_inv_n, active, n_episodes, HW, n_cells, sums, variant, st);
    case 256: return dispatch<256>(feat, layout, idx, samp, frame_cnt, pix_inv_n, active, n_episodes, HW, n_cells, sums, variant, st);
    case 512: return dispatch<512>(feat, layout, idx, samp, frame_cnt, pix_inv_n, active, n_episodes, HW, n_cells, sums, variant, st);
    default:
        eod_set_error("eod_write_mean: C=%d not compiled in (128, 256, 512)", C);
        return EOD_ERR_UNSUPPORTED;
    }
}

extern "C" int eod_box_to_image_features(const float *box_features, const uint8_t *masks, int K, int C, int HW,
                                         float *image_features, uint8_t *observed, eod_stream_t stream)
{
    EOD_REQUIRE(box_features && masks && image_features, EOD_ERR_BADARG, "eod_box_to_image_features: null pointer");
    EOD_REQUIRE(K > 0 && K <= 256 && C > 0 && HW > 0, EOD_ERR_BADARG, "eod_box_to_image_features: bad sizes (K must be 1..256)");
    dim3 grid((HW + 255) / 256, (C + 15) / 16);
    box_to_image_kernel<<<grid, 256, (size_t)K * 16 * sizeof(float), (cudaStream_t)stream>>>(box_features, masks, K, C, HW, image_features, observed);
    return eod_check_launch("eod_box_to_image_features");
}
