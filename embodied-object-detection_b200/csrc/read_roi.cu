// Per-ROI memory read (BASELINE north star, subsystem 3): the map feature of a detection proposal = ROIAlign of the pooled
// memory levels over the proposal's box.
//
// The reference never forms this tensor on its own: it sums the projected memory into the FPN levels p3-p5 (timm.py:170-189)
// and the ROI heads then pool the FUSED levels per proposal (detic_roi_heads.py:331-334: self.box_pooler(features, boxes) =
// detectron2 ROIPooler: ROIAlignV2 = aligned, sampling_ratio 0, 7x7 bins, scales 1/8, 1/16, 1/32, FPN level assignment).
// ROIAlign is linear in its input, so  pool(res + w * (conv(L) + b)) = pool(res) + w * (conv(pool(L)) + b):  pooling the
// memory levels L (what eod_read_pool produces) with the same boxes gives the per-ROI map feature that the fused path
// carries implicitly.  This kernel is that pooling, for all proposals of all episodes in one launch:
//   * level assignment in the kernel, detectron2 assign_boxes_to_levels: floor(4 + log2(sqrt(area) / 224 + eps)) clamped
//     to [min_level, max_level] - fp32 like torch.  A box with no level there (NaN size: inverted in exactly one axis, or a NaN
//     coordinate) and a box whose batch_idx names no episode pool nothing: zero bins, valid 0, level -1;
//   * bilinear sampling with the exact point set, clamping rules and operation order of the ROIAlign CPU kernel
//     (torchvision/csrc/ops/cpu/roi_align_kernel.cpp, which tests/ execute as the oracle): per bin, samples row-major,
//     val = w1*v1 + w2*v2 + w3*v3 + w4*v4 accumulated in fp32, then / count;
//   * a warp owns one (proposal, bin); lanes own C/32 consecutive channels, so every tap is one coalesced C*2-byte row of a
//     channels-last fp16 level (the levels of a frame, 6 300 pixels x C, live in L2).
// Output: (R, P, P, C) fp32 channels-last (logical (R, C, P, P)), plus the level each proposal was assigned to (-1: none).
#include "eod_common.cuh"

namespace {

struct RoiLevels {
    const __half *ptr[4];      // (E, h, w, C) fp16 channels-last
    int h[4], w[4];
    float scale[4];            // 1 / stride
    int n;
};

template <int V>
__device__ __forceinline__ void load_tap(const __half *row, int lane, float (&v)[V])
{
#pragma unroll
    for (int i = 0; i < V / 8; ++i) {
        const uint4 q = __ldg(reinterpret_cast<const uint4 *>(row + (size_t)lane * V) + i);
        const uint32_t w[4] = {q.x, q.y, q.z, q.w};
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            const float2 f = __half22float2(*reinterpret_cast<const __half2 *>(&w[k]));
            v[8 * i + 2 * k] = f.x;
            v[8 * i + 2 * k + 1] = f.y;
        }
    }
}
template <>
__device__ __forceinline__ void load_tap<4>(const __half *row, int lane, float (&v)[4])
{
    const uint2 q = __ldg(reinterpret_cast<const uint2 *>(row) + lane);
    const float2 a = __half22float2(*reinterpret_cast<const __half2 *>(&q.x)), b = __half22float2(*reinterpret_cast<const __half2 *>(&q.y));
    v[0] = a.x; v[1] = a.y; v[2] = b.x; v[3] = b.y;
}

// detectron2 modeling/poolers.py assign_boxes_to_levels (fp32 tensor arithmetic); -1 for no level
__device__ __forceinline__ int assign_level(float x1, float y1, float x2, float y2, int n_levels, int min_level, float canonical_size,
                                            int canonical_level)
{
    const float area = __fmul_rn(__fsub_rn(x2, x1), __fsub_rn(y2, y1));
    const float s = __fsqrt_rn(area);
    const float lg = log2f(__fadd_rn(__fdiv_rn(s, canonical_size), 2.220446049250313e-16f));
    float lvl = floorf(__fadd_rn((float)canonical_level, lg));
    // NaN (negative area, NaN coordinate): torch.clamp keeps the NaN and the cast to int64 after it yields an integer outside every
    // level, so ROIPooler pools the box from no level
    if (!(lvl == lvl)) return -1;
    lvl = fminf(fmaxf(lvl, (float)min_level), (float)(min_level + n_levels - 1));
    return (int)lvl - min_level;
}

template <int C>
__global__ void __launch_bounds__(256) read_roi_kernel(RoiLevels L, const float *__restrict__ boxes, const int32_t *__restrict__ batch_idx, int n_episodes, int P,
                                                       int sampling_ratio, int min_level, float canonical_size, int canonical_level,
                                                       float *__restrict__ out, int32_t *__restrict__ out_level, float *__restrict__ out_valid)
{
    constexpr int V = C / 32;
    const int r = blockIdx.x;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, n_warps = blockDim.x >> 5;
    const float x1 = __ldg(boxes + 4 * r), y1 = __ldg(boxes + 4 * r + 1), x2 = __ldg(boxes + 4 * r + 2), y2 = __ldg(boxes + 4 * r + 3);
    int lv = assign_level(x1, y1, x2, y2, L.n, min_level, canonical_size, canonical_level);
    const int e = batch_idx ? __ldg(batch_idx + r) : 0;
    if (e < 0 || e >= n_episodes) lv = -1;
    if (threadIdx.x == 0 && out_level) out_level[r] = lv;
    const bool none = lv < 0;                       // takes no samples below: zero bins, valid 0
    const int h = L.h[none ? 0 : lv], w = L.w[none ? 0 : lv];
    const float sc = L.scale[none ? 0 : lv];
    const __half *base = L.ptr[none ? 0 : lv] + (size_t)(none ? 0 : e) * h * w * C;
    // ROIAlign, aligned = true (detectron2 ROIAlignV2): half-pixel offset, no minimum roi size
    const float rsw = __fsub_rn(__fmul_rn(x1, sc), 0.5f), rsh = __fsub_rn(__fmul_rn(y1, sc), 0.5f);
    const float rew = __fsub_rn(__fmul_rn(x2, sc), 0.5f), reh = __fsub_rn(__fmul_rn(y2, sc), 0.5f);
    const float roi_w = __fsub_rn(rew, rsw), roi_h = __fsub_rn(reh, rsh);
    const float bin_h = __fdiv_rn(roi_h, (float)P), bin_w = __fdiv_rn(roi_w, (float)P);
    const int gh = none ? 0 : sampling_ratio > 0 ? sampling_ratio : (int)ceilf(__fdiv_rn(roi_h, (float)P));
    const int gw = none ? 0 : sampling_ratio > 0 ? sampling_ratio : (int)ceilf(__fdiv_rn(roi_w, (float)P));
    const float count = (float)max(gh * gw, 1);

    for (int bin = warp; bin < P * P; bin += n_warps) {
        const int ph = bin / P, pw = bin - ph * P;
        float acc[V];
#pragma unroll
        for (int k = 0; k < V; ++k) acc[k] = 0.f;
        int n_valid = 0;
        for (int iy = 0; iy < gh; ++iy) {
            const float yy = __fadd_rn(__fadd_rn(rsh, __fmul_rn((float)ph, bin_h)), __fdiv_rn(__fmul_rn(__fadd_rn((float)iy, 0.5f), bin_h), (float)gh));
            for (int ix = 0; ix < gw; ++ix) {
                const float xx = __fadd_rn(__fadd_rn(rsw, __fmul_rn((float)pw, bin_w)), __fdiv_rn(__fmul_rn(__fadd_rn((float)ix, 0.5f), bin_w), (float)gw));
                float y = yy, x = xx;
                if (y < -1.0f || y > (float)h || x < -1.0f || x > (float)w) continue;        // empty sample: contributes 0
                ++n_valid;
                if (y <= 0.f) y = 0.f;
                if (x <= 0.f) x = 0.f;
                int y_low = (int)y, x_low = (int)x, y_high, x_high;
                if (y_low >= h - 1) { y_high = y_low = h - 1; y = (float)y_low; } else y_high = y_low + 1;
                if (x_low >= w - 1) { x_high = x_low = w - 1; x = (float)x_low; } else x_high = x_low + 1;
                const float ly = __fsub_rn(y, (float)y_low), lx = __fsub_rn(x, (float)x_low);
                const float hy = __fsub_rn(1.f, ly), hx = __fsub_rn(1.f, lx);
                const float w1 = __fmul_rn(hy, hx), w2 = __fmul_rn(hy, lx), w3 = __fmul_rn(ly, hx), w4 = __fmul_rn(ly, lx);
                float v1[V], v2[V], v3[V], v4[V];
                load_tap<V>(base + ((size_t)y_low * w + x_low) * C, lane, v1);
                load_tap<V>(base + ((size_t)y_low * w + x_high) * C, lane, v2);
                load_tap<V>(base + ((size_t)y_high * w + x_low) * C, lane, v3);
                load_tap<V>(base + ((size_t)y_high * w + x_high) * C, lane, v4);
#pragma unroll
                for (int k = 0; k < V; ++k) {
                    const float val = __fadd_rn(__fadd_rn(__fadd_rn(__fmul_rn(w1, v1[k]), __fmul_rn(w2, v2[k])), __fmul_rn(w3, v3[k])), __fmul_rn(w4, v4[k]));
                    acc[k] = __fadd_rn(acc[k], val);
                }
            }
        }
        // what ROIAlign makes of a constant-1 plane: the share of this bin's sample points that fall on the level (the bias of a 1x1
        // projection applied BEFORE the pooling survives it with exactly this factor; 0 for empty / inverted boxes and boxes without a level)
        if (out_valid && lane == 0) out_valid[(size_t)r * P * P + bin] = __fdiv_rn((float)n_valid, count);
        float *dst = out + ((size_t)r * P * P + bin) * C + (size_t)lane * V;
#pragma unroll
        for (int k = 0; k < V; k += 4)
            *reinterpret_cast<float4 *>(dst + k) = make_float4(__fdiv_rn(acc[k], count), __fdiv_rn(acc[k + 1], count), __fdiv_rn(acc[k + 2], count),
                                                               __fdiv_rn(acc[k + 3], count));
    }
}

}  // namespace

extern "C" int eod_read_roi(int n_levels, const void *const *levels, const int *level_h, const int *level_w, const float *level_scale,
                            int n_episodes, int C, const float *boxes, const int32_t *batch_idx, int n_rois, int pooled, int sampling_ratio,
                            int min_level, float canonical_size, int canonical_level, float *out, int32_t *out_level, float *out_valid, eod_stream_t stream)
{
    EOD_REQUIRE(levels && level_h && level_w && level_scale && boxes && out, EOD_ERR_BADARG, "eod_read_roi: null pointer");
    EOD_REQUIRE(n_levels >= 1 && n_levels <= 4 && n_episodes > 0 && n_rois >= 0 && pooled > 0 && pooled <= 32 && sampling_ratio >= 0,
                EOD_ERR_BADARG, "eod_read_roi: bad sizes (1..4 levels, pooled 1..32)");
    EOD_REQUIRE(canonical_size > 0.f, EOD_ERR_BADARG, "eod_read_roi: canonical box size must be positive");
    if (n_rois == 0) return EOD_OK;
    RoiLevels L;
    L.n = n_levels;
    for (int l = 0; l < 4; ++l) {
        const int k = l < n_levels ? l : n_levels - 1;
        EOD_REQUIRE(levels[k] && level_h[k] > 0 && level_w[k] > 0 && level_scale[k] > 0.f, EOD_ERR_BADARG, "eod_read_roi: bad level %d", k);
        EOD_REQUIRE(eod_aligned16(levels[k]), EOD_ERR_ALIGN, "eod_read_roi: levels must be 16-byte aligned");
        L.ptr[l] = (const __half *)levels[k]; L.h[l] = level_h[k]; L.w[l] = level_w[k]; L.scale[l] = level_scale[k];
    }
    EOD_REQUIRE(eod_aligned16(out), EOD_ERR_ALIGN, "eod_read_roi: out must be 16-byte aligned");
    cudaStream_t st = (cudaStream_t)stream;
    switch (C) {
    case 128: read_roi_kernel<128><<<n_rois, 256, 0, st>>>(L, boxes, batch_idx, n_episodes, pooled, sampling_ratio, min_level, canonical_size, canonical_level, out, out_level, out_valid); break;
    case 256: read_roi_kernel<256><<<n_rois, 256, 0, st>>>(L, boxes, batch_idx, n_episodes, pooled, sampling_ratio, min_level, canonical_size, canonical_level, out, out_level, out_valid); break;
    case 512: read_roi_kernel<512><<<n_rois, 256, 0, st>>>(L, boxes, batch_idx, n_episodes, pooled, sampling_ratio, min_level, canonical_size, canonical_level, out, out_level, out_valid); break;
    default:
        eod_set_error("eod_read_roi: C=%d not compiled in (128, 256, 512)", C);
        return EOD_ERR_UNSUPPORTED;
    }
    return eod_check_launch("eod_read_roi");
}
