// Depth back-projection + pose transform + quantisation to map-cell indices (SURVEY 8a rows A2-A5).
//
// One thread per pixel; every access is coalesced (depth read, idx/mask/height writes).  ~9 B/pixel of
// HBM traffic, so the kernel is a small streaming pass; it exists to be BIT-EXACT with torch-CPU:
//   x_scale = ((u + 0.5) - cx) / fx         IEEE divide          (core.py:107)
//   world_r = fma(T3,1, fma(T2,z, fma(T1,y, T0*x)))              (core.py:175, torch.bmm K=4 on CPU)
//   q       = rint((world - shift0 - shift1) / cell)             (core.py:220, build_memory_data.py:135-136)
// All arithmetic uses explicit _rn intrinsics so nvcc can neither contract nor reassociate (the per-pixel helpers live in
// backproject.cuh, shared with the height-max contest of write_max.cu).
#include "backproject.cuh"

namespace {

struct BackprojectParams {
    const void *depth;
    double depth_div;
    const float *pose;
    const float *shifts;
    int32_t *idx;
    int32_t *q2;
    uint8_t *outlier;
    float *height;
    float *world;
    int H, W;
    float fx, fy, cx, cy, cell, z_clip;
    int map_w, map_h, order;
    // optional, 4-pixel kernel only: per-cell pixel counts of the frame (eod_frame_count without a sample mask) folded into this launch
    uint32_t *frame_cnt;
    const int32_t *active;
    int64_t n_cells;
};

template <bool U16>
__global__ void __launch_bounds__(256) backproject_quantize_kernel(const BackprojectParams P)
{
    const int e = blockIdx.y;
    const int HW = P.H * P.W;
    const int p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= HW) return;
    const int v = p / P.W, u = p - v * P.W;

    const float *T = P.pose + 12 * e;       // uniform across the block: served by the constant/L1 path
    const float *S = P.shifts + 6 * e;

    const float xs = pixel_scale(u, P.cx, P.fx);
    const float ys = pixel_scale(v, P.cy, P.fy);
    const size_t g = (size_t)e * HW + p;
    const float z = load_depth<U16>(P.depth, P.depth_div, g);
    const float x = __fmul_rn(z, xs);
    const float y = __fmul_rn(z, ys);

    float w[3];
#pragma unroll
    for (int r = 0; r < 3; ++r) {
        const float t0 = __ldg(T + 4 * r), t1 = __ldg(T + 4 * r + 1), t2 = __ldg(T + 4 * r + 2), t3 = __ldg(T + 4 * r + 3);
        w[r] = pose_row(t0, t1, t2, t3, x, y, z);
    }
    const float p0x = __fsub_rn(w[0], __ldg(S + 0)), p0y = __fsub_rn(w[1], __ldg(S + 1)), p0z = __fsub_rn(w[2], __ldg(S + 2));
    if (P.world) {
        float *o = P.world + 3 * g;
        o[0] = p0x; o[1] = p0y; o[2] = p0z;
    }
    const float p1x = __fsub_rn(p0x, __ldg(S + 3)), p1y = __fsub_rn(p0y, __ldg(S + 4)), p1z = __fsub_rn(p0z, __ldg(S + 5));
    const float qx = quantize(p1x, P.cell);
    const float qz = quantize(p1z, P.cell);
    if (P.q2) {
        P.q2[2 * g] = (int32_t)qx;
        P.q2[2 * g + 1] = (int32_t)qz;
    }
    if (P.outlier) {
        const float thr = __fadd_rn(__ldg(T + 7), P.z_clip);
        P.outlier[g] = is_outlier(qx, qz, p1y, thr, z, P.map_w, P.map_h) ? 1 : 0;
    }
    if (P.height) P.height[g] = p1y;
    if (P.idx) {
        const int ix = clip_cell(qx, P.map_w), iz = clip_cell(qz, P.map_h);
        P.idx[g] = P.order == EOD_ORDER_XZ ? ix * P.map_h + iz : iz * P.map_w + ix;
    }
}

// Same arithmetic, four consecutive pixels of one image row per thread (W % 4 == 0, 16-byte aligned planes): 128-bit depth loads
// and index stores, the pose / shift scalars and the row's y_scale are fetched and computed once per thread instead of
// once per pixel (the scalar kernel issued 18 uniform loads and 4 IEEE divides per pixel).
template <bool U16>
__global__ void __launch_bounds__(256) backproject_quantize_vec4_kernel(const BackprojectParams P)
{
    const int e = blockIdx.y;
    const int HW = P.H * P.W;
    const int p = (blockIdx.x * blockDim.x + threadIdx.x) * 4;
    if (p >= HW) return;
    const int v = p / P.W, u0 = p - v * P.W;

    const float *T = P.pose + 12 * e;
    const float *S = P.shifts + 6 * e;
    float t[12], sh[6];
#pragma unroll
    for (int i = 0; i < 12; ++i) t[i] = __ldg(T + i);
#pragma unroll
    for (int i = 0; i < 6; ++i) sh[i] = __ldg(S + i);
    const float ys = pixel_scale(v, P.cy, P.fy);
    const float thr = __fadd_rn(t[7], P.z_clip);
    const size_t g = (size_t)e * HW + p;
    float zz[4];
    if (U16) {
        const uint2 d = __ldg(reinterpret_cast<const uint2 *>(reinterpret_cast<const uint16_t *>(P.depth) + g));
        const uint32_t raw[4] = {d.x & 0xffffu, d.x >> 16, d.y & 0xffffu, d.y >> 16};
#pragma unroll
        for (int k = 0; k < 4; ++k) zz[k] = __double2float_rn(__ddiv_rn((double)raw[k], P.depth_div));
    } else {
        const float4 d4 = __ldg(reinterpret_cast<const float4 *>(reinterpret_cast<const float *>(P.depth) + g));
        zz[0] = d4.x; zz[1] = d4.y; zz[2] = d4.z; zz[3] = d4.w;
    }
    int idx4[4], q2v[8];
    uint32_t out4 = 0;
    float h4[4], w12[12];
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        const float z = zz[k];
        float p0[3], p1[3];
        world_point(z, pixel_scale(u0 + k, P.cx, P.fx), ys, t, sh, p0, p1);
        w12[3 * k] = p0[0]; w12[3 * k + 1] = p0[1]; w12[3 * k + 2] = p0[2];
        const float qx = quantize(p1[0], P.cell);
        const float qz = quantize(p1[2], P.cell);
        q2v[2 * k] = (int32_t)qx; q2v[2 * k + 1] = (int32_t)qz;
        out4 |= (is_outlier(qx, qz, p1[1], thr, z, P.map_w, P.map_h) ? 1u : 0u) << (8 * k);
        h4[k] = p1[1];
        const int ix = clip_cell(qx, P.map_w), iz = clip_cell(qz, P.map_h);
        idx4[k] = P.order == EOD_ORDER_XZ ? ix * P.map_h + iz : iz * P.map_w + ix;
    }
    if (P.world) {
        float4 *o = reinterpret_cast<float4 *>(P.world + 3 * g);
        o[0] = make_float4(w12[0], w12[1], w12[2], w12[3]);
        o[1] = make_float4(w12[4], w12[5], w12[6], w12[7]);
        o[2] = make_float4(w12[8], w12[9], w12[10], w12[11]);
    }
    if (P.q2) {
        int4 *o = reinterpret_cast<int4 *>(P.q2 + 2 * g);
        o[0] = make_int4(q2v[0], q2v[1], q2v[2], q2v[3]);
        o[1] = make_int4(q2v[4], q2v[5], q2v[6], q2v[7]);
    }
    if (P.outlier) *reinterpret_cast<uint32_t *>(P.outlier + g) = out4;
    if (P.height) *reinterpret_cast<float4 *>(P.height + g) = make_float4(h4[0], h4[1], h4[2], h4[3]);
    if (P.idx) *reinterpret_cast<int4 *>(P.idx + g) = make_int4(idx4[0], idx4[1], idx4[2], idx4[3]);
    if (P.frame_cnt && (!P.active || __ldg(P.active + e) > 0)) {
        // Per-cell pixel counts over the warp's 128 consecutive pixels with ONE integer atomic per run of equal cell id (the host only
        // asks for this when H * W % 128 == 0: warps are full).  A lane issues the atomics of the runs that START among its four pixels;
        // a run that reaches the lane's last pixel also takes the pixels it continues into: four from every following lane it swallows
        // whole, then the leading pixels of the first lane where it ends.  Equals frame_count_kernel without a sample mask (sums of 1).
        const unsigned lane = threadIdx.x & 31;
        const int c0 = idx4[0], c1 = idx4[1], c2 = idx4[2], c3 = idx4[3];
        const int prev3 = __shfl_up_sync(0xffffffffu, c3, 1);
        const bool h0 = lane == 0 || prev3 != c0, h1 = c1 != c0, h2 = c2 != c1, h3 = c3 != c2;
        const int lead = h1 ? 1 : (h2 ? 2 : (h3 ? 3 : 4));                 // pixels before the lane's first internal run head
        const unsigned cont_mask = __ballot_sync(0xffffffffu, !h0);        // lanes whose first pixel continues the previous lane's run
        const unsigned full_mask = __ballot_sync(0xffffffffu, !h0 && lead == 4);
        const unsigned above = lane == 31 ? 0u : (0xffffffffu << (lane + 1));
        const unsigned stop = ~full_mask & above;
        const int M = stop ? (__ffs(stop) - 1) : 32;                       // first following lane that is not swallowed whole
        const int lead_m = __shfl_sync(0xffffffffu, lead, M & 31);
        const int ext = 4 * (M - (int)lane - 1) + ((M < 32 && ((cont_mask >> M) & 1u)) ? lead_m : 0);
        uint32_t *cnt = P.frame_cnt + (size_t)e * P.n_cells;
        const int end1 = h2 ? 2 : (h3 ? 3 : 4), end2 = h3 ? 3 : 4;          // end of a run starting at pixel 1 / 2
        if (h0) atomicAdd(cnt + c0, (uint32_t)(lead + (lead == 4 ? ext : 0)));
        if (h1) atomicAdd(cnt + c1, (uint32_t)(end1 - 1 + (end1 == 4 ? ext : 0)));
        if (h2) atomicAdd(cnt + c2, (uint32_t)(end2 - 2 + (end2 == 4 ? ext : 0)));
        if (h3) atomicAdd(cnt + c3, (uint32_t)(1 + ext));
    }
}

// World xyz (as stored in sensor_data/*.h5 'projection_indices', SMNet/build_data.py:209-213,280) -> flat clipped cell
// index: exactly SMNet/build_memory_data.py:135-143 (shift, IEEE divide, round-half-even, clip, z*map_w + x).
__global__ void __launch_bounds__(256) quantize_world_kernel(const float *__restrict__ world, int64_t n, float sx, float sz, float cell,
                                                             int map_w, int map_h, int order, int32_t *__restrict__ idx)
{
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const float x = __ldg(world + 3 * i), z = __ldg(world + 3 * i + 2);
    idx[i] = flat_cell(quantize(__fsub_rn(x, sx), cell), quantize(__fsub_rn(z, sz), cell), map_w, map_h, order);
}

}  // namespace

extern "C" int eod_quantize_world(const float *world, int64_t n_points, float shift_x, float shift_z, float cell, int map_w, int map_h,
                                  int order, int32_t *idx, eod_stream_t stream)
{
    EOD_REQUIRE(world && idx, EOD_ERR_BADARG, "eod_quantize_world: null pointer");
    EOD_REQUIRE(n_points > 0 && map_w > 0 && map_h > 0 && cell > 0.0f, EOD_ERR_BADARG, "eod_quantize_world: bad sizes");
    EOD_REQUIRE(order == EOD_ORDER_ZX || order == EOD_ORDER_XZ, EOD_ERR_BADARG, "eod_quantize_world: bad order");
    EOD_REQUIRE((int64_t)map_w * map_h < (int64_t)INT32_MAX, EOD_ERR_BADARG, "eod_quantize_world: map too large");
    const int64_t blocks = (n_points + 255) / 256;
    EOD_REQUIRE(blocks <= 0x7fffffff, EOD_ERR_BADARG, "eod_quantize_world: too many points for one launch");
    quantize_world_kernel<<<(unsigned)blocks, 256, 0, (cudaStream_t)stream>>>(world, n_points, shift_x, shift_z, cell, map_w, map_h, order, idx);
    return eod_check_launch("eod_quantize_world");
}

static int backproject_launch(const void *depth, bool u16, double depth_div, const float *pose, const float *shifts, int n_episodes,
                              int H, int W, float fx, float fy, float cx, float cy, float cell, int map_w,
                              int map_h, int order, float z_clip, int32_t *idx, int32_t *q2,
                              uint8_t *outlier, float *height, float *world, eod_stream_t stream, uint32_t *frame_cnt = nullptr,
                              const int32_t *active = nullptr)
{
    EOD_REQUIRE(depth && pose && shifts, EOD_ERR_BADARG, "eod_backproject_quantize: null input");
    EOD_REQUIRE(n_episodes > 0 && H > 0 && W > 0 && map_w > 0 && map_h > 0, EOD_ERR_BADARG,
                "eod_backproject_quantize: non-positive size");
    EOD_REQUIRE(order == EOD_ORDER_ZX || order == EOD_ORDER_XZ, EOD_ERR_BADARG, "eod_backproject_quantize: bad order");
    EOD_REQUIRE(cell > 0.0f && fx != 0.0f && fy != 0.0f, EOD_ERR_BADARG, "eod_backproject_quantize: bad cell/intrinsics");
    EOD_REQUIRE((int64_t)map_w * map_h < (int64_t)INT32_MAX, EOD_ERR_BADARG, "eod_backproject_quantize: map too large");
    EOD_REQUIRE(n_episodes <= 65535, EOD_ERR_BADARG, "eod_backproject_quantize: n_episodes > 65535");
    BackprojectParams P{depth, depth_div, pose, shifts, idx, q2, outlier, height, world, H, W, fx, fy, cx, cy, cell, z_clip, map_w, map_h, order,
                        frame_cnt, active, (int64_t)map_w * map_h};
    const bool vec = W % 4 == 0 && eod_aligned16(depth) && (!idx || eod_aligned16(idx)) && (!q2 || eod_aligned16(q2)) &&
                     (!outlier || (reinterpret_cast<uintptr_t>(outlier) & 3u) == 0) && (!height || eod_aligned16(height)) && (!world || eod_aligned16(world));
    EOD_REQUIRE(!frame_cnt || (vec && (H * W) % 128 == 0), EOD_ERR_UNSUPPORTED,
                "eod_backproject_count: the fused count needs W %% 4 == 0, H * W %% 128 == 0 and 16-byte aligned planes (run eod_frame_count instead)");
    if (vec) {
        dim3 grid((H * W / 4 + 255) / 256, n_episodes);
        if (u16) backproject_quantize_vec4_kernel<true><<<grid, 256, 0, (cudaStream_t)stream>>>(P);
        else backproject_quantize_vec4_kernel<false><<<grid, 256, 0, (cudaStream_t)stream>>>(P);
    } else {
        dim3 grid((H * W + 255) / 256, n_episodes);
        if (u16) backproject_quantize_kernel<true><<<grid, 256, 0, (cudaStream_t)stream>>>(P);
        else backproject_quantize_kernel<false><<<grid, 256, 0, (cudaStream_t)stream>>>(P);
    }
    return eod_check_launch("eod_backproject_quantize");
}

extern "C" int eod_backproject_quantize(const float *depth, const float *pose, const float *shifts, int n_episodes,
                                        int H, int W, float fx, float fy, float cx, float cy, float cell, int map_w,
                                        int map_h, int order, float z_clip, int32_t *idx, int32_t *q2,
                                        uint8_t *outlier, float *height, float *world, eod_stream_t stream)
{
    return backproject_launch(depth, false, 1.0, pose, shifts, n_episodes, H, W, fx, fy, cx, cy, cell, map_w, map_h, order, z_clip, idx, q2,
                              outlier, height, world, stream);
}

extern "C" int eod_backproject_quantize_u16(const uint16_t *depth, double depth_div, const float *pose, const float *shifts, int n_episodes,
                                            int H, int W, float fx, float fy, float cx, float cy, float cell, int map_w,
                                            int map_h, int order, float z_clip, int32_t *idx, int32_t *q2,
                                            uint8_t *outlier, float *height, float *world, eod_stream_t stream)
{
    EOD_REQUIRE(depth_div > 0.0, EOD_ERR_BADARG, "eod_backproject_quantize_u16: depth_div must be positive");
    return backproject_launch(depth, true, depth_div, pose, shifts, n_episodes, H, W, fx, fy, cx, cy, cell, map_w, map_h, order, z_clip, idx, q2,
                              outlier, height, world, stream);
}

extern "C" int eod_backproject_count(const void *depth, int depth_is_u16, double depth_div, const float *pose, const float *shifts, int n_episodes,
                                     int H, int W, float fx, float fy, float cx, float cy, float cell, int map_w, int map_h, int order,
                                     const int32_t *active, int32_t *idx, uint32_t *frame_cnt, eod_stream_t stream)
{
    EOD_REQUIRE(idx && frame_cnt, EOD_ERR_BADARG, "eod_backproject_count: null output");
    EOD_REQUIRE(!depth_is_u16 || depth_div > 0.0, EOD_ERR_BADARG, "eod_backproject_count: depth_div must be positive");
    return backproject_launch(depth, depth_is_u16 != 0, depth_is_u16 ? depth_div : 1.0, pose, shifts, n_episodes, H, W, fx, fy, cx, cy, cell, map_w, map_h,
                              order, 0.5f, idx, nullptr, nullptr, nullptr, nullptr, stream, frame_cnt, active);
}
