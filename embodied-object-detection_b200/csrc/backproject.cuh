// Per-pixel geometry of the back-projection (SURVEY 8a rows A2-A5), shared by the back-projection kernels (backproject.cu) and the
// height-max contest that computes its cells from depth (write_max.cu): one definition keeps both bit-exact with torch-CPU.
// All arithmetic uses explicit _rn intrinsics so nvcc can neither contract nor reassociate.
#pragma once
#include "eod_common.cuh"

namespace {

// build_memory_data.py:136-142 / robot_demo.py:527-530: q.round().long() and THEN the clip.  On the x86 hosts the reference runs on,
// float -> int64 of NaN, +-inf or anything beyond +-2^63 yields INT64_MIN, which clips to cell 0; finite values clip as usual.
// (The outlier mask of core.py:253-256 compares the rounded FLOATS, so it needs no such rule.)
__device__ __forceinline__ bool q_overflows(float q) { return !(fabsf(q) < 9.223372036854775808e18f); }
__device__ __forceinline__ int clip_cell(float q, int n)
{
    return q_overflows(q) ? 0 : (int)fminf(fmaxf(q, 0.0f), (float)(n - 1));
}

// Depth as the sensor delivers it: fp32 metres (habitat: build_data.py:205-207), or uint16 sensor units divided by `depth_div`
// (robot_demo.py:515: depth_image / 1000 - numpy true division in fp64, then torch.FloatTensor rounds to fp32).
template <bool U16>
__device__ __forceinline__ float load_depth(const void *depth, double div, size_t g)
{
    if (U16) return __double2float_rn(__ddiv_rn((double)__ldg(reinterpret_cast<const uint16_t *>(depth) + g), div));
    return __ldg(reinterpret_cast<const float *>(depth) + g);
}

// x_scale / y_scale of a pixel column / row: ((u + 0.5) - cx) / fx, IEEE divide (core.py:107)
__device__ __forceinline__ float pixel_scale(int u, float c, float f) { return __fdiv_rn(__fsub_rn(__fadd_rn((float)u, 0.5f), c), f); }

// one row of the camera-to-world transform: torch.bmm with K=4 on CPU is an FMA chain (core.py:175)
__device__ __forceinline__ float pose_row(float t0, float t1, float t2, float t3, float x, float y, float z)
{
    return __fmaf_rn(t3, 1.0f, __fmaf_rn(t2, z, __fmaf_rn(t1, y, __fmul_rn(t0, x))));
}

// q = rint((world - shift0 - shift1) / cell): round-half-even of an IEEE quotient (core.py:220, build_memory_data.py:135-136)
__device__ __forceinline__ float quantize(float p, float cell) { return rintf(__fdiv_rn(p, cell)); }

// core.py:253-256: outside the map, above the camera height + z_clip, or no depth
__device__ __forceinline__ bool is_outlier(float qx, float qz, float y, float thr, float z, int map_w, int map_h)
{
    return (qx >= (float)map_w) || (qz >= (float)map_h) || (qx < 0.0f) || (qz < 0.0f) || (y > thr) || (z == 0.0f);
}

// clipped flat cell index in the map's order (the back-projection kernels spell the same expression out: as a call it changed their SASS)
__device__ __forceinline__ int flat_cell(float qx, float qz, int map_w, int map_h, int order)
{
    const int ix = clip_cell(qx, map_w), iz = clip_cell(qz, map_h);
    return order == EOD_ORDER_XZ ? ix * map_h + iz : iz * map_w + ix;
}

// One pixel from its depth z and column / row scales, the 12 pose scalars t and the 6 shifts sh held in registers:
// p0 = world point after world_shift_origin, p1 = after map_world_shift as well.
__device__ __forceinline__ void world_point(float z, float xs, float ys, const float (&t)[12], const float (&sh)[6], float (&p0)[3], float (&p1)[3])
{
    const float x = __fmul_rn(z, xs);
    const float y = __fmul_rn(z, ys);
#pragma unroll
    for (int r = 0; r < 3; ++r) p0[r] = __fsub_rn(pose_row(t[4 * r], t[4 * r + 1], t[4 * r + 2], t[4 * r + 3], x, y, z), sh[r]);
#pragma unroll
    for (int r = 0; r < 3; ++r) p1[r] = __fsub_rn(p0[r], sh[3 + r]);
}

}  // namespace
