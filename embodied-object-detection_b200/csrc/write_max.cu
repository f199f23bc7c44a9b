// Memory write, SMNet height-max mode (SURVEY 8a row A7': SMNet.encode, bytecode only).
//
//   height_map, arg = scatter_max(heights[inliers] + 1000, flat_idx[inliers], out=height_map)
//   m = arg >= 0 ; observed |= m ; state[m] = feature[inliers][arg[m]]            ('replace' update)
//
// Deterministic argmax by packing: key = (orderable(height+1000) << 32) | (raster pixel index + 1);
// atomicMax on a u64 scratch word per cell makes the highest pixel index win among equal heights; the
// winner thread then compares against the persistent fp32 height map with >= (an equal later value
// replaces), which is the canonical torch_scatter-1.4 CPU rule fixed in SURVEY 8(c).
//   pass 1  one thread per lattice pixel: atomicMax(key64[cell], key)                   [index plane only]
//   pass 2  one WARP per lattice pixel: if it is its cell's winner and raises the map, update
//           height_map / arg / observed, copy the pixel's C-vector into state[cell] (lanes over
//           channels) and clear the scratch word.
//
// Lock-step height-max regime (eod_heightmax_contest_* / eod_heightmax_update / eod_heightmax_reset): the same contest and rule
// without the per-pixel planes, the arg_pix plane or a scan over the cells.
//   contest  one thread per lattice pixel: the cell, outlier bit and height come from the depth (the back-projection's own device
//            functions, backproject.cuh) or from precomputed planes; the same 64-bit key is max-reduced inside the warp over
//            runs of equal cell id and issued as ONE atomicMax per run.  The atomic that finds the word still 0 is the frame's
//            first touch of the cell (keys are never 0) and appends the cell to the episode's list.
//   update   the listed cells only, 32 per warp: decode the winning height and pixel from the key (a bijection), apply the
//            '>=' rule, clear the key, and copy the winner's feature row (fp32 / bf16 / fp16, CHW / HWC) into state - or emit
//            the (source offset, destination row) list that eod_linear_rows takes.  The last block of an episode resets its list.
#include "backproject.cuh"

namespace {

__device__ __forceinline__ uint32_t orderable(float f)
{
    const uint32_t b = __float_as_uint(f);
    return (b & 0x80000000u) ? ~b : (b | 0x80000000u);
}

__global__ void __launch_bounds__(256) max_pass1_kernel(const float *__restrict__ height, const int32_t *__restrict__ idx,
                                                        const uint8_t *__restrict__ outlier, int H, int W, int stride, int Hs,
                                                        int Ws, int64_t n_cells, unsigned long long *__restrict__ key64)
{
    const int e = blockIdx.y;
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= Hs * Ws) return;
    const int v = (i / Ws) * stride, u = (i % Ws) * stride;
    const int p = v * W + u;
    const size_t g = (size_t)e * H * W + p;
    if (outlier && __ldg(outlier + g)) return;
    const float h = __fadd_rn(__ldg(height + g), 1000.0f);
    if (h != h) return;          // NaN never satisfies `src >= out`: it may neither raise the cell nor shadow the finite candidates
    const unsigned long long key = ((unsigned long long)orderable(h) << 32) | (unsigned)(p + 1);
    atomicMax(key64 + (size_t)e * n_cells + __ldg(idx + g), key);
}

__global__ void __launch_bounds__(256) max_pass2_kernel(const float *__restrict__ height, const int32_t *__restrict__ idx,
                                                        const uint8_t *__restrict__ outlier, const float *__restrict__ feat,
                                                        int layout, int C, int H, int W, int stride, int Hs, int Ws, int64_t n_cells,
                                                        float *__restrict__ height_map, unsigned long long *__restrict__ key64,
                                                        int32_t *__restrict__ arg_pix, uint8_t *__restrict__ observed,
                                                        float *__restrict__ state)
{
    const int e = blockIdx.y;
    const unsigned lane = threadIdx.x & 31;
    const int warp_global = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    // each warp scans 32 lattice pixels with one lane each, then serves the winners among them cooperatively
    const int i = warp_global * 32 + lane;
    const int HW = H * W;
    bool win = false;
    int p = 0, cell = 0;
    float h = 0.f;
    if (i < Hs * Ws) {
        const int v = (i / Ws) * stride, u = (i % Ws) * stride;
        p = v * W + u;
        const size_t g = (size_t)e * HW + p;
        if (!(outlier && __ldg(outlier + g))) {
            cell = __ldg(idx + g);
            const unsigned long long k = key64[(size_t)e * n_cells + cell];
            if ((unsigned)(k & 0xffffffffull) == (unsigned)(p + 1)) {      // this pixel won the in-frame contest
                h = __fadd_rn(__ldg(height + g), 1000.0f);
                key64[(size_t)e * n_cells + cell] = 0ull;                   // only the winner resets
                win = h >= height_map[(size_t)e * n_cells + cell];          // '>=': equal later value replaces
                if (win) {
                    height_map[(size_t)e * n_cells + cell] = h;
                    arg_pix[(size_t)e * n_cells + cell] = p;
                    if (observed) observed[(size_t)e * n_cells + cell] = 1;
                }
            }
        }
    }
    if (!feat || !state) return;
    unsigned todo = __ballot_sync(0xffffffffu, win);
    while (todo) {
        const int src = __ffs(todo) - 1;
        todo &= todo - 1;
        const int wp = __shfl_sync(0xffffffffu, p, src);
        const int wc = __shfl_sync(0xffffffffu, cell, src);
        float *dst = state + ((size_t)e * n_cells + wc) * C;
        if (layout == EOD_LAYOUT_HWC) {
            const float4 *row = reinterpret_cast<const float4 *>(feat + ((size_t)e * HW + wp) * C);
            for (int k = lane; k < C / 4; k += 32) reinterpret_cast<float4 *>(dst)[k] = __ldg(row + k);
        } else {
            const float *col = feat + (size_t)e * C * HW + wp;
            for (int c = lane; c < C; c += 32) dst[c] = __ldg(col + (size_t)c * HW);
        }
    }
}

// inverse of orderable(): the key's high word back to the fp32 height it was built from
__device__ __forceinline__ float from_orderable(uint32_t b) { return __uint_as_float((b & 0x80000000u) ? (b & 0x7fffffffu) : ~b); }

__device__ __forceinline__ unsigned long long height_key(float h, int p) { return ((unsigned long long)orderable(h) << 32) | (unsigned)(p + 1); }

enum { HM_PLANES = 0, HM_DEPTH_F32 = 1, HM_DEPTH_U16 = 2 };

struct ContestParams {
    const float *height;          // HM_PLANES: (E,H,W) world height, (E,H,W) clipped cell id, (E,H,W) u8 outlier (nullable)
    const int32_t *idx;
    const uint8_t *outlier;
    const void *depth;            // HM_DEPTH_*: (E,H,W) depth, pose (E,12), shifts (E,6) and the back-projection's scalars
    double depth_div;
    const float *pose;
    const float *shifts;
    float fx, fy, cx, cy, cell, z_clip;
    int map_w, map_h, order;
    const int32_t *active;
    int H, W, stride, Hs, Ws;
    int64_t n_cells, list_cap;
    unsigned long long *key64;
    int32_t *cell_list;
    int32_t *n_list;
    int32_t *raised;
};

template <int SRC>
__global__ void __launch_bounds__(256) heightmax_contest_kernel(const ContestParams P)
{
    const int e = blockIdx.y;
    if (blockIdx.x == 0 && e == 0 && threadIdx.x == 0) *P.raised = 0;         // the update of this frame counts from 0
    if (P.active && __ldg(P.active + e) <= 0) return;                          // idle slot: reads nothing, appends nothing
    const unsigned lane = threadIdx.x & 31;
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    int cell = -1;                                                             // -1: no candidate (outside, outlier, NaN)
    unsigned long long key = 0ull;
    if (i < P.Hs * P.Ws) {
        const int v = (i / P.Ws) * P.stride, u = (i % P.Ws) * P.stride;
        const int p = v * P.W + u;
        const size_t g = (size_t)e * P.H * P.W + p;
        bool out;
        float h;
        int c;
        if constexpr (SRC == HM_PLANES) {
            out = P.outlier && __ldg(P.outlier + g);
            h = __fadd_rn(__ldg(P.height + g), 1000.0f);
            c = __ldg(P.idx + g);
        } else {
            const float *T = P.pose + 12 * e;
            const float *S = P.shifts + 6 * e;
            float t[12], sh[6];
#pragma unroll
            for (int k = 0; k < 12; ++k) t[k] = __ldg(T + k);
#pragma unroll
            for (int k = 0; k < 6; ++k) sh[k] = __ldg(S + k);
            const float z = load_depth<SRC == HM_DEPTH_U16>(P.depth, P.depth_div, g);
            float p0[3], p1[3];
            world_point(z, pixel_scale(u, P.cx, P.fx), pixel_scale(v, P.cy, P.fy), t, sh, p0, p1);
            const float qx = quantize(p1[0], P.cell), qz = quantize(p1[2], P.cell);
            out = is_outlier(qx, qz, p1[1], __fadd_rn(t[7], P.z_clip), z, P.map_w, P.map_h);
            h = __fadd_rn(p1[1], 1000.0f);
            c = flat_cell(qx, qz, P.map_w, P.map_h, P.order);
        }
        if (!out && h == h) {                                                  // NaN never satisfies `src >= out` (max_pass1_kernel)
            cell = c;
            key = height_key(h, p);
        }
    }
    // segmented max over runs of equal cell id: Hillis-Steele scan that never crosses the head of the lane's run
    const int prev = __shfl_up_sync(0xffffffffu, cell, 1);
    const unsigned heads = __ballot_sync(0xffffffffu, lane == 0 || prev != cell);
    const int start = 31 - __clz(heads & (0xffffffffu >> (31 - lane)));
#pragma unroll
    for (int off = 1; off < 32; off <<= 1) {
        const unsigned long long o = __shfl_up_sync(0xffffffffu, key, off);
        if ((int)lane - off >= start && o > key) key = o;
    }
    const bool tail = lane == 31 || ((heads >> (lane + 1)) & 1u);
    const bool fresh = tail && cell >= 0 && atomicMax(P.key64 + (size_t)e * P.n_cells + cell, key) == 0ull;
    const unsigned fm = __ballot_sync(0xffffffffu, fresh);
    if (!fm) return;
    const int leader = __ffs(fm) - 1;
    int base = 0;
    if ((int)lane == leader) base = atomicAdd(P.n_list + 2 * e, __popc(fm));
    base = __shfl_sync(0xffffffffu, base, leader);
    if (fresh) P.cell_list[(size_t)e * P.list_cap + base + __popc(fm & ((1u << lane) - 1u))] = cell;
}

struct UpdateParams {
    const void *feat;
    int C, HW;
    int64_t n_cells, list_cap;
    const int32_t *cell_list;
    int32_t *n_list;
    unsigned long long *key64;
    float *height_map;
    uint8_t *observed;
    float *state;                 // copy update (nullable when the winner list is requested)
    int64_t *src_off;             // 'replace' update through eod_linear_rows: winner list (nullable)
    int64_t *dst_row;
    int64_t win_cap;
    int32_t *raised;
};

// four consecutive channels (c4 = channel / 4) of a channels-last row, widened exactly
template <int F>
__device__ __forceinline__ float4 row4(const void *row, int c4)
{
    if constexpr (F == FEAT_F32) return __ldg(reinterpret_cast<const float4 *>(row) + c4);
    const uint2 q = __ldg(reinterpret_cast<const uint2 *>(row) + c4);
    const float2 a = widen2<F>(q.x), b = widen2<F>(q.y);
    return make_float4(a.x, a.y, b.x, b.y);
}

template <int F, bool HWC>
__global__ void __launch_bounds__(256) heightmax_update_kernel(const UpdateParams P)
{
    using T = typename FeatElem<F>::T;
    const int e = blockIdx.y;
    const unsigned lane = threadIdx.x & 31;
    const int n = P.n_list[2 * e];
    const int warps = gridDim.x * (blockDim.x >> 5);
    for (int j0 = (blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5)) * 32; j0 < n; j0 += warps * 32) {
        const int j = j0 + lane;
        bool win = false;
        int cell = 0, p = 0;
        if (j < n) {
            cell = P.cell_list[(size_t)e * P.list_cap + j];
            const size_t r = (size_t)e * P.n_cells + cell;
            const unsigned long long k = P.key64[r];
            P.key64[r] = 0ull;
            p = (int)(unsigned)(k & 0xffffffffull) - 1;
            const float h = from_orderable((uint32_t)(k >> 32));
            win = h >= P.height_map[r];                                       // '>=': equal later value replaces (SURVEY 8c)
            if (win) {
                P.height_map[r] = h;
                P.observed[r] = 1;
            }
        }
        const unsigned wm = __ballot_sync(0xffffffffu, win);
        if (!wm) continue;
        int base = 0;
        if (lane == 0) base = atomicAdd(P.raised, __popc(wm));
        if (P.src_off) {
            base = __shfl_sync(0xffffffffu, base, 0);
            const int64_t slot = base + __popc(wm & ((1u << lane) - 1u));
            if (win && slot < P.win_cap) {
                P.src_off[slot] = HWC ? ((int64_t)e * P.HW + p) * P.C : (int64_t)e * P.C * P.HW + p;
                P.dst_row[slot] = (int64_t)e * P.n_cells + cell;
            }
            continue;
        }
        for (unsigned todo = wm; todo; todo &= todo - 1) {
            const int src = __ffs(todo) - 1;
            const int wp = __shfl_sync(0xffffffffu, p, src);
            const int wc = __shfl_sync(0xffffffffu, cell, src);
            float *dst = P.state + ((size_t)e * P.n_cells + wc) * P.C;
            if constexpr (HWC) {
                const T *row = reinterpret_cast<const T *>(P.feat) + ((size_t)e * P.HW + wp) * P.C;
                for (int k = lane; k < P.C / 4; k += 32) reinterpret_cast<float4 *>(dst)[k] = row4<F>(row, k);
            } else {
                const T *col = reinterpret_cast<const T *>(P.feat) + (size_t)e * P.C * P.HW + wp;
                for (int c = lane; c < P.C; c += 32) dst[c] = widen1<F>(__ldg(col + (size_t)c * P.HW));
            }
        }
    }
    // every block of the episode has read n above: the last one to finish leaves the list empty for the next frame
    __syncthreads();
    if (threadIdx.x == 0 && atomicAdd(P.n_list + 2 * e + 1, 1) == (int)gridDim.x - 1) {
        P.n_list[2 * e] = 0;
        P.n_list[2 * e + 1] = 0;
    }
}

// per-slot reset: 32 rows per warp; height and observed bit of every row of a masked episode, state rows of observed cells only
__global__ void __launch_bounds__(256) heightmax_reset_kernel(const int32_t *__restrict__ mask, int64_t n_cells, int64_t n_rows, int C,
                                                              float *__restrict__ height_map, uint8_t *__restrict__ observed, float *__restrict__ state)
{
    const unsigned lane = threadIdx.x & 31;
    const int64_t step = (int64_t)gridDim.x * blockDim.x;
    for (int64_t r0 = ((int64_t)blockIdx.x * blockDim.x + (threadIdx.x & ~31u)); r0 < n_rows; r0 += step) {
        const int64_t r = r0 + lane;
        bool clear_row = false;
        if (r < n_rows && __ldg(mask + r / n_cells) != 0) {
            clear_row = observed[r] != 0;
            height_map[r] = 0.0f;
            observed[r] = 0;
        }
        for (unsigned todo = __ballot_sync(0xffffffffu, clear_row); todo; todo &= todo - 1) {
            float4 *dst = reinterpret_cast<float4 *>(state + (r0 + __ffs(todo) - 1) * C);
            for (int k = lane; k < C / 4; k += 32) dst[k] = make_float4(0.f, 0.f, 0.f, 0.f);
        }
    }
}

int contest_launch(int src, ContestParams P, int n_episodes, const char *what, cudaStream_t st)
{
    EOD_REQUIRE(P.key64 && P.cell_list && P.n_list && P.raised, EOD_ERR_BADARG, "%s: null scratch pointer", what);
    EOD_REQUIRE(n_episodes > 0 && n_episodes <= 65535 && P.H > 0 && P.W > 0 && P.n_cells > 0 && P.stride > 0, EOD_ERR_BADARG, "%s: bad sizes", what);
    P.Hs = (P.H + P.stride - 1) / P.stride;
    P.Ws = (P.W + P.stride - 1) / P.stride;
    const int64_t lattice = (int64_t)P.Hs * P.Ws;
    EOD_REQUIRE(P.list_cap >= (lattice < P.n_cells ? lattice : P.n_cells), EOD_ERR_BADARG,
                "%s: list_cap must hold min(n_cells, lattice pixels) = %lld cells", what, (long long)(lattice < P.n_cells ? lattice : P.n_cells));
    dim3 grid((unsigned)((lattice + 255) / 256), n_episodes);
    if (src == HM_PLANES) heightmax_contest_kernel<HM_PLANES><<<grid, 256, 0, st>>>(P);
    else if (src == HM_DEPTH_U16) heightmax_contest_kernel<HM_DEPTH_U16><<<grid, 256, 0, st>>>(P);
    else heightmax_contest_kernel<HM_DEPTH_F32><<<grid, 256, 0, st>>>(P);
    return eod_check_launch(what);
}

}  // namespace

extern "C" int eod_write_max(const float *height, const int32_t *idx, const uint8_t *outlier, const float *feat, int layout,
                             int n_episodes, int C, int H, int W, int pix_stride, int64_t n_cells, float *height_map,
                             uint64_t *key64, int32_t *arg_pix, uint8_t *observed, float *state, eod_stream_t stream)
{
    EOD_REQUIRE(height && idx && height_map && key64 && arg_pix, EOD_ERR_BADARG, "eod_write_max: null pointer");
    EOD_REQUIRE(n_episodes > 0 && n_episodes <= 65535 && H > 0 && W > 0 && n_cells > 0 && pix_stride > 0, EOD_ERR_BADARG, "eod_write_max: bad sizes");
    EOD_REQUIRE(layout == EOD_LAYOUT_CHW || layout == EOD_LAYOUT_HWC, EOD_ERR_BADARG, "eod_write_max: bad layout");
    EOD_REQUIRE(!feat || (C > 0 && C % 4 == 0 && eod_aligned16(feat) && eod_aligned16(state)), EOD_ERR_ALIGN, "eod_write_max: C %% 4 and 16-byte alignment required");
    cudaStream_t st = (cudaStream_t)stream;
    const int Hs = (H + pix_stride - 1) / pix_stride, Ws = (W + pix_stride - 1) / pix_stride;
    const int n = Hs * Ws;
    cudaError_t err = cudaMemsetAsync(arg_pix, 0xff, (size_t)n_episodes * n_cells * sizeof(int32_t), st);   // arg := -1
    EOD_REQUIRE(err == cudaSuccess, EOD_ERR_LAUNCH, "eod_write_max: memset failed: %s", cudaGetErrorString(err));
    dim3 grid((n + 255) / 256, n_episodes);
    max_pass1_kernel<<<grid, 256, 0, st>>>(height, idx, outlier, H, W, pix_stride, Hs, Ws, n_cells, (unsigned long long *)key64);
    int rc = eod_check_launch("eod_write_max[pass1]");
    if (rc) return rc;
    max_pass2_kernel<<<grid, 256, 0, st>>>(height, idx, outlier, feat, layout, C, H, W, pix_stride, Hs, Ws, n_cells, height_map,
                                           (unsigned long long *)key64, arg_pix, observed, state);
    return eod_check_launch("eod_write_max[pass2]");
}

extern "C" int eod_heightmax_contest_depth(const void *depth, int depth_is_u16, double depth_div, const float *pose, const float *shifts,
                                           int n_episodes, int H, int W, float fx, float fy, float cx, float cy, float cell, int map_w,
                                           int map_h, int order, float z_clip, int pix_stride, const int32_t *active, uint64_t *key64,
                                           int32_t *cell_list, int64_t list_cap, int32_t *n_list, int32_t *raised, eod_stream_t stream)
{
    EOD_REQUIRE(depth && pose && shifts, EOD_ERR_BADARG, "eod_heightmax_contest_depth: null input");
    EOD_REQUIRE(!depth_is_u16 || depth_div > 0.0, EOD_ERR_BADARG, "eod_heightmax_contest_depth: depth_div must be positive");
    EOD_REQUIRE(map_w > 0 && map_h > 0 && (int64_t)map_w * map_h < (int64_t)INT32_MAX, EOD_ERR_BADARG, "eod_heightmax_contest_depth: bad map size");
    EOD_REQUIRE(order == EOD_ORDER_ZX || order == EOD_ORDER_XZ, EOD_ERR_BADARG, "eod_heightmax_contest_depth: bad order");
    EOD_REQUIRE(cell > 0.0f && fx != 0.0f && fy != 0.0f, EOD_ERR_BADARG, "eod_heightmax_contest_depth: bad cell/intrinsics");
    ContestParams P{nullptr, nullptr, nullptr, depth, depth_is_u16 ? depth_div : 1.0, pose, shifts, fx, fy, cx, cy, cell, z_clip, map_w, map_h,
                    order, active, H, W, pix_stride, 0, 0, (int64_t)map_w * map_h, list_cap, (unsigned long long *)key64, cell_list, n_list, raised};
    return contest_launch(depth_is_u16 ? HM_DEPTH_U16 : HM_DEPTH_F32, P, n_episodes, "eod_heightmax_contest_depth", (cudaStream_t)stream);
}

extern "C" int eod_heightmax_contest_planes(const float *height, const int32_t *idx, const uint8_t *outlier, int n_episodes, int H, int W,
                                            int pix_stride, int64_t n_cells, const int32_t *active, uint64_t *key64, int32_t *cell_list,
                                            int64_t list_cap, int32_t *n_list, int32_t *raised, eod_stream_t stream)
{
    EOD_REQUIRE(height && idx, EOD_ERR_BADARG, "eod_heightmax_contest_planes: null input");
    ContestParams P{height, idx, outlier, nullptr, 1.0, nullptr, nullptr, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0, 0, 0, active, H, W, pix_stride, 0, 0,
                    n_cells, list_cap, (unsigned long long *)key64, cell_list, n_list, raised};
    return contest_launch(HM_PLANES, P, n_episodes, "eod_heightmax_contest_planes", (cudaStream_t)stream);
}

extern "C" int eod_heightmax_update(const void *feat, int layout, int n_episodes, int C, int H, int W, int64_t n_cells, const int32_t *cell_list,
                                    int64_t list_cap, int32_t *n_list, uint64_t *key64, float *height_map, uint8_t *observed, float *state,
                                    int64_t *src_off, int64_t *dst_row, int64_t win_cap, int32_t *raised, eod_stream_t stream)
{
    EOD_REQUIRE(feat || src_off, EOD_ERR_BADARG, "eod_heightmax_update: null feat");
    EOD_REQUIRE(cell_list && n_list && key64 && height_map && observed && raised, EOD_ERR_BADARG, "eod_heightmax_update: null pointer");
    EOD_REQUIRE(src_off ? (dst_row && win_cap > 0) : state != nullptr, EOD_ERR_BADARG, "eod_heightmax_update: state, or src_off + dst_row + win_cap");
    EOD_REQUIRE(n_episodes > 0 && n_episodes <= 65535 && H > 0 && W > 0 && n_cells > 0 && list_cap > 0, EOD_ERR_BADARG, "eod_heightmax_update: bad sizes");
    EOD_REQUIRE(layout >= EOD_LAYOUT_CHW && layout <= EOD_LAYOUT_CHW_F16, EOD_ERR_BADARG, "eod_heightmax_update: bad layout");
    EOD_REQUIRE(!src_off || layout == EOD_LAYOUT_CHW || layout == EOD_LAYOUT_HWC, EOD_ERR_UNSUPPORTED,
                "eod_heightmax_update: the winner list indexes fp32 features (eod_linear_rows reads fp32)");
    EOD_REQUIRE(C > 0 && C % 4 == 0 && (src_off || (eod_aligned16(feat) && eod_aligned16(state))), EOD_ERR_ALIGN,
                "eod_heightmax_update: C %% 4 and 16-byte alignment required");
    UpdateParams P{feat, C, H * W, n_cells, list_cap, cell_list, n_list, (unsigned long long *)key64, height_map, observed, state,
                   src_off, dst_row, win_cap, raised};
    // enough warps for a frame's new cells without a grid sized for the worst case (blocks loop over the list)
    int64_t bx = (list_cap + 255) / 256;
    const int64_t cap = ((int64_t)eod_num_sms() * 8 + n_episodes - 1) / n_episodes;
    if (bx > cap) bx = cap;
    dim3 grid((unsigned)bx, n_episodes);
    cudaStream_t st = (cudaStream_t)stream;
    switch (layout) {
    case EOD_LAYOUT_CHW: heightmax_update_kernel<FEAT_F32, false><<<grid, 256, 0, st>>>(P); break;
    case EOD_LAYOUT_HWC: heightmax_update_kernel<FEAT_F32, true><<<grid, 256, 0, st>>>(P); break;
    case EOD_LAYOUT_HWC_BF16: heightmax_update_kernel<FEAT_BF16, true><<<grid, 256, 0, st>>>(P); break;
    case EOD_LAYOUT_HWC_F16: heightmax_update_kernel<FEAT_F16, true><<<grid, 256, 0, st>>>(P); break;
    case EOD_LAYOUT_CHW_BF16: heightmax_update_kernel<FEAT_BF16, false><<<grid, 256, 0, st>>>(P); break;
    default: heightmax_update_kernel<FEAT_F16, false><<<grid, 256, 0, st>>>(P); break;
    }
    return eod_check_launch("eod_heightmax_update");
}

extern "C" int eod_heightmax_reset(const int32_t *mask, int n_episodes, int64_t n_cells, int C, float *height_map, uint8_t *observed, float *state,
                                   eod_stream_t stream)
{
    EOD_REQUIRE(mask && height_map && observed && state, EOD_ERR_BADARG, "eod_heightmax_reset: null pointer");
    EOD_REQUIRE(n_episodes > 0 && n_cells > 0 && C > 0 && C % 4 == 0, EOD_ERR_BADARG, "eod_heightmax_reset: bad sizes (C %% 4 == 0)");
    EOD_REQUIRE(eod_aligned16(state), EOD_ERR_ALIGN, "eod_heightmax_reset: state rows must be 16-byte aligned");
    const int64_t n_rows = (int64_t)n_episodes * n_cells;
    int64_t blocks = (n_rows + 255) / 256;
    const int64_t cap = (int64_t)eod_num_sms() * 16;
    if (blocks > cap) blocks = cap;
    heightmax_reset_kernel<<<(unsigned)blocks, 256, 0, (cudaStream_t)stream>>>(mask, n_cells, n_rows, C, height_map, observed, state);
    return eod_check_launch("eod_heightmax_reset");
}
