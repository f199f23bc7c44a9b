// Memory write, object-feature regime, fused (SURVEY 8a rows A6 + A7; 8f rank 1).
//
// The reference builds a (1, C, 480, 640) fp32 image of per-pixel object-feature means (629 MB at C=512,
// custom_rcnn.py:884-901, one host sync per object), compacts the observed pixels, keeps every 8th and reduces
// them per map cell with a dense one-hot matmul (:903-936).  Only the SAMPLED pixels ever reach the grid, so the
// image is never needed:
//
//   eod_masks_observed   observed[p] = any_k masks[k][p]                                  (K*HW bytes read once)
//   eod_sample_mask      every stride-th observed pixel in raster order (write_mean.cu)
//   eod_frame_count      per-cell sample counts + visibility bits; the first sample of a cell claims a compact
//                        SLOT for it (write_mean.cu)
//   eod_write_objects    for each sampled pixel: g = (sum over the covering objects, in index order, of f_k) / n_obj
//                        - the value box_to_image_features would have stored, bit for bit - then
//                        scratch[slot(cell)] += g   (fp32 reductions into a zeroed per-frame row)
//   eod_flush_slots      sums[cell] += scratch[slot] / n_cell ; scratch row, slot map and slot counter := 0
//   eod_finalize_counts  counts += 1 for every visible cell                (write_mean.cu)
//
// Deterministic variant (eod_write_objects[_pasted]_det): eod_frame_count without slots, then the run pre-passes of the dense
// deterministic write (det.cuh), write_objects_det_kernel storing one partial per run of equal cell id, and the dense write's
// segmented reduce - the bits of eod_write_mean_det on the box_to_image_features image, reproducible run to run.
//
// The per-frame scratch keeps the arithmetic of the reference: the frame's samples of a cell are summed on their own,
// divided by their count, and only that mean meets the (much larger) running sum - one rounding at grid magnitude per
// frame instead of one per sample.
//
// Work is ~P'(=observed/8) * K * C adds per frame (a few 10^8): the kernel is latency-, not bandwidth-bound;
// what matters is that the 629 MB image and the K host round trips are gone.
//
// Mask pasting (8f rank 1, second half).  The reference turns the mask head's (K,28,28) probabilities into (K,480,640)
// bools with detectron2's paste_masks_in_image (custom_rcnn.py:880): per object, pixel centres of the box's integer
// neighbourhood are mapped into the 28x28 map, bilinearly sampled with F.grid_sample(align_corners=False, zero
// padding) and thresholded at 0.5.  Here that test is a pure function of (object, pixel) - paste_covers() - with the
// exact fp32 operation sequence of ATen's vectorised CPU sampler (canonical: torch CPU, AVX2/AVX-512 build:
// ix = fma(gx + 1, S/2, -0.5); out = fma(se_v, se, fma(sw_v, sw, fma(ne_v, ne, nw_v * nw)))), so the (K,480,640)
// masks need never exist: eod_paste_masks folds them straight into `observed`, and the pasted variant of the write
// re-evaluates the test for the ~1/8 sampled pixels only.
#include "det.cuh"
#include "eod_common.cuh"

namespace {

// One kept detection prepared for pasting (detectron2 _do_paste_mask with skip_empty=True, one chunk per mask).
struct PasteObj {
    float x0, y0, dx, dy;      // box corner and extents x1 - x0, y1 - y0 (fp32 subtraction as torch does it)
    int rx0, ry0, rx1, ry1;    // integer region [rx0, rx1) x [ry0, ry1) outside of which the pasted mask is False
};

// thr >= 0.5: the integer neighbourhood of the box (detectron2's skip_empty=True CPU path) - for probabilities <= 1 the bilinear value
// outside it is below 0.5, so this is also what the skip_empty=False path the reference takes on CUDA tensors (custom_rcnn.py:880)
// produces.  thr < 0.5: the two paths differ up to extent/(2S) pixels outside the box, so the WHOLE image is sampled, as the
// reference's CUDA path does.
__device__ __forceinline__ PasteObj paste_prepare(const float *__restrict__ box, int H, int W, float thr)
{
    PasteObj o;
    const float x0 = __ldg(box), y0 = __ldg(box + 1), x1 = __ldg(box + 2), y1 = __ldg(box + 3);
    o.x0 = x0; o.y0 = y0;
    o.dx = __fsub_rn(x1, x0); o.dy = __fsub_rn(y1, y0);
    // clamp(floor(x0) - 1, min=0), clamp(ceil(x1) + 1, max=W); the extra clamps only keep the float->int conversion defined
    o.rx0 = (int)fminf(fmaxf(__fsub_rn(floorf(x0), 1.f), 0.f), (float)W);
    o.ry0 = (int)fminf(fmaxf(__fsub_rn(floorf(y0), 1.f), 0.f), (float)H);
    o.rx1 = (int)fmaxf(fminf(__fadd_rn(ceilf(x1), 1.f), (float)W), 0.f);
    o.ry1 = (int)fmaxf(fminf(__fadd_rn(ceilf(y1), 1.f), (float)H), 0.f);
    if (!(thr >= 0.5f)) { o.rx0 = 0; o.ry0 = 0; o.rx1 = W; o.ry1 = H; }
    return o;
}

// source coordinate of pixel centre c + 0.5 along one axis: ((c + 0.5 - b0) / extent * 2 - 1) un-normalised for an S-wide map
__device__ __forceinline__ float paste_coord(int c, float b0, float extent, float half_S)
{
    const float g = __fsub_rn(__fmul_rn(__fdiv_rn(__fsub_rn(__fadd_rn((float)c, 0.5f), b0), extent), 2.f), 1.f);
    return __fmaf_rn(__fadd_rn(g, 1.f), half_S, -0.5f);
}

// one axis of the bilinear tap: source coordinate i -> near tap floor(i) with weight 1 - frac, far tap floor(i) + 1 with weight frac
struct PasteAxis {
    float w_near, w_far;
    int i_near, i_far;
    bool in_near, in_far;
};
__device__ __forceinline__ PasteAxis paste_axis(int c, float b0, float extent, int S)
{
    const float fS = (float)S;
    const float i = paste_coord(c, b0, extent, fS * 0.5f);
    const float f = floorf(i), f1 = __fadd_rn(f, 1.f);
    PasteAxis a;
    a.w_far = __fsub_rn(i, f);
    a.w_near = __fsub_rn(1.f, a.w_far);
    a.in_near = f > -1.f && f < fS;                     // comparisons in the float domain: false for inf / NaN coordinates
    a.in_far = f1 > -1.f && f1 < fS;
    a.i_near = a.in_near ? (int)f : 0;
    a.i_far = a.in_far ? (int)f1 : 0;
    return a;
}
// sampled value >= thr, in the operation order of ATen's vectorised CPU grid_sample; padding taps contribute 0 * weight
// (NaN for non-finite coordinates, which then compares false)
__device__ __forceinline__ bool paste_eval(const float *__restrict__ m, int S, const PasteAxis &x, const PasteAxis &y, float thr)
{
    const float v_nw = (x.in_near && y.in_near) ? __ldg(m + y.i_near * S + x.i_near) : 0.f;
    const float v_ne = (x.in_far && y.in_near) ? __ldg(m + y.i_near * S + x.i_far) : 0.f;
    const float v_sw = (x.in_near && y.in_far) ? __ldg(m + y.i_far * S + x.i_near) : 0.f;
    const float v_se = (x.in_far && y.in_far) ? __ldg(m + y.i_far * S + x.i_far) : 0.f;
    float acc = __fmul_rn(v_nw, __fmul_rn(y.w_near, x.w_near));
    acc = __fmaf_rn(v_ne, __fmul_rn(y.w_near, x.w_far), acc);
    acc = __fmaf_rn(v_sw, __fmul_rn(y.w_far, x.w_near), acc);
    acc = __fmaf_rn(v_se, __fmul_rn(y.w_far, x.w_far), acc);
    return acc >= thr;
}
// pasted-mask value test for one (object, pixel); m = the object's (S,S) probabilities
__device__ __forceinline__ bool paste_covers(const float *__restrict__ m, const PasteObj &o, int S, int px, int py, float thr)
{
    if (px < o.rx0 || px >= o.rx1 || py < o.ry0 || py >= o.ry1) return false;
    return paste_eval(m, S, paste_axis(px, o.x0, o.dx, S), paste_axis(py, o.y0, o.dy, S), thr);
}

constexpr int kPasteChunk = 128;      // objects staged in shared memory at a time

// thread per 4 consecutive pixels; masks (E,Kmax,HW) u8 and / or observed (E,HW) u8
__global__ void __launch_bounds__(256) paste_masks_kernel(const float *__restrict__ probs, const float *__restrict__ boxes,
                                                          const int32_t *__restrict__ n_obj, int Kmax, int S, int H, int W, float thr,
                                                          uint8_t *__restrict__ masks, uint8_t *__restrict__ observed)
{
    __shared__ PasteObj s_obj[kPasteChunk];
    __shared__ uint32_t s_hit[kPasteChunk / 32];           // observed-only: objects whose row range meets this CTA's pixel rows
    const int e = blockIdx.y, HW = H * W;
    const int p0 = (blockIdx.x * 256 + threadIdx.x) * 4;
    const int K = n_obj ? max(0, min(__ldg(n_obj + e), Kmax)) : Kmax;
    int px[4], py[4];
    {
        const int v = p0 / W, u0 = p0 - v * W;                 // one integer division per thread; the quad rarely wraps a row
        if (u0 + 3 < W) {
#pragma unroll
            for (int b = 0; b < 4; ++b) { px[b] = u0 + b; py[b] = v; }
        } else {
#pragma unroll
            for (int b = 0; b < 4; ++b) { px[b] = (p0 + b) % W; py[b] = (p0 + b) / W; }
        }
    }
    uint32_t any = 0;
    for (int k0 = 0; k0 < Kmax; k0 += kPasteChunk) {
        const int kn = min(kPasteChunk, Kmax - k0);
        __syncthreads();
        if ((int)threadIdx.x < kPasteChunk) {
            bool hit = false;
            if ((int)threadIdx.x < kn && k0 + (int)threadIdx.x < K) {
                const PasteObj o = paste_prepare(boxes + ((size_t)e * Kmax + k0 + threadIdx.x) * 4, H, W, thr);
                s_obj[threadIdx.x] = o;
                const int row_lo = (int)(blockIdx.x * 1024) / W, row_hi = min(HW - 1, (int)(blockIdx.x * 1024) + 1023) / W;
                hit = !(row_hi < o.ry0 || row_lo >= o.ry1);
            }
            const unsigned hits = __ballot_sync(0xffffffffu, hit);
            if ((threadIdx.x & 31) == 0) s_hit[threadIdx.x >> 5] = hits;
        }
        __syncthreads();
        if (p0 >= HW) continue;
        if (!masks) {
            // observed only (the fused object write never builds the masks): walk just the objects that reach this CTA's rows, and stop
            // as soon as all four pixels are covered - overlapping detections are the rule
            for (int w = 0; w < kPasteChunk / 32 && any != 0x01010101u; ++w) {
                unsigned todo = s_hit[w];
                while (todo && any != 0x01010101u) {
                    const int j = w * 32 + __ffs(todo) - 1;
                    todo &= todo - 1;
                    const PasteObj o = s_obj[j];
                    if (py[3] < o.ry0 || py[0] >= o.ry1 || (py[0] == py[3] && (px[3] < o.rx0 || px[0] >= o.rx1))) continue;
                    const float *m = probs + ((size_t)e * Kmax + k0 + j) * S * S;
                    if (py[0] == py[3]) {
                        const PasteAxis ay = paste_axis(py[0], o.y0, o.dy, S);
#pragma unroll
                        for (int b = 0; b < 4; ++b)
                            if (!((any >> (8 * b)) & 1u) && p0 + b < HW && px[b] >= o.rx0 && px[b] < o.rx1 &&
                                paste_eval(m, S, paste_axis(px[b], o.x0, o.dx, S), ay, thr))
                                any |= 1u << (8 * b);
                    } else {
#pragma unroll
                        for (int b = 0; b < 4; ++b)
                            if (!((any >> (8 * b)) & 1u) && p0 + b < HW && paste_covers(m, o, S, px[b], py[b], thr)) any |= 1u << (8 * b);
                    }
                }
            }
            continue;
        }
        for (int j = 0; j < kn; ++j) {
            const int k = k0 + j;
            uint32_t bits = 0;
            if (k < K) {
                const PasteObj o = s_obj[j];
                // whole quad outside the object's rows / columns: skip (the common case)
                if (!(py[3] < o.ry0 || py[0] >= o.ry1 || (py[0] == py[3] && (px[3] < o.rx0 || px[0] >= o.rx1)))) {
                    const float *m = probs + ((size_t)e * Kmax + k) * S * S;
                    if (py[0] == py[3]) {                      // the usual case (W % 4 == 0): one row, the y axis is shared
                        const PasteAxis ay = paste_axis(py[0], o.y0, o.dy, S);
#pragma unroll
                        for (int b = 0; b < 4; ++b)
                            if (p0 + b < HW && px[b] >= o.rx0 && px[b] < o.rx1 && paste_eval(m, S, paste_axis(px[b], o.x0, o.dx, S), ay, thr))
                                bits |= 1u << (8 * b);
                    } else {
#pragma unroll
                        for (int b = 0; b < 4; ++b)
                            if (p0 + b < HW && paste_covers(m, o, S, px[b], py[b], thr)) bits |= 1u << (8 * b);
                    }
                }
            }
            any |= bits;
            if (masks) {                                   // objects beyond n_obj[e] get all-False planes
                uint8_t *dst = masks + ((size_t)e * Kmax + k) * HW + p0;
                if (p0 + 3 < HW && (reinterpret_cast<uintptr_t>(dst) & 3u) == 0) *reinterpret_cast<uint32_t *>(dst) = bits;
                else
                    for (int b = 0; b < 4 && p0 + b < HW; ++b) dst[b] = (bits >> (8 * b)) & 1u;
            }
        }
    }
    if (observed && p0 < HW) {
        uint8_t *dst = observed + (size_t)e * HW + p0;
        if (p0 + 3 < HW && (reinterpret_cast<uintptr_t>(dst) & 3u) == 0) *reinterpret_cast<uint32_t *>(dst) = any;
        else
            for (int b = 0; b < 4 && p0 + b < HW; ++b) dst[b] = (any >> (8 * b)) & 1u;
    }
}

// one thread per 4 pixels (uchar4 mask loads): observed = OR over the episode's objects
__global__ void __launch_bounds__(256) masks_observed_kernel(const uint8_t *__restrict__ masks, const int32_t *__restrict__ n_obj, int Kmax,
                                                             int HW, uint8_t *__restrict__ observed)
{
    const int e = blockIdx.y;
    const int p4 = blockIdx.x * blockDim.x + threadIdx.x;
    if (p4 * 4 >= HW) return;
    const int K = n_obj ? min(__ldg(n_obj + e), Kmax) : Kmax;
    const uint8_t *m = masks + (size_t)e * Kmax * HW;
    uint32_t acc = 0;
    for (int k = 0; k < K; ++k) acc |= __ldg(reinterpret_cast<const uint32_t *>(m + (size_t)k * HW) + p4);
    uint32_t out = 0;
#pragma unroll
    for (int b = 0; b < 4; ++b) out |= ((acc >> (8 * b)) & 0xffu) ? (1u << (8 * b)) : 0u;
    reinterpret_cast<uint32_t *>(observed + (size_t)e * HW)[p4] = out;
}

// CTA = 2048 consecutive pixels of one episode (the sampled ones are ~2 % of them: compacted first, then processed in
// rounds of up to 256).  Two phases per round, so that the dependent global loads of all sampled pixels of
// the CTA are in flight together instead of one pixel after the other (the kernel is latency-, not bandwidth-bound):
//   A  thread per (sampled pixel, object): cover test -> one 32-object bitmask word per warp ballot, kept in shared memory;
//      thread per sampled pixel: cell index and slot;
//   B  warp per sampled pixel, lanes own channels c = lane + 32*j: the covering objects' features are added in ascending
//      object index (custom_rcnn.py:890-895), divided by their number, and reduced into the cell's scratch slot.
// kPasted: the cover test is paste_covers() on the (Kmax,S,S) probabilities + boxes instead of a byte of the (Kmax,HW) masks.
// Frames with more than kCoverObjs kept objects (the reference caps at 100, custom_rcnn.py:860) take the
// one-pixel-at-a-time path at the end of the kernel.
constexpr int kCoverObjs = 128;

constexpr int kObjSpan = 2048;            // pixels per CTA (8 per thread); ~1/50 of them are sampled in the reference's regime

template <int C, bool kPasted>
__global__ void __launch_bounds__(256) write_objects_kernel(const float *__restrict__ box_features, const uint8_t *__restrict__ masks,
                                                            const float *__restrict__ probs, const float *__restrict__ boxes, int Sm, int W,
                                                            float thr, const int32_t *__restrict__ n_obj, int Kmax, const int32_t *__restrict__ idx,
                                                            const uint8_t *__restrict__ samp, const int32_t *__restrict__ slot_of_cell, int HW,
                                                            int64_t n_cells, int S, float *__restrict__ scratch)
{
    constexpr int J = C / 32;
    __shared__ int s_list[kObjSpan];
    __shared__ int s_slot[256];
    __shared__ __align__(16) uint32_t s_cover[256][kCoverObjs / 32];
    __shared__ PasteObj s_obj[kPasted ? kCoverObjs : 1];
    __shared__ int s_wcnt[8];
    const int e = blockIdx.y;
    const unsigned lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    int n;
    {   // raster-ordered list of the CTA's sampled pixels (neighbours in the list are neighbours in the image row)
        const int p0 = blockIdx.x * kObjSpan + threadIdx.x * 8;
        const uint8_t *sp = samp + (size_t)e * HW + p0;
        uint32_t lo = 0, hi = 0;
        if (p0 + 7 < HW && (reinterpret_cast<uintptr_t>(sp) & 7u) == 0) {
            const uint2 q = __ldg(reinterpret_cast<const uint2 *>(sp));
            lo = q.x; hi = q.y;
        } else {
            for (int b = 0; b < 8 && p0 + b < HW; ++b) {
                const uint32_t v = __ldg(sp + b);
                if (b < 4) lo |= v << (8 * b); else hi |= v << (8 * (b - 4));
            }
        }
        unsigned bits = 0;                                            // bit b: pixel p0 + b is sampled
#pragma unroll
        for (int b = 0; b < 4; ++b) bits |= (((lo >> (8 * b)) & 0xffu) ? 1u : 0u) << b | (((hi >> (8 * b)) & 0xffu) ? 1u : 0u) << (b + 4);
        const int cnt = __popc(bits);
        int incl = cnt;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const int up = __shfl_up_sync(0xffffffffu, incl, o);
            if ((int)lane >= o) incl += up;
        }
        if (lane == 31) s_wcnt[warp] = incl;
        __syncthreads();
        int pre = 0, tot = 0;
#pragma unroll
        for (int w = 0; w < 8; ++w) { pre += w < (int)warp ? s_wcnt[w] : 0; tot += s_wcnt[w]; }
        int pos = pre + incl - cnt;
        while (bits) {
            s_list[pos++] = p0 + __ffs(bits) - 1;
            bits &= bits - 1;
        }
        n = tot;
        __syncthreads();
    }
    if (n == 0) return;
    const int K = n_obj ? min(__ldg(n_obj + e), Kmax) : Kmax;
    const uint8_t *m = kPasted ? nullptr : masks + (size_t)e * Kmax * HW;
    const float *f = box_features + (size_t)e * Kmax * C;

    if (K <= kCoverObjs) {
        if (kPasted) {
            if ((int)threadIdx.x < K) s_obj[threadIdx.x] = paste_prepare(boxes + ((size_t)e * Kmax + threadIdx.x) * 4, HW / W, W, thr);
            __syncthreads();
        }
        const int Kpad = (K + 31) & ~31;
        constexpr int J4 = C / 128;
        const int n_words = Kpad >> 5;
        for (int base = 0; base < n; base += 256) {                      // rounds of up to 256 sampled pixels
            const int nn = min(256, n - base);
            // ---- phase A: thread per sampled pixel ----
            // Cell and slot of the pixel, then the objects one after the other: an integer box-region test from shared memory and,
            // for the one or two objects that pass it, the sampler.  (The first version spent a warp trip per (pixel, 32 objects)
            // - 53 trips per CTA with one or two useful lanes each, an integer division per lane and trip; this is ~3 trips.)
            if ((int)threadIdx.x < nn) {
                const int px = s_list[base + threadIdx.x];
                const int cell = __ldg(idx + (size_t)e * HW + px);
                const int my_slot = __ldg(slot_of_cell + (size_t)e * n_cells + cell) - 1;
                const int x = px % W, y = px / W;
                static_assert(kCoverObjs == 128, "four cover words");
                unsigned w0 = 0u, w1 = 0u, w2 = 0u, w3 = 0u;
                for (int k = 0; k < K; ++k) {
                    bool mine;
                    if (kPasted) {
                        const PasteObj &o = s_obj[k];
                        mine = x >= o.rx0 && x < o.rx1 && y >= o.ry0 && y < o.ry1 &&
                               paste_eval(probs + ((size_t)e * Kmax + k) * Sm * Sm, Sm, paste_axis(x, o.x0, o.dx, Sm), paste_axis(y, o.y0, o.dy, Sm), thr);
                    } else {
                        mine = __ldg(m + (size_t)k * HW + px) != 0;
                    }
                    if (mine) {
                        const unsigned bit = 1u << (k & 31);
                        const int wd = k >> 5;
                        w0 |= wd == 0 ? bit : 0u; w1 |= wd == 1 ? bit : 0u; w2 |= wd == 2 ? bit : 0u; w3 |= wd == 3 ? bit : 0u;
                    }
                }
                s_cover[threadIdx.x][0] = w0; s_cover[threadIdx.x][1] = w1; s_cover[threadIdx.x][2] = w2; s_cover[threadIdx.x][3] = w3;
                s_slot[threadIdx.x] = my_slot;
            }
            __syncthreads();
            const int chunk = (nn + 7) >> 3;                              // warp w owns pixels [w*chunk, i_end)
            const int i_beg = (int)warp * chunk, i_end = min(nn, ((int)warp + 1) * chunk);
            // ---- phase B ----
            // Lanes own float4 channel groups 4*lane + 128*j.  Consecutive samples that fall into the same cell are summed in
            // registers and leave as ONE 128-bit reduction per lane and group (the scratch row is an unordered fp32 sum either way).
            float4 agg[J4];
            int agg_slot = -1;
            auto flush = [&]() {
                if (agg_slot >= 0) {
                    float *dst = scratch + ((size_t)e * S + agg_slot) * C + 4 * lane;
#pragma unroll
                    for (int j = 0; j < J4; ++j) red_add_v4(dst + 128 * j, agg[j].x, agg[j].y, agg[j].z, agg[j].w);
                }
            };
            // The pixel's value depends only on WHICH objects cover it: consecutive samples (8 observed pixels apart in raster order)
            // mostly sit inside the same objects, so the value is recomputed only when the cover set changes (bit-identical either way).
            float4 acc[J4];
            uint4 have = make_uint4(0u, 0u, 0u, 0u);                       // cover set `acc` was computed for (all-zero: none yet)
            int cnt = 0;
            for (int i = i_beg; i < i_end; ++i) {
                const uint4 cw = *reinterpret_cast<const uint4 *>(&s_cover[i][0]);
                if (cw.x != have.x || cw.y != have.y || cw.z != have.z || cw.w != have.w) {
                    have = cw;
#pragma unroll
                    for (int j = 0; j < J4; ++j) acc[j] = make_float4(0.f, 0.f, 0.f, 0.f);
                    cnt = 0;
                    const unsigned words[4] = {cw.x, cw.y, cw.z, cw.w};
#pragma unroll
                    for (int wd = 0; wd < 4; ++wd) {
                        unsigned todo = words[wd];
                        cnt += __popc(todo);
                        while (todo) {                                     // ascending object index
                            const int kk = wd * 32 + __ffs(todo) - 1;
                            todo &= todo - 1;
                            const float4 *row = reinterpret_cast<const float4 *>(f + (size_t)kk * C) + lane;
#pragma unroll
                            for (int j = 0; j < J4; ++j) {
                                const float4 x = __ldg(row + 32 * j);
                                acc[j].x = __fadd_rn(acc[j].x, x.x); acc[j].y = __fadd_rn(acc[j].y, x.y);
                                acc[j].z = __fadd_rn(acc[j].z, x.z); acc[j].w = __fadd_rn(acc[j].w, x.w);
                            }
                        }
                    }
                    // / number of covering objects (custom_rcnn.py:899).  Almost always 1 or 2: a power of two divides exactly like the
                    // multiplication by its (exact) reciprocal, so the 4*J4 IEEE divides are only paid for 3, 5, 6, 7, ... objects
                    if (cnt > 1) {
                        if ((cnt & (cnt - 1)) == 0) {
                            const float r = 1.0f / (float)cnt;
#pragma unroll
                            for (int j = 0; j < J4; ++j)
                                acc[j] = make_float4(__fmul_rn(acc[j].x, r), __fmul_rn(acc[j].y, r), __fmul_rn(acc[j].z, r), __fmul_rn(acc[j].w, r));
                        } else {
                            const float n_px = (float)cnt;
#pragma unroll
                            for (int j = 0; j < J4; ++j)
                                acc[j] = make_float4(__fdiv_rn(acc[j].x, n_px), __fdiv_rn(acc[j].y, n_px), __fdiv_rn(acc[j].z, n_px), __fdiv_rn(acc[j].w, n_px));
                        }
                    }
                }
                const int slot = s_slot[i];
                if (cnt == 0 || slot < 0 || slot >= S) continue;           // cnt == 0 cannot happen for a sampled pixel; slot overflow: caller error
                if (slot != agg_slot) {
                    flush();
                    agg_slot = slot;
#pragma unroll
                    for (int j = 0; j < J4; ++j) agg[j] = acc[j];
                } else {
#pragma unroll
                    for (int j = 0; j < J4; ++j) {
                        agg[j].x = __fadd_rn(agg[j].x, acc[j].x); agg[j].y = __fadd_rn(agg[j].y, acc[j].y);
                        agg[j].z = __fadd_rn(agg[j].z, acc[j].z); agg[j].w = __fadd_rn(agg[j].w, acc[j].w);
                    }
                }
            }
            flush();
            __syncthreads();                                               // s_cover / s_slot are rewritten by the next round
        }
        return;
    }

    // ---- more than kCoverObjs objects: one sampled pixel at a time per warp ----
    for (int i = warp; i < n; i += 8) {
        const int px = s_list[i];
        float acc[J];
#pragma unroll
        for (int j = 0; j < J; ++j) acc[j] = 0.f;
        int cnt = 0;
        for (int k0 = 0; k0 < K; k0 += 32) {                       // lanes test 32 objects at once
            const int k = k0 + (int)lane;
            bool mine = false;
            if (k < K) {
                if (kPasted) {
                    const PasteObj o = paste_prepare(boxes + ((size_t)e * Kmax + k) * 4, HW / W, W, thr);
                    mine = paste_covers(probs + ((size_t)e * Kmax + k) * Sm * Sm, o, Sm, px % W, px / W, thr);
                } else {
                    mine = __ldg(m + (size_t)k * HW + px) != 0;
                }
            }
            const unsigned cover = __ballot_sync(0xffffffffu, mine);
            unsigned todo = cover;
            while (todo) {                                         // ascending object index
                const int kk = k0 + __ffs(todo) - 1;
                todo &= todo - 1;
                const float *row = f + (size_t)kk * C + lane;
#pragma unroll
                for (int j = 0; j < J; ++j) acc[j] = __fadd_rn(acc[j], __ldg(row + 32 * j));
            }
            cnt += __popc(cover);
        }
        if (cnt == 0) continue;                                    // cannot happen for a sampled pixel; defensive
        const int cell = __ldg(idx + (size_t)e * HW + px);
        const int slot = __ldg(slot_of_cell + (size_t)e * n_cells + cell) - 1;
        if (slot < 0 || slot >= S) continue;                       // slot table overflow (S < #sampled pixels): caller error
        const float n_px = (float)cnt;
        float *dst = scratch + ((size_t)e * S + slot) * C + lane;
#pragma unroll
        for (int j = 0; j < J; ++j) red_add_f32(dst + 32 * j, __fdiv_rn(acc[j], n_px));
    }
}

// warp per slot: sums[cell] += scratch[slot] / n_cell (custom_rcnn.py:931-934, :696-697,742); scratch and slot map back to zero
__global__ void __launch_bounds__(256) flush_slots_kernel(const uint32_t *__restrict__ frame_cnt, int32_t *__restrict__ slot_of_cell,
                                                          const int32_t *__restrict__ slot_cell, const int32_t *__restrict__ n_slots, int S, int C,
                                                          int64_t n_cells, float *__restrict__ scratch, float *__restrict__ sums)
{
    // the number of claimed slots is only known on the device (a few hundred of the S = HW/8 possible ones): a fixed, small grid walks
    // them with a stride (one CTA per 8 possible slots was 307 k mostly empty CTAs at E=64: 0.17 ms of block scheduling)
    const int e = blockIdx.y;
    const unsigned lane = threadIdx.x & 31;
    const int n = min(__ldg(n_slots + e), S);
    for (int slot = blockIdx.x * 8 + (threadIdx.x >> 5); slot < n; slot += (int)gridDim.x * 8) {
        const int cell = __ldg(slot_cell + (size_t)e * S + slot);
        const float n_cell = (float)(__ldg(frame_cnt + (size_t)e * n_cells + cell) & 0x7fffffffu);
        float4 *src = reinterpret_cast<float4 *>(scratch + ((size_t)e * S + slot) * C);
        float4 *dst = reinterpret_cast<float4 *>(sums + ((size_t)e * n_cells + cell) * C);
        for (int k = lane; k < C / 4; k += 32) {
            const float4 a = src[k];
            float4 d = dst[k];
            d.x = __fadd_rn(d.x, __fdiv_rn(a.x, n_cell)); d.y = __fadd_rn(d.y, __fdiv_rn(a.y, n_cell));
            d.z = __fadd_rn(d.z, __fdiv_rn(a.z, n_cell)); d.w = __fadd_rn(d.w, __fdiv_rn(a.w, n_cell));
            dst[k] = d;
            src[k] = make_float4(0.f, 0.f, 0.f, 0.f);
        }
        if (lane == 0) slot_of_cell[(size_t)e * n_cells + cell] = 0;
    }
}

// Deterministic variant (eod_write_objects[_pasted]_det): the main pass of det.cuh for the object regime.  It stores exactly the run
// partials the dense deterministic write would store for the image eod_box_to_image_features builds - a run's sum, from +0, of the
// values g of its sampled pixels in raster order - without building that image, so the pre-passes and the segmented reduce of the
// dense write finish the job and the result is bitwise reproducible.
// The CTA span, the sampled-pixel compaction and phase A's cover words are those of write_objects_kernel; phase B gives warps whole
// 32-pixel tiles (one warp must own a run) in rounds of tiles whose sampled pixels fit the 256 cover rows.  Tiles without a sampled
// pixel have no run and are skipped.  More than kCoverObjs objects: warp per tile, the cover set of a pixel by warp ballots.
template <int C, bool kPasted>
__global__ void __launch_bounds__(256) write_objects_det_kernel(const float *__restrict__ box_features, const uint8_t *__restrict__ masks,
                                                                const float *__restrict__ probs, const float *__restrict__ boxes, int Sm, int W,
                                                                float thr, const int32_t *__restrict__ n_obj, int Kmax, const int32_t *__restrict__ idx,
                                                                const uint8_t *__restrict__ samp, const uint32_t *__restrict__ frame_cnt, int HW,
                                                                int64_t n_cells, float *__restrict__ sums, const DetArgs det)
{
    constexpr int J = C / 32, J4 = C / 128;
    constexpr int kTiles = kObjSpan / TILE_PX;
    __shared__ int s_list[kObjSpan];
    __shared__ __align__(16) uint32_t s_cover[256][kCoverObjs / 32];
    __shared__ PasteObj s_obj[kPasted ? kCoverObjs : 1];
    __shared__ int s_wcnt[8];
    __shared__ int s_tstart[kTiles + 1];         // s_list index of each tile's first sampled pixel
    __shared__ int s_busy[kTiles];               // tiles with a sampled pixel, in raster order
    __shared__ int s_nbusy;
    const int e = blockIdx.y;
    const unsigned lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    if (n_obj && __ldg(n_obj + e) <= 0) return;  // idle slot: the pre-passes gave it no runs; nothing of it is read
    {   // raster-ordered list of the CTA's sampled pixels, as in write_objects_kernel, plus where each tile's pixels start in it
        const int p0 = blockIdx.x * kObjSpan + threadIdx.x * 8;
        const uint8_t *sp = samp + (size_t)e * HW + p0;
        uint32_t lo = 0, hi = 0;
        if (p0 + 7 < HW && (reinterpret_cast<uintptr_t>(sp) & 7u) == 0) {
            const uint2 q = __ldg(reinterpret_cast<const uint2 *>(sp));
            lo = q.x; hi = q.y;
        } else {
            for (int b = 0; b < 8 && p0 + b < HW; ++b) {
                const uint32_t v = __ldg(sp + b);
                if (b < 4) lo |= v << (8 * b); else hi |= v << (8 * (b - 4));
            }
        }
        unsigned bits = 0;
#pragma unroll
        for (int b = 0; b < 4; ++b) bits |= (((lo >> (8 * b)) & 0xffu) ? 1u : 0u) << b | (((hi >> (8 * b)) & 0xffu) ? 1u : 0u) << (b + 4);
        const int cnt = __popc(bits);
        int incl = cnt;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const int up = __shfl_up_sync(0xffffffffu, incl, o);
            if ((int)lane >= o) incl += up;
        }
        if (lane == 31) s_wcnt[warp] = incl;
        __syncthreads();
        int pre = 0, tot = 0;
#pragma unroll
        for (int w = 0; w < 8; ++w) { pre += w < (int)warp ? s_wcnt[w] : 0; tot += s_wcnt[w]; }
        int pos = pre + incl - cnt;
        if ((threadIdx.x & 3) == 0) s_tstart[threadIdx.x >> 2] = pos;          // four threads (32 pixels) per tile
        if (threadIdx.x == 0) s_tstart[kTiles] = tot;
        while (bits) {
            s_list[pos++] = p0 + __ffs(bits) - 1;
            bits &= bits - 1;
        }
        __syncthreads();
        if (warp == 0) {
            const bool b0 = s_tstart[lane + 1] > s_tstart[lane], b1 = s_tstart[lane + 33] > s_tstart[lane + 32];
            const unsigned m0 = __ballot_sync(0xffffffffu, b0), m1 = __ballot_sync(0xffffffffu, b1);
            if (b0) s_busy[__popc(m0 & ((1u << lane) - 1u))] = (int)lane;
            if (b1) s_busy[__popc(m0) + __popc(m1 & ((1u << lane) - 1u))] = (int)lane + 32;
            if (lane == 0) s_nbusy = __popc(m0) + __popc(m1);
        }
        __syncthreads();
    }
    const int n_busy = s_nbusy;
    if (n_busy == 0) return;
    const int K = n_obj ? min(__ldg(n_obj + e), Kmax) : Kmax;
    const uint8_t *m = kPasted ? nullptr : masks + (size_t)e * Kmax * HW;
    const float *f = box_features + (size_t)e * Kmax * C;
    const int tiles_per_ep = HW / TILE_PX;

    // warp-level run walk of one tile: for every run with a sampled pixel (det_run_mask order), value(p, acc) adds the pixel's g into the
    // run's accumulator, then the run's sum is stored at its raster rank - or, past the workspace, reduced into sums as sum / n_cell
    auto walk_tile = [&](int tt, auto &&begin_run, auto &&add_pixel, auto &&end_run) {
        const int tile = (int)blockIdx.x * kTiles + tt;
        int cell;
        unsigned heads, samps;
        det_tile_masks(idx, samp, (size_t)e * HW + (size_t)tile * TILE_PX, lane, cell, heads, samps);
        int run_pos = __ldg(det.tile_off + (size_t)e * tiles_per_ep + tile);
        while (heads) {
            const int p0 = __ffs(heads) - 1;
            heads &= heads - 1;
            unsigned mr = det_run_mask(heads, samps, p0);
            if (mr == 0) continue;
            begin_run();
            do {
                const int p = __ffs(mr) - 1;
                mr &= mr - 1;
                add_pixel(tile * TILE_PX + p, __popc(samps & ((1u << p) - 1u)));
            } while (mr);
            end_run(__shfl_sync(0xffffffffu, cell, p0), run_pos++);
        }
    };
    auto fallback_n = [&](int rc) {
        if (lane == 0) *det.status = 1;                                    // workspace too small: correct, but not reproducible
        return (float)(__ldg(frame_cnt + (size_t)e * n_cells + rc) & 0x7fffffffu);
    };

    if (K <= kCoverObjs) {
        if (kPasted) {
            if ((int)threadIdx.x < K) s_obj[threadIdx.x] = paste_prepare(boxes + ((size_t)e * Kmax + threadIdx.x) * 4, HW / W, W, thr);
            __syncthreads();
        }
        for (int b0 = 0; b0 < n_busy;) {
            // round: busy tiles [b0, b1) whose sampled pixels (contiguous in s_list) fit the 256 cover rows; one tile has at most 32
            const int base = s_tstart[s_busy[b0]];
            int b1 = b0 + 1;
            while (b1 < n_busy && s_tstart[s_busy[b1] + 1] - base <= 256) ++b1;
            const int nn = s_tstart[s_busy[b1 - 1] + 1] - base;
            // ---- phase A: thread per sampled pixel, its cover words (write_objects_kernel's test) ----
            if ((int)threadIdx.x < nn) {
                const int px = s_list[base + threadIdx.x];
                const int x = px % W, y = px / W;
                unsigned w0 = 0u, w1 = 0u, w2 = 0u, w3 = 0u;
                for (int k = 0; k < K; ++k) {
                    bool mine;
                    if (kPasted) {
                        const PasteObj &o = s_obj[k];
                        mine = x >= o.rx0 && x < o.rx1 && y >= o.ry0 && y < o.ry1 &&
                               paste_eval(probs + ((size_t)e * Kmax + k) * Sm * Sm, Sm, paste_axis(x, o.x0, o.dx, Sm), paste_axis(y, o.y0, o.dy, Sm), thr);
                    } else {
                        mine = __ldg(m + (size_t)k * HW + px) != 0;
                    }
                    if (mine) {
                        const unsigned bit = 1u << (k & 31);
                        const int wd = k >> 5;
                        w0 |= wd == 0 ? bit : 0u; w1 |= wd == 1 ? bit : 0u; w2 |= wd == 2 ? bit : 0u; w3 |= wd == 3 ? bit : 0u;
                    }
                }
                s_cover[threadIdx.x][0] = w0; s_cover[threadIdx.x][1] = w1; s_cover[threadIdx.x][2] = w2; s_cover[threadIdx.x][3] = w3;
            }
            __syncthreads();
            // ---- phase B: warp per busy tile; lanes own float4 channel groups 4*lane + 128*j ----
            // g is recomputed only when the cover set changes (bit-identical either way); the empty set's g is +0, the image's value
            // at a pixel no object covers
            float4 g[J4], acc[J4];
#pragma unroll
            for (int j = 0; j < J4; ++j) g[j] = make_float4(0.f, 0.f, 0.f, 0.f);
            uint4 have = make_uint4(0u, 0u, 0u, 0u);
            for (int bt = b0 + (int)warp; bt < b1; bt += 8) {
                const int tt = s_busy[bt];
                const int row0 = s_tstart[tt] - base;
                walk_tile(
                    tt,
                    [&]() {
#pragma unroll
                        for (int j = 0; j < J4; ++j) acc[j] = make_float4(0.f, 0.f, 0.f, 0.f);
                    },
                    [&](int, int rank) {
                        const uint4 cw = *reinterpret_cast<const uint4 *>(&s_cover[row0 + rank][0]);
                        if (cw.x != have.x || cw.y != have.y || cw.z != have.z || cw.w != have.w) {
                            have = cw;
#pragma unroll
                            for (int j = 0; j < J4; ++j) g[j] = make_float4(0.f, 0.f, 0.f, 0.f);
                            int cnt = 0;
                            const unsigned words[4] = {cw.x, cw.y, cw.z, cw.w};
#pragma unroll
                            for (int wd = 0; wd < 4; ++wd) {
                                unsigned todo = words[wd];
                                cnt += __popc(todo);
                                while (todo) {                             // ascending object index
                                    const int kk = wd * 32 + __ffs(todo) - 1;
                                    todo &= todo - 1;
                                    const float4 *row = reinterpret_cast<const float4 *>(f + (size_t)kk * C) + lane;
#pragma unroll
                                    for (int j = 0; j < J4; ++j) {
                                        const float4 v = __ldg(row + 32 * j);
                                        g[j].x = __fadd_rn(g[j].x, v.x); g[j].y = __fadd_rn(g[j].y, v.y);
                                        g[j].z = __fadd_rn(g[j].z, v.z); g[j].w = __fadd_rn(g[j].w, v.w);
                                    }
                                }
                            }
                            if (cnt > 1) {                                 // / #objects; a power of two as the exact reciprocal
                                if ((cnt & (cnt - 1)) == 0) {
                                    const float r = 1.0f / (float)cnt;
#pragma unroll
                                    for (int j = 0; j < J4; ++j)
                                        g[j] = make_float4(__fmul_rn(g[j].x, r), __fmul_rn(g[j].y, r), __fmul_rn(g[j].z, r), __fmul_rn(g[j].w, r));
                                } else {
                                    const float n_px = (float)cnt;
#pragma unroll
                                    for (int j = 0; j < J4; ++j)
                                        g[j] = make_float4(__fdiv_rn(g[j].x, n_px), __fdiv_rn(g[j].y, n_px), __fdiv_rn(g[j].z, n_px), __fdiv_rn(g[j].w, n_px));
                                }
                            }
                        }
#pragma unroll
                        for (int j = 0; j < J4; ++j) {
                            acc[j].x = __fadd_rn(acc[j].x, g[j].x); acc[j].y = __fadd_rn(acc[j].y, g[j].y);
                            acc[j].z = __fadd_rn(acc[j].z, g[j].z); acc[j].w = __fadd_rn(acc[j].w, g[j].w);
                        }
                    },
                    [&](int rc, int pos) {
                        if (pos < det.cap) {
                            float *d = det.partials + ((size_t)e * det.cap + pos) * C + 4 * lane;
#pragma unroll
                            for (int j = 0; j < J4; ++j) *reinterpret_cast<float4 *>(d + 128 * j) = acc[j];
                            if (lane == 0) det.run_cell[(size_t)e * det.cap + pos] = rc;
                            return;
                        }
                        const float n = fallback_n(rc);
                        float *d = sums + ((size_t)e * n_cells + rc) * C + 4 * lane;
#pragma unroll
                        for (int j = 0; j < J4; ++j)
                            red_add_v4(d + 128 * j, __fdiv_rn(acc[j].x, n), __fdiv_rn(acc[j].y, n), __fdiv_rn(acc[j].z, n), __fdiv_rn(acc[j].w, n));
                    });
            }
            __syncthreads();                                               // s_cover is rewritten by the next round
            b0 = b1;
        }
        return;
    }

    // ---- more than kCoverObjs objects: warp per busy tile, lanes test 32 objects at once; lanes own channels lane + 32*j ----
    float acc[J];
    for (int bt = (int)warp; bt < n_busy; bt += 8) {
        walk_tile(
            s_busy[bt],
            [&]() {
#pragma unroll
                for (int j = 0; j < J; ++j) acc[j] = 0.f;
            },
            [&](int px, int) {
                float g[J];
#pragma unroll
                for (int j = 0; j < J; ++j) g[j] = 0.f;
                int cnt = 0;
                for (int k0 = 0; k0 < K; k0 += 32) {
                    const int k = k0 + (int)lane;
                    bool mine = false;
                    if (k < K) {
                        if (kPasted) {
                            const PasteObj o = paste_prepare(boxes + ((size_t)e * Kmax + k) * 4, HW / W, W, thr);
                            mine = paste_covers(probs + ((size_t)e * Kmax + k) * Sm * Sm, o, Sm, px % W, px / W, thr);
                        } else {
                            mine = __ldg(m + (size_t)k * HW + px) != 0;
                        }
                    }
                    unsigned todo = __ballot_sync(0xffffffffu, mine);
                    cnt += __popc(todo);
                    while (todo) {                                         // ascending object index
                        const int kk = k0 + __ffs(todo) - 1;
                        todo &= todo - 1;
                        const float *row = f + (size_t)kk * C + lane;
#pragma unroll
                        for (int j = 0; j < J; ++j) g[j] = __fadd_rn(g[j], __ldg(row + 32 * j));
                    }
                }
                const float n_px = (float)cnt;
#pragma unroll
                for (int j = 0; j < J; ++j) acc[j] = __fadd_rn(acc[j], cnt ? __fdiv_rn(g[j], n_px) : 0.f);
            },
            [&](int rc, int pos) {
                if (pos < det.cap) {
                    float *d = det.partials + ((size_t)e * det.cap + pos) * C + lane;
#pragma unroll
                    for (int j = 0; j < J; ++j) d[32 * j] = acc[j];
                    if (lane == 0) det.run_cell[(size_t)e * det.cap + pos] = rc;
                    return;
                }
                const float n = fallback_n(rc);
                float *d = sums + ((size_t)e * n_cells + rc) * C + lane;
#pragma unroll
                for (int j = 0; j < J; ++j) red_add_f32(d + 32 * j, __fdiv_rn(acc[j], n));
            });
    }
}

__global__ void zero_i32_kernel(int32_t *p, int n)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) p[i] = 0;
}

}  // namespace

extern "C" int eod_masks_observed(const uint8_t *masks, const int32_t *n_obj, int n_episodes, int Kmax, int HW, uint8_t *observed,
                                  eod_stream_t stream)
{
    EOD_REQUIRE(masks && observed, EOD_ERR_BADARG, "eod_masks_observed: null pointer");
    EOD_REQUIRE(n_episodes > 0 && n_episodes <= 65535 && Kmax >= 0 && HW > 0, EOD_ERR_BADARG, "eod_masks_observed: bad sizes");
    EOD_REQUIRE(HW % 4 == 0 && (reinterpret_cast<uintptr_t>(masks) & 3u) == 0 && (reinterpret_cast<uintptr_t>(observed) & 3u) == 0, EOD_ERR_ALIGN,
                "eod_masks_observed: HW %% 4 == 0 and 4-byte aligned planes required");
    dim3 grid((HW / 4 + 255) / 256, n_episodes);
    masks_observed_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(masks, n_obj, Kmax, HW, observed);
    return eod_check_launch("eod_masks_observed");
}

static int launch_write_objects(const char *what, bool pasted, const float *box_features, const uint8_t *masks, const float *probs,
                                const float *boxes, int S, int W, float thr, const int32_t *n_obj, int Kmax, const int32_t *idx,
                                const uint8_t *samp, const int32_t *slot_of_cell, int n_episodes, int C, int HW, int64_t n_cells,
                                int n_slots_max, float *scratch, cudaStream_t st)
{
    dim3 grid((HW + kObjSpan - 1) / kObjSpan, n_episodes);
#define EOD_WO(CC)                                                                                                                      \
    case CC:                                                                                                                            \
        if (pasted)                                                                                                                     \
            write_objects_kernel<CC, true><<<grid, 256, 0, st>>>(box_features, masks, probs, boxes, S, W, thr, n_obj, Kmax, idx, samp,  \
                                                                 slot_of_cell, HW, n_cells, n_slots_max, scratch);                     \
        else                                                                                                                            \
            write_objects_kernel<CC, false><<<grid, 256, 0, st>>>(box_features, masks, probs, boxes, S, W, thr, n_obj, Kmax, idx, samp, \
                                                                  slot_of_cell, HW, n_cells, n_slots_max, scratch);                    \
        break;
    switch (C) {
        EOD_WO(128)
        EOD_WO(256)
        EOD_WO(512)
    default:
        eod_set_error("%s: C=%d not compiled in (128, 256, 512)", what, C);
        return EOD_ERR_UNSUPPORTED;
    }
#undef EOD_WO
    return eod_check_launch(what);
}

extern "C" int eod_write_objects(const float *box_features, const uint8_t *masks, const int32_t *n_obj, int Kmax, const int32_t *idx,
                                 const uint8_t *samp, const int32_t *slot_of_cell, int n_episodes, int C, int HW, int64_t n_cells,
                                 int n_slots_max, float *scratch, eod_stream_t stream)
{
    EOD_REQUIRE(box_features && masks && idx && samp && slot_of_cell && scratch, EOD_ERR_BADARG, "eod_write_objects: null pointer");
    EOD_REQUIRE(n_episodes > 0 && n_episodes <= 65535 && Kmax > 0 && HW > 0 && n_cells > 0 && n_slots_max > 0, EOD_ERR_BADARG,
                "eod_write_objects: bad sizes");
    return launch_write_objects("eod_write_objects", false, box_features, masks, nullptr, nullptr, 0, 1, 0.f, n_obj, Kmax, idx, samp,
                                slot_of_cell, n_episodes, C, HW, n_cells, n_slots_max, scratch, (cudaStream_t)stream);
}

extern "C" int eod_paste_masks(const float *mask_probs, const float *boxes, const int32_t *n_obj, int n_episodes, int Kmax, int S, int H,
                               int W, float threshold, uint8_t *masks, uint8_t *observed, eod_stream_t stream)
{
    EOD_REQUIRE(mask_probs && boxes && (masks || observed), EOD_ERR_BADARG, "eod_paste_masks: null pointer");
    EOD_REQUIRE(n_episodes > 0 && n_episodes <= 65535 && Kmax > 0 && S > 0 && S <= 4096 && H > 0 && W > 0 && (int64_t)H * W < (1ll << 31) - 1024,
                EOD_ERR_BADARG, "eod_paste_masks: bad sizes");
    EOD_REQUIRE(threshold >= 0.f, EOD_ERR_UNSUPPORTED, "eod_paste_masks: threshold < 0 (uint8 soft masks) is not supported");
    dim3 grid((H * W + 1023) / 1024, n_episodes);
    paste_masks_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(mask_probs, boxes, n_obj, Kmax, S, H, W, threshold, masks, observed);
    return eod_check_launch("eod_paste_masks");
}

extern "C" int eod_write_objects_pasted(const float *box_features, const float *mask_probs, const float *boxes, const int32_t *n_obj,
                                        int Kmax, int S, int H, int W, float threshold, const int32_t *idx, const uint8_t *samp,
                                        const int32_t *slot_of_cell, int n_episodes, int C, int64_t n_cells, int n_slots_max,
                                        float *scratch, eod_stream_t stream)
{
    EOD_REQUIRE(box_features && mask_probs && boxes && idx && samp && slot_of_cell && scratch, EOD_ERR_BADARG,
                "eod_write_objects_pasted: null pointer");
    EOD_REQUIRE(n_episodes > 0 && n_episodes <= 65535 && Kmax > 0 && S > 0 && S <= 4096 && H > 0 && W > 0 && (int64_t)H * W < (1ll << 31) - 1024 &&
                    n_cells > 0 && n_slots_max > 0,
                EOD_ERR_BADARG, "eod_write_objects_pasted: bad sizes");
    EOD_REQUIRE(threshold >= 0.f, EOD_ERR_UNSUPPORTED, "eod_write_objects_pasted: threshold < 0 is not supported");
    return launch_write_objects("eod_write_objects_pasted", true, box_features, nullptr, mask_probs, boxes, S, W, threshold, n_obj, Kmax, idx,
                                samp, slot_of_cell, n_episodes, C, H * W, n_cells, n_slots_max, scratch, (cudaStream_t)stream);
}

static int launch_write_objects_det(const char *what, bool pasted, const float *box_features, const uint8_t *masks, const float *probs,
                                    const float *boxes, int S, int W, float thr, const int32_t *n_obj, int Kmax, const int32_t *idx,
                                    const uint8_t *samp, const uint32_t *frame_cnt, int n_episodes, int C, int HW, int64_t n_cells, float *sums,
                                    void *ws, int64_t ws_bytes, cudaStream_t st)
{
    EOD_REQUIRE(C == 128 || C == 256 || C == 512, EOD_ERR_UNSUPPORTED, "%s: C=%d not compiled in (128, 256, 512)", what, C);
    EOD_REQUIRE(eod_aligned16(box_features) && eod_aligned16(sums), EOD_ERR_ALIGN, "%s: box_features and sums must be 16-byte aligned", what);
    DetWorkspace w;
    int rc = det_prepass(what, idx, samp, n_obj, n_episodes, C, HW, n_cells, ws, (size_t)ws_bytes, &w, st);
    if (rc) return rc;
    const DetArgs det = det_args(w);
    dim3 grid((HW + kObjSpan - 1) / kObjSpan, n_episodes);
#define EOD_WOD(CC)                                                                                                                        \
    case CC:                                                                                                                               \
        if (pasted)                                                                                                                        \
            write_objects_det_kernel<CC, true><<<grid, 256, 0, st>>>(box_features, masks, probs, boxes, S, W, thr, n_obj, Kmax, idx, samp,  \
                                                                     frame_cnt, HW, n_cells, sums, det);                                  \
        else                                                                                                                               \
            write_objects_det_kernel<CC, false><<<grid, 256, 0, st>>>(box_features, masks, probs, boxes, S, W, thr, n_obj, Kmax, idx, samp, \
                                                                      frame_cnt, HW, n_cells, sums, det);                                 \
        break;
    switch (C) {
        EOD_WOD(128)
        EOD_WOD(256)
        EOD_WOD(512)
    }
#undef EOD_WOD
    if ((rc = eod_check_launch(what))) return rc;
    return det_reduce(what, w, C, n_episodes, n_cells, frame_cnt, sums, st);
}

extern "C" int eod_write_objects_det(const float *box_features, const uint8_t *masks, const int32_t *n_obj, int Kmax, const int32_t *idx,
                                     const uint8_t *samp, const uint32_t *frame_cnt, int n_episodes, int C, int HW, int64_t n_cells, float *sums,
                                     void *workspace, int64_t workspace_bytes, eod_stream_t stream)
{
    EOD_REQUIRE(box_features && masks && idx && samp && frame_cnt && sums && workspace, EOD_ERR_BADARG, "eod_write_objects_det: null pointer");
    EOD_REQUIRE(n_episodes > 0 && n_episodes <= 65535 && Kmax > 0 && HW > 0 && n_cells > 0 && workspace_bytes > 0, EOD_ERR_BADARG,
                "eod_write_objects_det: bad sizes");
    return launch_write_objects_det("eod_write_objects_det", false, box_features, masks, nullptr, nullptr, 0, 1, 0.f, n_obj, Kmax, idx, samp,
                                    frame_cnt, n_episodes, C, HW, n_cells, sums, workspace, workspace_bytes, (cudaStream_t)stream);
}

extern "C" int eod_write_objects_pasted_det(const float *box_features, const float *mask_probs, const float *boxes, const int32_t *n_obj,
                                            int Kmax, int S, int H, int W, float threshold, const int32_t *idx, const uint8_t *samp,
                                            const uint32_t *frame_cnt, int n_episodes, int C, int64_t n_cells, float *sums, void *workspace,
                                            int64_t workspace_bytes, eod_stream_t stream)
{
    EOD_REQUIRE(box_features && mask_probs && boxes && idx && samp && frame_cnt && sums && workspace, EOD_ERR_BADARG,
                "eod_write_objects_pasted_det: null pointer");
    EOD_REQUIRE(n_episodes > 0 && n_episodes <= 65535 && Kmax > 0 && S > 0 && S <= 4096 && H > 0 && W > 0 && (int64_t)H * W < (1ll << 31) - 1024 &&
                    n_cells > 0 && workspace_bytes > 0,
                EOD_ERR_BADARG, "eod_write_objects_pasted_det: bad sizes");
    EOD_REQUIRE(threshold >= 0.f, EOD_ERR_UNSUPPORTED, "eod_write_objects_pasted_det: threshold < 0 is not supported");
    return launch_write_objects_det("eod_write_objects_pasted_det", true, box_features, nullptr, mask_probs, boxes, S, W, threshold, n_obj, Kmax,
                                    idx, samp, frame_cnt, n_episodes, C, H * W, n_cells, sums, workspace, workspace_bytes, (cudaStream_t)stream);
}

extern "C" int eod_flush_slots(const uint32_t *frame_cnt, int32_t *slot_of_cell, const int32_t *slot_cell, int32_t *n_slots, int n_episodes,
                               int C, int64_t n_cells, int n_slots_max, float *scratch, float *sums, eod_stream_t stream)
{
    EOD_REQUIRE(frame_cnt && slot_of_cell && slot_cell && n_slots && scratch && sums, EOD_ERR_BADARG, "eod_flush_slots: null pointer");
    EOD_REQUIRE(n_episodes > 0 && n_episodes <= 65535 && C > 0 && C % 4 == 0 && n_cells > 0 && n_slots_max > 0, EOD_ERR_BADARG, "eod_flush_slots: bad sizes");
    EOD_REQUIRE(eod_aligned16(scratch) && eod_aligned16(sums), EOD_ERR_ALIGN, "eod_flush_slots: rows must be 16-byte aligned");
    cudaStream_t st = (cudaStream_t)stream;
    const int per_ep = (n_slots_max + 7) / 8;
    int gx = (eod_num_sms() * 16 + n_episodes - 1) / n_episodes;          // ~16 CTAs per SM over all episodes, at least 8 per episode
    if (gx < 8) gx = 8;
    if (gx > per_ep) gx = per_ep;
    dim3 grid(gx, n_episodes);
    flush_slots_kernel<<<grid, 256, 0, st>>>(frame_cnt, slot_of_cell, slot_cell, n_slots, n_slots_max, C, n_cells, scratch, sums);
    int rc = eod_check_launch("eod_flush_slots");
    if (rc) return rc;
    zero_i32_kernel<<<(n_episodes + 255) / 256, 256, 0, st>>>(n_slots, n_episodes);
    return eod_check_launch("eod_flush_slots[reset]");
}
