// Memory read (SURVEY 8a rows A10-A12): normalise (sum/count where count>1) -> fp16 -> gather to the
// image plane -> avg-pool 4 -> three times (avg-pool 2 -> fp16): one kernel for levels 0 and 1 (the (480,640,C)
// image-plane tensors are never materialised) and a small second one that pools level 2 from level 1.
//
// Work decomposition: a warp owns one 16x16-pixel quadrant of one episode's frame (= four L0 pixels, one L1 pixel)
// and ALL channels (lane = C/32 consecutive channels), so the cell id is warp-uniform, every table access is one
// coalesced C*2-byte (fp16) / C*4-byte (fp32) cell row, and consecutive pixels that hit the same cell reuse the value
// from registers.  The 1.2 MB index plane is read once; table rows come from L1/L2 after the first touch (a frame sees a
// few hundred to a few thousand distinct cells).  The kernel is instruction-issue bound, not bandwidth bound: what it
// optimises is scalar bookkeeping per gathered row (see read_pool_kernel).
//
// Summation order == ATen CPU avg_pool2d: fp32, start from 0, row-major over the window, then / k^2;
// the fp16 roundings between levels (timm.py:168) are reproduced, so outputs are bit-identical.
#include <stdlib.h>

#include "eod_common.cuh"

namespace {

// ---- V channels per lane (V = 4 or 8) as packed fp32x2 pairs -------------------------------------------------------
// FADD2 / FMUL2 (sm_100): two IEEE round-to-nearest operations per instruction, the same bits as the scalar ones.
template <int V>
struct Vec { float2 p[V / 2]; };

template <int V>
__device__ __forceinline__ Vec<V> vzero()
{
    Vec<V> r;
#pragma unroll
    for (int i = 0; i < V / 2; ++i) r.p[i] = make_float2(0.f, 0.f);
    return r;
}
template <int V>
__device__ __forceinline__ Vec<V> vadd(const Vec<V> &a, const Vec<V> &b)
{
    Vec<V> r;
#pragma unroll
    for (int i = 0; i < V / 2; ++i) r.p[i] = __fadd2_rn(a.p[i], b.p[i]);
    return r;
}
template <int V>
__device__ __forceinline__ Vec<V> vscale(const Vec<V> &a, float s)
{
    Vec<V> r;
#pragma unroll
    for (int i = 0; i < V / 2; ++i) r.p[i] = __fmul2_rn(a.p[i], make_float2(s, s));
    return r;
}
template <int V>
__device__ __forceinline__ Vec<V> vround_half(const Vec<V> &a)
{
    Vec<V> r;
#pragma unroll
    for (int i = 0; i < V / 2; ++i) r.p[i] = __half22float2(__float22half2_rn(a.p[i]));
    return r;
}
// V halves, 2*V bytes, one store
template <int V>
__device__ __forceinline__ void vstore_half(__half *dst, const Vec<V> &a)
{
    uint32_t w[V / 2];
#pragma unroll
    for (int i = 0; i < V / 2; ++i) {
        const __half2 h = __float22half2_rn(a.p[i]);
        w[i] = *reinterpret_cast<const uint32_t *>(&h);
    }
    if (V >= 8) {
#pragma unroll
        for (int i = 0; i < V / 8; ++i) reinterpret_cast<uint4 *>(dst)[i] = make_uint4(w[(4 * i) % (V / 2)], w[(4 * i + 1) % (V / 2)], w[(4 * i + 2) % (V / 2)], w[(4 * i + 3) % (V / 2)]);
    } else {
        *reinterpret_cast<uint2 *>(dst) = make_uint2(w[0], w[1]);
    }
}

// Rows of a two-cell window in summation order: for each of `reps` rows, s += (bit k of pat ? b : a) for k = 0..3.  pat and reps are
// warp-uniform; one dispatch to one of 16 straight-line variants (no predicated-off additions, no per-run bookkeeping).  reps = 4
// serves the commonest mixed window - a vertical edge, all four rows alike - with a single dispatch.
template <int V>
__device__ __forceinline__ void vadd_row2(Vec<V> &s, const Vec<V> &a, const Vec<V> &b, unsigned pat, int reps)
{
#define EOD_R4(x0, x1, x2, x3)                                                                                         \
    _Pragma("unroll 1") for (int r = 0; r < reps; ++r) { s = vadd<V>(s, x0); s = vadd<V>(s, x1); s = vadd<V>(s, x2); s = vadd<V>(s, x3); } \
    break;
    switch (pat & 15u) {
    case 0: EOD_R4(a, a, a, a)
    case 1: EOD_R4(b, a, a, a)
    case 2: EOD_R4(a, b, a, a)
    case 3: EOD_R4(b, b, a, a)
    case 4: EOD_R4(a, a, b, a)
    case 5: EOD_R4(b, a, b, a)
    case 6: EOD_R4(a, b, b, a)
    case 7: EOD_R4(b, b, b, a)
    case 8: EOD_R4(a, a, a, b)
    case 9: EOD_R4(b, a, a, b)
    case 10: EOD_R4(a, b, a, b)
    case 11: EOD_R4(b, b, a, b)
    case 12: EOD_R4(a, a, b, b)
    case 13: EOD_R4(b, a, b, b)
    case 14: EOD_R4(a, b, b, b)
    default: EOD_R4(b, b, b, b)
    }
#undef EOD_R4
}

// Split row fetch: the global load of a row is issued (load_raw) before its consumer (finish: normalise + fp16
// rounding) runs, so the next run's row is in flight under the current run's adds.
template <int V> struct RawF32 { float4 v[V / 4]; float n; };
template <int V> struct RawF16 { uint32_t w[V / 2]; };

template <int V>
__device__ __forceinline__ RawF32<V> load_raw(const float *table, const float *counts, size_t cell, int C, int g)
{
    RawF32<V> r;
#pragma unroll
    for (int i = 0; i < V / 4; ++i) r.v[i] = __ldg(reinterpret_cast<const float4 *>(table + cell * C + (size_t)g * V) + i);
    r.n = counts ? __ldg(counts + cell) : 0.f;
    return r;
}
template <int V>
__device__ __forceinline__ RawF16<V> load_raw(const __half *table, const float *, size_t cell, int C, int g)
{
    RawF16<V> r;
    if (V >= 8) {
#pragma unroll
        for (int i = 0; i < V / 8; ++i) {
            const uint4 q = __ldg(reinterpret_cast<const uint4 *>(table + cell * C + (size_t)g * V) + i);
            r.w[(4 * i) % (V / 2)] = q.x; r.w[(4 * i + 1) % (V / 2)] = q.y; r.w[(4 * i + 2) % (V / 2)] = q.z; r.w[(4 * i + 3) % (V / 2)] = q.w;
        }
    } else {
        const uint2 q = __ldg(reinterpret_cast<const uint2 *>(table + cell * C) + g);
        r.w[0] = q.x; r.w[1] = q.y;
    }
    return r;
}
template <int V>
__device__ __forceinline__ Vec<V> finish(const RawF32<V> &r)
{
    Vec<V> v;
#pragma unroll
    for (int i = 0; i < V / 4; ++i) {
        float4 x = r.v[i];
        if (r.n > 1.0f) {        // custom_rcnn.py:774 (cells seen once or never are left as-is)
            x.x = __fdiv_rn(x.x, r.n); x.y = __fdiv_rn(x.y, r.n); x.z = __fdiv_rn(x.z, r.n); x.w = __fdiv_rn(x.w, r.n);
        }
        v.p[2 * i] = make_float2(x.x, x.y);
        v.p[2 * i + 1] = make_float2(x.z, x.w);
    }
    return vround_half<V>(v);    // custom_rcnn.py:1036
}
template <int V>
__device__ __forceinline__ Vec<V> finish(const RawF16<V> &r)
{
    Vec<V> v;
#pragma unroll
    for (int i = 0; i < V / 2; ++i) v.p[i] = __half22float2(*reinterpret_cast<const __half2 *>(&r.w[i]));
    return v;
}
template <typename T, int V> struct RawOf;
template <int V> struct RawOf<float, V> { using type = RawF32<V>; };
template <int V> struct RawOf<__half, V> { using type = RawF16<V>; };

// Warp-autonomous read: a work item = one 16x16-pixel quadrant (4 L0 pixels, 1 L1 pixel) x all C channels, owned by ONE
// warp (lane = group of V = C/32 consecutive channels: the per-run bookkeeping below is scalar work that every lane
// repeats, so wider lanes amortise it over more channels - V = 4 -> 8 took C=256 from 0.40 to 0.27 ms, V = 8 -> 16 took
// C=512 from 0.51 to 0.40 ms at E=64).  No CTA barrier anywhere; the ids of the NEXT item are already in flight (registers)
// while the current one is processed.  Level 2 needs four L1 pixels of different quadrants; it is pooled from the stored L1
// by pool_level2_kernel instead of through a CTA-wide exchange.
//
// v3 (round 2) - the kernel is issue-bound, so this version removes instructions, not bytes:
//  * the run structure of the 16 4x4 windows is derived IN PARALLEL: lane -> (window, half) loads its two 4-pixel row
//    segments straight from global memory, compares neighbours in summation order (8 compares + one shuffle) and the
//    pair of lanes of a window combines its 16-bit "run head" mask with one more shuffle.  v2 had lanes 0-15 walk their
//    window serially and write run lists to shared memory (~200 warp instructions per item, half of them predicated off);
//  * windows are numbered L0-block-major, so the four masks / first cells an L0 pixel needs come back with one LDS each;
//    runs are then enumerated from the mask in registers (ffs) and only a run's cell id is read from shared memory;
//  * item -> (episode, quadrant) is stepped incrementally in 32-bit arithmetic (v2 decoded every item - and the
//    prefetched one - with 64-bit divisions: six software-division calls per item).
//
// v4 (round 2): windows that hold exactly two cells (an edge: 89 % of the mixed windows) keep both rows in registers and are summed
// row by row through one of 16 straight-line 4-pixel variants (vadd_row2), one dispatch when all four rows are alike; shared memory
// is addressed through one opaque base register, the row pointer / L0 base / lane are opaque too (the compiler re-derived them inside
// the loops); uniform windows enter the common tail as 16 * x (exact) so that the L0 accumulator has a single join point.
//
// Summation order == ATen CPU avg_pool2d: fp32, start from 0, row-major over the window, then / k^2; the fp16 roundings
// between levels (timm.py:168) are reproduced, so outputs are bit-identical.
constexpr int kReadWarps = 8;

struct QuadIdx { int a[4], b[4]; };      // two 4-pixel row segments of this lane's window half

template <typename IdxT>
__device__ __forceinline__ QuadIdx load_quad_idx(const IdxT *src, int W)
{
    QuadIdx q;
    if (sizeof(IdxT) == 4) {
        const int4 a = __ldg(reinterpret_cast<const int4 *>(src)), b = __ldg(reinterpret_cast<const int4 *>(src + W));
        q.a[0] = a.x; q.a[1] = a.y; q.a[2] = a.z; q.a[3] = a.w; q.b[0] = b.x; q.b[1] = b.y; q.b[2] = b.z; q.b[3] = b.w;
    } else {
#pragma unroll
        for (int k = 0; k < 2; ++k) {
            const longlong2 a = __ldg(reinterpret_cast<const longlong2 *>(src) + k), b = __ldg(reinterpret_cast<const longlong2 *>(src + W) + k);
            q.a[2 * k] = (int)a.x; q.a[2 * k + 1] = (int)a.y; q.b[2 * k] = (int)b.x; q.b[2 * k + 1] = (int)b.y;
        }
    }
    return q;
}

// per-warp slice: ids window-major (1024 B) | window descriptors {first cell, second cell or -1, run-head mask, 0} (16 x 16 B) |
// first cells (16 x 4 B) | run-head masks (16 x 2 B)
constexpr int kRpIdx = 0, kRpDesc = 1024, kRpWc = 1280, kRpWm = 1344, kRpSlice = 1376;

template <int C, typename TableT, typename IdxT>
__global__ void __launch_bounds__(kReadWarps * 32, (C >= 512 ? 2 : (C >= 256 ? 3 : 4))) read_pool_kernel(const TableT *__restrict__ table, const float *__restrict__ counts,
                                                                                        const IdxT *__restrict__ idx, int H, int W, int64_t n_cells, int E,
                                                                                        __half *__restrict__ L0, __half *__restrict__ L1)
{
    constexpr int V = C >= 512 ? 16 : (C >= 256 ? 8 : 4);      // channels per lane
    static_assert(C == 32 * V, "one warp covers all channels of a quadrant");
    using Raw = typename RawOf<TableT, V>::type;
    __shared__ __align__(16) unsigned char s_raw[kReadWarps * kRpSlice];

    unsigned lane = threadIdx.x & 31;
    const unsigned warp = threadIdx.x >> 5;
    asm volatile("" : "+r"(lane));
    uint32_t sm = smem_u32(s_raw) + warp * kRpSlice;                         // this warp's slice
    asm volatile("" : "+r"(sm));                                             // opaque: one register, not a %tid / %cluster_ctaid recomputation per use
    const int nqy = H / 16, nqx = W / 16, per_ep = nqy * nqx;
    const int n_items = E * per_ep;                                          // the host guarantees it fits 31 bits
    const int stride = (int)gridDim.x * kReadWarps;
    const int h0 = H / 8, w0 = W / 8, h1 = H / 16, w1 = W / 16;

    int item = (int)blockIdx.x * kReadWarps + (int)warp;
    if (item >= n_items) return;
    // item -> (episode, quadrant row, quadrant column), then stepped with carries: no division inside the loop
    int e = item / per_ep, qy = (item - e * per_ep) / nqx, qx = item - e * per_ep - qy * nqx;
    const int se = stride / per_ep, sqy = (stride - se * per_ep) / nqx, sqx = stride - se * per_ep - sqy * nqx;
    // this lane's share of a quadrant: window w = lane >> 1 in L0-block-major order (w = l0 * 4 + win), rows 2h, 2h+1 of the window
    const int w = lane >> 1, hh = lane & 1;
    const int lane_off = (((w >> 3) * 8 + ((w >> 1) & 1) * 4 + 2 * hh) * W) + ((w >> 2) & 1) * 8 + (w & 1) * 4;
    auto src_of = [&](int e_, int qy_, int qx_) { return idx + ((size_t)e_ * H + (size_t)qy_ * 16) * W + qx_ * 16 + lane_off; };
    QuadIdx nxt = load_quad_idx<IdxT>(src_of(e, qy, qx), W);
    const int g = (int)lane;                                // group of V channels
    uint32_t sm_ids = sm + kRpIdx + (w * 16 + hh * 8) * 4;
    asm volatile("" : "+r"(sm_ids));
    const size_t ep_rows = (size_t)n_cells * C;

    for (; item < n_items; item += stride) {
        const QuadIdx q = nxt;
        const int ce = e, cqy = qy, cqx = qx;
        // advance to the next item of this warp and start its loads
        qx += sqx; if (qx >= nqx) { qx -= nqx; ++qy; }
        qy += sqy; if (qy >= nqy) { qy -= nqy; ++e; }
        e += se;
        if (item + stride < n_items) nxt = load_quad_idx<IdxT>(src_of(e, qy, qx), W);
        // stage the ids window-major; derive the window's run heads in summation (row-major) order
        sts128(sm_ids, q.a[0], q.a[1], q.a[2], q.a[3]);
        sts128(sm_ids + 16, q.b[0], q.b[1], q.b[2], q.b[3]);
        const int prev = __shfl_up_sync(0xffffffffu, q.b[3], 1);             // last pixel of the window's second row (for hh == 1)
        unsigned m8 = (hh == 0 || q.a[0] != prev) ? 1u : 0u;
        m8 |= (q.a[1] != q.a[0]) << 1 | (q.a[2] != q.a[1]) << 2 | (q.a[3] != q.a[2]) << 3 | (q.b[0] != q.a[3]) << 4 | (q.b[1] != q.b[0]) << 5 |
              (q.b[2] != q.b[1]) << 6 | (q.b[3] != q.b[2]) << 7;
        const unsigned other = __shfl_xor_sync(0xffffffffu, m8, 1);
        // two-cell windows (an edge between two map cells: 89 % of the mixed windows of the synthetic episodes, typically 8 runs
        // A A B B / A A B B / ...): the pixels take one of TWO rows, so the walk below keeps both in registers and pays nothing per
        // run.  B = any id != A; valid iff every id of the window is A or B.
        const int cA = __shfl_sync(0xffffffffu, q.a[0], lane & ~1u);
        int bsel = cA;
        bsel = q.b[3] != cA ? q.b[3] : bsel; bsel = q.b[2] != cA ? q.b[2] : bsel; bsel = q.b[1] != cA ? q.b[1] : bsel; bsel = q.b[0] != cA ? q.b[0] : bsel;
        bsel = q.a[3] != cA ? q.a[3] : bsel; bsel = q.a[2] != cA ? q.a[2] : bsel; bsel = q.a[1] != cA ? q.a[1] : bsel; bsel = q.a[0] != cA ? q.a[0] : bsel;
        const int bsel_o = __shfl_xor_sync(0xffffffffu, bsel, 1);
        const int b_first = hh == 0 ? bsel : bsel_o, b_second = hh == 0 ? bsel_o : bsel;
        const int cB = b_first != cA ? b_first : b_second;
        const bool in2 = (q.a[0] == cA || q.a[0] == cB) && (q.a[1] == cA || q.a[1] == cB) && (q.a[2] == cA || q.a[2] == cB) && (q.a[3] == cA || q.a[3] == cB) &&
                         (q.b[0] == cA || q.b[0] == cB) && (q.b[1] == cA || q.b[1] == cB) && (q.b[2] == cA || q.b[2] == cB) && (q.b[3] == cA || q.b[3] == cB);
        const bool in2_o = __shfl_xor_sync(0xffffffffu, (int)in2, 1) != 0;
        if (hh == 0) {
            const unsigned m16 = m8 | (other << 8);
            sts128(sm + kRpDesc + w * 16, cA, (in2 && in2_o && cB != cA) ? cB : -1, m16, 0);
            sts32(sm + kRpWc + w * 4, cA);
            sts16(sm + kRpWm + w * 2, m16);
        }
        __syncwarp();

        const char *rows = reinterpret_cast<const char *>(table + (size_t)ce * ep_rows + (size_t)g * V);   // this lane's channel group of row 0
        asm volatile("" : "+l"(rows));      // opaque: keep the pointer in registers (the compiler re-derived it - 12 instructions - before every fetch)
        const float *counts_e = counts ? counts + (size_t)ce * n_cells : nullptr;
        auto fetch = [&](int cell) { return load_raw<V>(reinterpret_cast<const TableT *>(rows), counts_e, (size_t)cell, C, 0); };
        int cur_cell = -1, oth_cell = -1;
        Vec<V> cur = vzero<V>(), oth = vzero<V>();
        Vec<V> l1acc = vzero<V>();
        __half *l0_dst = L0 + (((size_t)ce * h0 + cqy * 2) * w0 + cqx * 2) * C + V * g;     // L0 pixel (2 qy, 2 qx): the other three are at + C, + w0 * C, + (w0 + 1) * C
        asm volatile("" : "+l"(l0_dst));
#pragma unroll 1
        for (int l0 = 0; l0 < 4; ++l0) {                   // L0 pixels of the quadrant, row-major
            // The four 4x4 windows of this L0 pixel.  A window whose 16 pixels hit ONE cell needs no additions: the
            // gathered value x is an fp16 number, so the sequential fp32 sum 0+x+x+...+x is exact at every step
            // (k*x, k <= 16, has at most 15 significant bits) and avg_pool2d(4) returns x itself - except that -0.0
            // becomes +0.0 (0 + -0 = +0), which the shortcuts reproduce by adding +0 (found by the read stress sweep).
            const uint4 wc4 = lds128(sm + kRpWc + l0 * 16);
            const uint2 wm2 = lds64(sm + kRpWm + l0 * 8);
            Vec<V> v0;
            if (wm2.x == 0x00010001 && wm2.y == 0x00010001 && wc4.x == wc4.y && wc4.x == wc4.z && wc4.x == wc4.w) {
                // whole 8x8 block in one cell: pool(4), pool(2) and the fp16 rounding all return the gathered value
                if ((int)wc4.x != cur_cell) cur = finish<V>(fetch((int)wc4.x));
                cur_cell = (int)wc4.x;
                v0 = vadd<V>(cur, vzero<V>());               // the reference's sums start from +0: a gathered -0.0 comes out as +0.0
            } else {
                Vec<V> s2 = vzero<V>();
                // NOT unrolled: the window body holds the 16 row variants of vadd_row2 and the generic run walk; four copies of it
                // (r2 v4a) ran slower than v3 despite fewer instructions - the warps of an SM sit in different windows and the
                // instruction cache could not hold the unrolled body.  One LDS.128 brings the window's descriptor.
                uint32_t dsc = sm + kRpDesc + l0 * 64;
#pragma unroll 1
                for (int win = 0; win < 4; ++win, dsc += 16) {   // 4x4 windows of the avg_pool2d(4) (timm.py:152), row-major
                    const uint4 d = lds128(dsc);
                    const int wc = (int)d.x, wb = (int)d.y;
                    unsigned rest = d.z & ~1u;        // run heads after the first pixel
                    if (wc != cur_cell) cur = finish<V>(fetch(wc));
                    cur_cell = wc;
                    Vec<V> s4;
                    if (rest == 0u) {
                        // one cell for the whole window: 16 * x is exact for an fp16-valued x, so the common tail below adds exactly x
                        // (one join point for s2: the separate `s2 += cur; continue` cost eight register moves per window)
                        s4 = vscale<V>(cur, 16.0f);
                    } else if (wb >= 0) {
                        s4 = vzero<V>();
                        // exactly two cells: cur = row of A (first pixel), oth = row of B
                        if (wb != oth_cell) oth = finish<V>(fetch(wb));
                        oth_cell = wb;
                        // bit p of bm: pixel p belongs to B = parity of the run heads in (0, p] (prefix xor over the 16-bit head mask)
                        unsigned bm = rest;
                        bm ^= bm << 1; bm ^= bm << 2; bm ^= bm << 4; bm ^= bm << 8;
                        bm &= 0xffffu;
                        if (bm == (bm & 15u) * 0x1111u) {
                            vadd_row2<V>(s4, cur, oth, bm, 4);      // all four rows alike
                        } else {
#pragma unroll 1
                            for (int r = 0; r < 4; ++r, bm >>= 4) vadd_row2<V>(s4, cur, oth, bm, 1);
                        }
                    } else {
                        s4 = vzero<V>();
                        // three or more cells in the window: 2-8 runs instead of 16 pixels; the walk pays the fetch / fp16->fp32
                        // conversion / bookkeeping per RUN and V/2 packed adds per pixel.  (A straight-line per-pixel walk with a
                        // head-bit test per pixel was tried in r2: the compiler if-converts it into predicated copies, 52.6 M
                        // instead of 40.0 M warp instructions per E=16 launch.)
                        const uint32_t cells = sm + kRpIdx + (uint32_t)(l0 * 4 + win) * 64;
                        int p = 0;
#pragma unroll 1
                        while (true) {
                            const int pn = rest ? (__ffs(rest) - 1) : 16;
                            rest &= rest - 1;
                            Raw raw;
                            int ncell = cur_cell;
                            if (pn < 16) {                   // next run's row in flight under the adds
                                ncell = (int)lds32(cells + pn * 4);
                                raw = fetch(ncell);
                            }
                            int len = pn - p;                // 1..15, warp-uniform; sequential fp32 sum: `len` times + cur
#pragma unroll 1
                            for (; len >= 4; len -= 4) { s4 = vadd<V>(s4, cur); s4 = vadd<V>(s4, cur); s4 = vadd<V>(s4, cur); s4 = vadd<V>(s4, cur); }
                            if (len & 2) { s4 = vadd<V>(s4, cur); s4 = vadd<V>(s4, cur); }
                            if (len & 1) s4 = vadd<V>(s4, cur);
                            if (pn >= 16) break;
                            cur = finish<V>(raw);
                            cur_cell = ncell;
                            p = pn;
                        }
                    }
                    s2 = vadd<V>(s2, vscale<V>(s4, 0.0625f));    // / 16 (exact)
                }
                v0 = vround_half<V>(vscale<V>(s2, 0.25f));      // avg_pool2d(2) -> half (timm.py:168, level 0)
            }
            vstore_half<V>(l0_dst + ((l0 >> 1) * w0 + (l0 & 1)) * C, v0);
            l1acc = vadd<V>(l1acc, v0);
        }
        const Vec<V> v1 = vround_half<V>(vscale<V>(l1acc, 0.25f));  // level 1
        vstore_half<V>(L1 + (((size_t)ce * h1 + cqy) * w1 + cqx) * C + V * g, v1);
        __syncwarp();                                       // the slices are rewritten by the next item
    }
}

// level 2 = avg_pool2d(level 1, 2) -> half (timm.py:168): the four L1 pixels in row-major order, fp32, then / 4
__global__ void __launch_bounds__(256) pool_level2_kernel(const __half *__restrict__ L1, int E, int h1, int w1, int C4, __half *__restrict__ L2)
{
    const int h2 = h1 / 2, w2 = w1 / 2;
    const int64_t total = (int64_t)E * h2 * w2 * C4, step = (int64_t)gridDim.x * blockDim.x;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += step) {
        const int g = (int)(i % C4);
        int64_t p = i / C4;
        const int x = (int)(p % w2); p /= w2;
        const int y = (int)(p % h2);
        const int e = (int)(p / h2);
        Vec<4> s = vzero<4>();
#pragma unroll
        for (int k = 0; k < 4; ++k)
            s = vadd<4>(s, finish<4>(load_raw<4>(L1, nullptr, ((size_t)e * h1 + 2 * y + (k >> 1)) * w1 + 2 * x + (k & 1), C4 * 4, g)));
        vstore_half<4>(L2 + (((size_t)e * h2 + y) * w2 + x) * C4 * 4 + 4 * g, vscale<4>(s, 0.25f));
    }
}


// Full-grid normalise (create_implicit_memory, custom_rcnn.py:764-774) for callers that want the table
// itself (the reference API returns it); the read kernel above never needs it.  Streaming, float4.
template <bool HALF_OUT>
__global__ void __launch_bounds__(256) normalize_kernel(const float4 *__restrict__ sums, const float *__restrict__ counts, int64_t n_rows, int C4,
                                                        float4 *__restrict__ out32, uint2 *__restrict__ out16)
{
    const int64_t total = n_rows * C4, stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += stride) {
        const int64_t row = i / C4;
        float4 v = __ldg(sums + i);
        const float n = __ldg(counts + row);
        if (n > 1.0f) { v.x = __fdiv_rn(v.x, n); v.y = __fdiv_rn(v.y, n); v.z = __fdiv_rn(v.z, n); v.w = __fdiv_rn(v.w, n); }
        if (HALF_OUT) {
            __half2 a = __floats2half2_rn(v.x, v.y), b = __floats2half2_rn(v.z, v.w);
            uint2 raw; raw.x = *reinterpret_cast<uint32_t *>(&a); raw.y = *reinterpret_cast<uint32_t *>(&b);
            out16[i] = raw;
        } else out32[i] = v;
    }
}

template <int C>
int launch(const void *table, int mem_is_f16, const float *counts, const void *idx, int idx_is_i64, int E, int H, int W,
           int64_t n_cells, void *L0, void *L1, void *L2, cudaStream_t st)
{
    const int64_t n_items = (int64_t)E * (H / 16) * (W / 16);      // C in {128, 256, 512}: one warp covers all channels of a quadrant (V = C / 32 per lane)
    EOD_REQUIRE(n_items < (1ll << 31) - (1ll << 24), EOD_ERR_BADARG, "eod_read_pool: too many quadrants for one launch");
    int64_t blocks = (n_items + kReadWarps - 1) / kReadWarps;
    static const int cap_env = [] { const char *v = getenv("EOD_READ_CTAS_PER_SM"); const int k = v ? atoi(v) : 16; return k > 0 ? k : 16; }();   // tuning knob
    const int64_t cap = (int64_t)eod_num_sms() * cap_env;        // default 16: 3-4 resident CTAs per SM, a few waves: each warp walks several items with prefetch
    if (blocks > cap) blocks = cap;
    dim3 grid((unsigned)blocks), block(kReadWarps * 32);
    __half *l0 = (__half *)L0, *l1 = (__half *)L1, *l2 = (__half *)L2;
    if (mem_is_f16) {
        if (idx_is_i64) read_pool_kernel<C, __half, int64_t><<<grid, block, 0, st>>>((const __half *)table, nullptr, (const int64_t *)idx, H, W, n_cells, E, l0, l1);
        else read_pool_kernel<C, __half, int32_t><<<grid, block, 0, st>>>((const __half *)table, nullptr, (const int32_t *)idx, H, W, n_cells, E, l0, l1);
    } else {
        if (idx_is_i64) read_pool_kernel<C, float, int64_t><<<grid, block, 0, st>>>((const float *)table, counts, (const int64_t *)idx, H, W, n_cells, E, l0, l1);
        else read_pool_kernel<C, float, int32_t><<<grid, block, 0, st>>>((const float *)table, counts, (const int32_t *)idx, H, W, n_cells, E, l0, l1);
    }
    int rc = eod_check_launch("eod_read_pool");
    if (rc) return rc;
    const int64_t total = (int64_t)E * (H / 32) * (W / 32) * (C / 4);
    int64_t b2 = (total + 255) / 256;
    if (b2 > (int64_t)eod_num_sms() * 8) b2 = (int64_t)eod_num_sms() * 8;
    pool_level2_kernel<<<(unsigned)b2, 256, 0, st>>>(l1, E, H / 16, W / 16, C / 4, l2);
    return eod_check_launch("eod_read_pool[level 2]");
}

}  // namespace

extern "C" int eod_read_pool(const void *table, int mem_is_f16, const float *counts, const void *idx, int idx_is_i64,
                             int n_episodes, int C, int H, int W, int64_t n_cells, void *L0, void *L1, void *L2,
                             eod_stream_t stream)
{
    EOD_REQUIRE(table && idx && L0 && L1 && L2, EOD_ERR_BADARG, "eod_read_pool: null pointer");
    EOD_REQUIRE(n_episodes > 0 && n_episodes <= 65535 && n_cells > 0, EOD_ERR_BADARG, "eod_read_pool: bad sizes");
    EOD_REQUIRE(H > 0 && W > 0 && H % 32 == 0 && W % 32 == 0, EOD_ERR_BADARG, "eod_read_pool: H and W must be multiples of 32 (got %dx%d)", H, W);
    EOD_REQUIRE(H / 32 <= 65535, EOD_ERR_BADARG, "eod_read_pool: H too large");
    EOD_REQUIRE(eod_aligned16(table) && eod_aligned16(idx) && eod_aligned16(L0) && eod_aligned16(L1) && eod_aligned16(L2),
                EOD_ERR_ALIGN, "eod_read_pool: pointers must be 16-byte aligned");
    cudaStream_t st = (cudaStream_t)stream;
    switch (C) {
    case 128: return launch<128>(table, mem_is_f16, counts, idx, idx_is_i64, n_episodes, H, W, n_cells, L0, L1, L2, st);
    case 256: return launch<256>(table, mem_is_f16, counts, idx, idx_is_i64, n_episodes, H, W, n_cells, L0, L1, L2, st);
    case 512: return launch<512>(table, mem_is_f16, counts, idx, idx_is_i64, n_episodes, H, W, n_cells, L0, L1, L2, st);
    default:
        eod_set_error("eod_read_pool: C=%d not compiled in (128, 256, 512)", C);
        return EOD_ERR_UNSUPPORTED;
    }
}

extern "C" int eod_normalize_memory(const float *sums, const float *counts, int64_t n_rows, int C, void *out, int out_is_f16,
                                    eod_stream_t stream)
{
    EOD_REQUIRE(sums && counts && out, EOD_ERR_BADARG, "eod_normalize_memory: null pointer");
    EOD_REQUIRE(n_rows > 0 && C > 0 && C % 4 == 0, EOD_ERR_BADARG, "eod_normalize_memory: bad sizes (C %% 4 == 0)");
    EOD_REQUIRE(eod_aligned16(sums) && eod_aligned16(out), EOD_ERR_ALIGN, "eod_normalize_memory: pointers must be 16-byte aligned");
    const int64_t total = n_rows * (C / 4);
    int64_t blocks = (total + 255) / 256;
    const int64_t cap = (int64_t)eod_num_sms() * 16;
    if (blocks > cap) blocks = cap;
    if (out_is_f16) normalize_kernel<true><<<(int)blocks, 256, 0, (cudaStream_t)stream>>>((const float4 *)sums, counts, n_rows, C / 4, nullptr, (uint2 *)out);
    else normalize_kernel<false><<<(int)blocks, 256, 0, (cudaStream_t)stream>>>((const float4 *)sums, counts, n_rows, C / 4, (float4 *)out, nullptr);
    return eod_check_launch("eod_normalize_memory");
}
