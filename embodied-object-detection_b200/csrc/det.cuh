// Deterministic write (EOD_WRITE_DET), the part every layout shares: a run of equal cell id over a 32-pixel tile is the unit of
// the segmented reduce, and a write is three host-side pieces -
//
//   det_prepass   carve the caller's workspace, then det_tile_runs -> det_scan_tiles -> det_cell_runs -> det_scan_list
//   main pass     the layout's own kernel: for every run that holds a sampled pixel, in the tile's raster order r = 0, 1, ...,
//                 partials[tile_off[tile] + r] = the run's value sum (from +0, sampled pixels in raster order) and run_cell = cell;
//                 a run at or past cap adds sum / n_cell into sums with reductions and sets *status = 1
//   det_reduce    det_claim -> det_reduce -> det_chunk -> det_final: every cell adds its runs' partials in run order, divides by
//                 n_cell and adds the mean ONCE to sums[cell]
//
// The pre-passes and the reduce live in write_mean.cu; the dense write (write_mean.cu) and the object write (write_objects.cu)
// bring a main pass each.  Both main passes must find the runs of det_tile_masks / det_run_mask in the same order as the pre-passes:
// a run's rank is its row in partials.
#pragma once

#include "eod_common.cuh"

namespace {

constexpr int TILE_PX = 32;

// a main pass's view of the workspace: a run's (unscaled) sums are STORED to partials[tile_off[tile] + r] (raster run order, no
// atomics) for the segmented reduce of det_reduce_kernel; runs beyond the workspace capacity fall back to reductions and raise *status.
struct DetArgs {
    const int32_t *tile_off;     // (E, tiles) exclusive scan of the per-tile run counts, restarting per episode
    float *partials;             // (E, cap, C)
    int32_t *run_cell;           // (E, cap)
    int32_t *status;             // set to 1 when a run did not fit
    int cap;                     // runs per episode the workspace holds
};

// The sampled pixels (bit p = pixel p of a 32-pixel tile) of the deterministic run that starts at head p0; `later` holds the heads
// after p0 only.  The run pre-passes (det_run_sampled) and every main pass must find the same runs in the same order: a run's
// rank among them is its slot in partials.
__device__ __forceinline__ unsigned det_run_mask(unsigned later, unsigned samps, int p0)
{
    const int p1 = later ? (__ffs(later) - 1) : TILE_PX;
    return samps & (0xffffffffu >> (32 - p1)) & (0xffffffffu << p0);
}

// lane p of a warp looks at pixel g0 + p of a tile: its cell, the tile's run heads (bit p: a run starts at p) and sampled pixels
__device__ __forceinline__ void det_tile_masks(const int32_t *idx, const uint8_t *samp, size_t g0, unsigned lane, int &cell, unsigned &heads,
                                               unsigned &samps)
{
    cell = __ldg(idx + g0 + lane);
    const int prev = __shfl_up_sync(0xffffffffu, cell, 1);
    heads = __ballot_sync(0xffffffffu, lane == 0 || prev != cell);
    samps = samp ? __ballot_sync(0xffffffffu, __ldg(samp + g0 + lane) != 0) : 0xffffffffu;
}

}  // namespace

// The caller's workspace carved for one call (det_prepass fills it).  cell_runs is all-zero between calls.
struct DetWorkspace {
    int32_t *tile_off, *n_runs, *n_list, *status, *cell_runs, *cell_off, *run_cell, *seg, *cell_list, *list_off;
    float *partials;
    // long segments (> 256 runs): sorted positions, chunk tasks and chunk sums (det_reduce_kernel -> det_chunk -> det_final)
    int32_t *seg2, *task_start, *task_len, *long_i, *long_base, *chunk_rows, *n_long;
    float *cparts;
    int rows;
    int cap;                     // runs per episode the workspace holds
};

// Checks the shape (HW % 32 == 0, 16-byte aligned samp: EOD_ERR_UNSUPPORTED) and the workspace (EOD_ERR_BADARG), carves the workspace
// into *w and launches the four run pre-passes.  active (E) i32 nullable: slots with active[e] <= 0 get no runs.  `what` names the
// entry point in error messages.
int det_prepass(const char *what, const int32_t *idx, const uint8_t *samp, const int32_t *active, int E, int C, int HW, int64_t n_cells,
                void *ws, size_t ws_bytes, DetWorkspace *w, cudaStream_t st);

// The segmented reduce of the partials a main pass stored: sums[cell] += (sum of the cell's runs in run order) / n_cell.
int det_reduce(const char *what, const DetWorkspace &w, int C, int E, int64_t n_cells, const uint32_t *frame_cnt, float *sums, cudaStream_t st);

static inline DetArgs det_args(const DetWorkspace &w) { return DetArgs{w.tile_off, w.partials, w.run_cell, w.status, w.cap}; }
