/*
 * eod_memory.h - C ABI of the B200-native spatial feature memory (libeod_memory.so).
 *
 * This is the drop-in boundary for ONE path of nhcha6/embodied-object-detection: back-project ->
 * memory write -> memory read -> fusion.  The reference has no FFI for this path today: it is a chain
 * of torch ops inside two Python classes.  Each entry point below names the reference lines it
 * replaces (paths relative to <reference>/Detic); INTEGRATION.md shows the ctypes stub a maintainer
 * adds on the reference side.
 *
 * Conventions
 *   - every pointer is a DEVICE pointer owned by the caller (torch allocates); the library allocates no
 *     persistent memory and keeps no global state apart from a thread-local error string;
 *   - all work is enqueued on `stream` (a cudaStream_t passed as void*); calls are asynchronous and
 *     thread-safe for distinct streams;
 *   - return value: EOD_OK or a negative EOD_ERR_*; eod_last_error() describes the last failure of the
 *     calling thread;
 *   - leading dimension E = number of independent episodes processed by one launch ("batch x64");
 *     tensors of different episodes are E-contiguous: element (e, i) lives at base + e*stride + i;
 *   - grid state of one episode: sums (cells, C) fp32 row = cell, counts (cells) fp32 (integer valued),
 *     frame_cnt (cells) u32 scratch that is all-zero between frames;
 *   - cell indices are int32 (cells < 2^31); int64 indices of the reference API are accepted where
 *     stated (idx_is_i64).
 */
#ifndef EOD_MEMORY_H
#define EOD_MEMORY_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define EOD_OK 0
#define EOD_ERR_BADARG (-1)      /* null pointer / non-positive size / unsupported enum            */
#define EOD_ERR_ALIGN (-2)       /* pointer or row stride not 16-byte aligned                       */
#define EOD_ERR_LAUNCH (-3)      /* CUDA launch / driver error (message in eod_last_error)          */
#define EOD_ERR_UNSUPPORTED (-4) /* shape not compiled in (C must be one of 128, 256, 512)          */

#define EOD_ORDER_ZX 0 /* flat = q_z * map_w + q_x   SMNet/build_memory_data.py:143 */
#define EOD_ORDER_XZ 1 /* flat = q_x * map_h + q_z   robot_demo.py:533               */

#define EOD_LAYOUT_CHW 0 /* features (E, C, H*W): the reference's image_features, custom_rcnn.py:886 */
#define EOD_LAYOUT_HWC 1 /* features (E, H*W, C): channels-last                                         */
#define EOD_LAYOUT_HWC_BF16 2 /* channels-last bf16 features (a bf16 backbone's output): widened exactly, summed in fp32 */
#define EOD_LAYOUT_HWC_F16 3  /* channels-last fp16 features                                                             */
#define EOD_LAYOUT_CHW_BF16 4 /* (E, C, H*W) bf16 features (what a bf16 / autocast backbone emits in NCHW): widened exactly  */
#define EOD_LAYOUT_CHW_F16 5  /* (E, C, H*W) fp16 features                                                                 */

#define EOD_FUSE_SUM 0        /* res + w*mem   timm.py:181-182 */
#define EOD_FUSE_MEM_ONLY 1   /* w*mem         timm.py:183-184 */
#define EOD_FUSE_IMAGE_ONLY 2 /* res           timm.py:185-186 */

#define EOD_WRITE_AUTO 0 /* TMA-staged kernel when the shape allows it, else LDG-staged */
#define EOD_WRITE_LDG 1  /* force the LDG-staged kernel                                  */
#define EOD_WRITE_TMA 2  /* force the TMA-staged kernel (error if shape unsupported)     */
#define EOD_WRITE_TMA_DRY 3 /* profiling only: stream the tiles, no accumulation (no result) */
#define EOD_WRITE_DET 4  /* host-side selector of eod_write_mean_det (deterministic segmented reduce)   */

typedef void *eod_stream_t;

int eod_version(void);
const char *eod_last_error(void);

/* ---------------------------------------------------------------------------------------------------
 * (1) Geometry.  Replaces SMNet/projector/core.py:107-175,220 (pixel_to_world_mapping),
 * core.py:227-271 (discretize_point_cloud), projector.py:88-101, SMNet/build_memory_data.py:135-143,
 * robot_demo.py:526-533.
 *   depth  (E,H,W) f32 metres (0 = no depth)      pose (E,12) rows 0..2 of the 4x4 camera-to-world T
 *   shifts (E,6): world_shift_origin xyz, map_world_shift xyz
 *   intrinsics fx,fy,cx,cy are the fp32 values of core.py:68-77 (host computes them; the kernel does not)
 * Outputs, each nullable: idx (E,H,W) clipped flat cell index; q2 (E,H,W,2) unclipped (x,z);
 * outlier (E,H,W) u8; height (E,H,W) world y; world (E,H,W,3) xyz after world_shift_origin only.
 * Bit-exact with torch-CPU execution of the cited lines (FMA-chain bmm, IEEE divide, round-half-even).
 */
int eod_backproject_quantize(const float *depth, const float *pose, const float *shifts, int n_episodes, int H,
                             int W, float fx, float fy, float cx, float cy, float cell, int map_w, int map_h,
                             int order, float z_clip, int32_t *idx, int32_t *q2, uint8_t *outlier, float *height,
                             float *world, eod_stream_t stream);

/* Same launch on RAW sensor depth: uint16 sensor units divided by depth_div (1000 for millimetres) exactly as
 * robot_demo.py:515-517 does it on the host (numpy true division in fp64, then torch.FloatTensor rounds to fp32), so the
 * online robot path uploads 2 bytes per pixel and no host-side conversion remains.  Bit-exact with the float entry point
 * fed `FloatTensor(depth_u16 / depth_div)`. */
int eod_backproject_quantize_u16(const uint16_t *depth, double depth_div, const float *pose, const float *shifts, int n_episodes,
                                 int H, int W, float fx, float fy, float cx, float cy, float cell, int map_w, int map_h,
                                 int order, float z_clip, int32_t *idx, int32_t *q2, uint8_t *outlier, float *height,
                                 float *world, eod_stream_t stream);

/* eod_backproject_quantize (idx only) and eod_frame_count without a sample mask in ONE launch: the dense frame-step's per-cell pixel
 * counts are taken while the cell ids are still in registers (one integer atomic per run of equal id over 128 consecutive pixels)
 * instead of in a second pass over the index plane.  depth: f32 metres, or uint16 sensor words / depth_div (depth_is_u16);
 * active (E) nullable: episodes with active <= 0 get their idx but are not counted; frame_cnt (E, map_w*map_h) u32 accumulates.
 * Needs W % 4 == 0, H*W % 128 == 0 and 16-byte aligned planes, else EOD_ERR_UNSUPPORTED (then call the two entry points). */
int eod_backproject_count(const void *depth, int depth_is_u16, double depth_div, const float *pose, const float *shifts, int n_episodes,
                          int H, int W, float fx, float fy, float cx, float cy, float cell, int map_w, int map_h, int order,
                          const int32_t *active, int32_t *idx, uint32_t *frame_cnt, eod_stream_t stream);

/* Offline builder's quantise step on STORED world coordinates (sensor_data/<name>.h5 'projection_indices'):
 * SMNet/build_memory_data.py:135-143.  world (n_points,3) f32 -> idx (n_points) i32, clipped, bit-exact. */
int eod_quantize_world(const float *world, int64_t n_points, float shift_x, float shift_z, float cell, int map_w, int map_h,
                       int order, int32_t *idx, eod_stream_t stream);

/* ---------------------------------------------------------------------------------------------------
 * (2) Write, mean mode.
 */

/* Raster-order "every stride-th observed pixel" selection, custom_rcnn.py:905-914.
 * observed (E,HW) u8 -> samp (E,HW) u8 (1 = pixel is sampled).  n_sampled (E) i32 nullable. */
int eod_sample_mask(const uint8_t *observed, int n_episodes, int HW, int stride, uint8_t *samp, int32_t *n_sampled,
                    eod_stream_t stream);

/* Per-frame pre-pass: frame_cnt[cell] += #sampled pixels of the cell; bit 31 marks cells that are
 * visible but have no sampled pixel (torch.unique(proj_indices), custom_rcnn.py:699).  samp nullable
 * (= every pixel sampled).  active (E) i32 nullable: episodes with active[e] <= 0 are skipped altogether
 * (a frame without kept detections writes nothing, not even visibility: custom_rcnn.py:686,872-873).
 * frame_cnt must be zero on entry.
 * Slot table (all nullable together; used by eod_write_objects): the first sample of a cell claims the next
 * free slot of its episode: slot_of_cell (E,cells) i32 := slot + 1, slot_cell (E,n_slots_max) i32 := cell,
 * n_slots (E) i32 += 1.  slot_of_cell and n_slots must be zero on entry (eod_flush_slots leaves them so). */
int eod_frame_count(const int32_t *idx, const uint8_t *samp, const int32_t *active, int n_episodes, int HW,
                    int64_t n_cells, uint32_t *frame_cnt, int32_t *slot_of_cell, int32_t *slot_cell, int32_t *n_slots,
                    int n_slots_max, eod_stream_t stream);

/* Optional companion of the pre-pass: pix_inv_n[p] = 1 / frame_cnt[idx[p]] (sample count of p's cell, IEEE
 * reciprocal; 0 where the cell has no sample), (E,HW) f32.  Given to eod_write_mean, the scale of a run of
 * pixels travels with the feature tile instead of being a dependent global load per run. */
int eod_expand_counts(const int32_t *idx, const uint32_t *frame_cnt, int n_episodes, int HW, int64_t n_cells,
                      float *pix_inv_n, eod_stream_t stream);

/* Main pass: sums[cell] += (sum of the sampled pixels' feature vectors) / n_cell, i.e. the per-cell mean
 * of custom_rcnn.py:917-934 accumulated as in :696-697,742.  Warp-aggregated fp32 reductions
 * (red.global.add.f32, one per run of equal cell id and channel): run-to-run results agree to ~1e-7 of
 * scale, not bitwise.  pix_inv_n: nullable, output of eod_expand_counts for this frame.
 * feat is fp32 for EOD_LAYOUT_CHW / _HWC and bf16 / fp16 for EOD_LAYOUT_HWC_BF16 / _HWC_F16 / _CHW_BF16 / _CHW_F16 (half the
 * bytes of the dominant stream: the 16-bit values are widened exactly and everything downstream is the fp32 arithmetic of the fp32
 * layouts).  16-bit CHW rows must be 16-byte aligned (HW % 8 == 0, else EOD_ERR_ALIGN); their TMA kernel takes 64-pixel tiles
 * (HW % 64 == 0 and a 16-byte aligned samp, else the LDG kernel - or EOD_ERR_UNSUPPORTED for EOD_WRITE_TMA / _TMA_DRY);
 * pix_inv_n with a 16-bit CHW layout is EOD_ERR_UNSUPPORTED.  eod_write_mean_det_layout takes every layout but the 16-bit CHW ones.
 * active (E) i32 nullable: the same mask eod_frame_count takes - slots of the lock-step batch with active[e] <= 0 (an episode
 * that has ended, custom_rcnn.py:441-443 iterates ragged sequences) are skipped without reading their features. */
int eod_write_mean(const void *feat, int layout, const int32_t *idx, const uint8_t *samp, const uint32_t *frame_cnt,
                   int n_episodes, int C, int HW, int64_t n_cells, float *sums, int variant, const float *pix_inv_n,
                   const int32_t *active, eod_stream_t stream);

/* Deterministic variant of the main pass (HW %% 32 == 0): run sums are stored in raster run order
 * (no atomics), then every touched cell adds the partial sums of its runs in ascending run position, divides by
 * n_cell and adds the mean ONCE to sums[cell] - bitwise reproducible run to run and independent of how episodes are
 * batched, and the arithmetic shape of custom_rcnn.py:930-934,742 (sum, divide, add).
 * layout: EOD_LAYOUT_CHW, _HWC, _HWC_BF16 or _HWC_F16 (EOD_LAYOUT_CHW_BF16 / _F16: EOD_ERR_UNSUPPORTED).  Every layout sums a run's
 * sampled pixels in raster order from +0 with 16-bit values widened exactly, so the result does not depend on the layout: channels-last
 * x gives the bits of CHW x, bf16 / fp16 x those of CHW fp32 x.float().
 * active (E) i32 nullable: the mask eod_frame_count took - slots with active[e] <= 0 get no runs, their features are not read and
 * their sums are left alone.  eod_write_mean_det is eod_write_mean_det_layout with EOD_LAYOUT_CHW and no mask.
 * workspace: caller-owned, 256-byte aligned, zero-filled ONCE before first use (the library leaves its persistent
 * planes zero again after every call); eod_write_mean_det_workspace_bytes(E, C, HW, cells, runs_per_episode) sizes
 * it for runs_per_episode runs of equal cell id per episode and frame (<= 0: HW/4).  Runs that do not fit fall back
 * to the fp32 reductions of eod_write_mean (still correct) and set the int32 at byte offset
 * eod_write_mean_det_status_offset(E, cells) of the workspace to 1. */
int64_t eod_write_mean_det_workspace_bytes(int n_episodes, int C, int HW, int64_t n_cells, int runs_per_episode);
int64_t eod_write_mean_det_status_offset(int n_episodes, int64_t n_cells);
int eod_write_mean_det(const float *feat, const int32_t *idx, const uint8_t *samp, const uint32_t *frame_cnt, int n_episodes,
                       int C, int HW, int64_t n_cells, float *sums, void *workspace, int64_t workspace_bytes,
                       eod_stream_t stream);
int eod_write_mean_det_layout(const void *feat, int layout, const int32_t *idx, const uint8_t *samp, const uint32_t *frame_cnt,
                              const int32_t *active, int n_episodes, int C, int HW, int64_t n_cells, float *sums, void *workspace,
                              int64_t workspace_bytes, eod_stream_t stream);

/* Post-pass: counts[cell] += 1 for every visible cell (custom_rcnn.py:699-701,743) and frame_cnt := 0.
 * touched (E,cells) u8 nullable: |= 1 where the cell received samples this frame (observed_mem, :922).
 * norm16 (E,cells,C) f16 nullable: when given (with sums, C), the normalised fp16 row of every visible cell
 * is refreshed, norm16[cell] = half(sums[cell] / counts[cell] if counts[cell] > 1 else sums[cell])
 * (custom_rcnn.py:764-774,1036), so eod_read_pool can gather from an always-current fp16 table. */
int eod_finalize_counts(const int32_t *idx, int n_episodes, int HW, int64_t n_cells, uint32_t *frame_cnt,
                        float *counts, uint8_t *touched, const float *sums, void *norm16, int C,
                        eod_stream_t stream);

/* Per-pixel mean of the kept objects' features, custom_rcnn.py:884-901 (objects added in index order,
 * then / count): box_features (K,C) f32, masks (K,HW) u8 -> image_features (C,HW) f32 (zeros where
 * unobserved), observed (HW) u8.  Bit-exact (same fp32 add order). */
int eod_box_to_image_features(const float *box_features, const uint8_t *masks, int K, int C, int HW,
                              float *image_features, uint8_t *observed, eod_stream_t stream);

/* Fused object-regime write (custom_rcnn.py:884-936 without the (C,H,W) image): observed[p] = any_k masks[k][p].
 * masks (E,Kmax,HW) u8, n_obj (E) i32 nullable (= Kmax objects everywhere) -> observed (E,HW) u8.  HW %% 4 == 0. */
int eod_masks_observed(const uint8_t *masks, const int32_t *n_obj, int n_episodes, int Kmax, int HW, uint8_t *observed,
                       eod_stream_t stream);

/* For every sampled pixel (samp from eod_sample_mask(observed, 8); slots from eod_frame_count):
 *   g = (sum over the objects covering the pixel, ascending index, of box_features[k]) / #objects   - bit-identical
 *       to the value eod_box_to_image_features / custom_rcnn.py:890-899 stores for that pixel;
 *   scratch[slot(cell)] += g.
 * box_features (E,Kmax,C) f32, masks (E,Kmax,HW) u8, scratch (E,n_slots_max,C) f32 zero on entry;
 * n_slots_max >= number of sampled pixels per episode (HW/stride rounded up is always enough). */
int eod_write_objects(const float *box_features, const uint8_t *masks, const int32_t *n_obj, int Kmax, const int32_t *idx,
                      const uint8_t *samp, const int32_t *slot_of_cell, int n_episodes, int C, int HW, int64_t n_cells,
                      int n_slots_max, float *scratch, eod_stream_t stream);

/* Mask pasting, detectron2 layers/mask_ops.py paste_masks_in_image as called at custom_rcnn.py:880 (threshold 0.5):
 * mask_probs (E,Kmax,S,S) f32 (the mask head's probabilities, S = 28), boxes (E,Kmax,4) f32 XYXY in image pixels ->
 * masks (E,Kmax,H*W) u8 (nullable; planes of objects >= n_obj[e] are all zero) and / or observed (E,H*W) u8 = OR over
 * the episode's objects (nullable; what eod_masks_observed would return for the pasted masks).  Per object the CPU
 * code path of the reference's dependency is followed: only pixels of [max(floor(x0)-1,0), min(ceil(x1)+1,W)) x (same
 * in y) are sampled, pixel centre -> box-normalised coordinate -> F.grid_sample(bilinear, zero padding,
 * align_corners=False) -> value >= threshold, in the fp32 operation order of ATen's vectorised CPU sampler.
 * Bit-exact with torch-CPU on the pasted bools.  The reference calls the function on CUDA tensors, where the dependency
 * samples the WHOLE image (skip_empty=False); for probabilities <= 1 and threshold >= 0.5 (the reference's 0.5) the value
 * outside the integer neighbourhood is below the threshold and both paths give the same bools.  For 0 <= threshold < 0.5 they
 * differ up to extent/(2S) pixels outside the box, and this library then samples the whole image like the CUDA path.
 * threshold must be >= 0 (negative = detectron2's uint8 soft masks: EOD_ERR_UNSUPPORTED). */
int eod_paste_masks(const float *mask_probs, const float *boxes, const int32_t *n_obj, int n_episodes, int Kmax, int S, int H,
                    int W, float threshold, uint8_t *masks, uint8_t *observed, eod_stream_t stream);

/* eod_write_objects with the pasted-mask test evaluated on the fly for the sampled pixels (samp from
 * eod_sample_mask(observed of eod_paste_masks)): the (K,H,W) masks are never built.  Same result, bit for bit, as
 * eod_paste_masks followed by eod_write_objects. */
int eod_write_objects_pasted(const float *box_features, const float *mask_probs, const float *boxes, const int32_t *n_obj,
                             int Kmax, int S, int H, int W, float threshold, const int32_t *idx, const uint8_t *samp,
                             const int32_t *slot_of_cell, int n_episodes, int C, int64_t n_cells, int n_slots_max,
                             float *scratch, eod_stream_t stream);

/* Deterministic object-regime write (custom_rcnn.py:903-934 accumulated as in :696-697,742): eod_write_objects /
 * eod_write_objects_pasted, then the per-cell mean added to sums, bitwise reproducible run to run and independent of how episodes
 * are batched (HW %% 32 == 0, 16-byte aligned samp, else EOD_ERR_UNSUPPORTED).  The result is, bit for bit, what
 * eod_write_mean_det_layout(EOD_LAYOUT_CHW) gives for the (C,HW) image eod_box_to_image_features builds from the same objects
 * (the pasted masks for the _pasted entry), with the same samp, frame_cnt and active = n_obj - without building that image.
 * frame_cnt: from eod_frame_count WITHOUT the slot table, with n_obj as its active mask: a slot with n_obj[e] <= 0 gets no runs,
 * its inputs are not read and its sums are left alone.  Any Kmax; box_features and sums 16-byte aligned.
 * workspace: the workspace of eod_write_mean_det - the same eod_write_mean_det_workspace_bytes sizing, zero-filled once, one
 * workspace may serve both writes; runs that do not fit fall back to fp32 reductions and set the int32 at byte offset
 * eod_write_mean_det_status_offset(E, cells) to 1. */
int eod_write_objects_det(const float *box_features, const uint8_t *masks, const int32_t *n_obj, int Kmax, const int32_t *idx,
                          const uint8_t *samp, const uint32_t *frame_cnt, int n_episodes, int C, int HW, int64_t n_cells, float *sums,
                          void *workspace, int64_t workspace_bytes, eod_stream_t stream);
int eod_write_objects_pasted_det(const float *box_features, const float *mask_probs, const float *boxes, const int32_t *n_obj,
                                 int Kmax, int S, int H, int W, float threshold, const int32_t *idx, const uint8_t *samp,
                                 const uint32_t *frame_cnt, int n_episodes, int C, int64_t n_cells, float *sums, void *workspace,
                                 int64_t workspace_bytes, eod_stream_t stream);

/* sums[cell] += scratch[slot] / n_cell for every claimed slot (the per-cell mean of custom_rcnn.py:931-934 added
 * once, :696-697,742); scratch rows, slot_of_cell entries and n_slots return to zero.  Run before
 * eod_finalize_counts (which clears frame_cnt). */
int eod_flush_slots(const uint32_t *frame_cnt, int32_t *slot_of_cell, const int32_t *slot_cell, int32_t *n_slots, int n_episodes,
                    int C, int64_t n_cells, int n_slots_max, float *scratch, float *sums, eod_stream_t stream);

/* Front end of the dense backbone-feature write (SURVEY 8a row A7'', bytecode-only CustomMapFPN.forward):
 * out = F.interpolate(src, (H_out, W_out), mode='bilinear', align_corners=True)[:, :, ::step, ::step] without building the
 * upsampled tensor.  src (E,C,h,w) f32 -> out (E,C,ceil(H_out/step),ceil(W_out/step)) f32; bit-exact with ATen CPU.
 * The samples then go through eod_frame_count / eod_write_mean with idx = proj_indices[::step, ::step] into a ZEROED
 * table (the reference replaces the memory: memory[observed_mem] = per-cell mean). */
int eod_bilinear_lattice(const float *src, int n_episodes, int C, int h, int w, int H_out, int W_out, int step, float *out,
                         eod_stream_t stream);

/* ---------------------------------------------------------------------------------------------------
 * (2b) Write, SMNet height-max mode (bytecode-only SMNet.encode, SURVEY 8a row A7').
 * Per frame: for inlier pixels (outlier == 0) on the [::pix_stride, ::pix_stride] lattice,
 * height_map[cell] = max(height_map[cell], height + 1000) with the canonical tie rule (highest raster
 * index wins; an equal later value replaces).  arg_pix (E,cells) i32: winning raster pixel index or -1;
 * observed (E,cells) u8 |= raised; state (E,cells,C) f32: raised cells := the winner's feature vector
 * ('replace' update).  key64 (E,cells) u64 scratch, all-zero between frames.  feat nullable (then state
 * is not touched). */
int eod_write_max(const float *height, const int32_t *idx, const uint8_t *outlier, const float *feat, int layout,
                  int n_episodes, int C, int H, int W, int pix_stride, int64_t n_cells, float *height_map,
                  uint64_t *key64, int32_t *arg_pix, uint8_t *observed, float *state, eod_stream_t stream);

/* 'replace' update of the SMNet encoder (SMNet/__pycache__/model.cpython-310.pyc, bytecode listing smnet_encode_model_py310.txt src
 * lines 104-128: tmp_memory = feature[proj_index[m]]; state[m] = linlayer(tmp_memory)): the raised cells of eod_write_max as a
 * compact list - src_off[i] = element offset of the winner pixel's feature vector inside feat (E,H,W,C) [HWC: channels contiguous]
 * or (E,C,H,W) [CHW: channel stride H*W], dst_row[i] = e * n_cells + cell - in arbitrary order; count[0] (device int32) = number of
 * winners.  capacity = entries src_off / dst_row can hold (winners beyond it are counted but not listed). */
int eod_max_winner_list(const int32_t *arg_pix, int n_episodes, int64_t n_cells, int H, int W, int C, int layout, int64_t *src_off,
                        int64_t *dst_row, int32_t *count, int capacity, eod_stream_t stream);

/* Lock-step height-max regime: the contest and rule of eod_write_max (same key, same '>=' update, same results bit for bit)
 * without the per-pixel idx / outlier / height planes, the arg_pix plane or its memset, and without a scan over the cells.
 * Per frame: one contest entry point, then eod_heightmax_update.  Scratch, all-zero between frames (the update leaves it so):
 *   key64 (E,cells) u64; n_list (E,2) i32 [listed cells, internal ticket]; cell_list (E,list_cap) i32 with
 *   list_cap >= min(cells, lattice pixels) (else EOD_ERR_BADARG): the cells the frame touched, one entry each, in arbitrary order.
 * raised (1) i32 device: set to 0 by the contest, = number of cells the update raised (all episodes) after it.
 * active (E) i32 nullable: episodes with active <= 0 read nothing and list nothing (their state is left alone).
 *
 * Contest from DEPTH: geometry of eod_backproject_quantize (same device functions, bit-exact) computed in registers for the
 * [::pix_stride, ::pix_stride] lattice; depth f32 metres or uint16 / depth_div (depth_is_u16); cells = map_w * map_h. */
int eod_heightmax_contest_depth(const void *depth, int depth_is_u16, double depth_div, const float *pose, const float *shifts,
                                int n_episodes, int H, int W, float fx, float fy, float cx, float cy, float cell, int map_w, int map_h,
                                int order, float z_clip, int pix_stride, const int32_t *active, uint64_t *key64, int32_t *cell_list,
                                int64_t list_cap, int32_t *n_list, int32_t *raised, eod_stream_t stream);
/* Contest from PLANES: height (E,H,W) f32 world height, idx (E,H,W) i32 cell ids in [0, n_cells), outlier (E,H,W) u8 nullable -
 * what create_coco_mp3d.py:157-165 stores, and what eod_write_max takes. */
int eod_heightmax_contest_planes(const float *height, const int32_t *idx, const uint8_t *outlier, int n_episodes, int H, int W,
                                 int pix_stride, int64_t n_cells, const int32_t *active, uint64_t *key64, int32_t *cell_list,
                                 int64_t list_cap, int32_t *n_list, int32_t *raised, eod_stream_t stream);
/* Update of the listed cells: height_map (E,cells) f32 and observed (E,cells) u8 of every raised cell, then either
 *   copy:    state (E,cells,C) f32 row := the winner pixel's feature row; feat (E,C,H,W) [CHW] or (E,H,W,C) [HWC] in fp32
 *            (EOD_LAYOUT_CHW / _HWC) or bf16 / fp16 (EOD_LAYOUT_*_BF16 / _F16, widened exactly: the state of feat.float());
 *            C %% 4 == 0, feat and state 16-byte aligned (EOD_ERR_ALIGN);
 *   replace: (src_off != NULL, state ignored) the compact winner list of eod_max_winner_list - src_off[i] element offset of the
 *            winner's fp32 feature vector, dst_row[i] = e * cells + cell, count = raised - for eod_linear_rows (fp32 layouts only,
 *            else EOD_ERR_UNSUPPORTED); win_cap entries. */
int eod_heightmax_update(const void *feat, int layout, int n_episodes, int C, int H, int W, int64_t n_cells, const int32_t *cell_list,
                         int64_t list_cap, int32_t *n_list, uint64_t *key64, float *height_map, uint8_t *observed, float *state,
                         int64_t *src_off, int64_t *dst_row, int64_t win_cap, int32_t *raised, eod_stream_t stream);
/* Per-slot reset of the height-max state (mask (E) i32, mask[e] != 0): height_map := 0 and observed := 0 for every cell, state rows
 * := 0 for the observed cells only (the others are zero already), as eod_reset_episodes does for the mean grid.  C %% 4 == 0. */
int eod_heightmax_reset(const int32_t *mask, int n_episodes, int64_t n_cells, int C, float *height_map, uint8_t *observed, float *state,
                        eod_stream_t stream);

/* Row GEMM with fp32 accuracy on tcgen05 tensor cores (3xTF32 split, fp32 accumulation in TMEM):
 *   Y[dst(i) * y_row_stride + j] = scale * ( sum_l A(i,l) * B(j,l) + bias[j] ),  i < min(M, *m_count), j < N, l < K
 *   A(i,l) = A[(a_off ? a_off[i] : i * a_row_stride) + l * a_k_stride]      B(j,l) = B[j * b_row_stride + l * b_k_stride]
 *   dst(i) = y_dst ? y_dst[i] : i ;  a_off, bias, m_count, y_dst nullable ;  N % 16 == 0.
 * Replaces the nn.Linear of the 'replace' update above (with the lists of eod_max_winner_list), the 1x1 forward projection of the
 * dense backbone-feature write (A7''), the projection of per-ROI memory features and the fp32 conv1x1 of timm.py:174 on the
 * training path (forward and, through the strides, both gradients).  |error| <= 1e-5 * scale of the result vs fp64.  A non-finite
 * operand makes its output row non-finite (inf or NaN - the operand split can turn inf * 0 into NaN), never another row. */
int eod_linear_rows(const float *A, int64_t a_row_stride, int64_t a_k_stride, const int64_t *a_off, const float *B, int64_t b_row_stride,
                    int64_t b_k_stride, const float *bias, float scale, int M, const int32_t *m_count, int N, int K, float *Y,
                    int64_t y_row_stride, const int64_t *y_dst, eod_stream_t stream);

/* ---------------------------------------------------------------------------------------------------
 * (3) Read.  Replaces create_implicit_memory (custom_rcnn.py:764-774), the fp16 cast (:1036) and
 * timm.py:147-168 (gather to the image plane, avg-pool 4, then per level avg-pool 2 -> half) in one
 * kernel for levels 0 and 1 plus a small second one that pools level 2 from level 1; the (480,640,C)
 * image-plane tensors are never materialised.
 *   table: mem_is_f16 == 0: sums (E,cells,C) f32 with counts (E,cells) f32 (nullable = no normalise);
 *          mem_is_f16 == 1: already normalised fp16 table (E,cells,C) (reference API: map_memory list)
 *   idx (E,H,W) int32 or int64.  H, W multiples of 32.
 *   L0 (E,H/8,W/8,C), L1 (E,H/16,W/16,C), L2 (E,H/32,W/32,C) fp16, channels-last.
 * Bit-exact with torch-CPU (sequential row-major window sums, fp16 rounding between levels).
 */
int eod_read_pool(const void *table, int mem_is_f16, const float *counts, const void *idx, int idx_is_i64,
                  int n_episodes, int C, int H, int W, int64_t n_cells, void *L0, void *L1, void *L2,
                  eod_stream_t stream);


/* Per-ROI read (north star subsystem 3): ROIAlign of the pooled memory levels over each proposal's box - the pooling the
 * reference's ROI heads apply to the FUSED levels (detic_roi_heads.py:331-334, self.box_pooler = detectron2 ROIPooler:
 * ROIAlignV2 (aligned, half-pixel offset), sampling_ratio 0 (adaptive ceil(roi / pooled)), 7x7 bins, scales 1/8, 1/16, 1/32,
 * FPN level assignment floor(canonical_level + log2(sqrt(area) / canonical_size + eps)) clamped to the available levels).
 * ROIAlign is linear, so pooling the memory levels with the proposals' boxes yields the per-ROI map feature that the fused
 * path carries implicitly: pool(res + w (conv(L) + b)) = pool(res) + w (conv(pool(L)) + b).
 *   levels / level_h / level_w / level_scale: HOST arrays of n_levels (<= 4) entries; levels[l] = device pointer of an
 *     (E, h_l, w_l, C) fp16 channels-last level exactly as eod_read_pool stores it; level_scale[l] = 1 / stride
 *   boxes (R,4) f32 XYXY in image pixels, batch_idx (R) i32 episode of each box (nullable = 0)
 *   out (R, pooled, pooled, C) f32 channels-last (logical (R, C, pooled, pooled)); out_level (R) i32 nullable: assigned level
 * Sample points, clamping and summation order of torchvision's CPU ROIAlign (ops/cpu/roi_align_kernel.cpp); accumulated fp32:
 * within 1e-5 of scale of the executed reference op, level assignments exact.  min_level: index of levels[0] in the pyramid
 * (3 for p3); canonical_size 224, canonical_level 4 in detectron2.  out_valid (nullable, (R,P,P) f32): per bin, the share of its sample
 * points that lie on the level = ROIAlign of a constant-1 plane (1 for boxes inside the image, 0 for empty / inverted boxes): the factor
 * with which the bias of a 1x1 projection applied before the pooling survives it. */
int eod_read_roi(int n_levels, const void *const *levels, const int *level_h, const int *level_w, const float *level_scale,
                 int n_episodes, int C, const float *boxes, const int32_t *batch_idx, int n_rois, int pooled, int sampling_ratio,
                 int min_level, float canonical_size, int canonical_level, float *out, int32_t *out_level, float *out_valid, eod_stream_t stream);

/* Stand-alone create_implicit_memory (custom_rcnn.py:764-774, and the half cast of :1036 when out_is_f16):
 * out[row] = sums[row] / counts[row] where counts[row] > 1 else sums[row].  n_rows = E*cells.  Only for
 * callers that need the normalised table itself; eod_read_pool fuses this step. */
int eod_normalize_memory(const float *sums, const float *counts, int64_t n_rows, int C, void *out, int out_is_f16,
                         eod_stream_t stream);

/* ---------------------------------------------------------------------------------------------------
 * Explicit semantic map (custom_rcnn.py:747-756 and visualise_clip_image_features :938-978), maintained
 * incrementally.  eod_semmap_update: for every cell visible in the current frame (frame_cnt != 0; call it after
 * the write and BEFORE eod_finalize_counts) refresh intensity[cell] = mean_ch|sums| (/ n if n > 1, n = counts + 1)
 * and cls[cell] = argmax_{k < n_cls} <sums[cell], zs_weight[:, k]> (zs_weight (C, ldz) f32 row-major, the
 * reference's zs_weight; n_cls = 20 there, <= 32 here).  eod_semmap_decode: semmap[cell] = cls[cell], or -1 where
 * (intensity - min) / (max - min) < thresh with the min / max taken over the episode's whole grid (:751,968).
 * minmax_ws: (E,2) f32 scratch. */
int eod_semmap_update(const uint32_t *frame_cnt, const float *counts, const float *sums, const float *zs_weight, int ldz,
                      int n_cls, int n_episodes, int C, int64_t n_cells, float *intensity, int32_t *cls,
                      eod_stream_t stream);
int eod_semmap_decode(const float *intensity, const int32_t *cls, int n_episodes, int64_t n_cells, float thresh,
                      float *minmax_ws, int32_t *semmap, eod_stream_t stream);

/* memory_reset (custom_rcnn.py:470-477) for state maintained by this library: clears counts, the sums row and
 * (if given) the norm16 row of every cell whose count is non-zero - equivalent to zero-filling the grid because
 * rows of never-visible cells are zero already.  n_rows = E*cells. */
int eod_reset_touched(float *counts, float *sums, void *norm16, int64_t n_rows, int C, eod_stream_t stream);

/* Per-slot memory_reset of a lock-step batch: the same as eod_reset_touched for the episodes with mask[e] != 0 only
 * (frame['memory_reset'] is per sequence: custom_rcnn.py:470-477, SMNet/loader.py:289-293).  mask (E) i32. */
int eod_reset_episodes(float *counts, float *sums, void *norm16, const int32_t *mask, int n_episodes, int64_t n_cells, int C,
                       eod_stream_t stream);

/* Re-derive the normalised fp16 rows (custom_rcnn.py:764-774,1036) of every cell with a non-zero count from the current
 * sums / counts, for the episodes with mask[e] != 0 (mask nullable = all).  TEST_TYPE 'longterm' reads a snapshot of the
 * memory taken at the first frame of each sequence (custom_rcnn.py:482-486): the write then runs eod_finalize_counts WITHOUT
 * norm16 and this refresh runs once per sequence start. */
int eod_refresh_norm16(const float *counts, const float *sums, void *norm16, const int32_t *mask, int n_episodes, int64_t n_cells,
                       int C, eod_stream_t stream);

/* Range check of an externally supplied index plane (proj_indices of memory_data/<name>.h5, SMNet/loader.py:185-186; the reference
 * raises IndexError on a bad id, timm.py:147).  Every kernel here uses a cell id as a row offset, so ids outside [0, n_cells)
 * must not reach them: err[0] (device int32, caller zeroes it) += number of out-of-range ids; idx32_out (nullable, n int32)
 * receives the ids with out-of-range ones clamped into the grid.  idx: n ids, int32 or int64 (idx_is_i64). */
int eod_check_indices(const void *idx, int idx_is_i64, int64_t n, int64_t n_cells, int32_t *idx32_out, int32_t *err,
                      eod_stream_t stream);

/* explicit_map read mode (SMNet/loader.py:233-246: `proj_indices = semmap_real[proj_indices]` with `semmap_real = semmap + 1`, memory =
 * [zero row; class-embedding table]; consumed by create_explicit_memory of the older custom_rcnn revision, bytecode listing
 * oracle/disasm/create_explicit_memory_custom_rcnn_py39.txt): out32[i] = lut[idx[i]] + add, the row of the (n_rows, C) table
 * that eod_read_pool then gathers.  idx: n cell ids (int32 / int64), lut: n_cells class ids (int32 / int64).  err[0] (device int32,
 * caller zeroes it) += number of ids outside [0, n_cells) or rows outside [0, n_rows); those come out as row 0. */
int eod_remap_indices(const void *idx, int idx_is_i64, int64_t n, const void *lut, int lut_is_i64, int64_t n_cells, int add, int64_t n_rows,
                      int32_t *out32, int32_t *err, eod_stream_t stream);

/* ---------------------------------------------------------------------------------------------------
 * (4) Fusion epilogue, timm.py:177-189: out = res + weight*mem | weight*mem | res (two roundings, no
 * FMA contraction, as torch computes it).  n elements, fp32. */
int eod_fuse(const float *res, const float *mem, float weight, int mode, int64_t n, float *out, eod_stream_t stream);

/* 1x1 projection + fusion in one tensor-core kernel (timm.py:170-189 with the modules of :78-86):
 *   out = res + weight * (level . W^T + bias)   (EOD_FUSE_SUM)   |   weight * (level . W^T + bias)   (EOD_FUSE_MEM_ONLY)
 * level   (E, h*w, K) f16  - a pooled level exactly as eod_read_pool stores it (channels-last), K = memory feature dim
 * w_split (2N, K) f16      - eod_project_split_weights(weight (N,K) f32): W = W_hi + 2^-11 * W_lo, two fp16 terms per weight,
 *                            so that the fp16 tensor-core products reproduce the fp32 GEMM (every product exact in fp32;
 *                            |error| <= ~2^-22 |W| per weight).  Re-run it whenever the weights change.
 * bias    (N) f32 nullable; res, out (E, N, h*w) f32 NCHW (res nullable for MEM_ONLY).  N % 128 == 0, K % 64 == 0.
 * The conv output, the scaling and the sum are rounded separately, as torch does (no contraction across the three ops).
 * Accumulated fp32: within 1e-5 of scale of the fp32 reference (tolerance stated in the tests), not bit-exact. */
int eod_project_split_weights(const float *weight, int N, int K, void *w_split, eod_stream_t stream);
/* All pyramid levels (<= 3) in ONE persistent launch.  level / w_split / bias / res / out / hw are HOST arrays of n_levels
 * entries (device pointers inside; bias and res arrays nullable, and so is each bias[l]).  variant: 0 = auto (persistent
 * kernel when every hw[l] % 4 == 0, else one tile-per-CTA launch per level), 1 = tile per CTA, 2 = persistent. */
int eod_project_fuse_levels(int n_levels, const void *const *level, const void *const *w_split, const float *const *bias,
                            const float *const *res, float *const *out, const int *hw, float weight, int mode, int n_episodes,
                            int K, int N, int variant, eod_stream_t stream);
int eod_project_fuse(const void *level, const void *w_split, const float *bias, const float *res, float weight, int mode,
                     int n_episodes, int hw, int K, int N, float *out, eod_stream_t stream);

#ifdef __cplusplus
}
#endif
#endif /* EOD_MEMORY_H */
