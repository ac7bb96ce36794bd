/*
 * a3d.h — C ABI of the B200-native temporal articulation optimizer hot path.
 *
 * Drop-in scope: the data-parallel part of JasonQSY/Articulation3D's
 * post-detection temporal optimisation, i.e. everything inside
 *     articulation3d/utils/opt_utils.py:382-682  optimize_planes_3dc
 *     articulation3d/utils/opt_utils.py:685-959  optimize_planes_3d_trans
 * that touches pixels:  get_pcd / project2D (articulation3d/utils/vis.py:62-102),
 * the pytorch3d transform chain, the point-splat loops and the IoU/argmax loops.
 * The reference has no FFI for this path (SURVEY.md §8b): the host side that
 * binds these symbols is articulation3d_b200/opt_utils.py, which keeps the
 * reference's Python signatures (track_planes / optimize_planes).
 *
 * Conventions
 *   - every function returns 0 on success, a negative A3D_E* code on failure;
 *     a3d_last_error_string() describes the last failure on the calling thread;
 *   - all buffers are caller-owned DEVICE pointers unless marked HOST;
 *   - `stream` is a cudaStream_t passed as void* (NULL = default stream);
 *     every call is asynchronous with respect to the host;
 *   - no global state, re-entrant, no C++ exceptions cross the boundary.
 *
 * Bit-packed mask layout ("bits"): uint32 [n][H][pitch], pitch =
 * a3d_pitch_words(W) = ceil(W/32) rounded up to a multiple of 4 words so that
 * rows are 16-byte aligned (TMA / bulk-copy granularity); bit i of word j of
 * row r is pixel (r, 32*j + i); padding bits are zero.
 */
#ifndef A3D_H_
#define A3D_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define A3D_VERSION 100            /* 0.1.0 */

enum {
    A3D_OK = 0,
    A3D_EINVAL = -1,               /* bad argument */
    A3D_ECUDA = -2,                /* CUDA runtime error (see error string) */
    A3D_ELIMIT = -3                /* shape exceeds what the kernels support */
};

/* mask element types accepted by a3d_pack_masks / produced by a3d_emit_masks */
enum { A3D_F32 = 0, A3D_U8 = 1 };
/* what a3d_project / a3d_pass write of every projected mask */
enum { A3D_OUT_FULL = 0, A3D_OUT_BBOX_ROWS = 1 };

/* floats of point-cloud workspace per point: X | Y | Z planes, the packed source pixel and the
 * error-bound coefficient of the filtered projection */
#define A3D_PCD_PLANES 5
/* floats of homography workspace per candidate (filtered projection) */
#define A3D_HOM_FLOATS 12

/* candidate transform modes (one per job) */
enum {
    A3D_MODE_SEQ = 0,        /* q=p-a; r=q*R; s=r+a  — cluster phase, opt_utils.py:433-435   */
    A3D_MODE_COMPOSED = 1,   /* s=p*R+t            — final phase, opt_utils.py:571-572       */
    A3D_MODE_TRANSLATE = 2   /* s=p+t              — translation tracks, opt_utils.py:726-728 */
};

/* Pinhole camera of get_pcd / project2D (vis.py:62-68, 86-95).  HOST struct. */
typedef struct {
    double  kinv[9];         /* row-major inverse intrinsics exactly as numpy.linalg.inv returns them */
    float   f, cx, cy;       /* project2D: K = [[f,0,cx],[0,f,cy],[0,0,1]] in fp32 */
    int32_t H, W;            /* mask size */
} a3d_camera_t;

/* One scoring job = one source frame of one track: its mask is unprojected onto
 * its plane, moved by n_cand candidate transforms, re-projected, and every
 * candidate is scored against n_tgt target masks (opt_utils.py:397-488). */
typedef struct {
    int32_t src_mask;        /* index into the source mask pool                         */
    int32_t mode;            /* A3D_MODE_*                                               */
    int32_t cand_begin;      /* first global candidate slot (xform / proj_* arrays)     */
    int32_t n_cand;
    int32_t tgt_begin;       /* first global target slot (tgt_index / best_* arrays)    */
    int32_t n_tgt;
    float   normal[3];       /* unit plane normal, camera frame (opt_utils.py:410)      */
    float   offset;          /* plane offset                      (opt_utils.py:411)    */
    float   pivot[3];        /* fp32 axis point a = Translate(verts_axis_3d[0]) (:420)  */
    int32_t pcd_cap;         /* capacity (points, multiple of 32) of this job's slice of
                                the point-cloud workspace; >= popcount of the source    */
    int64_t tab_begin;       /* first element of this job's [n_tgt][n_cand] table       */
    int64_t pcd_begin;       /* first point of this job's slice (multiple of 32)        */
} a3d_job_t;                 /* 72 bytes */

int         a3d_version(void);
const char* a3d_last_error_string(void);

/* words per packed row for an image of width W */
int a3d_pitch_words(int W);

/* Largest number of candidates one projection CTA can hold in shared memory for
 * an HxW mask on the current device (>=1), or A3D_ELIMIT. */
int a3d_project_max_tile(int H, int W);

/* HOST helper: split of a pass into projection CTAs ("tile map" of a3d_project / a3d_pass) when the
 * grid is about one wave, so that jobs whose source masks differ in size get tiles of different size
 * and every CTA carries about the same number of (point, candidate) pairs.
 *   jobs_host     [n_jobs] HOST copy of the jobs (n_cand and pcd_cap are read)
 *   tile_max      a3d_project_max_tile(H, W);  sm_count  SMs of the device
 *   tile_map_out  HOST [cap_tiles][4] int32, cap_tiles >= 2 * sm_count
 *   tile_cand_out candidates per CTA to pass as tile_cand (the largest tile of the map)
 * Returns the number of tiles written, 0 when the grid is several waves anyway (use uniform tiles of
 * *tile_cand_out = tile_max and no map), or a negative A3D_E* code.                              */
int a3d_plan_tiles(const a3d_job_t* jobs_host, int n_jobs, int tile_max, int sm_count,
                   int32_t* tile_map_out, int cap_tiles, int* tile_cand_out);

/* HOST helper: run lengths of n COCO compressed RLE strings (the `counts` of the reference's prediction records,
 * evaluation/arti_evaluation.py:153-180; decoded there with pycocotools' C extension, utils/arti_vis.py:135,182)
 * — the input of a3d_rle_to_bits.
 *   chars            HOST the n strings back to back;  begin  HOST [n+1] byte offsets into chars
 *   counts_out       HOST uint32 [cap], or NULL to only count (first of two calls)
 *   count_begin_out  HOST int64 [n+1] first count of every mask (may be NULL)
 *   run_sum_out      HOST int64 [n] sum of the mask's runs — must equal H*W (may be NULL)
 * Returns the total number of counts, or a negative A3D_E* code (truncated / malformed string, cap too small). */
int64_t a3d_host_rle_counts(const uint8_t* chars, const int64_t* begin, int64_t n, uint32_t* counts_out, int64_t cap,
                            int64_t* count_begin_out, int64_t* run_sum_out);

/* HOST helper: the 3x3 rotation entries of n unit quaternions, as pytorch3d's quaternion_to_matrix evaluates
 * them in float64 (the reference's axis_angle_to_matrix, utils/opt_utils.py:428-431), rounded once to fp32
 * (what Rotate stores) into the first nine floats of each 12-float candidate row.
 *   q      HOST [n][4] float64 {r, i, j, k};  two_s  HOST [n] float64 = 2 / |q|^2
 *   xform_out  HOST [n][12] fp32 (entries 9..11 untouched)                                          */
int a3d_host_quat_to_xform(const double* q, const double* two_s, int64_t n, float* xform_out);

/* Dense HOST masks of a clip -> packed bits, as one call: what `a3d_pack_masks` does for device-resident masks,
 * with the host-to-device copies in front.  chunks[i] points at chunk_masks[i] contiguous H x W masks of `dtype`
 * in host memory (pinned for asynchronous copies); they are copied one after the other into the device staging
 * block stage_dev (room for stage_cap_masks masks; every chunk must fit), which is packed into the next slots of
 * bits_gt / bits_nz (as a3d_pack_masks) whenever the next chunk does not fit and at the end.  At most `depth`
 * chunk copies are in flight (0 = no limit): submitted all at once, a gigabyte of copies fills the copy
 * engine's queue and the submitting call blocks inside the driver, holding up every other thread's CUDA calls.
 * Everything is enqueued on `stream`; the call returns when the last copy is SUBMITTED (not done).
 * Replaces the `.cuda()` of the per-frame `pred_masks` (reference utils/opt_utils.py:409, 471-473).            */
int a3d_upload_masks(const void* const* chunks, const int64_t* chunk_masks, int n_chunks, int dtype, int H, int W,
                     float thresh, void* stage_dev, int64_t stage_cap_masks, uint32_t* bits_gt, uint32_t* bits_nz,
                     int depth, void* stream);

/* Copies a block of PINNED host memory (cudaHostAlloc / cudaHostRegister: e.g. torch's pin_memory) into device
 * memory with a kernel that reads the host block over PCIe, instead of a cudaMemcpyAsync.  For the per-pass
 * descriptor block (jobs | candidate transforms | target indices, a3d_job_t above) of a caller that uploads
 * masks on another stream at the same time: a DMA copy of the descriptors queues on the host-to-device copy
 * engine behind every mask copy already submitted (measured: the submitting thread blocks for 14 ms per video,
 * the pass starts a whole upload late); the kernel is ordered by `stream` alone.  Both blocks 16-byte aligned;
 * the tail up to the next multiple of 16 bytes is copied too (size the blocks accordingly).
 * No reference counterpart (the reference keeps everything in torch tensors).                       */
int a3d_fetch_host_block(void* dst_dev, const void* src_host_pinned, int64_t nbytes, void* stream);

/* (a7/a8 input stage) threshold + bit-pack.  Replaces the per-visit
 * `(pred_mask > 0.5)` of opt_utils.py:471-473 and `pred_mask.nonzero()` of :409.
 *   src      [n][H][W] of dtype (A3D_F32 | A3D_U8), contiguous
 *   bits_gt  [n][H][pitch]  bit = src > thresh
 *   bits_nz  [n][H][pitch]  bit = src != 0        (may be NULL)               */
int a3d_pack_masks(const void* src, int dtype, int64_t n, int H, int W, float thresh,
                   uint32_t* bits_gt, uint32_t* bits_nz, void* stream);

/* population count and bounding box of packed masks.
 *   popc [n];  bbox [n][4] = {row_min, row_max, word_min, word_max} inclusive,
 *   {0,-1,0,-1} for an empty mask.                                             */
int a3d_mask_meta(const uint32_t* bits, int64_t n, int H, int W,
                  int32_t* popc, int32_t* bbox, void* stream);

/* (a4-a7) unproject + transform + project + splat.  Replaces get_pcd
 * (vis.py:86-102), the Transform3d chain (opt_utils.py:420-435, 553-574,
 * 724-728), project2D (vis.py:71-75) and the splat loop (opt_utils.py:438-457).
 * Two launches: k_unproject (source pixels -> compacted fp32 point cloud, float64
 * ray/plane intersection) and k_project (transform, project, splat per candidate).
 *   cam        HOST
 *   jobs       [n_jobs] device
 *   max_cand   max over jobs of n_cand
 *   tile_cand  candidates per CTA, 1..a3d_project_max_tile(H,W) (0 = choose)
 *   src_bits   source mask pool, src_bbox its a3d_mask_meta boxes
 *   xform      [n_cand_total][12] fp32: rows 0-2 of R (row-vector convention,
 *              p' = p*R), then t
 *   pcd_ws     workspace, A3D_PCD_PLANES * sum(pcd_cap) floats (planes of pcd_cap floats per job slice)
 *   pcd_count  workspace, [n_jobs + 1] int32 (points actually produced per job; the last entry is the
 *              work counter of the persistent projection kernel)
 *   hom_ws     workspace, [n_cand_total][A3D_HOM_FLOATS] floats: per candidate the plane-induced
 *              homography source pixel -> projected pixel and its error bound, from which the
 *              filtered projection kernel takes every pixel it can PROVE equal to the reference
 *              chain's (the others run that chain; results are identical either way).  NULL or
 *              A3D_PROJECT_KERNEL=exact: the reference chain for every point; by default the
 *              filter is taken when the grid is more than two waves of CTAs.
 *   tile_map   optional [n_tiles][4] int32, 16-byte aligned: the caller's split of the work into
 *              CTAs, {job, first candidate, candidates (<= tile_cand), role}; role 1 marks the CTA
 *              that takes the job's exact-only candidates (one per job, first/count ignored).
 *              Every candidate of every job must be covered exactly once by role-0 entries.
 *              NULL: uniform tiles of tile_cand candidates.  Jobs of very different size in a
 *              grid of about one wave are the case for it (see engine.plan_tiles).
 *   proj_bits  [n_cand_total][H][pitch]; proj_popc [n_cand_total];
 *   proj_bbox  [n_cand_total][4]
 *   out_mode   A3D_OUT_FULL: every word of every projected mask is written.
 *              A3D_OUT_BBOX_ROWS: for callers that keep proj_bits / proj_bbox between calls.  On entry the
 *              image of every slot must be zero outside the rows row_min..row_max of proj_bbox[slot] — true
 *              for a pair initialised to {proj_bits = 0, proj_bbox = {0,-1,0,-1}} and after every call in
 *              this mode; the call then writes only the 16-byte pieces that lie in a row of the slot's old
 *              box (zeros included) or are non-zero, and leaves the same invariant.  proj_bits is fully
 *              defined either way.
 *              (The zeros around a door-sized mask are 85 % of the projection's DRAM writes.)         */
int a3d_project(const a3d_camera_t* cam, const a3d_job_t* jobs, int n_jobs, int max_cand,
                int tile_cand, const uint32_t* src_bits, const int32_t* src_bbox,
                const float* xform, float* pcd_ws, int32_t* pcd_count, float* hom_ws,
                const int32_t* tile_map, int n_tiles,
                uint32_t* proj_bits, int32_t* proj_popc, int32_t* proj_bbox, int out_mode, void* stream);

/* (a8) mask-IoU scoring with fused arg-max over candidates.  Replaces the
 * `for idx in id_list` loops of opt_utils.py:464-477, 600-612, 757-770, 892-904.
 *   n_pool_masks, n_cand_total  sizes of the target pool / of proj_* (TMA tensor extents)
 *   tgt_index  [n_tgt_total] indices into the target pool (tgt_bits/popc/bbox)
 *   key_ws     [n_tgt_total] uint64 workspace
 *   inter_tab  optional [sum n_tgt*n_cand] int32 table of intersections (NULL ok)
 * outputs, per target slot:
 *   best_cand  index of the first candidate with maximal IoU (NaN counts as max)
 *   best_inter, best_union  integer counts at that candidate
 *   best_iou   fp32 inter/union (IEEE division)                                */
int a3d_score(int H, int W, const a3d_job_t* jobs, int n_jobs, int max_tgt, int max_cand,
              int64_t n_tgt_total, int64_t n_pool_masks, int64_t n_cand_total,
              const uint32_t* tgt_bits, const int32_t* tgt_popc, const int32_t* tgt_bbox,
              const int32_t* tgt_index,
              const uint32_t* proj_bits, const int32_t* proj_popc, const int32_t* proj_bbox,
              uint64_t* key_ws, int32_t* inter_tab,
              int32_t* best_cand, int32_t* best_inter, int32_t* best_union, float* best_iou,
              void* stream);

/* One whole pass = a3d_project followed by a3d_score on the same stream, as one call: the arg-max keys
 * are cleared first, so k_project, the scoring kernel and k_finalize run as programmatic dependent
 * launches of their predecessors (their launch latency and prologue overlap the predecessor's tail).
 * Same results as the two calls.  pool_* = target pool; src_bits/src_bbox = source pool
 * (NULL: the target pool is also the source pool).                                              */
int a3d_pass(const a3d_camera_t* cam, const a3d_job_t* jobs, int n_jobs, int max_tgt, int max_cand,
             int tile_cand, int64_t n_tgt_total, int64_t n_pool_masks, int64_t n_cand_total,
             const uint32_t* pool_bits, const int32_t* pool_popc, const int32_t* pool_bbox,
             const uint32_t* src_bits, const int32_t* src_bbox, const float* xform, const int32_t* tgt_index,
             float* pcd_ws, int32_t* pcd_count, float* hom_ws, const int32_t* tile_map, int n_tiles,
             uint32_t* proj_bits, int32_t* proj_popc, int32_t* proj_bbox,
             uint64_t* key_ws, int32_t* inter_tab,
             int32_t* best_cand, int32_t* best_inter, int32_t* best_union, float* best_iou,
             int out_mode, void* stream);

/* (a11) materialise selected packed masks as dense images: out[i] =
 * unpack(bits[index[i]]) as A3D_F32 (0.0/1.0) or A3D_U8 (0/1).  Replaces
 * `proj_masks[angle_id].cpu()` of opt_utils.py:614, 906 (index may be NULL =
 * identity).                                                                   */
int a3d_emit_masks(const uint32_t* bits, const int32_t* index, int64_t n, int H, int W,
                   int out_dtype, void* out, void* stream);

/* (f2, SURVEY.md 8f) COCO RLE -> packed masks on the device.  Replaces
 * pycocotools mask_util.decode in create_instances (utils/arti_vis.py:182) and
 * override_depth (:135).
 *   counts  concatenated run lengths of all masks (runs alternate 0/1, start with 0,
 *           column-major order); begin [n+1] offsets into counts
 *   bits    [n][H][pitch]                                                          */
int a3d_rle_to_bits(const uint32_t* counts, const int64_t* begin, int64_t n, int H, int W,
                    uint32_t* bits, void* stream);

/* (f2, SURVEY.md 8f) packed masks -> COCO RLE run lengths on the device, the inverse of a3d_rle_to_bits: the
 * `counts` rle.encode computes (pycocotools mask_util.encode in the reference), runs alternating 0/1 in
 * column-major order, starting with 0s (a set pixel (0,0) gives a first run of 0); every mask's runs sum to
 * H*W.  Two calls, both asynchronous on `stream`; `index` selects the masks as in a3d_emit_masks (NULL =
 * identity).  Any H, W >= 1 with H*W <= 2^31 - 1 (A3D_ELIMIT beyond), any n.
 *   runs_out   [n] int64: number of runs of every selected mask (first call)
 *   begin      [n+1] int64: exclusive scan of runs_out (begin[0] = 0)
 *   counts_out [begin[n]] uint32: mask i's runs go to counts_out[begin[i] .. begin[i+1])               */
int a3d_rle_count_runs(const uint32_t* bits, const int32_t* index, int64_t n, int H, int W,
                       int64_t* runs_out, void* stream);
int a3d_bits_to_rle(const uint32_t* bits, const int32_t* index, int64_t n, int H, int W,
                    const int64_t* begin, uint32_t* counts_out, void* stream);

/* HOST helper: COCO compressed strings of n masks' run lengths (the inverse of a3d_host_rle_counts; byte for
 * byte what rle.counts_to_string writes).
 *   counts          HOST uint32, mask i's runs at counts[begin[i] .. begin[i+1]);  begin  HOST [n+1]
 *   chars_out       HOST [cap] (7 * total counts always suffices)
 *   char_begin_out  HOST [n+1] first byte of every mask's string (may be NULL)
 * Returns the total number of bytes, or a negative A3D_E* code (bad offsets, cap too small).          */
int64_t a3d_host_rle_strings(const uint32_t* counts, const int64_t* begin, int64_t n,
                             uint8_t* chars_out, int64_t cap, int64_t* char_begin_out);

/* (f1, SURVEY.md 8f) plane offset implied by the depth map: for every instance the mean
 * over its mask of normal . (rays * depth).  Replaces the per-instance loop of
 * override_depth (utils/arti_vis.py:125-149) and depth2XYZ (:90-99).
 *   depth     [n_frames][H][W] fp32, or NULL when `rays` already holds XYZ
 *   rays      [3][H][W] fp32  K^-1 [x y 1] table (get_K_inv_dot_xy_1, :101-122)
 *   bits/bbox mask pool and its a3d_mask_meta boxes
 *   inst_mask [n_inst] pool index, inst_frame [n_inst] depth frame, normals [n_inst][3]
 *   offset_out [n_inst] fp32 mean (0 when the mask is empty), count_out [n_inst] pixels */
int a3d_plane_offsets(const float* depth, const float* rays, int H, int W, const uint32_t* bits,
                      const int32_t* bbox, const int32_t* inst_mask, const int32_t* inst_frame,
                      const float* normals, int64_t n_inst, float* offset_out, int32_t* count_out,
                      void* stream);

/* (f5) what a3d_render draws: a mask of the pool, filled or as its outline, blended with alpha rgba[3] */
enum { A3D_LAYER_FILL = 0, A3D_LAYER_OUTLINE = 1 };
typedef struct { int32_t mask; int32_t kind; uint8_t rgba[4]; } a3d_layer_t;                       /* 12 bytes */
/* an opaque line segment of half-width `radius`; |coordinates| <= 2^14, 0 <= radius <= 256 */
typedef struct { int32_t x0, y0, x1, y1; int32_t radius; uint8_t rgb[3], pad; } a3d_segment_t;    /* 24 bytes */
#define A3D_RENDER_MAX_SIDE 16384

/* (f5) the fitted result drawn into the clip's frames (reference tools/inference.py:253-278, there with
 * detectron2's Visualizer): n_frames RGB frames out [n_frames][H][W][3] uint8, every byte defined as
 *   1. the background pixel: background + f * bg_frame_stride (bytes; 0 = one H x W x 3 image for all frames);
 *   2. frame f's layers layers[layer_begin[f] .. layer_begin[f+1]) in order: FILL covers the mask's set pixels,
 *      OUTLINE its set pixels with at least one unset 4-neighbour (outside the frame = unset); a covered
 *      channel o becomes (c * a + o * (255 - a) + 127) / 255 (uint32, floor);  a layer whose mask is outside
 *      [0, n_masks) draws nothing;
 *   3. frame f's segments segs[seg_begin[f] .. seg_begin[f+1]) in order, opaque: pixel q is on segment (p0, p1)
 *      when its squared distance to the closed segment is <= radius^2, decided in int64 with d = p1 - p0,
 *      t = (q - p0).d, L = d.d: t <= 0 -> |q - p0|^2, t >= L -> |q - p1|^2, else cross(q - p0, d)^2 <= r^2 L.
 *   bits/bbox  the mask pool and its a3d_mask_meta boxes (bbox may be NULL: same output, no culling)
 *   layers, layer_begin [n_frames + 1], segs, seg_begin [n_frames + 1]  DEVICE
 * H, W <= A3D_RENDER_MAX_SIDE.  One CTA per (frame, band of rows): the band's background and output bytes
 * are streamed once, the list entries whose box misses the band are culled first.                      */
int a3d_render(const uint8_t* background, int64_t bg_frame_stride, int n_frames, int H, int W,
               const uint32_t* bits, const int32_t* bbox, int64_t n_masks,
               const a3d_layer_t* layers, const int64_t* layer_begin,
               const a3d_segment_t* segs, const int64_t* seg_begin, uint8_t* out, void* stream);

/* (f6) a mask of the pool lying on the plane n . X = offset (camera frame of get_pcd), drawn in colour rgb */
typedef struct { int32_t mask; float normal[3]; float offset; uint8_t rgb[3], pad; } a3d_plane_layer_t;   /* 24 bytes */

/* (f6) per-frame depth and colour (e.g. surface-normal) maps of planar masks (reference tools/inference.py:231-243
 * shows the planes as a normal map).  For pixel (x, y) of frame f and every layer of
 * layers[layer_begin[f] .. layer_begin[f+1]) whose mask has the pixel set, in float64 with every product and sum
 * rounded separately, left to right (k_unproject's chain):
 *     ray = kinv [x, y, 1]   (rx = (k0 x + k1 y) + k2, ry = (k3 x + k4 y) + k5, rz = (k6 x + k7 y) + k8;
 *                             with k1 = k3 = k6 = k7 = 0, k8 = 1: rx = k0 x + k2, ry = k4 y + k5, rz = 1)
 *     dot = (n0 rx + n1 ry) + n2 rz,  depth = offset / dot,  z = fp32_rn(depth * rz)
 * (n, offset: the layer's fp32 values widened).  The layer covers the pixel when z is finite and z > 0 (a plane
 * behind the camera, an edge-on ray and a NaN plane cover nothing); a layer whose mask is outside [0, n_masks)
 * covers nothing.  The covering layer of smallest z wins the pixel, the earlier one in the list on equal z:
 *     depth_out [n_frames][H][W] fp32   the winner's z, 0.0f where no layer covers the pixel
 *     rgb_out   [n_frames][H][W][3] u8  the winner's rgb, bg_rgb (HOST, 3 bytes) where none does
 * Either output may be NULL (not written).  bits/bbox: the mask pool [n_masks][H][pitch] of the camera's H x W
 * and its a3d_mask_meta boxes (bbox may be NULL: same output, no culling).  layers, layer_begin [n_frames + 1]
 * DEVICE.  H, W <= A3D_RENDER_MAX_SIDE, any number of frames and layers.  One CTA per (frame, band of rows):
 * the frame's layers whose box misses the band are culled first, in batches, and the band's running best
 * (z, colour) stays in shared memory until its outputs are written once.                                  */
int a3d_plane_maps(const a3d_camera_t* cam, int n_frames, const uint32_t* bits, const int32_t* bbox, int64_t n_masks,
                   const a3d_plane_layer_t* layers, const int64_t* layer_begin, const uint8_t bg_rgb[3],
                   float* depth_out, uint8_t* rgb_out, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* A3D_H_ */
