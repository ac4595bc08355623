/*
 * mrx.h -- C ABI of the B200 (sm_100a) Mask R-CNN serving hot path.
 *
 * The reference (huyhoang17/matterport-maskrcnn-with-tensorflow-serving) has NO
 * FFI / plugin interface: its boundary is three plain Python call sites in
 * serve.py.  Each entry point below names the Python call it stands behind:
 *
 *   mrx_anchors            <- api_utils.get_anchors(image_shape)          serve.py:105
 *   mrx_unmold_prologue    <- api_utils.unmold_detections(...) steps 1-6  serve.py:147-154
 *   mrx_gather_tiles       <- mrcnn_mask[arange(N),:,:,class_ids]         (same call)
 *   mrx_unmold_prepare     (the two above in one launch)
 *   mrx_mask_expand        <- per-instance unmold_mask + np.stack(axis=-1)(same call)
 *   mrx_mask_expand_values    (parity instrumentation of the kernel above)
 *   mrx_cv2_resize_u8c3[_batch] <- cv2.resize(img, (S, S))                serve.py:88-89
 *   mrx_mold_image[_batch] <- resize_image + mold_image                   serve.py:91-98
 *   mrx_composite_masks    <- visualize.display_instances (mask overlay)  serve.py:160-169
 *   mrx_pack_masks         (extension: bit-packed transport of the masks of serve.py:147)
 *   mrx_mask_expand_packed (extension: the expand step writing that packed layout directly)
 *   mrx_rle_count / _write (extension: the same masks as COCO run-length encodings)
 *   mrx_contours_count / _write <- the contour polygons display_instances traces  serve.py:160-169
 *   mrx_peer_*             (multi-GPU: the final gather of the masks to rank 0, SURVEY.md 8e)
 *
 * Conventions
 *   - every pointer named d_* is DEVICE memory owned by the caller (the Python
 *     side holds them as torch tensors and passes data_ptr()); nothing here
 *     allocates, frees or synchronises -- all work is ordered on `stream`
 *     (a cudaStream_t passed as void*; NULL = legacy default stream).
 *   - return value: MRX_OK (0) or a negative MRX_E_* code; mrx_last_error()
 *     returns a thread-local description of the last failure.
 *   - dtype codes: MRX_F32 = 0, MRX_F64 = 1.
 *   - there is no CPU fallback behind any of these calls.
 */
#ifndef MRX_H_
#define MRX_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define MRX_ABI_VERSION 6

#define MRX_OK              0
#define MRX_E_INVALID      -1   /* bad argument (null pointer, size out of range) */
#define MRX_E_UNSUPPORTED  -2   /* shape outside what the kernels are built for   */
#define MRX_E_CUDA         -3   /* a CUDA runtime call failed                      */

#define MRX_F32 0
#define MRX_F64 1

/* per-image status bits written by mrx_unmold_prologue into d_status[b] */
#define MRX_ST_CLASS_RANGE  1   /* class id outside [-C, C): numpy would raise IndexError */
#define MRX_ST_BOX_RANGE    2   /* kept box outside the canvas: numpy paste would raise   */

/* limits (compile-time properties of the kernels) */
#define MRX_MAX_LEVELS   8
#define MRX_MAX_RATIOS   8
#define MRX_MAX_BATCH    4096    /* images per mrx_mask_expand launch */
#define MRX_MAX_MASK_DIM 64      /* mask tile side (28 upstream); width must be a multiple of 4 */

int         mrx_abi_version(void);
const char *mrx_last_error(void);

/* Device properties the host-side planner needs (SM count, opt-in smem per block). */
int mrx_device_props(int device, int *sm_count, int *cc_major, int *cc_minor,
                     int *max_smem_optin);

/* ---------------------------------------------------------------- anchors (a5) */
/* Number of anchors for an image of img_h x img_w:  R * sum_l ceil(ceil(H/s_l)/as) * ceil(ceil(W/s_l)/as). */
int mrx_anchor_count(int img_h, int img_w, const int *strides, int n_levels,
                     int n_ratios, int anchor_stride, long long *count);

/* d_out: [A,4] float32 (y1,x1,y2,x2) normalised by norm_boxes; level-major, then
 * y, x, ratio innermost.  scales[n_levels], ratios[n_ratios] are HOST arrays.
 * Arithmetic is fp64 with numpy's operation order, rounded once to fp32. */
int mrx_anchors(float *d_out, int img_h, int img_w,
                const double *scales, const double *ratios, const int *strides,
                int n_levels, int n_ratios, int anchor_stride, void *stream);

/* ---------------------------------------------------------------- unmold (a1-a4) */
/* Geometry per image, 8 x int32:
 *   [0] orig_h [1] orig_w   original image (canvas) size
 *   [2] img_h  [3] img_w    molded image size
 *   [4..7]  window y1,x1,y2,x2 in molded pixels                                  */
#define MRX_GEOM_INTS 8

/* Steps 1-6 of unmold_detections for a batch of B images, one CTA per image:
 * trim at the first class_id==0 row, class ids, window normalisation (float32),
 * box affine + denorm (float64, round-half-even), zero-area drop with
 * order-preserving compaction.
 *   d_detections [B,R,6] det_dtype      d_geom [B,8] int32
 *   d_boxes [B,R,4] int32   d_class_ids [B,R] int32   d_scores [B,R] det_dtype
 *   d_src_index [B,R] int32 (kept row -> original row)
 *   d_counts [B] int32 (N per image)    d_status [B] int32 (MRX_ST_* bits)
 * C = number of classes in mrcnn_mask's last axis (for the class-range check).
 * d_sched (may be NULL): the scheduler words of the expand kernels (MRX_SCHED_WORDS x uint32),
 * zeroed here as well. */
int mrx_unmold_prologue(const void *d_detections, int det_dtype, int B, int R, int C,
                        const int *d_geom,
                        int *d_boxes, int *d_class_ids, void *d_scores,
                        int *d_src_index, int *d_counts, int *d_status,
                        unsigned int *d_sched, void *stream);

/* masks = mrcnn_mask[src_index, :, :, class_id] packed to float32 tiles.
 *   d_mrcnn_mask [B,R,mh,mw,C] mask_dtype  ->  d_tiles [B,R,mh,mw] float32      */
int mrx_gather_tiles(const void *d_mrcnn_mask, int mask_dtype,
                     int B, int R, int mh, int mw, int C,
                     const int *d_class_ids, const int *d_src_index,
                     const int *d_counts, float *d_tiles, void *stream);

/* Scheduler scratch of the expand kernels: MRX_SCHED_WORDS x uint32 of device memory that the
 * caller zeroes ONCE after allocating it; every launch hands out its work through it and leaves
 * it zeroed (no memset between launches).  One scratch per stream of launches. */
#define MRX_SCHED_WORDS 4

/* mrx_unmold_prologue and mrx_gather_tiles in ONE launch (what the engine uses): the prologue's
 * outputs as above; the class tiles are stored by ORIGINAL detection row,
 *   d_tiles[b][t] = float32(mrcnn_mask[b, t, :, :, class_id of row t])      (rows with class 0: untouched)
 * which needs nothing from the prologue, so both run side by side in the same grid.  The expand
 * entry points then take d_tile_index = d_src_index (kept instance k -> its row). */
int mrx_unmold_prepare(const void *d_detections, int det_dtype, const void *d_mrcnn_mask,
                       int mask_dtype, int B, int R, int mh, int mw, int C,
                       const int *d_geom, int *d_boxes, int *d_class_ids, void *d_scores,
                       int *d_src_index, int *d_counts, int *d_status,
                       float *d_tiles, unsigned int *d_sched, void *stream);

/* The hot kernel.  For every image b writes the bool canvas [H_b, W_b, N_b]
 * (N innermost, 1 byte per element, values 0/1) at d_canvas + d_canvas_off[b]:
 * zero fill, zero-border half-pixel bilinear resize of each tile to its box,
 * >= 0.5 threshold and paste, fused so each output byte is written once.
 *   d_canvas_off [B] int64, each a multiple of 16; slot b must hold at least
 *   round_up(H_b*W_b*N_b, 16) bytes (bytes past H_b*W_b*N_b may or may not be written).
 *   chunk_bytes: upper bound, in bytes, of the canvas tile a team of warps builds in
 *   shared memory and stores with one bulk copy per tile row (a tile is P pixels x
 *   10 rows x N instances; it is raised to the minimum that holds 16 pixels of R
 *   instances per row); multiple of 16, >= 1024; 0 = as large as fits (library default).
 *   ctas_per_sm: used by the generic kernel only (R too large for the tile buffers, or
 *   mask tiles wider than 30 columns); 0 = as many as fit.
 *   d_tile_index [B,R] int32 or NULL: kept instance k of image b resizes
 *   d_tiles[b][d_tile_index[b][k]] (NULL: d_tiles[b][k], the layout mrx_gather_tiles writes;
 *   d_src_index: the layout mrx_unmold_prepare writes).                              */
int mrx_mask_expand(const float *d_tiles, const int *d_tile_index, const int *d_boxes,
                    const int *d_counts, const int *d_geom, const long long *d_canvas_off,
                    unsigned char *d_canvas, int B, int R, int mh, int mw,
                    int chunk_bytes, int ctas_per_sm,
                    unsigned int *d_sched, void *stream);

/* Parity instrumentation: the SAME kernel template as mrx_mask_expand (same culling, source
 * coordinates, interpolation and row walk -- a second instantiation of it), which in addition
 * stores every pre-threshold sample it evaluates: d_values is float32, indexed exactly like
 * d_canvas (element d_canvas_off[b] + (y*W_b + x)*N_b + n); only elements inside box n are
 * written.  The canvas is written as usual.  Tests compare these values with the float64
 * oracle (|diff| <= 1e-6).  Shapes the team kernel does not take (R > 200, mask tiles wider
 * than 30 columns) return MRX_E_UNSUPPORTED. */
int mrx_mask_expand_values(const float *d_tiles, const int *d_tile_index, const int *d_boxes,
                           const int *d_counts, const int *d_geom, const long long *d_canvas_off,
                           unsigned char *d_canvas, float *d_values, int B, int R, int mh, int mw,
                           unsigned int *d_sched, void *stream);

/* ---------------------------------------------------------------- mold (a6) */
/* cv2.resize(src, (dst_w, dst_h)) for uint8 HxWx3, default INTER_LINEAR
 * (OpenCV's 11-bit fixed-point path, incl. its exact-2x INTER_AREA shortcut). */
int mrx_cv2_resize_u8c3(const unsigned char *d_src, int src_h, int src_w,
                        unsigned char *d_dst, int dst_h, int dst_w, void *stream);

/* The same for a batch in ONE launch (the reference resizes every request image to
 * (IMAGE_SIZE, IMAGE_SIZE), serve.py:88-89, 114): sources of any sizes, image b at
 * d_src + d_src_off[b] (int64 byte offsets) with (h, w) = d_src_hw[2b], d_src_hw[2b+1];
 * destinations densely packed [B, dst_h, dst_w, 3]. */
int mrx_cv2_resize_u8c3_batch(const unsigned char *d_src, const long long *d_src_off,
                              const int *d_src_hw, unsigned char *d_dst, int B,
                              int dst_h, int dst_w, void *stream);

/* resize_image(mode square/pad64/none geometry precomputed by the host) fused
 * with mold_image: scale src (uint8 HxWx3) to new_h x new_w with the zero-border
 * bilinear of a4 in fp64, truncate to uint8, place at (top,left) in an
 * out_h x out_w canvas of zeros, subtract mean_pixel.
 *   out_dtype MRX_F32: float32( float64(u8) - mean )   (what serve.py:117 sends)
 *   out_dtype MRX_F64: float64(u8) - mean              (what preprocess_input returns)
 *   d_molded_u8 (optional, may be NULL): the uint8 image before mean subtraction. */
int mrx_mold_image(const unsigned char *d_src, int src_h, int src_w,
                   int new_h, int new_w, int top, int left, int out_h, int out_w,
                   const double *mean_pixel /* host, 3 */, int out_dtype,
                   void *d_out, unsigned char *d_molded_u8, void *stream);

/* The same for B equally sized images in ONE launch: d_src [B,src_h,src_w,3] ->
 * d_out [B,out_h,out_w,3] (and d_molded_u8 likewise). */
int mrx_mold_image_batch(const unsigned char *d_src, int B, int src_h, int src_w,
                         int new_h, int new_w, int top, int left, int out_h, int out_w,
                         const double *mean_pixel /* host, 3 */, int out_dtype,
                         void *d_out, unsigned char *d_molded_u8, void *stream);

/* ---------------------------------------------------------------- compositing (8f) */
/* Mask part of visualize.display_instances(img, boxes, masks, ...) (serve.py:160-169), on
 * the canvas mrx_mask_expand wrote: for every image b, per instance i in order (skipped when
 * its box is all zeros), per channel c,
 *     v = uint32( float64(v) * one_minus_alpha + blend[b][i][c] )      where mask[.,.,i] == 1
 * starting from the uint8 image and ending with astype(uint8).
 *   d_images / d_out: uint8 H_b x W_b x 3 images of the batch, image b at byte offset
 *   d_image_off[b] (int64) in both;  d_blend [B,R,3] float64 = alpha * color[c] * 255,
 *   evaluated by the caller in float64 in that order;  d_boxes [B,R,4] as written by
 *   mrx_unmold_prologue;  max_pixels = max_b H_b * W_b (grid sizing). */
int mrx_composite_masks(const unsigned char *d_canvas, const long long *d_canvas_off,
                        const int *d_counts, const int *d_geom, const int *d_boxes,
                        const unsigned char *d_images, const long long *d_image_off,
                        const double *d_blend, double one_minus_alpha,
                        unsigned char *d_out, int B, int R, long long max_pixels,
                        void *stream);

/* ---------------------------------------------------------------- packed masks (8f) */
/* EXTENSION (not the reference layout): bit-packed copy of the canvases for transport.
 * For image b:  d_packed + d_packed_off[b]  holds  uint8 [N_b, H_b, ceil(W_b/8)]  with
 *     packed[n, y, :] = np.packbits(masks[y, :, n])          (most significant bit first)
 * so that np.unpackbits(packed, axis=-1, count=W).transpose(1, 2, 0) is the bool [H,W,N] array
 * unmold_detections returns.  Slot b must hold R * H_b * ceil(W_b/8) bytes; d_packed_off int64.
 * max_h / max_w: largest H_b / W_b of the batch (grid sizing). */
int mrx_pack_masks(const unsigned char *d_canvas, const long long *d_canvas_off,
                   const int *d_counts, const int *d_geom, unsigned char *d_packed,
                   const long long *d_packed_off, int B, int R, int max_h, int max_w,
                   void *stream);

/* EXTENSION: the expand step with bit-packed output, without ever writing the byte canvas
 * (expand_bits.cu).  Same inputs as mrx_mask_expand (tiles, boxes, counts, geometry as left by
 * mrx_unmold_prologue / mrx_gather_tiles); output layout exactly that of mrx_pack_masks:
 * image b at d_packed + d_packed_off[b] as uint8 [N_b, H_b, ceil(W_b/8)] (slot capacity
 * R * H_b * ceil(W_b/8)); planes n >= N_b are not written.  The samples are computed with the
 * same arithmetic as mrx_mask_expand, so  packed == np.packbits(canvas)  bit for bit.
 * d_packed may be memory of ANOTHER GPU mapped with mrx_peer_open (fused compute + gather).
 * max_w: widest W_b of the batch.  Mask tiles wider than 30 columns: MRX_E_UNSUPPORTED
 * (use mrx_mask_expand + mrx_pack_masks). */
int mrx_mask_expand_packed(const float *d_tiles, const int *d_tile_index, const int *d_boxes,
                           const int *d_counts,
                           const int *d_geom, const long long *d_packed_off,
                           unsigned char *d_packed, int B, int R, int mh, int mw, int max_w,
                           unsigned int *d_sched, void *stream);

/* EXTENSION: COCO run-length masks (pycocotools' "uncompressed RLE": the mask in COLUMN-major
 * order as alternating run lengths of zeros and ones, starting with zeros), computed from the
 * tiles with the arithmetic of mrx_mask_expand -- decoding them gives that kernel's masks bit
 * for bit -- without materialising any mask (rle.cu).  Two calls around one host read:
 *   mrx_rle_count:  d_col_count [B,R,max_w] int32 scratch; d_inst_off [B*R+1] int64: on return
 *                   (stream-ordered) d_inst_off[i] = number of value changes of all instances
 *                   before i = b*R + k, d_inst_off[B*R] = their total T.  The caller reads T and
 *                   allocates d_positions [T] and d_run_lengths [T + B*R] (uint32).
 *   mrx_rle_write:  instance i's runs are d_run_lengths[d_inst_off[i] + i ...], one more than
 *                   its value changes (d_inst_off[i+1] - d_inst_off[i] + 1); they sum to H*W.
 * Inputs as for mrx_mask_expand_packed.  Mask tiles wider than 30 columns: MRX_E_UNSUPPORTED. */
int mrx_rle_count(const float *d_tiles, const int *d_tile_index, const int *d_boxes,
                  const int *d_counts, const int *d_geom, int *d_col_count,
                  long long *d_inst_off, int B, int R, int mh, int mw, int max_w, void *stream);
int mrx_rle_write(const float *d_tiles, const int *d_tile_index, const int *d_boxes,
                  const int *d_counts, const int *d_geom, int *d_col_count,
                  long long *d_inst_off, unsigned int *d_positions, unsigned int *d_run_lengths,
                  int B, int R, int mh, int mw, int max_w, void *stream);

/* ---------------------------------------------------------------- contour polygons (f5) */
/* The outline step of visualize.display_instances (serve.py:160-169): for every instance,
 *     padded = zeros((H+2, W+2)); padded[1:-1, 1:-1] = mask
 *     [np.fliplr(v) - 1 for v in skimage.measure.find_contours(padded, 0.5)]
 * (fully_connected='low', positive_orientation='low'), computed from the bit-packed masks:
 * image b at d_packed + d_packed_off[b] as uint8 [N_b, H_b, ceil(W_b/8)] (the layout of
 * mrx_mask_expand_packed / mrx_pack_masks / np.packbits; bits past W_b are ignored).  A mask is
 * read as zero outside its box d_boxes[b][k] (y1, x1, y2, x2) -- only the box's cells and one ring
 * around them are scanned; an instance k >= d_counts[b] or with an empty box has no contours.
 *
 * Marching squares: cell (r, c) of the padded mask P is (ul, ur, ll, lr) = P[r..r+1, c..c+1],
 * case = ul + 2 ur + 4 ll + 8 lr; segments (from, to) between edge midpoints top (r, c+1/2),
 * bottom (r+1, c+1/2), left (r+1/2, c), right (r+1/2, c+1), cells in row-major order:
 *     1 (T,L)  2 (R,T)  3 (R,L)  4 (L,B)  5 (T,B)  6 (R,T),(L,B)  7 (R,B)
 *     8 (B,R)  9 (T,L),(B,R)  10 (B,T)  11 (B,L)  12 (L,R)  13 (T,R)  14 (L,T)
 * Every edge midpoint has one segment in and one out, so the segments form cycles.  Each cycle
 * is one polygon: it starts at the `to` point of the cycle's last-emitted segment, follows the
 * segments and repeats its start point at the end; polygons are ordered by the emission index
 * of each cycle's first-emitted segment.  This is the order and the start vertex skimage's
 * contour assembly produces.  Islands run counter-clockwise in (x, y) with y down (positive
 * shoelace area), holes the other way.  Vertices are exact halves (float32).
 *
 * Two calls around one host read, like the RLE pair:
 *   mrx_contours_count:  d_row_seg [B, R, max_h+1] int32 scratch (kept for the write call);
 *                        d_seg_off [B*R+1] int64: on return (stream-ordered) d_seg_off[i] = number
 *                        of segments S of all instances before i = b*R + k, d_seg_off[B*R] = T.
 *   mrx_contours_write:  total_segments = T as read back;  with  o_i = d_seg_off[i]:
 *     d_scratch        int32 [2*T]                    (successor and end point of every segment)
 *     d_vertices       float32 [T + T/4, 2] (x, y)    instance i's polygons, one after the other,
 *                                                     from vertex o_i + o_i/4 (integer division)
 *     d_contour_len    int32 [T/4]                    vertices per polygon (closing one included),
 *                                                     instance i's from o_i/4
 *     d_inst_contours  int32 [B*R]                    number of polygons of instance i
 *   A cycle has at least 4 segments, so instance i has at most S_i/4 polygons and S_i + S_i/4
 *   vertices: the regions above never overlap.  (d_scratch / d_vertices / d_contour_len may be
 *   NULL when T == 0.)
 * Limits: max_h, max_w (largest H_b / W_b of the batch) <= MRX_CONTOUR_MAX_DIM
 * (MRX_E_UNSUPPORTED otherwise): the doubled padded coordinates fit 16 bits and an instance's
 * segment count (at most 2 (H+1)(W+1)) fits 31. */
#define MRX_CONTOUR_MAX_DIM 32766
int mrx_contours_count(const unsigned char *d_packed, const long long *d_packed_off,
                       const int *d_boxes, const int *d_counts, const int *d_geom,
                       int *d_row_seg, long long *d_seg_off, int B, int R, int max_h, int max_w,
                       void *stream);
int mrx_contours_write(const unsigned char *d_packed, const long long *d_packed_off,
                       const int *d_boxes, const int *d_counts, const int *d_geom,
                       int *d_row_seg, const long long *d_seg_off, int *d_scratch,
                       float *d_vertices, int *d_contour_len, int *d_inst_contours,
                       long long total_segments, int B, int R, int max_h, int max_w, void *stream);

/* ---------------------------------------------------------------- multi-GPU gather (8e) */
/* Peer-memory plumbing for the final gather of the canvases to rank 0 (one process per GPU).
 * Rank 0: mrx_peer_alloc a receive buffer + mrx_peer_export its 64-byte handle; other ranks:
 * mrx_peer_open the handle and pass the mapped address as the OUTPUT pointer of
 * mrx_mask_expand / mrx_mask_expand_packed -- the kernels store over NVLink straight into
 * rank 0's HBM.  mrx_peer_signal(flag, v, stream): after everything queued on `stream` so far,
 * store v to *flag (system scope, release).  mrx_peer_wait(flags, n, v, stream): `stream`
 * proceeds once flags[0..n) are all >= v (acquire).  Flags live in peer-allocated memory. */
#define MRX_PEER_HANDLE_BYTES 64
int mrx_peer_alloc(unsigned long long bytes, void **d_ptr);
int mrx_peer_free(void *d_ptr);
int mrx_peer_export(void *d_ptr, unsigned char *handle64);
int mrx_peer_open(const unsigned char *handle64, void **d_ptr);
int mrx_peer_close(void *d_ptr);
int mrx_peer_signal(unsigned int *d_flag, unsigned int value, void *stream);
int mrx_peer_wait(const unsigned int *d_flags, int n_flags, unsigned int value, void *stream);

#ifdef __cplusplus
}
#endif
#endif /* MRX_H_ */
