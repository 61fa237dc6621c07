/* bevk.h -- C ABI of libbevk.so, the B200 (sm_100a) surround-BEV warping engine.
 *
 * Drop-in boundary for the per-pixel hot path of dyfcalid/CameraCalibration.  The
 * reference has no FFI of its own (it is pure Python over OpenCV); each entry
 * point below replaces the OpenCV call(s) the reference makes at the cited
 * file:line (paths relative to the reference tree).  INTEGRATION.md shows the
 * ctypes binding a maintainer of the reference would add.
 *
 * Conventions
 *   - plain C, no torch / C++ types; every call returns 0 on success or a negative
 *     bevk_status; bevk_last_error() gives the thread-local message.
 *   - images are uint8, interleaved channels (BGR as cv2.imread gives), row-major,
 *     explicit row stride in bytes.  3x3 matrices are row-major double[9].
 *   - "host" entry points take host pointers and do H2D / D2H inside the call;
 *     "_device" entry points take device pointers on the ctx's device and only
 *     enqueue work on the ctx stream (no synchronisation).
 *   - the caller owns every buffer it passes in (inputs and outputs).
 *   - a ctx is not thread-safe; use one ctx per thread.  No CPU fallback exists:
 *     without a CUDA device bevk_ctx_create fails.
 */
#ifndef BEVK_H
#define BEVK_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct bevk_ctx bevk_ctx;

typedef enum {
  BEVK_OK = 0,
  BEVK_ERR_ARG = -1,         /* bad argument / call order                       */
  BEVK_ERR_CUDA = -2,        /* CUDA runtime error (message has the details)    */
  BEVK_ERR_OOM = -3,
  BEVK_ERR_UNSUPPORTED = -4
} bevk_status;

enum { BEVK_INTER_NEAREST = 0, BEVK_INTER_LINEAR = 1 };          /* cv2.INTER_* values */
enum { BEVK_MAPS_UNDISTORT = 0, BEVK_MAPS_BEV = 1 };
enum { BEVK_MODEL_FISHEYE = 0, BEVK_MODEL_PINHOLE = 1 };
enum { BEVK_FLAG_BALANCE = 1 };                                   /* bevk_bev_run flags */
#define BEVK_MAX_CAMERAS 8

int bevk_version(void);
const char *bevk_last_error(void);

/* ---- context ------------------------------------------------------------- */
int bevk_ctx_create(int device, bevk_ctx **out);
int bevk_ctx_destroy(bevk_ctx *ctx);
/* Run on an externally owned cudaStream_t (e.g. torch's current stream); NULL
 * restores the ctx's own stream. */
int bevk_ctx_set_stream(bevk_ctx *ctx, void *cuda_stream);
int bevk_ctx_sync(bevk_ctx *ctx);
/* PCI bus id ("0000:1b:00.0") of a CUDA device: lets a multi-process launcher bind each rank to the CPUs and memory
 * of its GPU's NUMA node (/sys/bus/pci/devices/<id>/local_cpulist) before it allocates page-locked buffers. */
int bevk_device_pci_bus_id(int device, char *out, int len);
/* Pinned host memory for callers who want full-rate PCIe copies. */
int bevk_host_alloc(uint64_t bytes, void **out);
int bevk_host_free(void *p);

/* ---- K1: undistortion maps ------------------------------------------------
 * cv2.fisheye.initUndistortRectifyMap(K, D, eye(3), P, (w,h), CV_16SC2)
 *   SurroundBirdEyeView/surroundBEV.py:98-103, Tools/undistort.py:50-52,
 *   IntrinsicCalibration/intrinsicCalib.py:98-103            (model FISHEYE, 4 coeffs)
 * cv2.initUndistortRectifyMap(K, D5, eye(3), P, (w,h), CV_16SC2)
 *   IntrinsicCalibration/intrinsicCalib.py:158-163           (model PINHOLE, 5 coeffs)
 * map1: int16[h][w][2] (x,y integer part), map2: uint16[h][w] (fy*32+fx).        */
int bevk_undistort_map(bevk_ctx *ctx, int model, const double K[9], const double *D, int n_dist,
                       const double P[9], int w, int h, int16_t *map1, uint16_t *map2);

/* ---- K3: cv2.remap(src, map1, map2, interp), BORDER_CONSTANT 0 --------------
 *   surroundBEV.py:110-111,116-117; undistort.py:66; intrinsicCalib.py:193-195
 * channels in {1,3,4}; map2 may be NULL for NEAREST with integer maps.          */
int bevk_remap(bevk_ctx *ctx, const uint8_t *src, int sw, int sh, int64_t sstride, int channels,
               const int16_t *map1, const uint16_t *map2, int dw, int dh,
               uint8_t *dst, int64_t dstride, int interp);

/* ---- cached-map undistortion (the per-frame call of InCalibrator.undistort /
 * Camera.undistort / Tools/undistort.py's loop).  The map is built on the device
 * once per "slot" and never leaves HBM; each frame is one H2D, one gather kernel,
 * one D2H.  fused!=0 skips the map entirely and evaluates the camera model inside
 * the gather kernel (no 6 B/px map traffic; same results).                      */
int bevk_undistorter_set(bevk_ctx *ctx, int slot, int model, const double K[9], const double *D, int n_dist,
                         const double P[9], int dw, int dh, int fused);
int bevk_undistorter_maps(bevk_ctx *ctx, int slot, int16_t *map1, uint16_t *map2);   /* D2H, for parity tests */
/* dw x dh: the destination size the caller allocated; must equal the slot's map size (checked, so a stale handle to
 * a slot that was re-set can never make the library write past dst). */
int bevk_undistort(bevk_ctx *ctx, int slot, const uint8_t *src, int sw, int sh, int64_t sstride, int channels,
                   uint8_t *dst, int dw, int dh, int64_t dstride, int interp);

/* ---- K4: cv2.warpPerspective(src, H, (dw,dh), flags=interp), border 0 --------
 *   ExtrinsicCalibration/extrinsicCalib.py:166-169, surroundBEV.py:113-114      */
int bevk_warp_perspective(bevk_ctx *ctx, const uint8_t *src, int sw, int sh, int64_t sstride, int channels,
                          const double H[9], uint8_t *dst, int dw, int dh, int64_t dstride, int interp);
/* The same call applied to a 16SC2 / 16UC1 map pair (Camera.get_bev_maps,
 * surroundBEV.py:105-108): float-table bilinear, rounded, saturated.            */
int bevk_warp_maps(bevk_ctx *ctx, const int16_t *map1, const uint16_t *map2, int sw, int sh,
                   const double H[9], int dw, int dh, int16_t *out1, uint16_t *out2);

/* ---- the BEV engine (BevGenerator, surroundBEV.py:282-325) ----------------- */
int bevk_bev_configure(bevk_ctx *ctx, int n_cam, int frame_w, int frame_h, int bev_w, int bev_h);
/* Camera.__init__ (surroundBEV.py:82-108): K, D, P = camera_mat_dst, undistorted
 * size (und_w x und_h) and H.  Builds the camera's BEV LUT on the device with the
 * reference's semantics (the undistortion maps themselves warped by H, SURVEY A4)
 * without materialising the und_w x und_h intermediate map.                      */
int bevk_bev_set_camera(bevk_ctx *ctx, int cam, const double K[9], const double D[4], const double P[9],
                        int und_w, int und_h, const double H[9]);
/* Inject / read back a camera's BEV maps (int16[bev_h][bev_w][2], uint16[bev_h][bev_w]). */
int bevk_bev_set_maps(bevk_ctx *ctx, int cam, const int16_t *map1, const uint16_t *map2);
int bevk_bev_get_maps(bevk_ctx *ctx, int cam, int16_t *map1, uint16_t *map2);
/* Mask / BlendMask (surroundBEV.py:119-162, 164-280): uint8[bev_h][bev_w]; 0/255 for
 * the plain path, 0..255 blend weights otherwise (weight = float32(mask/255.0)). */
int bevk_bev_set_mask(bevk_ctx *ctx, int cam, const uint8_t *mask);
/* Interpolation of raw2bev's cv2.remap (surroundBEV.py:116-117 uses INTER_LINEAR; INTER_NEAREST is
 * offered with cv2.remap's exact fixed-point-map semantics).  Call before bevk_bev_finalize. */
int bevk_bev_set_interpolation(bevk_ctx *ctx, int interp);
/* BlendMask.get_blend_mask (surroundBEV.py:270-277) for the 4-camera layout, on the
 * device: polys = the four *unblended* 6-gon masks (uint8[4][bev_h][bev_w], order
 * front,back,left,right), lines = the 8 seam segments FL,FR,BL,BR,LF,LB,RF,RB as
 * int32[8][2][2].  Writes the four blend masks to out (same layout as polys).     */
int bevk_blend_masks(bevk_ctx *ctx, const uint8_t *polys, const int32_t *lines, int bev_w, int bev_h, uint8_t *out);
/* Compile LUTs + masks into the tile plan the fused kernel consumes. */
int bevk_bev_finalize(bevk_ctx *ctx);

/* BevGenerator.__call__ (surroundBEV.py:312-325) for `batch` frame-sets.
 * srcs: batch*n_cam host pointers (frame-set major: set0 cam0..camN-1, set1 ...),
 *       each uint8[frame_h][frame_w][3] with row stride src_stride bytes.
 * car : NULL or uint8[bev_h][bev_w][3] (dense), added after colour balance.
 * out : batch canvases uint8[bev_h][bev_w][3], dense, canvas b at out + b*bev_h*bev_w*3. */
int bevk_bev_run(bevk_ctx *ctx, const uint8_t *const *srcs, int64_t src_stride, int batch,
                 const uint8_t *car, int flags, uint8_t *out);
/* Device-resident variant: d_srcs is a DEVICE array of batch*n_cam device pointers
 * (dense frames, row stride frame_w*3); d_car NULL or device; d_out device.  Only
 * enqueues on the ctx stream.                                                    */
int bevk_bev_run_device(bevk_ctx *ctx, const void *d_srcs, int batch, const void *d_car, int flags, void *d_out);
/* Same with the table on the HOST: frames[batch*n_cam] are DEVICE pointers to dense frames (e.g. the
 * data pointers of torch / CuPy / NVDEC buffers; 4-byte aligned).  The library keeps the device copy of
 * the table and re-uploads it only when its contents change, so streaming into fixed buffers costs no
 * copy per call.  Replaces the host frames of BevGenerator.__call__ (surroundBEV.py:312-325) when the
 * decoder already left them on the GPU (SURVEY 8f-2).  Only enqueues on the ctx stream.             */
int bevk_bev_run_frames(bevk_ctx *ctx, const void *const *frames, int batch, const void *d_car, int flags, void *d_out);
/* Frame STACK on the device: frame i (= frame-set i / n_cam, camera i % n_cam) is the dense uint8[frame_h][frame_w][3]
 * at d_frames + i * frame_stride -- e.g. one uint8[batch][n_cam][H][W][3] tensor, or a decoder's surface pool.
 * Replaces the frames of BevGenerator.__call__ (surroundBEV.py:312-325, the cv2.remap inputs of :116-117).  With a
 * 16-byte aligned base and stride (and a row pitch frame_w*3 that is a multiple of 16) the TMA-staged kernel runs:
 * per (canvas tile, camera) one cp.async.bulk.tensor box per frame-set into shared memory; otherwise the
 * pointer-table gather.  bevk_bev_run_frames takes this path by itself when its table describes a stack, and so
 * does bevk_bev_run for its staging buffers.  Only enqueues on the ctx stream.                           */
int bevk_bev_run_stack(bevk_ctx *ctx, const void *d_frames, int64_t frame_stride, int batch, const void *d_car, int flags,
                       void *d_out);
/* Per-camera partial canvases for camera-sharded multi-GPU runs: rank r renders only
 * cameras [cam_lo, cam_hi) into d_out (zero elsewhere); the saturating sum of the
 * ranks' partials equals the full canvas (balance is not supported in this mode). */
int bevk_bev_run_device_cams(bevk_ctx *ctx, const void *d_srcs, int batch, int cam_lo, int cam_hi, void *d_out);
/* The same over a frame stack (see bevk_bev_run_stack). */
int bevk_bev_run_stack_cams(bevk_ctx *ctx, const void *d_frames, int64_t frame_stride, int batch, int cam_lo, int cam_hi,
                            void *d_out);
/* Saturating sum of n partial canvases (device), optional car, into d_out. */
int bevk_sat_sum_device(bevk_ctx *ctx, const void *const *d_parts_host_array, int n, uint64_t bytes,
                        const void *d_car, void *d_out);

/* ---- stand-alone forms of the reference's per-pixel helpers ----------------------
 * Mask.__call__ / BlendMask.__call__ (surroundBEV.py:161-162, 279-280): dense BGR image
 * uint8[h][w][3], mask uint8[h][w]; blend=0: mask ? px : 0, blend=1: trunc(px*f32(mask/255)). */
int bevk_apply_mask(bevk_ctx *ctx, const uint8_t *img, const uint8_t *mask, int w, int h, int blend, uint8_t *out);
/* color_balance (surroundBEV.py:43-55) of one dense BGR image. */
int bevk_color_balance(bevk_ctx *ctx, const uint8_t *img, int w, int h, uint8_t *out);
/* luminance_balance (surroundBEV.py:57-79) of n (<= 8) dense BGR frames of equal size. */
int bevk_luminance_balance(bevk_ctx *ctx, const uint8_t *const *imgs, int n, int w, int h, uint8_t *const *outs);

/* Introspection for tests / bench */
int bevk_bev_plan_info(bevk_ctx *ctx, int64_t *n_tiles, int64_t *n_items, int64_t *lut_bytes);
/* Bytes bevk_bev_run moves over PCIe per frame-set for the given flags: host->device (without
 * BALANCE only the rectangle of each frame its camera's LUT can sample is uploaded; with BALANCE
 * the whole frames, because the V means cover them) and device->host (the canvas). */
int bevk_bev_host_copy_bytes(bevk_ctx *ctx, int flags, int64_t *h2d_per_frame_set, int64_t *d2h_per_frame_set);
/* Host->device bytes the last bevk_bev_run call actually moved (page-locked frames are ingested span
 * by span by the SMs, pageable ones by DMA rectangles, BALANCE uploads whole frames). */
int64_t bevk_bev_last_h2d_bytes(bevk_ctx *ctx);
/* Which fused kernel the last BEV call launched: 1 = k_bev (pointer-table gather), 2 = k_bev_tma (TMA-staged). */
int bevk_bev_last_path(bevk_ctx *ctx);
/* The TMA-staged kernel's plan: work items, tensor-map box shapes, bytes one frame-set's boxes deliver, LUT entries
 * served from staged boxes / by global gathers.  All zero when the plan does not exist (row pitch not a multiple of
 * 16 bytes, or the environment variable BEVK_TMA=0 at bevk_bev_finalize, which leaves every call to k_bev). */
int bevk_bev_tma_plan_info(bevk_ctx *ctx, int64_t *n_items, int64_t *n_shapes, int64_t *box_bytes, int64_t *tma_entries,
                           int64_t *gather_entries);
/* ---- multi-GPU sharding: one process (one ctx) per GPU ---------------------------------------------------
 * The reference is a single process (no collective anywhere); the path shards two ways:
 *   BEVK_SHARD_FRAMES   every rank renders its own frame-sets with a replica of the plan -- no exchange at all;
 *   BEVK_SHARD_CAMERAS  rank r renders cameras [lo_r, hi_r) (contiguous blocks) of EVERY frame-set into a slab -- the
 *                       tile-aligned bounding box of the union of their masks -- ONE ncclAllGather moves the slabs
 *                       over NVLink, and each rank composes them with the saturating sum, which is exact because
 *                       the cv2.add chain of BevGenerator.__call__ (surroundBEV.py:316-320) is order-independent.
 * NCCL is dlopen'ed (libnccl.so.2) on first use.  Call order: bevk_bev_finalize, bevk_shard_configure on every rank,
 * bevk_shard_unique_id on ONE rank, its 128 bytes carried to the others by the launcher (file, MPI, torch.distributed),
 * bevk_shard_connect on every rank, then bevk_bev_run_sharded per step.  All work is enqueued on the ctx stream. */
enum { BEVK_SHARD_FRAMES = 0, BEVK_SHARD_CAMERAS = 1 };
int bevk_shard_configure(bevk_ctx *ctx, int policy, int rank, int world);
int bevk_shard_unique_id(void *id128, int len);
int bevk_shard_connect(bevk_ctx *ctx, const void *id128, int len);
/* Partition and slab geometry of `rank`: its cameras [cam_lo, cam_hi), its slab rectangle {x0, y0, x1, y1} in canvas
 * pixels, and the (padded, equal for all ranks) bytes of one frame-set's slab. */
int bevk_shard_info(bevk_ctx *ctx, int rank, int *cam_lo, int *cam_hi, int32_t rect[4], int64_t *slab_bytes);
/* BevGenerator.__call__ over a frame stack (see bevk_bev_run_stack) under the configured policy.  CAMERAS: every rank
 * passes the same batch; only the frames of its own cameras are read; every rank ends with all canvases in d_out. */
int bevk_bev_run_sharded(bevk_ctx *ctx, const void *d_frames, int64_t frame_stride, int batch, const void *d_car, int flags,
                         void *d_out);
/* CAMERAS policy, fused compute + exchange: frame-set b is OWNED by rank b % world.  Every rank renders its cameras'
 * slabs of all frame-sets and the fused kernel's write-out stores each slab straight into the owner's receive buffer
 * over NVLink (peer memory mapped with CUDA IPC); one 4-byte all-gather per step is the barrier, then each rank composes
 * the canvases it owns (d_out_own[*n_own][bev_h][bev_w][3], frame-sets rank, rank+world, ...).  Per step a rank sends
 * (and receives) (world-1)/world of one slab set, instead of receiving world-1 whole slab sets as the all-gather does.
 * Setup after bevk_shard_connect: bevk_shard_prepare(batch) on every rank gives a 64-byte handle; the launcher gathers
 * the handles of all ranks (rank order, world x 64 bytes) and gives them to bevk_shard_attach.  Frames must be a
 * 16-byte friendly stack (the TMA-staged kernel does the stores). */
int bevk_shard_prepare(bevk_ctx *ctx, int batch, void *handle64);
int bevk_shard_attach(bevk_ctx *ctx, const void *handles);
int bevk_bev_run_scattered(bevk_ctx *ctx, const void *d_frames, int64_t frame_stride, int batch, const void *d_car, int flags,
                           void *d_out_own, int *n_own);
/* Bytes this rank received (all-gather) or stored into its peers (scattered) over NVLink in the last sharded call. */
int64_t bevk_shard_last_link_bytes(bevk_ctx *ctx);
/* The two halves of the CAMERAS policy on their own (tests, custom exchanges): render the slabs of rank `as_rank`
 * into d_slabs[as_rank][batch][slab_bytes]; compose d_slabs[world][batch][slab_bytes] (+ car) into canvases. */
int bevk_shard_render(bevk_ctx *ctx, const void *d_frames, int64_t frame_stride, int batch, int as_rank, void *d_slabs);
int bevk_shard_compose(bevk_ctx *ctx, const void *d_slabs, int batch, const void *d_car, void *d_out);

/* ---- JPEG ingest on the device ------------------------------------------------------------------------------
 * Replaces cv2.imread in front of the path (surroundBEV.py:328-332, Tools/undistort.py:65): n baseline JPEG streams
 * (host memory) are decoded by nvJPEG (dlopen'ed on first use) into frames 0..n-1 of a device frame stack, BGR
 * interleaved, row pitch width*3 -- the layout bevk_bev_run_stack and the undistort entry points read.  Only the
 * compressed bytes cross PCIe.  Every stream must decode to width x height.  The pixels are nvJPEG's, which differ from
 * libjpeg-turbo's (cv2) by the decoders' IDCT / upsampling rounding; everything downstream is bit-exact on them.
 * The Huffman stage runs on the calling thread; GPU work is enqueued on the ctx stream. */
int bevk_jpeg_decode(bevk_ctx *ctx, const uint8_t *const *jpegs, const uint64_t *sizes, int n, int width, int height,
                     void *d_frames, int64_t frame_stride);

/* BevGenerator.__call__ (surroundBEV.py:312-325) on JPEG streams: jpegs[batch*n_cam] in frame-set-major order as in
 * bevk_bev_run; decoded on the device, rendered, canvases copied to `out` (host).  Synchronises. */
int bevk_bev_run_jpeg(bevk_ctx *ctx, const uint8_t *const *jpegs, const uint64_t *sizes, int batch, const uint8_t *car, int flags,
                      uint8_t *out);

/* ---- CUDA graphs over the device-pointer entry points ------------------------------------------------
 * Everything the "_device" / "_stack" / "_frames" entry points enqueue on the ctx stream between begin and end is
 * captured (stream capture) instead of executed, instantiated once, and replayed `times` times by one call --
 * BevGenerator.__call__ (surroundBEV.py:312-325) for a fixed set of device buffers costs one graph launch per
 * frame-set instead of up to five kernel launches and two memsets (BALANCE), and a host that stalls between calls
 * cannot starve the GPU.  Run the same calls once before capturing: a call that has to allocate or build tables
 * inside a capture fails, and bevk_graph_end reports it.  Host-pointer entry points cannot be captured.       */
int bevk_graph_begin(bevk_ctx *ctx);
int bevk_graph_end(bevk_ctx *ctx, int *graph_id);
int bevk_graph_launch(bevk_ctx *ctx, int graph_id, int times);
int bevk_graph_destroy(bevk_ctx *ctx, int graph_id);
/* Kernel launches issued by this ctx since creation (bench "gpu_launches"). */
int64_t bevk_launch_count(bevk_ctx *ctx);
/* Milliseconds spent in the last bevk_bev_run_device call's kernels, measured with
 * CUDA events on the ctx stream (synchronises). */
int bevk_last_kernel_ms(bevk_ctx *ctx, float *ms);

#ifdef __cplusplus
}
#endif
#endif /* BEVK_H */
