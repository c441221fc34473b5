/*
 * b200isp.h -- C ABI of the B200-native camera-ISP hot path.
 *
 * Drop-in boundary for uc-vision/taichi_image's `packed`, `bayer`, `tonemap`,
 * `interpolate` and `camera_isp` modules.  The reference has no FFI of its own:
 * its boundary is "Python wrapper -> cached Taichi kernel object called with
 * contiguous torch/numpy arrays" (e.g. bayer.py:202-219, packed.py:176-198).
 * Each entry point below replaces one such kernel object; the citation names it
 * (paths relative to /root/reference/taichi_image).
 *
 * Conventions
 *   - every pointer is a DEVICE pointer unless the name ends in `_host`;
 *   - images are row-major contiguous: (H, W) CFA planes, (H, W, 3) RGB,
 *     (H, W*3/2) bytes for packed12; sizes are in elements, never bytes;
 *   - launches are asynchronous on `stream` (a cudaStream_t); the caller owns
 *     all memory and keeps it alive until the stream has passed the call;
 *   - return value 0 = success, < 0 = b200isp_status; the calls never throw
 *     and never synchronise; b200isp_last_error() holds a thread-local message;
 *   - `workspace` is a caller-owned device buffer of at least
 *     b200isp_workspace_bytes() bytes, zero-initialised ONCE by the caller and
 *     then reused across calls on the same stream (the kernels leave it zeroed);
 *   - no global mutable state: thread-safe, multi-GPU by the caller's current
 *     device (cudaSetDevice / torch.cuda.device).
 */
#ifndef B200ISP_H
#define B200ISP_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define B200ISP_VERSION 103            /* 0.1.3 */
#define B200ISP_MAX_FRAMES 64          /* frames per batched call */
#define B200ISP_METRICS 9              /* camera_isp.py:102-115 */

typedef void* b200isp_stream;          /* cudaStream_t */

typedef enum {                         /* types.py:12-49 */
  B200ISP_U8 = 0, B200ISP_U16 = 1, B200ISP_I16 = 2, B200ISP_F16 = 3, B200ISP_F32 = 4
} b200isp_dtype;

typedef enum {                         /* bayer.py:75-79 (same values) */
  B200ISP_RGGB = 0, B200ISP_GRBG = 1, B200ISP_GBRG = 2, B200ISP_BGGR = 3
} b200isp_pattern;

typedef enum {                         /* interpolate.py:9-17 */
  B200ISP_T_NONE = 0, B200ISP_T_ROT90 = 1, B200ISP_T_ROT180 = 2, B200ISP_T_ROT270 = 3,
  B200ISP_T_TRANSPOSE = 4, B200ISP_T_FLIP_HORIZ = 5, B200ISP_T_FLIP_VERT = 6,
  B200ISP_T_TRANSVERSE = 7
} b200isp_transform_t;

typedef enum { B200ISP_TM_LINEAR = 0, B200ISP_TM_REINHARD = 1, B200ISP_TM_NONE = 2 } b200isp_tonemap_t;

typedef enum {
  B200ISP_OK = 0, B200ISP_E_ARG = -1, B200ISP_E_DTYPE = -2, B200ISP_E_SHAPE = -3,
  B200ISP_E_ALIGN = -4, B200ISP_E_CUDA = -5, B200ISP_E_FRAMES = -6, B200ISP_E_WORKSPACE = -7
} b200isp_status;

int         b200isp_version(void);
const char* b200isp_last_error(void);
size_t      b200isp_workspace_bytes(void);

/* ---- packed.py ---------------------------------------------------------- */
/* packed.py:59-89 encode12_kernel(in_type, scaled, ids_format)(values, encoded).
 * n_values even; encoded has n_values*3/2 bytes. */
int b200isp_encode12(const void* values, int in_dtype, int64_t n_values, uint8_t* encoded,
                     int scaled, int ids_format, b200isp_stream stream);
/* packed.py:122-131 decode12_kernel(out_type, scaled, ids_format)(encoded, out). */
int b200isp_decode12(const uint8_t* encoded, int64_t n_values, void* out, int out_dtype,
                     int scaled, int ids_format, b200isp_stream stream);
/* packed.py:36-44 then :12-20: re-pack IDS-layout 12-bit data into the standard layout (byte stream to byte
 * stream, n_bytes % 3 == 0) so that IDS frames can take b200isp_process_packed12. */
int b200isp_repack12_ids(const uint8_t* ids, uint8_t* standard, int64_t n_bytes, b200isp_stream stream);
/* packed.py:163-172 decode16_kernel(out_type, scaled)(encoded, out). */
int b200isp_decode16(const uint8_t* encoded, int64_t n_values, void* out, int out_dtype,
                     int scaled, b200isp_stream stream);

/* EXTENSION (SURVEY 8f-4 "10-bit packed"; the reference has no 10-bit format): MIPI CSI-2 RAW10, 5 bytes <-> 4 pixels --
 * bytes 0..3 = bits 9..2 of pixels 0..3, byte 4 = their bits 1..0 (pixel 0 in the lowest bit pair).  Value conventions of
 * packed.py:66-73 / :98-104 with 1023 in place of 4095.  n_values % 4 == 0; encoded has n_values*5/4 bytes. */
int b200isp_decode10(const uint8_t* encoded, int64_t n_values, void* out, int out_dtype,
                     int scaled, b200isp_stream stream);
int b200isp_encode10(const void* values, int in_dtype, int64_t n_values, uint8_t* encoded,
                     int scaled, b200isp_stream stream);

/* ---- bayer.py ----------------------------------------------------------- */
/* bayer.py:101-112 rgb_to_bayer_kernel(image, bayer, pixel_order). */
int b200isp_rgb_to_bayer(const void* rgb, void* bayer, int dtype, int height, int width,
                         int pattern, b200isp_stream stream);
/* bayer.py:179-190 bayer_to_rgb_kernel(pattern, correct_colors, in_dtype, out_dtype)(bayer, out).
 * ccm9_host: 9 row-major floats on the HOST, or NULL (no colour correction). */
int b200isp_bayer_to_rgb(const void* bayer, int in_dtype, void* rgb, int out_dtype,
                         int height, int width, int pattern, const float* ccm9_host,
                         b200isp_stream stream);

/* EXTENSION (north_star "bilinear demosaic"; the reference has only Malvar): 3x3 bilinear CFA interpolation with the
 * normalisation / CCM / clamp / cast rule of bayer.py:137-155 (mean of the in-bounds neighbours of each colour). */
int b200isp_bayer_to_rgb_bilinear(const void* bayer, int in_dtype, void* rgb, int out_dtype,
                                  int height, int width, int pattern, const float* ccm9_host,
                                  b200isp_stream stream);

/* ---- util.py / tonemap.py (stand-alone, per image) ---------------------- */
/* util.py:49-60 bounds_func: min/max over n_elems values -> bounds_out[2] (device). */
int b200isp_bounds(const void* src, int dtype, int64_t n_elems, float* bounds_out,
                   void* workspace, b200isp_stream stream);
/* tonemap.py:11-17 linear_func with bounds read from device memory (bounds[0]=min,[1]=max):
 * out = cast(clamp(((x-min)*(1/(max-min)))^(1/gamma),0,1)*scale[out_dtype]).
 * Used by tonemap.linear_kernel (tonemap.py:26-36) after b200isp_bounds and by the ISP
 * linear_kernel (camera_isp.py:220-227) with bounds = metrics[0:2]. */
int b200isp_linear(const void* src, int in_dtype, void* dst, int out_dtype, int64_t n_elems,
                   const float* bounds, float gamma, b200isp_stream stream);
/* tonemap.py:134-168 reinhard_kernel(in,out)(image,temp,dest,gamma,intensity,la,ca):
 * the five dependent passes of the stand-alone Reinhard operator, run as four reads of `src` that recompute the
 * normalised value / the map instead of keeping them in an f32 image (same arithmetic per value).
 * temp: NULL, or n_pixels*3 floats that receive the un-normalised Reinhard map (what the reference leaves in its
 * caller-owned temp image; costs one extra 12 B/px write). */
int b200isp_reinhard_standalone(const void* src, int in_dtype, float* temp, void* dst, int out_dtype,
                                int64_t n_pixels, float gamma, float intensity, float light_adapt,
                                float color_adapt, void* workspace, b200isp_stream stream);

/* ---- interpolate.py ----------------------------------------------------- */
/* interpolate.py:70-86 bilinear_kernel(in,out)(src,dst,scale); scale per axis (row, col). */
int b200isp_resize_bilinear(const void* src, int in_dtype, int src_h, int src_w,
                            void* dst, int out_dtype, int dst_h, int dst_w,
                            float scale_row, float scale_col, b200isp_stream stream);
/* EXTENSION (north_star "area resize"; no reference kernel): box filter over the source footprint. */
int b200isp_resize_area(const void* src, int in_dtype, int src_h, int src_w,
                        void* dst, int out_dtype, int dst_h, int dst_w, b200isp_stream stream);
/* interpolate.py:93-108 transform_kernel(dtype)(src,dst,transform); src is (H,W,3). */
int b200isp_transform(const void* src, void* dst, int dtype, int src_h, int src_w,
                      int transform, b200isp_stream stream);

/* ---- color/yuv_420.py (SURVEY 8f rank 2) -------------------------------- */
/* yuv_420.py:38-64 rgb_yuv420_kernel(in, out)(src, y_image, uv_image): rgb (H,W,3) -> one (3H/2, W) plane = Y rows
 * followed by the two (H/2, W/2) chroma planes.  matrix9_host = YCrCb_T_bgr (yuv_420.py:12-16), row-major, HOST. */
int b200isp_rgb_yuv420(const void* rgb, int in_dtype, void* yuv, int out_dtype, int height, int width,
                       const float* matrix9_host, b200isp_stream stream);
/* yuv_420.py:66-90 yuv420_rgb_kernel(in, out)(y_image, uv_image, rgb_image); matrix9_host = bgr_T_YCrCb (:18). */
int b200isp_yuv420_rgb(const void* yuv, int in_dtype, void* rgb, int out_dtype, int height, int width,
                       const float* matrix9_host, b200isp_stream stream);

/* ---- camera_isp.py (eager, per-stage; float RGB images of the ISP dtype) - */
/* camera_isp.py:82-99 load_16u / load_32f / load_16f: element-wise convert.
 * mode 0: out = cast(f32(u16)/65535)   (load_16u)
 * mode 1: out = cast(f32 in)           (load_32f)
 * mode 2: out = cast(f32(u16))         (load_16f as written, SURVEY 2.2 K10) */
int b200isp_load_convert(const void* src, void* dst, int out_dtype, int64_t n_elems, int mode,
                         b200isp_stream stream);
/* camera_isp.py:142-175 metering_kernel over stack([im[::stride, ::stride] for im in images]).
 * images_host: n_images device pointers (host array) of (H,W,3) tensors of `dtype` (F16|F32).
 * metrics: 9 floats on the device, updated in place: lerp(alpha, stats, prev). */
int b200isp_metering_update(const void* const* images_host, int n_images, int dtype,
                            int height, int width, int stride, float alpha, float* metrics,
                            void* workspace, b200isp_stream stream);
/* camera_isp.py:177-218 reinhard_kernel(image, output, metering, gamma, intensity, la, ca).
 * Like the reference, pass 1 overwrites `image` with the un-normalised map (ISP dtype). */
int b200isp_isp_reinhard(void* image, int dtype, void* output, int out_dtype, int64_t n_pixels,
                         const float* metrics, float gamma, float intensity, float light_adapt,
                         float color_adapt, void* workspace, b200isp_stream stream);

/* camera_isp.py:394-403: the same for a list of n_images same-size images (host arrays of device pointers),
 * one launch per pass for the whole list. */
int b200isp_isp_reinhard_batch(void* const* images_host, void* const* outputs_host, int n_images, int dtype,
                               int out_dtype, int64_t n_pixels, const float* metrics, float gamma,
                               float intensity, float light_adapt, float color_adapt, void* workspace,
                               b200isp_stream stream);

/* ---- fused path: packed12 frames -> tone-mapped RGB in one sweep --------- */
typedef enum { B200ISP_DEMOSAIC_MALVAR = 0, B200ISP_DEMOSAIC_BILINEAR = 1 } b200isp_demosaic_t;
typedef struct {
  int height, width;            /* sensor size; width % 8 == 0, height % 2 == 0 */
  int pattern;                  /* b200isp_pattern */
  int isp_dtype;                /* B200ISP_F16 (Camera16 rounding points) or B200ISP_F32 (Camera32) */
  int out_dtype;                /* U8 | U16 | F16 (tone-mapped) ; F16|F32 == isp_dtype for TM_NONE */
  int tonemap;                  /* b200isp_tonemap_t; TM_NONE = load_packed12 only (float RGB out) */
  int has_ccm;                  /* apply ccm (= color_correction * diag(white_balance)) */
  float ccm[9];                 /* row-major, camera_isp.py:360-369 */
  float gamma, intensity, light_adapt, color_adapt;   /* camera_isp.py:394-396 */
  int metering_stride;          /* camera_isp.py:251 (8) */
  float alpha;                  /* lerp weight of the PREVIOUS metrics: 0 on the first call,
                                   1 - moving_alpha afterwards (camera_isp.py:376-385) */
  int update_metering;          /* 1: run the two metering phases on these frames first */
  int rows_per_task;            /* 0 = default */
  int demosaic;                 /* b200isp_demosaic_t: 0 = Malvar-He-Cutler (bayer.py:30-55), 1 = bilinear (extension) */
  int out_yuv420;               /* 1: every output is a planar YUV 4:2:0 image, (3H/2, W) u8 (color/yuv_420.py:95-118), instead
                                   of RGB -- Camera16 + Reinhard + u8 with reinhard_scratch only; other combinations fail */
  int out_height, out_width;    /* > 0: bilinear resize of the demosaiced image BEFORE metering / tone map (camera_isp.py:302-315,
                                   :371-373; interpolate.py:59-66) fused into the pass: outputs are (out_height, out_width, 3) */
  float scale_r, scale_c;       /* source position of output (ro, co) = (ro / scale_r, co / scale_c) in f32, interpolate.py:60 */
  int resize_gather;            /* 1: force the per-output-pixel gather instead of the resizing sweep (testing / profiling) */
  int out_pitch;                /* elements per OUTPUT row; 0 = dense (3 * width).  Larger: every output frame is a tile of a bigger
                                   image (the rig's camera grid, scripts/tonemap_scan.py:91-100) -- the sweep writes the tile in place */
  int flip;                     /* ISP transform applied inside the call (interpolate.py:36-56): bit 0 = mirror columns, bit 1 = mirror
                                   rows, bit 2 = transpose (output (W, H), out_pitch counts elements of ITS rows):
                                   flip_horiz 1, flip_vert 2, rotate_180 3, transpose 4, rotate_270 5, rotate_90 6, transverse 7.
                                   1..3 are applied by the sweep's store (no resize, no YUV).  4..7 are applied by the normalise pass
                                   of a one-sweep Reinhard -> u8 form only: they need height % 8 == 0, height >= 16, a call for which
                                   b200isp_reinhard_scratch_bytes is not 0 and that scratch; any other call with bit 2 fails with
                                   B200ISP_E_ARG (run b200isp_transform on its result instead) */
  int reinhard_mode;            /* Camera32 Reinhard -> u8 with reinhard_scratch: 0 = one sweep that also stores the map as u16 fixed point
                                   + a normalise pass where it applies (b200isp_reinhard_scratch_bytes; u8 within 1 LSB of the
                                   two-sweep result, frames whose map leaves [0, 1) are redone exactly), 1 = always the exact max
                                   sweep + write sweep; any other value also takes the exact form */
  int ids_layout;               /* packed layout of the input frames: 0 = standard (packed.py:23-31), 1 = IDS (packed.py:36-44),
                                   decoded inside the row loader (4 instead of 2 instructions per sample, no re-pack pass) */
  void* profile_start;          /* optional cudaEvent_t pair recorded on `stream` immediately before / after */
  void* profile_stop;           /*   the dominant streaming kernel (bench.py's live roofline timing); NULL = off */
  void* meter_cache;            /* optional device scratch: >= n_frames*ceil(H/stride)*ceil(W/stride)*12 bytes; the second */
  size_t meter_cache_bytes;     /*   metering phase then re-reads the phase-1 samples instead of recomputing them */
  void* reinhard_scratch;       /* optional device scratch of b200isp_reinhard_scratch_bytes(params, n_frames) bytes: Reinhard then */
  size_t reinhard_scratch_bytes;/*   runs ONE sweep that stores the map (camera_isp.py:211) + an element-wise normalise / quantise
                                     pass.  YUV 4:2:0 output and Reinhard with resize require it */
} b200isp_fused_params;

/* camera_isp.py:333-340 load_packed12 + :376-385 update_metering + :394-413 tonemap_* over a
 * list of frames, without materialising the CFA or the float RGB.
 * packed_host / out_host: n_frames device pointers each (host arrays).
 * metrics: 9 floats (device), read and (if update_metering) updated in place. */
int b200isp_process_packed12(const uint8_t* const* packed_host, void* const* out_host, int n_frames,
                             const b200isp_fused_params* params, float* metrics,
                             void* workspace, b200isp_stream stream);
/* The bytes of reinhard_scratch with which b200isp_process_packed12(params, n_frames frames) runs its one-sweep Reinhard
 * form; 0 when that call uses no scratch (no Reinhard tone map, or the exact two-sweep form) or refuses the parameter
 * block whatever scratch it gets.  Reads only the scalar fields of params and makes no CUDA call. */
size_t b200isp_reinhard_scratch_bytes(const b200isp_fused_params* params, int n_frames);

/* EXTENSION (north_star "percentile histogram"; no reference counterpart): luminance histogram of the metering
 * samples (n_samples RGB float triples as written to fused_params.meter_cache), bin = min(bins-1, trunc(gray*bins)),
 * and percentiles of it: out[k] = upper edge of the first bin whose cumulative count reaches percents[k] %.
 * hist / percents / out are device pointers. */
int b200isp_sample_histogram(const float* samples, int64_t n_samples, int bins, uint32_t* hist, b200isp_stream stream);
int b200isp_histogram_percentiles(const uint32_t* hist, int bins, const float* percents, int n_percents, float* out,
                                  b200isp_stream stream);

/* ---- multi-GPU shared exposure (SURVEY 8e; no reference counterpart: the reference is single-GPU) ----
 * The reference meters all cameras of a time step jointly (camera_isp.py:168-175).  With one camera
 * shard per GPU the two dependent reductions of metering_kernel (camera_isp.py:149-166) are split at
 * their exchange points; between the calls the host all-gathers the per-rank records
 * (torch.distributed / NCCL, <= 32 bytes per rank) and every rank folds them in rank order, so all
 * ranks end with bit-identical metrics:
 *   record 1 (2 floats): {min, max} over this rank's samples
 *   record 2 (8 floats): {log_min, log_max, sum_log, sum_gray, sum_r, sum_g, sum_b, n_samples}
 *   phase1  -> rec1;  all_gather -> gathered1 [world][2]
 *   phase2(gathered1, alpha, metrics_prev) -> rec2 w.r.t. the blended joint bounds;  all_gather -> gathered2 [world][8]
 *   finalize(gathered1, gathered2, alpha, prev) -> metrics_out = lerp(alpha, joint stats, metrics_prev)
 *                                                  (metrics_out may be the same buffer as metrics_prev)
 * With world == 1 the three calls equal b200isp_metering_update. */
#define B200ISP_REC1 2
#define B200ISP_REC2 8
int b200isp_metering_phase1(const void* const* images_host, int n_images, int dtype, int height, int width,
                            int stride, float* rec1, void* workspace, b200isp_stream stream);
int b200isp_metering_phase2(const void* const* images_host, int n_images, int dtype, int height, int width,
                            int stride, const float* gathered1, int world, float alpha,
                            const float* metrics_prev, float* rec2, void* workspace, b200isp_stream stream);
int b200isp_metering_finalize(const float* gathered1, const float* gathered2, int world, float alpha,
                              const float* metrics_prev, float* metrics_out, b200isp_stream stream);
/* the same two phases straight from packed12 frames (the sampler of b200isp_process_packed12);
 * params->alpha, metering_stride, meter_cache as in the fused call. */
int b200isp_meter_packed12_phase1(const uint8_t* const* packed_host, int n_frames,
                                  const b200isp_fused_params* params, float* rec1,
                                  void* workspace, b200isp_stream stream);
int b200isp_meter_packed12_phase2(const uint8_t* const* packed_host, int n_frames,
                                  const b200isp_fused_params* params, const float* gathered1, int world,
                                  const float* metrics_prev, float* rec2, void* workspace, b200isp_stream stream);

/* ---- peer-memory exchange of the two records over NVLink (csrc/exchange.cu) ----
 * One process per GPU.  Every rank owns a small mailbox in device memory (b200isp_mailbox_create), exports it
 * with a 64-byte CUDA IPC handle, and opens the other ranks' mailboxes (b200isp_mailbox_open).  An exchange is
 * two 1-warp kernels on the metering stream -- post: write the record into every rank's mailbox and publish a
 * sequence number; wait: spin (bounded, ~2 s) until every rank's number has arrived, then copy the records to
 * `gathered` in rank order -- no host call, no NCCL, capturable in a CUDA graph.  kind = 1 | 2 (record 1 | 2). */
size_t b200isp_mailbox_bytes(int world);
int b200isp_mailbox_create(int world, void** mailbox_out, void* ipc_handle_out64);
int b200isp_mailbox_open(const void* ipc_handle64, void** mailbox_out);
int b200isp_mailbox_close(void* mailbox, int is_owner);
int b200isp_mailbox_post(const float* rec, int kind, void* const* peers_host, int world, int rank,
                         b200isp_stream stream);
int b200isp_mailbox_wait(void* mailbox, int kind, int world, float* gathered, b200isp_stream stream);
int b200isp_mailbox_exchange(const float* rec, int kind, void* const* peers_host, int world, int rank,
                             float* gathered, b200isp_stream stream);
/* 1 if a bounded wait has expired on this mailbox (a peer never posted); synchronises `stream` */
int b200isp_mailbox_error(const void* mailbox, int world, b200isp_stream stream);

/* The whole joint metering update (camera_isp.py:376-385 over the frames of ALL ranks) in two launches: the two
 * metering kernels run the record exchanges themselves (last block: post to every rank's mailbox, wait for every
 * rank's record, fold).  peers_host = the `world` mailbox pointers (entry `rank` = own).  params as for
 * b200isp_meter_packed12; every rank must call it once per time step, in the same order. */
int b200isp_meter_packed12_shared(const uint8_t* const* packed_host, int n_frames,
                                  const b200isp_fused_params* params, void* const* peers_host, int world, int rank,
                                  const float* metrics_prev, float* metrics_out, void* workspace, b200isp_stream stream);

/* camera_isp.py:376-385 update_metering on its own, straight from packed12 frames (what
 * b200isp_process_packed12 runs first when params->update_metering is set), with separate input / output
 * metrics so that the update for the NEXT batch can run on a side stream while the sweep of the current
 * batch still reads the current metrics ("look-ahead metering", camera_isp.process_packed12(lookahead=...)).
 * metrics_out may equal metrics_prev.  cooperative = 1: one cooperative launch (fastest on an idle GPU);
 * 0: two ordinary launches whose CTAs can interleave with a concurrently running sweep. */
int b200isp_meter_packed12(const uint8_t* const* packed_host, int n_frames,
                           const b200isp_fused_params* params, const float* metrics_prev,
                           float* metrics_out, int cooperative, void* workspace, b200isp_stream stream);

#ifdef __cplusplus
}
#endif
#endif /* B200ISP_H */
