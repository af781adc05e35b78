/*
 * vsc_b200.h — C ABI of libvsc_b200.so: the B200 (sm_100a) implementation of
 * Video-Stereo-Converter's SBS generation hot path.
 *
 * This is the drop-in boundary.  Every entry point replaces a piece of the reference's
 * Python interface in /root/reference/helper/stereo_core.py (cited per function); the
 * Python host shim (video-stereo-converter_b200/vsc_b200/stereo_core.py) binds them with
 * ctypes and re-exposes the reference's own names (StereoParams, StereoGenerator.process_frame,
 * ...).  INTEGRATION.md shows the binding a maintainer of the reference would add.
 *
 * Conventions: plain pointers and sizes only (no torch types); every function returns 0 on
 * success or a negative VSC_E_* code and never throws; vsc_last_error() returns a
 * thread-local, human-readable message for the last failure.  There is NO CPU fallback: with no
 * usable CUDA device vsc_create fails.
 */
#ifndef VSC_B200_H
#define VSC_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define VSC_ABI_VERSION 1

enum {
    VSC_OK = 0,
    VSC_E_INVALID = -1,   /* bad argument (NULL, size, dtype)                                  */
    VSC_E_PARAMS = -2,    /* stereo parameters give an invalid crop window: the reference raises
                             RuntimeError from _sharpen_image's reflect pad (stereo_core.py:291-296) */
    VSC_E_CUDA = -3,      /* CUDA runtime error; callers map this to exit code 100
                             (sbs_generator.py:41,317 GPU_ERROR_EXIT_CODE)                       */
    VSC_E_NOMEM = -4,
    VSC_E_STATE = -5      /* slot busy / not submitted                                          */
};

/* depth element types accepted by process_frame (stereo_core.py:254,328: any cv2.resize-able
 * numeric array that is then cast to float32) */
enum { VSC_DEPTH_U8 = 0, VSC_DEPTH_U16 = 1, VSC_DEPTH_F32 = 2 };

/* StereoParams (stereo_core.py:193-202) == config.json "stereo" block
 * (helper/config_manager.py:43-54).  Doubles, because the reference computes its integer
 * geometry from Python floats (stereo_core.py:249-251,275-289). */
typedef struct vsc_params {
    double max_disparity;      /* 50.0  */
    double convergence;        /* -10.0 */
    double super_sampling;     /* 3.0   */
    double edge_softness;      /* 20.0  */
    double artifact_smoothing; /* 1.0   */
    double depth_gamma;        /* 0.2   */
    double sharpen;            /* 14.0  */
} vsc_params;

/* Integer geometry of one frame, exactly as process_frame derives it
 * (stereo_core.py:249-251, :275-289, :364-365). */
typedef struct vsc_geom {
    int32_t height, width;          /* input frame                                           */
    int32_t stretched_w;            /* int(W * (1 + (2*md + |conv|)/W))                      */
    int32_t ss_h, ss_w;             /* super-sampled grid int(H*SS), int(stretched_w*SS)     */
    int32_t left_crop, right_crop;  /* first kept column of each eye on the SS grid          */
    int32_t crop_w;                 /* kept columns per eye on the SS grid                   */
    int32_t blur_k;                 /* depth blur taps (0 = off)  stereo_core.py:384         */
    int32_t bilateral_d;            /* bilateral diameter (0 = off) stereo_core.py:409       */
    int32_t super_sampled;          /* super_sampling > 1.0                                  */
} vsc_geom;

typedef struct vsc_ctx vsc_ctx;

/* -------- lifecycle: replaces StereoGenerator.__init__ (stereo_core.py:214-223) ------------ */
int vsc_abi_version(void);
const char *vsc_last_error(void);
void vsc_default_params(vsc_params *p);                       /* StereoParams() defaults :196-202 */
int vsc_create(int device, int n_slots, vsc_ctx **out);       /* n_slots frames may be in flight */
/* Grouped context: every slot takes up to `group_size` (<= 4) frames per submission.  The frames of a slot
 * share its CUDA stream and one hole-filling launch, so that n_slots * group_size frames overlap although the
 * device offers only 32 hardware queues.  vsc_create == group_size 1. */
int vsc_create_grouped(int device, int n_slots, int group_size, vsc_ctx **out);
int vsc_group_size(const vsc_ctx *ctx);
void vsc_destroy(vsc_ctx *ctx);
int vsc_device(const vsc_ctx *ctx);
int vsc_num_slots(const vsc_ctx *ctx);

/* host scalar geometry (stereo_core.py:249-251,275-289); VSC_E_PARAMS if the crop is invalid */
int vsc_geometry(int height, int width, const vsc_params *p, vsc_geom *out);

/* -------- the hot call: replaces StereoGenerator.process_frame (stereo_core.py:225-311) ---- */
/* Synchronous, host buffers.  rgb: H*W*3 uint8 RGB; depth: H*W of depth_dtype;
 * out_sbs: H*(2W)*3 uint8 RGB (left | right), caller-owned. */
int vsc_process_frame(vsc_ctx *ctx, const uint8_t *rgb, const void *depth, int depth_dtype,
                      int height, int width, const vsc_params *p, uint8_t *out_sbs);

/* -------- asynchronous variants for the frame loop (sbs_generator.py:304-328) -------------- */
/* pinned host memory for the double-buffered pipeline */
int vsc_host_alloc(size_t bytes, void **out);
int vsc_host_free(void *p);
/* enqueue H2D + the whole path + D2H on slot's stream; host buffers must stay valid (and
 * should be pinned) until vsc_wait(slot) returns. */
int vsc_submit(vsc_ctx *ctx, int slot, const uint8_t *rgb, const void *depth, int depth_dtype,
               int height, int width, const vsc_params *p, uint8_t *out_sbs);
/* group variants: n (<= group_size) frames of identical size and parameters per submission */
int vsc_submit_group(vsc_ctx *ctx, int slot, int n, const uint8_t *const *rgb, const void *const *depth, int depth_dtype,
                     int height, int width, const vsc_params *p, uint8_t *const *out_sbs);
int vsc_submit_device_group(vsc_ctx *ctx, int slot, int n, const uint8_t *const *d_rgb, const void *const *d_depth,
                            int depth_dtype, int height, int width, const vsc_params *p, uint8_t *const *d_out_sbs);
int vsc_wait(vsc_ctx *ctx, int slot);
/* non-blocking: 1 if the slot's frame has finished (vsc_wait will not block), 0 if it is still running */
int vsc_query(vsc_ctx *ctx, int slot);
/* Sleep (no polling) until one of the n in-flight slots has finished on the device, or timeout_ms has passed
 * (< 0: no timeout).  *which = that slot (still to be vsc_wait'ed, which then returns at once) or -1 on timeout.
 * The frame loop's replacement for the reference's blocking queue get (sbs_generator.py:243-246). */
int vsc_wait_any(vsc_ctx *ctx, const int *slots, int n, int timeout_ms, int *which);
/* device-resident variant: inputs/outputs are device pointers on ctx's device; enqueues only
 * (no copies, no synchronisation); vsc_wait(slot) or vsc_sync to complete. */
int vsc_submit_device(vsc_ctx *ctx, int slot, const uint8_t *d_rgb, const void *d_depth, int depth_dtype,
                      int height, int width, const vsc_params *p, uint8_t *d_out_sbs);
int vsc_sync(vsc_ctx *ctx);
/* CUDA stream (cudaStream_t) of a slot, for callers that time with events on that stream */
void *vsc_slot_stream(vsc_ctx *ctx, int slot);
/* device time of the last completed frame on `slot` in ms (events around the kernels only) */
int vsc_slot_elapsed_ms(vsc_ctx *ctx, int slot, float *ms);
/* number of kernel launches issued for the last frame submitted on `slot` */
int vsc_slot_launches(vsc_ctx *ctx, int slot);

/* -------- output layouts (no reference counterpart) -------------------------------------------- */
/* Every layout is a fixed function of the two final u8 eye images L, R [H,W,3] of the SBS layout:
 *   SBS        [H,2W,3]  hstack(L, R)                        (the reference's output, the default)
 *   HALF_SBS   [H,W,3]   hstack of both eyes at half width   (pixel pairs averaged, round half to even == cv2 INTER_AREA)
 *   TB         [2H,W,3]  vstack(L, R), left eye on top
 *   HALF_TB    [H,W,3]   vstack of both eyes at half height  (row pairs averaged, round half to even)
 *   ANAGLYPH   [H,W,3]   Dubois least-squares red-cyan, float32 in a fixed order (DESIGN.md section 2)
 * The half layouts take an even width (HALF_SBS) or height (HALF_TB) only. */
enum { VSC_LAYOUT_SBS = 0, VSC_LAYOUT_HALF_SBS = 1, VSC_LAYOUT_TB = 2, VSC_LAYOUT_HALF_TB = 3, VSC_LAYOUT_ANAGLYPH = 4 };
/* host only: output frame shape of a layout; VSC_E_INVALID for an unknown layout or an odd side a half layout halves */
int vsc_layout_shape(int layout, int height, int width, int *out_h, int *out_w);
/* layout of frames submitted to ctx from now on (vsc_process_frame, vsc_submit*, vsc_submit_device*);
 * frames already in flight keep theirs.  Default VSC_LAYOUT_SBS.  out buffers must hold out_h*out_w*3 bytes.
 * A submission whose frame size the layout cannot take fails with VSC_E_INVALID.  The layout adds no kernel launch:
 * it is the store epilogue of the back-end kernel.  vsc_stage_backend always writes SBS. */
int vsc_set_layout(vsc_ctx *ctx, int layout);

/* -------- output pixel formats (no reference counterpart) -------------------------------------- */
/* A pixel format is a fixed integer function of the final u8 RGB frame of the chosen layout (oh x ow,
 * vsc_layout_shape), so it inherits that frame's exactness.  All int32, no floats, no clamps; S = sum over a 2x2 block
 * (centre-sited chroma), cc = cu for Cb and cv for Cr, limited ("tv") range:
 *   Y8  = (cy.(r,g,b) + (16<<20) + (1<<19)) >> 20        C8  = (cc.(Sr,Sg,Sb) + (128<<22) + (1<<21)) >> 22
 *   Y10 = (cy.(r,g,b) + (16<<20) + (1<<17)) >> 18        C10 = (cc.(Sr,Sg,Sb) + (128<<22) + (1<<19)) >> 20
 *   BT709: cy = 191455 644068 65019   cu = -105533 -355018 460551   cv = 460551 -418321 -42230   (Kr .2126, Kb .0722, Q20)
 *   BT601: cy = 269484 528482 102760  cu = -155188 -305135 460324   cv = 460324 -385875 -74448   (OpenCV's RGB2YUV_I420)
 *   RGB24        [oh][ow][3] bytes (the default)
 *   YUV420P      I420: Y [oh][ow], U [oh/2][ow/2], V [oh/2][ow/2], bytes                      (oh*ow*3/2 bytes)
 *   YUV420P10LE  the same planes as little-endian uint16, the value in the low 10 bits    (oh*ow*3 bytes)
 * The YUV formats take an even H and W only, and also W % 4 == 0 with HALF_SBS and H % 4 == 0 with HALF_TB (each eye
 * then starts on an even coordinate of the output frame). */
enum { VSC_PIXFMT_RGB24 = 0, VSC_PIXFMT_YUV420P = 1, VSC_PIXFMT_YUV420P10LE = 2 };
enum { VSC_MATRIX_BT709 = 0, VSC_MATRIX_BT601 = 1 };
/* host only: bytes of one output frame of an H x W input in (layout, pixfmt); VSC_E_INVALID for an unknown layout or
 * format or a size they cannot take */
int vsc_output_size(int layout, int pixfmt, int height, int width, size_t *bytes);
/* pixel format and YUV matrix of frames submitted to ctx from now on (like vsc_set_layout: frames in flight keep
 * theirs).  Default VSC_PIXFMT_RGB24 / VSC_MATRIX_BT709.  out buffers must hold vsc_output_size bytes.  No kernel
 * launch is added: the conversion is the store epilogue of the back-end kernel.  vsc_stage_backend always writes RGB24. */
int vsc_set_pixfmt(vsc_ctx *ctx, int pixfmt, int matrix);

/* -------- encoded output (no reference counterpart) -------------------------------------------- */
/* VSC_ENCODE_PNG: every frame leaves the library as a complete PNG file of its rgb24 frame in the chosen layout
 * (oh x ow, 8-bit truecolour, chunks IHDR, IDAT..., IEND), encoded on the device by three kernels after the back end:
 *   filter   per row the PNG filter 0..4 of least sum(min(b, 256 - b)) over its filtered bytes (ties: the lowest type;
 *            row 0 against a zero row): the filtered stream, N = oh * (1 + 3 ow) bytes
 *   zlib     78 01, then per 32768-byte segment of the filtered stream (segments ignore row edges) one deflate block of
 *            its own: a greedy run-length parse (literals and distance-1 matches of 3..258, zlib's Z_RLE, no match
 *            reaching before the segment), dynamic Huffman (lit/len codes <= 15 bits, code-length codes <= 7 bits, one
 *            1-bit distance code), or stored when that is not larger; each segment is followed by an empty stored block
 *            (sync flush), so segments are byte-aligned.  Then a final empty fixed block (03 00) and the Adler-32.
 *   framing  one IDAT per segment; the first also holds the zlib header, the last the final block and the Adler-32.
 * Worst case (the capacity an output buffer must have), with nseg = ceil(N / 32768):
 *   bytes = 53 + N + 22 * nseg
 * PNG needs VSC_PIXFMT_RGB24: vsc_set_encode refuses PNG under a YUV format, vsc_set_pixfmt refuses a YUV format under
 * PNG, and a submission with both fails, all with VSC_E_INVALID. */
enum { VSC_ENCODE_NONE = 0, VSC_ENCODE_PNG = 1 };
/* encoding of frames submitted to ctx from now on (like vsc_set_layout: frames in flight keep theirs).  Default NONE.
 * With PNG every submit path (vsc_process_frame, vsc_submit*, vsc_submit_device*) writes the file into the out buffer,
 * which must hold vsc_encoded_capacity bytes.  A page-locked host buffer (vsc_host_alloc) is written by the device
 * directly, so that only the file's bytes cross the bus; a pageable one receives the whole capacity after the run. */
int vsc_set_encode(vsc_ctx *ctx, int encode);
/* host only: the worst-case file bytes of an H x W input in (layout, encode) (NONE: the rgb24 frame's bytes);
 * VSC_E_INVALID for an unknown layout or encoding or a size the layout cannot take */
int vsc_encoded_capacity(int layout, int encode, int height, int width, size_t *bytes);
/* bytes of the file of frame `index` of the slot's last completed submission (VSC_E_STATE while it is in flight or
 * if that submission was not encoded) */
int vsc_encoded_bytes(vsc_ctx *ctx, int slot, int index, size_t *bytes);

/* -------- stage-level entry points for per-stage parity tests (host buffers, synchronous) --- */
/* cv2.resize(src,(dst_w,H),INTER_LANCZOS4) (stereo_core.py:253-254); channels 1 or 3 for u8 */
int vsc_stage_lanczos(vsc_ctx *ctx, const void *src, int dtype, int channels, int height, int width,
                      int dst_w, void *dst);
/* normalize_depth -> _depth_upsampling -> _soft_depth_edges -> apply_depth_gamma
 * (stereo_core.py:258-268): depth_st f32 [H,SW] -> depth_ss f32 [ss_h,ss_w] */
int vsc_stage_depth(vsc_ctx *ctx, const float *depth_st, int height, int stretched_w, int ss_h, int ss_w,
                    const vsc_params *p, float *depth_ss);
/* F.interpolate(rgb) + forward_warp_stereo + uint8 truncation (stereo_core.py:262,270,405/482):
 * rgb_st u8 [H,SW,3], depth_ss f32 [ss_h,ss_w] -> per eye u8 [ss_h,ss_w,3] and mask u8 [ss_h,ss_w];
 * scale255 = the `max <= 1.0` branch of _smooth_warping_artifacts (stereo_core.py:406-407);
 * view_max (2 floats, may be NULL) = max of the float warped image per eye */
int vsc_stage_warp(vsc_ctx *ctx, const uint8_t *rgb_st, const float *depth_ss, int height, int stretched_w,
                   int ss_h, int ss_w, double max_disparity, int scale255,
                   uint8_t *left, uint8_t *left_mask, uint8_t *right, uint8_t *right_mask, float *view_max);
/* cv2.bilateralFilter(img, d, 30, 25*s) (stereo_core.py:409-410) on u8 [h,w,3] */
int vsc_stage_bilateral(vsc_ctx *ctx, const uint8_t *img, int height, int width, double artifact_smoothing,
                        uint8_t *out);
/* _inpaint_missing_regions (stereo_core.py:436-457): valid mask u8 [h,w] (1 = valid) ->
 * dilate(3x3) + cv2.inpaint(radius 3, TELEA) applied in place on img u8 [h,w,3].
 * Only hole clusters that reach columns [keep_x0, keep_x0+keep_w) are filled (pass 0,w for all). */
int vsc_stage_inpaint(vsc_ctx *ctx, uint8_t *img, const uint8_t *valid, int height, int width,
                      int keep_x0, int keep_w);
/* crop -> _sharpen_image -> area downsample -> uint8 truncation -> hstack
 * (stereo_core.py:275-311): two u8 [ss_h,ss_w,3] views -> u8 [H,2W,3] */
int vsc_stage_backend(vsc_ctx *ctx, const uint8_t *left, const uint8_t *right, int ss_h, int ss_w,
                      int left_crop, int right_crop, int crop_w, int height, int width, double sharpen,
                      uint8_t *out_sbs);

/* The PNG encoding of VSC_ENCODE_PNG applied to an arbitrary rgb24 frame rgb [H][W][3] (host buffers, synchronous):
 * the file goes to out (capacity >= vsc_encoded_capacity(VSC_LAYOUT_ANAGLYPH, VSC_ENCODE_PNG, H, W), the layout that
 * keeps H x W), its size to *bytes. */
int vsc_stage_png(vsc_ctx *ctx, const uint8_t *rgb, int height, int width, uint8_t *out, size_t capacity, size_t *bytes);

/* Depth-map post-processing of the producer stage (/root/reference/depth_map_generator.py:217-236, SURVEY.md 8(f) rank 3):
 * cv2.resize(depth f32 [h,w] -> [H,W], INTER_LINEAR), min/max normalise, x255 (bits 8) or x65535 (bits 16), round half to
 * even.  vsc_stage_depth_post: host buffers, synchronous; *ok = 0 when the resized map is flat (the reference then writes
 * no depth map at all).  vsc_depth_post_device: device buffers, enqueued on `slot`'s stream, so that a following
 * vsc_submit_device on the same slot can read d_out as its depth input without the map ever leaving the GPU. */
int vsc_stage_depth_post(vsc_ctx *ctx, const float *depth, int h, int w, int H, int W, int bits, void *out, int *ok);
int vsc_depth_post_device(vsc_ctx *ctx, int slot, const float *d_depth, int h, int w, int H, int W, int bits, void *d_out);

/* -------- the module-level helpers that stereo_core.__all__ exports (stereo_core.py:22-29) ---- */
/* normalize_depth (stereo_core.py:71-88) on n floats */
int vsc_stage_normalize_f32(vsc_ctx *ctx, const float *in, size_t n, float *out);
/* apply_depth_gamma (stereo_core.py:91-107) on n floats */
int vsc_stage_gamma_f32(vsc_ctx *ctx, const float *in, size_t n, double gamma, float *out);
/* forward_warp_stereo (stereo_core.py:110-190) on a float image [C,H,W] (B = 1) and depth [H,W]:
 * warped views [C,H,W] f32 (0 where never written) and masks [H,W] f32 in {0,1} */
int vsc_stage_warp_f32(vsc_ctx *ctx, const float *image, const float *depth, int channels, int height, int width,
                       double max_disparity, float *left, float *left_mask, float *right, float *right_mask);

/* -------- measurement / debugging helpers (no reference counterpart) -------------------------- */
/* record an event pair around every kernel launch of subsequently submitted frames */
int vsc_set_profiling(vsc_ctx *ctx, int on);
/* names and device milliseconds of the kernels of the last completed frame on `slot`; returns count */
int vsc_slot_kernel_times(vsc_ctx *ctx, int slot, int max_n, const char **names, float *ms);
/* device timer across all slot streams (CUDA events): begin gates every slot stream on a start
 * event, end records once every slot stream has drained and returns the elapsed milliseconds */
int vsc_timer_begin(vsc_ctx *ctx);
int vsc_timer_end(vsc_ctx *ctx, float *ms);
/* copies of slot 0's intermediates after a completed call, for stage bisection (which: 0 rgb_st, 1 depth_st,
 * 2 depth_ss, 3/4 pre-bilateral views, 5/6 filtered views, 7/8 hole bitmaps).  With artifact_smoothing > 0 the hole
 * filling reuses buffers 2, 3 and 4 as scratch, so they no longer hold the intermediate afterwards. */
int vsc_debug_fetch(vsc_ctx *ctx, int which, void *dst, size_t bytes);
/* after vsc_stage_inpaint: arrival times, state bytes and order words (index of every computed hole pixel in the
 * reference's computation order) of slot 0; any pointer may be null */
int vsc_debug_telea_state(vsc_ctx *ctx, int view, float *tt, uint8_t *st, uint32_t *ord, size_t n);
/* 64 phase counters of the hole-filling march (non-zero only in -DVSC_TELEA_STATS profiling builds) */
int vsc_debug_telea_stats(vsc_ctx *ctx, unsigned long long *out64);
/* test hook: set the hole-filling queue capacity (entries per view) to exercise the overflow/re-run path */
int vsc_debug_set_telea_capacity(vsc_ctx *ctx, size_t entries);
/* device-side check of two arithmetic identities the kernels use instead of library calls, over every float of
 * their range: which = 0 reciprocal (MUFU.RCP + one Newton step) against the correctly rounded 1/x on [1, 256);
 * which = 1 x/3 by multiply + two FMAs against the IEEE quotient on [0, 2295].  *mismatches must come back 0. */
int vsc_debug_selftest(vsc_ctx *ctx, int which, unsigned long long *mismatches);
/* counters of the last vsc_stage_png call: out[0] segments whose lit/len code needed the 15-bit limit, out[1] segments
 * whose code-length code needed the 7-bit limit, out[2] segments written as stored blocks */
int vsc_debug_png_stats(vsc_ctx *ctx, unsigned long long *out);

#ifdef __cplusplus
}
#endif
#endif /* VSC_B200_H */
