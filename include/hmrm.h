/* hmrm.h — C ABI of the B200-native heightmap ray-march path (libhmrm.so).
 *
 * The reference (Costava/heightmap-ray-marcher) has no library or FFI seam: its
 * hot path is inline in main() and parameterised by global variables
 * (main/hmap.cpp:28-112).  This header is the seam a maintainer would bind
 * instead: each entry point names the reference lines it replaces.  All
 * arguments are plain pointers, sizes and PODs; no C++ or torch types cross it.
 *
 * Conventions: every function returns 0 on success or an HMRM_ERR_* code;
 * hmrm_last_error() gives the message.  The caller owns every host buffer it
 * passes; the context owns all device memory.  A context is bound to one CUDA
 * device and must be used from one host thread at a time.  Nothing in this
 * library falls back to the CPU: without a CUDA device hmrm_create() fails.
 */
#ifndef HMRM_H
#define HMRM_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define HMRM_ABI_VERSION 2

/* image_plane values, main/hmap.cpp:104-107 */
#define HMRM_PERSPECTIVE  1
#define HMRM_SPHERICAL    2
#define HMRM_ORTHOGRAPHIC 3

/* arithmetic mode of the render kernel */
#define HMRM_FP64_EXACT 0   /* bit-exact to the reference's RGBA8 framebuffer */
#define HMRM_FP32_FAST  1   /* accepted, and an ALIAS of HMRM_FP64_EXACT: the production traversal already marches on a
                             * 32/64-bit integer model and keeps FP64 for ray set-up and for the few samples the model
                             * cannot decide, so there is nothing left for a lossy mode to win (DESIGN.md section 4).
                             * The north star's tolerance (>= 99.5 % identical pixels, |step delta| <= 1) is met
                             * with 100 % / 0 and is written out in the tests. */

/* traversal strategy (results are identical; this selects the kernel) */
#define HMRM_TRAVERSAL_AUTO  0
#define HMRM_TRAVERSAL_BRUTE 1   /* one height fetch per reference step (main/hmap.cpp:1000-1038 as written) */
#define HMRM_TRAVERSAL_SKIP  2   /* conservative max-mip empty-space skip in whole steps (integer linear model; default) */
#define HMRM_TRAVERSAL_SKIP_FP64 3   /* the same skip with exact FP64 positions at every decision (k2_render_skip.cuh) */
#define HMRM_TRAVERSAL_PACK  4   /* HMRM_TRAVERSAL_SKIP's traversal with lanes refilled from a per-warp stack of rays
                                  * (k2_render_pack.cuh) */

/* hmrm_frame.flags */
#define HMRM_FLAG_STATS      1u  /* count rays / steps / fetches (hmrm_get_stats) */
#define HMRM_FLAG_STEP_INDEX 2u  /* record the per-pixel first-hit step index (hmrm_get_step_index) */
#define HMRM_FLAG_RAY_DUMP   4u  /* record the device's ray / slab distance / entry point per pixel (hmrm_get_ray_dump) */
/* Supersampling (kernel K5, csrc/k5_downsample.cuh): bits 8-11 hold s - 1, s = 1..4 (0 = one ray per pixel, the
 * reference's frame).  screen_width x screen_height (W x H) stays the OUTPUT size: every buffer, bound and shape is the
 * one of the 1x frame.  A frame with factor s is the box filter of the reference's frame of the same camera at sW x sH:
 *   subsample (s px + i, s py + j), 0 <= i, j < s, is pixel (s px + i, s py + j) of that sW x sH frame (bit-exact to the
 *   reference, as every render here is);
 *   each of R, G, B = (sum + s*s/2) / (s*s) in integers (floor division; s*s/2 = 0, 2, 4, 8 for s = 1..4), with the sum
 *   of that channel over the s*s subsamples;  A = 255.
 * The subsample rays come from the sW x sH image plane (w = x / (sW - 1)), not jittered around the 1x pixel centres.
 * Accepted by hmrm_render, hmrm_render_async, hmrm_render_device, hmrm_render_png_async and hmrm_render_yuv420_async,
 * for whole frames only: s > 1 with cycle_period != 1, band_count > 1, a partial row band, HMRM_FLAG_STEP_INDEX or
 * HMRM_FLAG_RAY_DUMP, sW or sH above 65536, a field value above 3, or any s > 1 passed to hmrm_render_peer /
 * hmrm_render_peer_staged is HMRM_ERR_INVALID.  With HMRM_FLAG_STATS, hmrm_get_stats describes the sW x sH render
 * (rays = s*s*W*H; kernel_ms of the render kernel alone). */
#define HMRM_FLAG_SUPERSAMPLE_SHIFT 8
#define HMRM_FLAG_SUPERSAMPLE_MASK  (15u << HMRM_FLAG_SUPERSAMPLE_SHIFT)
#define HMRM_FLAG_SUPERSAMPLE(s)    ((uint32_t)((s) - 1) << HMRM_FLAG_SUPERSAMPLE_SHIFT)   /* s = 1..4 */

/* hmrm_frame.pixel_format: layout of the frame the render calls write */
#define HMRM_PIXEL_RGBA8 0       /* the reference's framebuf: [H][W][4], A = 255 (main/hmap.cpp:139-154) */
#define HMRM_PIXEL_RGB8  1       /* the same pixels without the constant alpha byte: [H][W][3] (25 % fewer bytes over
                                  * PCIe / NVLink; the north star's "RGB8 bands") */

/* memory layout of the 16-bit height pyramid the march fetches from (csrc/pyramid_layout.cuh); results are identical */
#define HMRM_LAYOUT_ROWMAJOR 0
#define HMRM_LAYOUT_TILE4    1   /* 4x4-texel (32-byte sector) tiles, tiles in row-major order */
#define HMRM_LAYOUT_ZORDER   2   /* 4x4-texel tiles in Z-order (Morton) inside 64x64-texel blocks */
#define HMRM_LAYOUT_DEFAULT  HMRM_LAYOUT_ROWMAJOR   /* measured: profiles/r02_layout_ab.txt — no layout wins */

#define HMRM_OK                  0
#define HMRM_ERR_INVALID         1   /* bad argument */
#define HMRM_ERR_CUDA            2   /* CUDA runtime error (message has the detail) */
#define HMRM_ERR_STATE           3   /* call order: maps / heightmap not set */
#define HMRM_ERR_NONTERMINATING  4   /* a ray can never leave the grid: the reference would hang (main/hmap.cpp:1000) */

typedef struct hmrm_ctx hmrm_ctx;

/* The reference's per-frame render state (globals, main/hmap.cpp:28-112), as one POD.
 * Angles are radians, as the reference stores them after DegreesToRads (:131-133). */
typedef struct hmrm_frame {
	int32_t projection;     /* image_plane :107 */
	int32_t screen_width;   /* :31 */
	int32_t screen_height;  /* :32 */
	int32_t precision;      /* HMRM_FP64_EXACT | HMRM_FP32_FAST */
	double cam_pos[3];      /* :75 */
	double hang;            /* :80 */
	double vang;            /* :85 */
	double hfov;            /* :35 */
	double ortho_width;     /* :98 */
	double grid_width;      /* :65 */
	double step_dist;       /* :68 */
	uint8_t bg[3];          /* bg_r, bg_g, bg_b :110-112 */
	uint8_t pixel_format;   /* HMRM_PIXEL_RGBA8 (0, the reference's framebuf) | HMRM_PIXEL_RGB8 */
	int32_t cycle;          /* first pixel index of this frame (:979), 0 <= cycle < cycle_period */
	int32_t cycle_period;   /* pixel stride (:71,:980); 1 = full frame */
	int32_t row_begin;      /* rows [row_begin,row_end) are rendered: row band of a multi-GPU frame */
	int32_t row_end;        /* 0,0 = all rows */
	int32_t traversal;      /* HMRM_TRAVERSAL_* */
	uint32_t flags;         /* HMRM_FLAG_* */
	int32_t band_count;     /* > 1: the 4-row tile rows of [row_begin,row_end) are dealt round-robin to band_count */
	int32_t band_index;     /*      renderers and this call renders those with (tile_row % band_count) == band_index */
} hmrm_frame;

typedef struct hmrm_stats {
	int64_t rays;           /* pixels rendered */
	int64_t box_hits;       /* rays that entered the AABB (src/AABB.cpp:30) */
	int64_t surf_hits;      /* rays that hit the terrain (main/hmap.cpp:1016) */
	int64_t steps;          /* reference-equivalent march steps = height fetches the reference performs (:1013) */
	int64_t fetches;        /* memory fetches this kernel actually issued on the march (any level) */
	int64_t max_steps;      /* longest single ray, in reference steps */
	int32_t status;         /* 0, or HMRM_ERR_NONTERMINATING if some ray was cut off */
	int32_t reserved0;
	double kernel_ms;       /* CUDA-event duration of the render kernel */
} hmrm_stats;

/* ---- lifetime -------------------------------------------------------------------------- */
int hmrm_abi_version(void);
int hmrm_device_count(void);
int hmrm_create(int device, hmrm_ctx **out);
void hmrm_destroy(hmrm_ctx *ctx);
const char *hmrm_last_error(const hmrm_ctx *ctx);   /* ctx may be NULL: last creation error */

/* ---- maps: replaces stbi_load results at main/hmap.cpp:320-321 (RGB8) and :341-342 (RGBA8) ---- */
int hmrm_set_maps(hmrm_ctx *ctx, const uint8_t *height_rgb8, const uint8_t *color_rgba8,
                  int32_t map_width, int32_t map_height);
/* same, from device memory of ctx's device (copied) */
int hmrm_set_maps_device(hmrm_ctx *ctx, const void *d_height_rgb8, const void *d_color_rgba8,
                         int32_t map_width, int32_t map_height);
/* synthetic fBm maps of size 2^log2n generated on the device (csrc/synth_fbm.h; bench / test input) */
int hmrm_synth_maps(hmrm_ctx *ctx, uint32_t log2n, uint32_t seed);
int hmrm_get_maps(hmrm_ctx *ctx, uint8_t *height_rgb8, uint8_t *color_rgba8);   /* download (either may be NULL) */

/* ---- 16-bit height maps: UpdateHeightmap (main/hmap.cpp:171-191) with 65535 in place of 255 ----
 * A 16-bit map has one channel, height [map_height][map_width] (uint16_t).  Its sample x is used as R = G = B, as stb
 * replicates a grey image, so lum keeps its meaning.  Each line is rounded separately, in this order, without FMA:
 *   v      = (lum_r*x + lum_g*x) + lum_b*x,  clamped to [0, 65535]
 *   height = (v / 65535) * (max_height - min_height) + min_height
 *   surf   = height + min_height          (what the march compares against)
 * For x = 257 * v8 and a unit lum vector, v / 65535 and v8 / 255 are the same correctly rounded number, so the heights
 * are bit-identical to those of the grey 8-bit map v8.  After any of these calls hmrm_update_heightmap builds the
 * pyramid as for 8-bit maps, and hmrm_get_heights returns the heights above.  hmrm_set_maps / hmrm_set_maps_device /
 * hmrm_synth_maps switch the context back to 8 bits.  hmrm_get_maps on a 16-bit map returns the colormap; a non-NULL
 * height_rgb8 is HMRM_ERR_STATE.  NULL pointers and sizes outside [1, 32768] are HMRM_ERR_INVALID. */
int hmrm_set_maps16(hmrm_ctx *ctx, const uint16_t *height, const uint8_t *color_rgba8,
                    int32_t map_width, int32_t map_height);
/* same, from device memory of ctx's device (copied) */
int hmrm_set_maps16_device(hmrm_ctx *ctx, const void *d_height, const void *d_color_rgba8,
                           int32_t map_width, int32_t map_height);
/* synthetic 16-bit map: hmrm_synth_height16 (csrc/synth_fbm.h) and exactly hmrm_synth_maps' colormap */
int hmrm_synth_maps16(hmrm_ctx *ctx, uint32_t log2n, uint32_t seed);

/* layout of the height pyramid (HMRM_LAYOUT_*; also the HMRM_LAYOUT environment variable at hmrm_create:
 * rowmajor | tile4 | zorder).  Takes effect at the next hmrm_update_heightmap, which must follow. */
int hmrm_set_layout(hmrm_ctx *ctx, int layout);
int hmrm_get_layout(hmrm_ctx *ctx);

/* ---- motion blur (kernel K5, csrc/k5_downsample.cuh): a frame averages the scene over several cameras ----
 * The state belongs to the context, as the layout does.  It is copied, so the caller may free `cams`.  Each render call
 * reads it when the frame is ENQUEUED: frames already in flight keep the cameras they were enqueued with.
 * With n >= 1, sub-frame j (0 <= j < n) is the reference's frame of `f` with cam_pos, hang and vang replaced by cams[j],
 * rendered at sW x sH when `f` has supersample factor s.  The fields of `f` that hold the camera are not used; every other
 * field comes from `f`.  Output pixel: each of R, G, B = (sum + N/2) / N in integers (floor division), N = n*s*s, with
 * the sum of that channel over the s x s subsamples of all n sub-frames (at most 16*16*255 = 65280);  A = 255.  There is
 * one rounding, not HMRM_FLAG_SUPERSAMPLE's box filter followed by an average.  Consequences:
 *   n = 1 is the supersampled frame of cams[0] (HMRM_FLAG_SUPERSAMPLE's definition);
 *   cams[0] equal to f's camera with n = 1 gives exactly the frame without blur;
 *   n identical cameras give the frame of that camera without blur, for every s <= 4 and n <= 16 (for every possible
 *   sum, the rounded mean of n copies of a rounded mean is that rounded mean).
 * Accepted by hmrm_render, hmrm_render_async, hmrm_render_device, hmrm_render_png_async, hmrm_render_yuv420_async and
 * hmrm_render_jpeg_async; while n >= 1 they refuse what HMRM_FLAG_SUPERSAMPLE refuses (cycle_period != 1,
 * band_count > 1, a partial row band, HMRM_FLAG_STEP_INDEX or HMRM_FLAG_RAY_DUMP) with HMRM_ERR_INVALID and nothing
 * written, and so do hmrm_render_peer and hmrm_render_peer_staged.  With HMRM_FLAG_STATS, hmrm_get_stats gives sums over
 * the n sub-frame renders (rays = n*s*s*W*H, steps and fetches summed, max_steps the maximum) and kernel_ms from the start
 * of the first sub-frame render to the end of the last. */
typedef struct hmrm_camera {
	double cam_pos[3];   /* as hmrm_frame.cam_pos */
	double hang, vang;   /* radians, as hmrm_frame */
} hmrm_camera;
/* n = 0 (the default): every render is as without this call.  n = 1..16: every whole-frame render on ctx averages n
 * sub-frames.  n < 0, n > 16 or NULL cams with n > 0 is HMRM_ERR_INVALID and leaves the previous state in place. */
int hmrm_set_motion_blur(hmrm_ctx *ctx, const hmrm_camera *cams, int32_t n);

/* ---- prepass: replaces UpdateHeightmap, main/hmap.cpp:171-191 (kernel K1) ---- */
int hmrm_update_heightmap(hmrm_ctx *ctx, const double lum[3], double min_height, double max_height);
/* heights exactly as the reference's heightmap_buf (double[H][W], main/hmap.cpp:53), for parity checks */
int hmrm_get_heights(hmrm_ctx *ctx, double *heights);

/* ---- render: replaces main/hmap.cpp:952-1058 (ImagePlane ctor + pixel loop; kernel K2) ---- */
void hmrm_frame_defaults(hmrm_frame *f);            /* the reference's defaults, :31-112, cycle_period 1 */
/* rgba_out: host RGBA8 [screen_height][screen_width][4], stride W*4 — the reference's framebuf (:612) — or, with
 * pixel_format = HMRM_PIXEL_RGB8, [screen_height][screen_width][3], stride W*3.
 * Only the pixels selected by cycle/cycle_period and the row band are written. Synchronous. */
int hmrm_render(hmrm_ctx *ctx, const hmrm_frame *f, uint8_t *rgba_out);
/* device output (same layout) on `stream` (a cudaStream_t, NULL = ctx's own stream); asynchronous.  d_rgba_out may
 * have any alignment (so may d_frame and d_stage of hmrm_render_peer / hmrm_render_peer_staged): an address that is
 * not a multiple of 4 is written byte by byte, as K3's and K5's device outputs already may be. */
int hmrm_render_device(hmrm_ctx *ctx, const hmrm_frame *f, void *d_rgba_out, void *stream);
/* render into the context's device framebuffer(s) and copy rows [row_begin,row_end) to (pinned or registered) host
 * memory asynchronously; hmrm_wait() joins.  rgba_out always addresses the WHOLE frame; with band_count > 1 only the
 * tile rows of this band are written (so several contexts / ranks can fill one host frame). */
int hmrm_render_async(hmrm_ctx *ctx, const hmrm_frame *f, uint8_t *rgba_out);
int hmrm_wait(hmrm_ctx *ctx);
/* Streaming: up to four whole frames (cycle_period 1) may be in flight; the copy-out of one overlaps the kernels
 * of the next ones.  hmrm_wait_pending(ctx, n) (n = 1..3) returns when every frame but the n most recent is complete
 * in its host buffer (so n + 1 host buffers are rotated); hmrm_wait_pending(ctx, 0) == hmrm_wait. */
int hmrm_wait_pending(hmrm_ctx *ctx, int max_pending);

/* ---- many cameras in one launch (kernel K2, csrc/k2_render_lin.cuh with kViews) ----
 * n views of f in one launch.  View j is exactly the frame hmrm_render would produce for f with cam_pos, hang and vang
 * replaced by cams[j] (set_camera's rule, as for motion blur); every other field comes from f, and f's own camera is
 * not used.  Output: [n][screen_height][screen_width][C], C = 4 (HMRM_PIXEL_RGBA8) or 3 (HMRM_PIXEL_RGB8); view j
 * starts at byte j * H * W * C.  cams is copied before the call returns.
 * Limits: 1 <= n <= 65536; f passes hmrm_render's frame checks; the batch has at most 2^26 tiles of 8x4 pixels
 * (n * ceil(W/8) * ceil(H/4)).  Outside them: HMRM_ERR_INVALID.
 * Refused with HMRM_ERR_INVALID, nothing written and the context left usable: what a motion-blurred frame refuses
 * (cycle_period != 1, band_count > 1, a partial row band, HMRM_FLAG_STEP_INDEX or HMRM_FLAG_RAY_DUMP); a supersample
 * field other than 0; a context with motion blur set; a non-finite value in any camera; NULL cams or output; a traversal
 * other than HMRM_TRAVERSAL_AUTO or HMRM_TRAVERSAL_SKIP; a grid_width so small that the skip traversal would fall back
 * to FP64 (views have no fallback path).  Maps whose height range could not be quantised: HMRM_ERR_STATE.
 * With HMRM_FLAG_STATS, hmrm_get_stats describes the batch: rays = n*W*H; box_hits, surf_hits, steps and fetches are
 * sums over the views, max_steps the maximum, status the OR of the views, kernel_ms the one launch.  Afterwards
 * hmrm_get_step_index and hmrm_get_ray_dump return HMRM_ERR_STATE.
 * d_out may have any alignment, as for hmrm_render_device; each view's base address has its own (with RGB8 and W*H*3
 * not a multiple of 4, consecutive views start at different offsets modulo 4) and is written accordingly. */
int hmrm_render_views_device(hmrm_ctx *ctx, const hmrm_frame *f, const hmrm_camera *cams, int32_t n,
                             void *d_out, void *stream);            /* stream-ordered; NULL = ctx's stream */
/* the same into any host memory, through a device buffer of the context on ctx's stream; synchronous.  Frames of
 * hmrm_render_async still in flight are not disturbed. */
int hmrm_render_views(hmrm_ctx *ctx, const hmrm_frame *f, const hmrm_camera *cams, int32_t n,
                      uint8_t *out);

/* ---- PNG frames, deflated on the device (kernel K3, csrc/k3_png.cuh) ----
 * The file is 8-bit, not interlaced, colour type 6 for 4 channels and 2 for 3; the decoded pixels are the frame's, byte
 * for byte.  The file is exactly this function of the pixels (C channels, W x H):
 * 1. Filter, per row: for each type t = 0 None, 1 Sub, 2 Up, 3 Average, 4 Paeth, the sum over the row's W C bytes of
 *    min(r, 256 - r), r = residual & 255; the row above row 0 is zero, a and c are zero for the first C bytes.  The
 *    smallest sum wins, the lowest type on a tie.  The filtered stream is H rows of 1 + W C bytes (type, residuals).
 * 2. Segments: the stream is cut into 4096-byte segments, the last one shorter; each is deflated on its own.
 * 3. Greedy parse of a segment: at position o each candidate distance, in the order 1, C, W C + 1 (the last only while
 *    W C + 1 <= 32768), has a run: the number of bytes from o on that equal the byte that many positions back.  A run
 *    may reach back before the segment's start, never before byte 0 of the stream, and stops at the segment's end; it
 *    is capped at 258.  The longest run, if it is at least 3, is a match (the earlier distance on a tie), else the byte
 *    is one literal.
 * 4. Coding: the segment is one fixed-Huffman block (RFC 1951: BFINAL 0, BTYPE 01, the tokens, EOB) followed by an
 *    empty stored block (3 header bits, alignment to a byte, 00 00 FF FF).  With n the segment's bytes and `bits` the
 *    tokens' bits, it stays so when 3 + bits + 10 <= 8 (n + 1), that is when its bytes do not exceed the n + 5 of a
 *    stored block (a tie stays coded); otherwise it is one stored block: 00, LEN, NLEN, the n bytes.
 * 5. Framing: signature; IHDR; one IDAT chunk per segment, the first one led by the zlib header 78 01; an IDAT of
 *    03 00 (a final empty fixed block) and the big-endian Adler-32 of the filtered stream; IEND. */
/* worst-case file size for width x height x channels (3 | 4), 0 for other shapes; host arithmetic, no device work:
 * with N = height * (width * channels + 1) and S = ceil(N / 4096) segments, N + 17 S + 65 */
size_t hmrm_png_bound(int32_t width, int32_t height, int32_t channels);
/* hmrm_render_async, but the frame leaves the device as a complete PNG file (colour type 6 for HMRM_PIXEL_RGBA8,
 * 2 for HMRM_PIXEL_RGB8).  Whole frames only (cycle_period 1, band_count <= 1, no STEP_INDEX / RAY_DUMP).  png_out:
 * pinned / registered host memory or device memory of ctx's device, capacity >= hmrm_png_bound; *png_bytes (same
 * kinds of memory, 8-byte aligned) receives the file size.  Both are valid once hmrm_wait / hmrm_wait_pending covers
 * the frame; up to four PNG frames may be in flight, as with hmrm_render_async. */
int hmrm_render_png_async(hmrm_ctx *ctx, const hmrm_frame *f, uint8_t *png_out, size_t capacity, uint64_t *png_bytes);
/* encode caller pixels (host memory, [height][width][channels], copied to the device); synchronous.  Sizes from 1 to
 * 65536 per axis; png_out / png_bytes as for hmrm_render_png_async. */
int hmrm_encode_png(hmrm_ctx *ctx, const uint8_t *pixels, int32_t width, int32_t height, int32_t channels,
                    uint8_t *png_out, size_t capacity, uint64_t *png_bytes);

/* ---- 4:2:0 video planes (kernel K4, csrc/k4_yuv.cuh): what every video encoder takes as input ----
 * Limited-range ("TV range") 8-bit YCbCr.  Coefficients are 2^-14 fixed point: round(k * 2^14 * 219/255) for Y and
 * round(k * 2^14 * 224/255) for Cb and Cr, with k the matrix's float coefficients:
 *              Y (R, G, B)           Cb (R, G, B)            Cr (R, G, B)
 *   BT.601     4207, 8260, 1604      -2428, -4768, 7196      7196, -6026, -1170
 *   BT.709     2991, 10064, 1016     -1649, -5547, 7196      7196, -6536, -660
 * Both chroma rows sum to 0: a grey pixel block gives exactly Cb = Cr = 128.
 *   luma, per pixel:          Y = ((yr R + yg G + yb B + 2^13) >> 14) + 16
 *   chroma, per 2x2 block:    sample (i, j) covers rows 2i, 2i+1 and columns 2j, 2j+1, indices clamped to H-1 and W-1
 *                             (odd sizes replicate the last row / column); with SR, SG, SB the sums over those four
 *                             pixels, Cb = ((cr SR + cg SG + cb SB + 2^15) >> 16) + 128, Cr the same with its own row.
 *                             >> is an arithmetic shift (floor).
 * Every output lies in [16, 240], within 0.51 of the float BT.601 / BT.709 value (of the block mean for chroma).
 * Layout: planar I420 without row padding: Y [H][W], then Cb [ceil(H/2)][ceil(W/2)], then Cr of the same shape.
 * The 2x2 box puts chroma at the centre of the block (Y4M's C420jpeg siting). */
#define HMRM_YUV_BT601 0
#define HMRM_YUV_BT709 1
/* W*H + 2*ceil(W/2)*ceil(H/2) bytes; 0 outside [1, 65536] per axis.  Host arithmetic, no device work. */
size_t hmrm_yuv420_bytes(int32_t width, int32_t height);
/* hmrm_render_async, but the frame leaves the device as I420 planes (HMRM_YUV_* matrix) of the RGBA8 or RGB8 frame.
 * Whole frames only (cycle_period 1, band_count <= 1, no row band, no STEP_INDEX / RAY_DUMP).  out: pinned / registered
 * host memory or device memory of ctx's device, capacity >= hmrm_yuv420_bytes; valid once hmrm_wait / hmrm_wait_pending
 * covers the frame.  Shares the ring with hmrm_render_async and hmrm_render_png_async: up to four frames of any of the
 * three kinds may be in flight. */
int hmrm_render_yuv420_async(hmrm_ctx *ctx, const hmrm_frame *f, int32_t matrix, uint8_t *out, size_t capacity);
/* convert caller pixels ([height][width][channels], channels 3 | 4, host or device memory, copied to the device);
 * synchronous.  Sizes from 1 to 65536 per axis; out as for hmrm_render_yuv420_async. */
int hmrm_convert_yuv420(hmrm_ctx *ctx, const uint8_t *pixels, int32_t width, int32_t height, int32_t channels,
                        int32_t matrix, uint8_t *out, size_t capacity);

/* ---- JPEG frames, encoded on the device (kernel K6, csrc/k6_jpeg.cuh) ----
 * A JPEG frame is exactly the file libjpeg-turbo writes for the frame's R, G, B (alpha ignored) with baseline coding,
 * the standard tables, IJG quality scaling and one restart interval per MCU row; in Pillow's words
 *   Image.fromarray(rgb).save(f, "JPEG", quality=q, subsampling=2 (4:2:0) or 0 (4:4:4), restart_marker_rows=1).
 * All integer; >> is an arithmetic shift:
 * 1. Colour, JFIF full-range BT.601 in 2^-16 fixed point (not K4's limited-range matrix):
 *      Y  = (19595 R + 38470 G + 7471 B + 32768) >> 16
 *      Cb = (-11059 R - 21709 G + 32768 B + 8421375) >> 16
 *      Cr = (32768 R - 27439 G - 5329 B + 8421375) >> 16
 * 2. Planes.  Y, and all three planes in 4:4:4: columns replicated to a multiple of 8, rows to whole MCU rows (16 rows
 *    for 4:2:0 luma, 8 otherwise).  4:2:0 chroma: source columns replicated to 16 ceil(ceil(W/2)/8), an odd last source
 *    row duplicated, each sample (a + b + c + d + bias) >> 2 over its 2x2 source block with bias 1, 2, 1, 2, ... by
 *    output column, then chroma rows replicated down to a multiple of 8 (libjpeg's order; not "pad, then downsample").
 * 3. Blocks: libjpeg's jfdctint ("islow") forward DCT on sample - 128; the Annex K.1 tables scaled by quality,
 *    s = q < 50 ? 5000 / q : 200 - 2q, entry = clamp((base s + 50) / 100, 1, 255); a coefficient c against entry t
 *    becomes (|c| + 4t) / (8t), truncated, with c's sign.  In 4:2:0 a luma block of an MCU outside
 *    ceil(W/8) x ceil(H/8) is a dummy block: AC 0, DC copied from the block to its left, or, in a bottom dummy row, from
 *    the last block of the MCU's row above.
 * 4. Entropy coding: the Annex K.3 Huffman tables; a DC predictor per component, reset at every restart; the restart
 *    interval is one MCU row (DRI = MCUs per row, RST0 .. RST7 cyclically); padding before a marker and at the end is
 *    1-bits; 0xFF in the data is stuffed as FF 00.
 * 5. Markers: SOI; APP0 JFIF 1.01 (density units 0, 1x1, no thumbnail); DQT 0 (luma), DQT 1 (chroma), zig-zag order;
 *    SOF0 (8 bit; components 1, 2, 3, sampling 0x22 / 0x11 / 0x11 or 0x11 x 3, tables 0 / 1 / 1); DHT DC0, AC0, DC1,
 *    AC1; DRI; SOS (03 01 00 02 11 03 11 00 3f 00); the data; EOI.  The header is 629 bytes, EOI adds 2.
 * Sizes run from 1 to 65535 per axis (SOF0's fields are 16 bits), quality from 1 to 100. */
#define HMRM_JPEG_420 0
#define HMRM_JPEG_444 1
/* Worst-case file size, 0 outside the limits; host arithmetic.  With B the blocks including 4:2:0's dummies (MCUs x 6
 * or x 3) and R the MCU rows: 631 + 415 B + 4 R.  Proof: a block codes at most 11 + 11 DC bits (code, then |diff| <=
 * 2047) and, per AC position, at most 16 + 10 bits (a ZRL covers 16 positions with 11 bits, EOB replaces a zero
 * position with at most 16), so 1660 bits; a row of b blocks is at most ceil(1660 b / 8) <= 207.5 b + 1 bytes with its
 * padding, at most 415 b + 2 after stuffing, + 2 for its RST marker; + 629 + 2 for the header and EOI. */
size_t hmrm_jpeg_bound(int32_t width, int32_t height, int32_t chroma);
/* hmrm_render_png_async, but the frame leaves the device as a JPEG file of quality 1..100 and chroma HMRM_JPEG_420 |
 * HMRM_JPEG_444: the same refusals (whole frames only), destinations (pinned / registered host or device memory, any
 * alignment; jpeg_bytes 8-byte aligned) and four-frame ring, shared with raw, PNG and YUV frames; HMRM_FLAG_SUPERSAMPLE
 * is accepted.  A frame above 65535 pixels per axis is HMRM_ERR_INVALID. */
int hmrm_render_jpeg_async(hmrm_ctx *ctx, const hmrm_frame *f, int32_t quality, int32_t chroma, uint8_t *jpeg_out,
                           size_t capacity, uint64_t *jpeg_bytes);
/* encode caller pixels ([height][width][channels], channels 3 | 4, host or device memory, copied to the device);
 * synchronous.  jpeg_out / jpeg_bytes as for hmrm_render_jpeg_async. */
int hmrm_encode_jpeg(hmrm_ctx *ctx, const uint8_t *pixels, int32_t width, int32_t height, int32_t channels,
                     int32_t quality, int32_t chroma, uint8_t *jpeg_out, size_t capacity, uint64_t *jpeg_bytes);

int hmrm_get_stats(hmrm_ctx *ctx, hmrm_stats *out);            /* of the last render */
/* traversal diagnostics of the last HMRM_FLAG_STATS render with a skip traversal: [0] jumps, [1] samples covered
 * by jumps, [2] single steps above a mip block, [3] level descents, [4] cell tests above the cell, [5] cell tests
 * below the quantised height (hits), [6] HMRM_TRAVERSAL_SKIP: warp-level loop iterations (lane utilisation of the
 * march loop = ([0]+[2]+[4]+[5]+[7]) / 32 / [6]); HMRM_TRAVERSAL_SKIP_FP64: refused jumps, [7] samples decided by the
 * exact FP64 expressions, [8]..[11] HMRM_TRAVERSAL_SKIP: warp-level iterations with 1-8 / 9-16 / 17-24 / 25-32 busy
 * lanes; HMRM_TRAVERSAL_SKIP_FP64: slowest 8x4 tile in SM clocks, sum of tile clocks, most loop iterations of any ray,
 * tiles above 100 k clocks */
int hmrm_get_debug_counters(hmrm_ctx *ctx, int64_t out[12]);
int hmrm_get_step_index(hmrm_ctx *ctx, int32_t *step_index);   /* int32 [H][W]: first-hit sample index,
                                                                  -1 box missed, -2 no surface hit */
/* of the last HMRM_FLAG_RAY_DUMP render: double [H][W][10] = what the DEVICE computed for each pixel: ray pos[3] and
 * dir[3] (ImagePlane::GetRay, src/Perspective.cpp:25-32 etc.), the slab entry distance (distance(), src/AABB.cpp:49-77;
 * -inf..inf as the reference leaves it when a slab test fails early), and the entry point (intersection(), :30-47; zeros
 * when the box is missed).  Pixels not rendered by that frame are NaN. */
int hmrm_get_ray_dump(hmrm_ctx *ctx, double *out);

/* ---- type-level API mirror (host side; no device work) ---- */
/* DegreesToRads, main/hmap.cpp:131-133 */
double hmrm_deg2rad(double degrees);
/* look/up from hang,vang, main/hmap.cpp:661-672 */
void hmrm_camera_basis(double hang, double vang, double look[3], double up[3]);
/* ImagePlane::GetRay (src/ImagePlane.hpp:10) of the plane the frame describes; w,h in [0,1] */
int hmrm_get_ray(const hmrm_frame *f, double w, double h, double pos[3], double dir[3]);

/* The device's own slab test (the function the render kernels call; src/AABB.cpp:30-77) on n caller-supplied rays
 * (pos[3], dir[3] each) and boxes (c0[3], c1[3] each): out[n][5] = distance(), intersection() as 0/1, entry point.
 * For known-answer tests against the reference's functions. */
int hmrm_debug_aabb(hmrm_ctx *ctx, int32_t n, const double *rays, const double *boxes, double *out);

/* pinned host memory helpers (so that callers without a CUDA binding can stage buffers) */
int hmrm_host_alloc(void **ptr, size_t bytes);
/* the same with HMRM_HOST_* flags; write-combined memory is fast to fill from the device and slow to read on the CPU */
#define HMRM_HOST_WRITE_COMBINED 1u
int hmrm_host_alloc_flags(void **ptr, size_t bytes, uint32_t flags);
void hmrm_host_free(void *ptr);
/* page-lock memory the caller owns (e.g. a POSIX shared-memory frame that several ranks fill with their bands) */
int hmrm_host_register(void *ptr, size_t bytes);
int hmrm_host_unregister(void *ptr);

/* ---- peer frames: one big frame rendered by several GPUs of one node (one process per GPU) ----
 * The root rank allocates the frame on its device and exports a 64-byte handle (CUDA IPC); every other rank opens it
 * and passes the mapped pointer to hmrm_render_device together with band_count / band_index: its kernel then stores
 * its tile rows straight into the root's frame over NVLink — no pack, no gather, no unpack; the only collective left
 * is the barrier that tells the root the frame is complete.  New surface: the reference has one OpenMP loop
 * (main/hmap.cpp:978) and no multi-GPU path. */
#define HMRM_IPC_HANDLE_BYTES 64
int hmrm_device_alloc(hmrm_ctx *ctx, size_t bytes, void **dptr);          /* zero-filled */
int hmrm_device_free(hmrm_ctx *ctx, void *dptr);
int hmrm_ipc_export(hmrm_ctx *ctx, void *dptr, uint8_t handle[HMRM_IPC_HANDLE_BYTES]);   /* dptr from hmrm_device_alloc */
int hmrm_ipc_open(hmrm_ctx *ctx, const uint8_t handle[HMRM_IPC_HANDLE_BYTES], void **dptr); /* in ANOTHER process */
int hmrm_ipc_close(hmrm_ctx *ctx, void *dptr);

/* Device-side completion of a peer frame (csrc/peer_sync.cuh): no collective, no host synchronisation.
 * The root allocates frame bytes + HMRM_PEER_CTRL_BYTES with hmrm_device_alloc (zero-filled); the control block is the
 * last HMRM_PEER_CTRL_BYTES of it (any 128-byte aligned place will do).  `use` counts the uses of ONE buffer, from 1.
 *   every rank:  hmrm_render_peer(ctx, f, d_frame, d_ctrl, use, stream)   waits (on the device) until the root has
 *                released use - 1, renders this rank's bands (f->band_count / band_index) into d_frame and counts the
 *                rank as arrived;
 *   the root:    hmrm_peer_wait(ctx, d_ctrl, use, ranks, stream)          stream-ordered: what follows on `stream`
 *                sees the complete frame;  hmrm_peer_release(ctx, d_ctrl, use, stream) when it has been read.
 * Two implementations of the same protocol on the same block, chosen once per context (hmrm_create):
 *   stream memory operations (the default when the driver has cuStreamWaitValue32 / cuStreamWriteValue32): the GPU's
 *     front end waits and writes, no SM is involved — a one-thread kernel needs a CTA slot, and the persistent render
 *     kernels of the frames in flight hold them all (measured, 8 GPUs: 0.2006 vs 0.2181 ms per 8K frame).  Every rank
 *     writes its own arrival word.  No timeout: a missing peer leaves the stream blocked (cudaStreamQuery says so);
 *   one-thread kernels (HMRM_PEER_SYNC=kernels in the environment): `arrived` is one counter; a wait that lasts
 *     longer than 5 s (HMRM_PEER_TIMEOUT_MS) sets the block's error word instead of hanging the GPU.
 * Every rank of a frame must use the same one.  hmrm_peer_status returns {arrived counter, released, error}. */
#define HMRM_PEER_CTRL_BYTES 256
int hmrm_render_peer(hmrm_ctx *ctx, const hmrm_frame *f, void *d_frame, void *d_ctrl, uint32_t use, void *stream);
/* The same with the exchange done by the copy engine: the rank renders its bands into d_stage (a frame-sized buffer
 * on ITS device), then pushes exactly its tile rows into d_frame with one strided device-to-device copy, then counts
 * itself in.  One more pass over the rank's rows, but NVLink sees large transfers instead of the kernel's 24- / 32-byte
 * row pieces: the faster exchange when many ranks write into one root (DESIGN.md section 6). */
int hmrm_render_peer_staged(hmrm_ctx *ctx, const hmrm_frame *f, void *d_stage, void *d_frame, void *d_ctrl, uint32_t use,
                            void *stream);
int hmrm_peer_wait(hmrm_ctx *ctx, void *d_ctrl, uint32_t use, int32_t ranks, void *stream);
int hmrm_peer_release(hmrm_ctx *ctx, void *d_ctrl, uint32_t use, void *stream);
int hmrm_peer_status(hmrm_ctx *ctx, void *d_ctrl, uint32_t out[3]);
#define HMRM_PEER_SYNC_KERNELS 0
#define HMRM_PEER_SYNC_MEMOPS 1
int hmrm_peer_sync_mode(const hmrm_ctx *ctx);     /* which implementation this context uses; < 0: ctx is NULL */

#ifdef __cplusplus
}
#endif

#endif
