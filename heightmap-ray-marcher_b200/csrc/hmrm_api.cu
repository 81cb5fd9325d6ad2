// libhmrm.so — C ABI (include/hmrm.h) over the sm_100a kernels.
//
// Host responsibilities (the reference does these inline in main(), see the
// line references in include/hmrm.h): own the device copies of the maps, run
// the K1 prepass when lum/min/max/maps change, build the per-frame image-plane
// constants with the host libm, launch K2, move the framebuffer.
// There is no CPU rendering path in this library.
#include <cuda.h>
#include <cuda_runtime.h>

#include <algorithm>
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <utility>
#include <vector>

#include "../../include/hmrm.h"
#include "frame_setup.h"
#include "k1_prepass.cuh"
#include "k2_render_brute.cuh"
#include "k2_render_skip.cuh"
#include "k2_render_lin.cuh"
#include "k2_render_pack.cuh"
#include "k3_png.cuh"
#include "k4_yuv.cuh"
#include "k5_downsample.cuh"
#include "k6_jpeg.cuh"
#include "peer_sync.cuh"
#include "render_params.h"
#include "synth_fbm.h"

using namespace hmrm;

namespace {

std::string g_create_error;

const int kLaunchSlots = 8;
const int kFrameRing = 4;      // device frame buffers (and compute streams) whole frames rotate through
const int kSubFrames = 4;      // sub-frame scratches of supersampled / motion-blurred frames, used round-robin
const int kBlurMax = 16;       // most motion-blur sub-frames (hmrm_set_motion_blur)

// Everything one launch writes before / while its kernel runs.  A slot is reused only after the kernel that used
// it last has finished (ev_end), so up to kLaunchSlots frames of one context may be in flight on any streams.
struct LaunchSlot {
	DeviceStats *d_stats;
	unsigned int *d_tile_counter;
	cudaEvent_t ev_begin, ev_end;
	bool used;
	double *sph_host;      // pinned staging of the spherical tables
	double *d_sph;
	size_t sph_cap;        // doubles
	int *d_row_order;
	int row_cap;
	double row_key[8];
	bool row_key_valid;
	int row_sky_first;           // schedule position of the first tile row that only looks above the horizon
	int32_t *d_step_index;       // HMRM_FLAG_STEP_INDEX output of the launch that used this slot
	size_t step_cap;             // pixels
	double *d_ray_dump;          // HMRM_FLAG_RAY_DUMP output, [pixels][10]
	size_t dump_cap;             // pixels
	uint8_t *view_host;          // hmrm_render_views: pinned staging of a batch's view records, schedule and spherical
	uint8_t *d_view;             // tables, and their device copy (view_pieces)
	size_t view_cap;             // bytes of each
};

// The sW x sH RGBA8 renders of one supersampled or motion-blurred frame, read by K5: up to kDownMaxPlanes planes, and
// K5's accumulator when a blurred frame has more sub-frames than planes.  Inside the frame the planes are reused in
// stream order; across frames the scratch is reused only after the filter that read it last has run (ev_read), so up to
// kSubFrames such frames of one context may be in flight on any streams.
struct SubFrame {
	uint32_t *d;
	size_t cap;                   // bytes
	uint2 *acc;                   // [H][W] sums (K5's kK5First .. kK5Last)
	size_t acc_cap;               // bytes
	cudaEvent_t ev_read;
	bool used;
};

} // namespace

// Experiment knobs (environment, read ONCE in hmrm_create): they never change a result, only how the work is
// scheduled / how many fetches are issued.
struct Knobs {
	bool no_row_order, no_batch, debug_sched, reset_kernel, peer_memops, views_view_major;
	int lmin_bias, lstride, lstart, sky_batch;
	float cell_exit, climb;
	bool zq_shrink_set;
	double zq_shrink;
	unsigned long long peer_timeout_ns;
};

struct hmrm_ctx {
	int device;
	Knobs knobs;
	int num_sms;
	cudaStream_t stream;          // compute stream of frame-buffer slot 0 (and of everything that is not a frame)
	cudaStream_t ring_stream[kFrameRing];   // compute stream of each frame buffer ([0] == stream): frame n+1 starts
	                                        // while frame n's tail drains
	std::string err;

	// maps
	int map_w, map_h;
	uint8_t *d_rgb;              // RGB8 [map_h][map_w][3], or with height_bits 16 the u16 plane [map_h][map_w] (2n <= 3n bytes)
	int height_bits;             // 8 (hmrm_set_maps, hmrm_synth_maps) or 16 (hmrm_set_maps16, hmrm_synth_maps16)
	uint32_t *d_color;           // RGBA8
	double *d_surf;              // fl(height + min_height)
	unsigned long long *d_max_bits;  // [0] max, [1] min of surf (order-preserving bits); [2] quantiser error flag
	bool maps_set, heights_set;
	double lum[3], min_height, max_height, max_surf, min_surf;
	// conservative fixed-point view for the skip traversal
	uint16_t *d_mip;             // what the traversal reads, levels 0..mip_levels-1 back to back: level 0 = Zq(surf)
	                             // per cell, level l >= 1 = 3x3-block dilation of the plain max-mip level l
	uint16_t *d_dil;             // scratch: the plain (undilated) max-mip levels 1.., input of the dilation
	size_t mip_offset[16];       // element offset of level l inside d_mip (sizes depend on the layout)
	size_t plain_offset[16];     // element offset of plain level l (>= 1) inside d_dil (row-major)
	int mip_w[16], mip_h[16];
	int mip_levels;
	int layout;                  // HMRM_LAYOUT_* of d_mip (pyramid_layout.cuh); fixed while maps are allocated
	int layout_wanted;           // takes effect at the next hmrm_update_heightmap
	unsigned int *d_k1_counter;  // k1_mip_upper's arrival counter
	double zq_scale, zq_offset;
	bool skip_ready;

	// per-resolution tables
	int tab_w, tab_h;
	std::vector<double> wtab, htab, sph;
	double *d_wtab, *d_htab;

	// outputs
	uint32_t *d_fb[kFrameRing];  // [0]: the persistent framebuffer (the reference's framebuf, main/hmap.cpp:612);
	                             // whole frames rotate through all of them so that frames n+1, n+2 render while frame
	                             // n is copied out
	int fb_w, fb_h;
	cudaStream_t copy_stream;
	cudaEvent_t ev_rendered[kFrameRing], ev_copied[kFrameRing];
	bool copy_pending[kFrameRing];
	int fb_format;               // pixel format of what the ring holds (a change re-zeroes it, like a new resolution)
	int slot;                    // buffer of the most recent hmrm_render_async
	// encoder scratch per ring slot, grown by the first frame that needs more: K3 (PNG), K4 (YUV) and K6 (JPEG) carve
	// their pieces from it (png_pieces, jpeg_pieces; K4's I420 planes are the whole of it)
	uint8_t *d_scratch[kFrameRing];
	size_t scratch_cap[kFrameRing];
	uint8_t *d_pixels;           // hmrm_encode_png's / _jpeg's / hmrm_convert_yuv420's device copy of the caller's pixels
	size_t pixels_cap;
	uint8_t *d_views;            // hmrm_render_views' device copy of the views before they go to the caller's memory
	size_t views_cap;
	// supersampled frames (K5): sub-frame scratches, allocated by the first supersampled frame that uses them
	SubFrame sub[kSubFrames];
	int sub_next;
	// motion blur (hmrm_set_motion_blur): blur_n sub-frame cameras, 0 = off; read when a frame is enqueued
	int blur_n;
	hmrm_camera blur_cams[kBlurMax];

	// per-launch resources, used round-robin so that up to kLaunchSlots kernels of this context may be in flight
	LaunchSlot slots[kLaunchSlots];
	int launch_next, launch_last;
	bool last_had_stats, last_had_step_index, last_had_ray_dump, timing_valid;
	int last_w, last_h;
	cudaStream_t last_stream;    // stream of the most recent render (the caller's, for hmrm_render_device)
};

namespace {

int fail(hmrm_ctx *ctx, int code, const char *fmt, ...) {
	char buf[512];
	va_list ap;
	va_start(ap, fmt);
	vsnprintf(buf, sizeof buf, fmt, ap);
	va_end(ap);
	if (ctx) ctx->err = buf;
	else g_create_error = buf;
	return code;
}

#define HMRM_CUDA(ctx, call)                                                                       \
	do {                                                                                           \
		cudaError_t e_ = (call);                                                                   \
		if (e_ != cudaSuccess)                                                                     \
			return fail((ctx), HMRM_ERR_CUDA, "%s failed: %s", #call, cudaGetErrorString(e_));     \
	} while (0)

bool finite3(const double *v) { return std::isfinite(v[0]) && std::isfinite(v[1]) && std::isfinite(v[2]); }

// Grows the device buffer *p of *cap bytes to at least `need` bytes.  Its contents are not kept; the caller makes sure
// no work in flight still uses it.
template <class T>
int grow(hmrm_ctx *c, T **p, size_t *cap, size_t need) {
	if (need <= *cap) return HMRM_OK;
	cudaFree(*p);
	*p = NULL;
	*cap = 0;
	HMRM_CUDA(c, cudaMalloc(p, need));
	*cap = need;
	return HMRM_OK;
}

__global__ void __launch_bounds__(256) k_synth_maps(uint32_t log2n, uint32_t seed, uint8_t *__restrict__ rgb,
                                                    uint32_t *__restrict__ rgba) {
	const uint32_t n = 1u << log2n;
	const unsigned long long total = (unsigned long long)n * n;
	const unsigned long long stride = (unsigned long long)gridDim.x * blockDim.x;
	for (unsigned long long p = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x; p < total; p += stride) {
		const uint32_t x = (uint32_t)(p & (n - 1u)), y = (uint32_t)(p >> log2n);
		const uint32_t v = hmrm_synth_height(x, y, log2n, seed);
		rgb[3ULL * p + 0] = (uint8_t)v;
		rgb[3ULL * p + 1] = (uint8_t)v;
		rgb[3ULL * p + 2] = (uint8_t)v;
		rgba[p] = hmrm_synth_color(v, x, y, n);
	}
}

// 16-bit height plane and the colormap of hmrm_synth_maps (the same seed gives the same colours)
__global__ void __launch_bounds__(256) k_synth_maps16(uint32_t log2n, uint32_t seed, uint16_t *__restrict__ h16,
                                                      uint32_t *__restrict__ rgba) {
	const uint32_t n = 1u << log2n;
	const unsigned long long total = (unsigned long long)n * n;
	const unsigned long long stride = (unsigned long long)gridDim.x * blockDim.x;
	for (unsigned long long p = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x; p < total; p += stride) {
		const uint32_t x = (uint32_t)(p & (n - 1u)), y = (uint32_t)(p >> log2n);
		h16[p] = (uint16_t)hmrm_synth_height16(x, y, log2n, seed);
		rgba[p] = hmrm_synth_color(hmrm_synth_height(x, y, log2n, seed), x, y, n);
	}
}

// the device's slab test on caller-supplied rays and boxes (hmrm_debug_aabb): the very function the render kernels call
__global__ void k_debug_aabb(int n, const double *rays, const double *boxes, double *out) {
	const int i = blockIdx.x * blockDim.x + threadIdx.x;
	if (i >= n) return;
	Ray r;
	r.ox = rays[6 * i + 0]; r.oy = rays[6 * i + 1]; r.oz = rays[6 * i + 2];
	r.dx = rays[6 * i + 3]; r.dy = rays[6 * i + 4]; r.dz = rays[6 * i + 5];
	double ex = 0.0, ey = 0.0, ez = 0.0, dist = 0.0;
	const bool hit = box_entry_at(boxes + 6 * i, boxes + 6 * i + 3, r, ex, ey, ez, dist);
	out[5 * i + 0] = dist;
	out[5 * i + 1] = hit ? 1.0 : 0.0;
	out[5 * i + 2] = hit ? ex : 0.0;
	out[5 * i + 3] = hit ? ey : 0.0;
	out[5 * i + 4] = hit ? ez : 0.0;
}

int drain(hmrm_ctx *c) {
	for (int i = 0; i < kFrameRing; ++i) HMRM_CUDA(c, cudaStreamSynchronize(c->ring_stream[i]));
	HMRM_CUDA(c, cudaStreamSynchronize(c->copy_stream));
	// kernels launched on the caller's streams (hmrm_render_device) are tracked by their slot's end event
	for (int i = 0; i < kLaunchSlots; ++i) {
		if (c->slots[i].used) HMRM_CUDA(c, cudaEventSynchronize(c->slots[i].ev_end));
	}
	// and so are the box filters that follow them
	for (int i = 0; i < kSubFrames; ++i) {
		if (c->sub[i].used) HMRM_CUDA(c, cudaEventSynchronize(c->sub[i].ev_read));
	}
	return HMRM_OK;
}

void free_maps(hmrm_ctx *c) {
	cudaFree(c->d_rgb);
	cudaFree(c->d_color);
	cudaFree(c->d_surf);
	cudaFree(c->d_mip);
	cudaFree(c->d_dil);
	c->d_mip = NULL;
	c->d_dil = NULL;
	c->d_rgb = NULL;
	c->d_color = NULL;
	c->d_surf = NULL;
	c->maps_set = c->heights_set = false;
}

// element offsets of the pyramid levels for `layout` (mip_w / mip_h / mip_levels are set); returns the total
size_t layout_pyramid(hmrm_ctx *c, int layout) {
	size_t total = 0;
	for (int l = 0; l < c->mip_levels; ++l) {
		c->mip_offset[l] = total;
		total += (pyr_level_elems(layout, c->mip_w[l], c->mip_h[l]) + 63) & ~(size_t)63;
	}
	return total;
}

int alloc_maps(hmrm_ctx *c, int32_t w, int32_t h) {
	if (w < 1 || h < 1 || w > 32768 || h > 32768)
		return fail(c, HMRM_ERR_INVALID, "map size %dx%d outside [1,32768]", w, h);
	HMRM_CUDA(c, cudaSetDevice(c->device));
	if (int rc = drain(c)) return rc;
	if (c->maps_set && c->map_w == w && c->map_h == h) {
		c->heights_set = false;
		return HMRM_OK;
	}
	free_maps(c);
	const size_t n = (size_t)w * (size_t)h;
	HMRM_CUDA(c, cudaMalloc(&c->d_rgb, n * 3));
	HMRM_CUDA(c, cudaMalloc(&c->d_color, n * 4));
	HMRM_CUDA(c, cudaMalloc(&c->d_surf, n * 8));
	// mip pyramid of 16-bit conservative heights: level l is ceil(w/2^l) x ceil(h/2^l), up to a single texel
	int lw = w, lh = h, levels = 0;
	size_t plain_total = 0;
	for (;;) {
		c->mip_w[levels] = lw;
		c->mip_h[levels] = lh;
		c->plain_offset[levels] = plain_total;
		if (levels >= 1) plain_total += ((size_t)lw * (size_t)lh + 63) & ~(size_t)63;
		levels += 1;
		if ((lw == 1 && lh == 1) || levels == 16) break;
		lw = (lw + 1) / 2;
		lh = (lh + 1) / 2;
	}
	c->mip_levels = levels;
	// the pyramid buffer fits whichever layout is selected later (hmrm_set_layout + hmrm_update_heightmap)
	size_t cap = 0;
	for (int layout = 0; layout < 3; ++layout) cap = std::max(cap, layout_pyramid(c, layout));
	c->layout = c->layout_wanted;
	layout_pyramid(c, c->layout);
	HMRM_CUDA(c, cudaMalloc(&c->d_mip, cap * 2));
	if (levels > 1) HMRM_CUDA(c, cudaMalloc(&c->d_dil, plain_total * 2));
	c->map_w = w;
	c->map_h = h;
	return HMRM_OK;
}

int ensure_tables(hmrm_ctx *c, int W, int H) {
	if (c->tab_w == W && c->tab_h == H) return HMRM_OK;
	if (int rc = drain(c)) return rc;
	cudaFree(c->d_wtab);
	cudaFree(c->d_htab);
	c->d_wtab = c->d_htab = NULL;
	c->tab_w = c->tab_h = 0;
	fill_wh_tables(W, H, &c->wtab, &c->htab);
	HMRM_CUDA(c, cudaMalloc(&c->d_wtab, (size_t)W * 8));
	HMRM_CUDA(c, cudaMalloc(&c->d_htab, (size_t)H * 8));
	HMRM_CUDA(c, cudaMemcpy(c->d_wtab, c->wtab.data(), (size_t)W * 8, cudaMemcpyHostToDevice));
	HMRM_CUDA(c, cudaMemcpy(c->d_htab, c->htab.data(), (size_t)H * 8, cudaMemcpyHostToDevice));
	c->tab_w = W;
	c->tab_h = H;
	return HMRM_OK;
}

int ensure_framebuffer(hmrm_ctx *c, int W, int H, int format) {
	if (c->d_fb[0] && c->fb_w == W && c->fb_h == H && c->fb_format == format) return HMRM_OK;
	if (int rc = drain(c)) return rc;
	for (int i = 0; i < kFrameRing; ++i) {
		c->copy_pending[i] = false;
		cudaFree(c->d_fb[i]);
		c->d_fb[i] = NULL;
	}
	c->fb_w = c->fb_h = 0;
	for (int i = 0; i < kFrameRing; ++i) {
		HMRM_CUDA(c, cudaMalloc(&c->d_fb[i], (size_t)W * (size_t)H * 4));
		// the reference's framebuf starts uninitialised (main/hmap.cpp:612); start from zeros instead
		HMRM_CUDA(c, cudaMemset(c->d_fb[i], 0, (size_t)W * (size_t)H * 4));
	}
	c->slot = 0;
	c->fb_w = W;
	c->fb_h = H;
	c->fb_format = format;
	return HMRM_OK;
}

int validate_frame(hmrm_ctx *c, const hmrm_frame *f, int *row_begin, int *row_end) {
	if (!f) return fail(c, HMRM_ERR_INVALID, "frame is NULL");
	if (!c->maps_set) return fail(c, HMRM_ERR_STATE, "hmrm_set_maps has not been called");
	if (!c->heights_set) return fail(c, HMRM_ERR_STATE, "hmrm_update_heightmap has not been called");
	if (f->projection < HMRM_PERSPECTIVE || f->projection > HMRM_ORTHOGRAPHIC)
		return fail(c, HMRM_ERR_INVALID, "projection %d is not 1, 2 or 3", f->projection);
	// w = px/(W-1), h = py/(H-1) (main/hmap.cpp:986-987) are 0/0 for a 1-pixel axis
	if (f->screen_width < 2 || f->screen_height < 2 || f->screen_width > 65536 || f->screen_height > 65536)
		return fail(c, HMRM_ERR_INVALID, "resolution %dx%d outside [2,65536]", f->screen_width, f->screen_height);
	if (!finite3(f->cam_pos) || !std::isfinite(f->hang) || !std::isfinite(f->vang) || !std::isfinite(f->hfov) ||
	    !std::isfinite(f->ortho_width))
		return fail(c, HMRM_ERR_INVALID, "camera parameters must be finite");
	if (!(f->grid_width > 0.0) || !std::isfinite(f->grid_width))
		return fail(c, HMRM_ERR_INVALID, "grid_width must be positive and finite");
	// step_dist <= 0 never terminates in the reference (main/hmap.cpp:1000-1038)
	if (!(f->step_dist > 0.0) || !std::isfinite(f->step_dist))
		return fail(c, HMRM_ERR_INVALID, "step_dist must be positive and finite");
	// cycle_period 0 is a division by zero in the reference (main/hmap.cpp:976)
	if (f->cycle_period < 1 || f->cycle < 0 || f->cycle >= f->cycle_period)
		return fail(c, HMRM_ERR_INVALID, "need cycle_period >= 1 and 0 <= cycle < cycle_period");
	if (f->precision != HMRM_FP64_EXACT && f->precision != HMRM_FP32_FAST)
		return fail(c, HMRM_ERR_INVALID, "unknown precision %d", f->precision);
	if (f->pixel_format != HMRM_PIXEL_RGBA8 && f->pixel_format != HMRM_PIXEL_RGB8)
		return fail(c, HMRM_ERR_INVALID, "unknown pixel_format %d", (int)f->pixel_format);
	int rb = f->row_begin, re = f->row_end;
	if (rb == 0 && re == 0) re = f->screen_height;
	if (rb < 0 || re > f->screen_height || rb >= re)
		return fail(c, HMRM_ERR_INVALID, "row band [%d,%d) outside the frame", rb, re);
	if (f->band_count < 0 || (f->band_count > 1 && (f->band_index < 0 || f->band_index >= f->band_count)))
		return fail(c, HMRM_ERR_INVALID, "need 0 <= band_index < band_count");
	*row_begin = rb;
	*row_end = re;
	return HMRM_OK;
}

// Zeroes a launch slot's tile-queue counter and statistics block (sizeof(DeviceStats) is a multiple of 4).
__global__ void k_reset_slot(unsigned int *tile_counter, unsigned int *stats_words) {
	if (threadIdx.x == 0) *tile_counter = 0u;
	for (unsigned i = threadIdx.x; i < sizeof(DeviceStats) / 4; i += 32) stats_words[i] = 0u;
}

// Takes a launch slot and waits (host side) for the kernel that used it kLaunchSlots launches ago.  A blurred frame's
// later sub-frames skip the slot that accumulates its statistics (acc_slot): its ev_end is their own latest kernel.
int take_slot(hmrm_ctx *c, int acc_slot, int *ls) {
	if (c->launch_next == acc_slot) c->launch_next = (acc_slot + 1) % kLaunchSlots;
	*ls = c->launch_next;
	c->launch_next = (*ls + 1) % kLaunchSlots;
	LaunchSlot &slot = c->slots[*ls];
	if (slot.used) HMRM_CUDA(c, cudaEventSynchronize(slot.ev_end));
	return HMRM_OK;
}

// The fields of P that one frame of `f` and every view of a batch of `f` share: screen, map, box, march constants,
// tables, pixel format and background; plus the camera constants of pc.
void frame_params(hmrm_ctx *c, const hmrm_frame *f, const PlaneConst &pc, RenderParams *P) {
	std::memset(P, 0, sizeof *P);
	P->projection = f->projection;
	P->W = f->screen_width;
	P->H = f->screen_height;
	P->tiles_x = (P->W + 7) / 8;
	P->inv_tiles_x = std::nextafterf(1.0f / (float)P->tiles_x, 0.0f) * (1.0f - 1.0e-6f);
	P->map_w = c->map_w;
	P->map_h = c->map_h;
	const Vec3 *src[5] = {&pc.cam, &pc.ul, &pc.pr, &pc.pd, &pc.look};
	double *dst[5] = {P->cam, P->ul, P->pr, P->pd, P->look};
	for (int i = 0; i < 5; ++i) {
		dst[i][0] = src[i]->x;
		dst[i][1] = src[i]->y;
		dst[i][2] = src[i]->z;
	}
	// main/hmap.cpp:967-974
	P->c0[0] = 0.0;
	P->c0[1] = 0.0;
	P->c0[2] = c->min_height;
	P->c1[0] = P->c0[0] + c->map_w * f->grid_width;
	P->c1[1] = P->c0[1] - c->map_h * f->grid_width;
	P->c1[2] = c->max_height;
	for (int i = 0; i < 3; ++i) {
		P->bmin[i] = std::fmin(P->c0[i], P->c1[i]);
		P->bmax[i] = std::fmax(P->c0[i], P->c1[i]);
	}
	P->gw = f->grid_width;
	P->nudge = f->grid_width * 0.01;
	P->step_dist = f->step_dist;
	P->max_surf = c->max_surf;
	P->wtab = c->d_wtab;
	P->htab = c->d_htab;
	P->row_order = NULL;
	P->batch_from_tile = 0xFFFFFFFFu;
	P->sky_batch = (unsigned)c->knobs.sky_batch;
	P->surf = c->d_surf;
	P->color = c->d_color;
	P->pixel_format = f->pixel_format;
	P->bg[0] = f->bg[0];
	P->bg[1] = f->bg[1];
	P->bg[2] = f->bg[2];
	P->bg_rgba = (uint32_t)f->bg[0] | ((uint32_t)f->bg[1] << 8) | ((uint32_t)f->bg[2] << 16) | 0xFF000000u;
}

// The skip traversals' constants of P (c->skip_ready).  The caller falls back to HMRM_TRAVERSAL_BRUTE when
// P->fx_bits < 1 or P->fx_scale is not finite.
void skip_params(hmrm_ctx *c, const hmrm_frame *f, RenderParams *P) {
	int dim = c->map_w > c->map_h ? c->map_w : c->map_h, clog = 0;
	while ((1 << clog) < dim) clog += 1;
	P->fx_bits = 30 - clog < 20 ? 30 - clog : 20;
	P->fx_scale = std::ldexp(1.0, P->fx_bits) / f->grid_width;
	if (P->fx_bits >= 1) {
		P->lin_grid_x = (unsigned)c->map_w << P->fx_bits;
		P->lin_grid_y = (unsigned)c->map_h << P->fx_bits;
		P->lin_span_x = P->lin_grid_x - 2u * HMRM_LIN_MARGIN;
		P->lin_span_y = P->lin_grid_y - 2u * HMRM_LIN_MARGIN;
	}
	P->zq_scale = c->zq_scale;
	P->zq_offset = c->zq_offset;
	P->inv_gw_up = (1.0 / f->grid_width) * 1.000001;
	P->ltop = c->mip_levels - 1;
	// lowest useful block: about one step wide (measured: profiles/r01_knob_sweep.txt)
	const double step_cells = f->step_dist / f->grid_width;
	int lmin = 1;
	while (lmin < P->ltop && (double)(1 << lmin) < step_cells) lmin += 1;
	// tuning knobs for experiments (never affect results, only how many fetches are issued): read once, hmrm_create
	lmin += c->knobs.lmin_bias;
	if (lmin < 1) lmin = 1;
	if (lmin > P->ltop) lmin = P->ltop;
	P->lmin = lmin;
	P->lstride = c->knobs.lstride < 1 ? 1 : c->knobs.lstride;
	P->cell_exit_scale = c->knobs.cell_exit;
	P->climb_ratio = c->knobs.climb;
	const int lstart = lmin + c->knobs.lstart * P->lstride;
	P->lstart = lstart > P->ltop ? P->ltop : (lstart < lmin ? lmin : lstart);
	P->lv = c->d_mip;
	P->lv_total = (unsigned long long)(c->mip_offset[c->mip_levels - 1] +
	                                   pyr_level_elems(c->layout, c->mip_w[c->mip_levels - 1], c->mip_h[c->mip_levels - 1]));
	P->layout = c->layout;
	for (int l = 0; l < 16; ++l) {
		P->lv_desc[l].x = (l < c->mip_levels) ? (unsigned)c->mip_offset[l] : 0u;
		P->lv_desc[l].y = (l < c->mip_levels) ? pyr_level_pitch(c->layout, c->mip_w[l]) : 0u;
	}
}

// Tile-row schedule: rows whose rays graze the terrain (direction just below the horizon) march for hundreds of
// steps at low clearance and cost ~50x the mean tile; rows that look up cost nothing.  Start the expensive rows
// first (cost proxy 1/|dir.z| of the centre ray for dir.z < 0).  Depends on the projection, W, H, hfov, vang and the
// rows only, not on the camera position or heading, so a flythrough computes it once and views with one vang share it.
// order[0 .. tiles_y) gets the tile rows t (frame tile row first + t * step) costliest first; `sky_first` the position
// in it from which on every row's lowest pixel row still looks up (cheap sky; a hint only).  `cost_scratch` is working
// space the caller may keep across calls.
void row_schedule(const PlaneConst &pc, int H, int row_begin, int first, int step, int tiles_y, int *order,
                  int *sky_first, std::vector<std::pair<double, int> > *cost_scratch) {
	std::vector<std::pair<double, int> > &cost = *cost_scratch;
	cost.resize((size_t)tiles_y);
	for (int t = 0; t < tiles_y; ++t) {
		int py = row_begin + (first + t * step) * 4 + 2;
		if (py > H - 1) py = H - 1;
		Vec3 pos, dir;
		plane_ray(pc, 0.5, (double)py / (H - 1), &pos, &dir);
		const double dz = dir.z;
		cost[(size_t)t].first = (dz < 0.0) ? -1.0 / std::fmax(-dz, 1e-3) : 1.0 + dz;   // ascending sort key
		cost[(size_t)t].second = t;
	}
	std::stable_sort(cost.begin(), cost.end());
	for (int t = 0; t < tiles_y; ++t) order[t] = cost[(size_t)t].second;
	*sky_first = tiles_y;
	for (int t = tiles_y - 1; t >= 0; --t) {
		int py = row_begin + (first + order[t] * step) * 4 + 3;
		if (py > H - 1) py = H - 1;
		Vec3 pos, dir;
		plane_ray(pc, 0.5, (double)py / (H - 1), &pos, &dir);
		if (!(dir.z >= 0.0) || !(cost[(size_t)t].first >= 1.0)) break;
		*sky_first = t;
	}
}

// The persistent lin kernel over P's tiles: HMRM_LIN_CTAS_LARGE CTAs per SM from HMRM_LIN_LARGE_TILES tiles on,
// HMRM_LIN_CTAS below, and no more CTAs than it takes to give every warp one tile.
template <bool kViews>
int launch_lin(hmrm_ctx *c, const RenderParams &P, bool stats_kernel, cudaStream_t stream) {
	const int n_tiles = P.tiles_x * P.tiles_y;
	const int lin_warps = HMRM_LIN_THREADS / 32;
	const bool large = n_tiles >= HMRM_LIN_LARGE_TILES;
	int lin_blocks = c->num_sms * (large ? HMRM_LIN_CTAS_LARGE : HMRM_LIN_CTAS);
	if (lin_blocks > (n_tiles + lin_warps - 1) / lin_warps) lin_blocks = (n_tiles + lin_warps - 1) / lin_warps;
	if (lin_blocks < 1) lin_blocks = 1;
#define HMRM_LAUNCH_LIN_SHAPE(LAYOUT, CTAS)                                                                              \
	do {                                                                                                                 \
		if (stats_kernel) k2_render_lin<true, LAYOUT, CTAS, kViews><<<lin_blocks, HMRM_LIN_THREADS, 0, stream>>>(P);     \
		else k2_render_lin<false, LAYOUT, CTAS, kViews><<<lin_blocks, HMRM_LIN_THREADS, 0, stream>>>(P);                 \
	} while (0)
#define HMRM_LAUNCH_LIN(LAYOUT)                                                                                          \
	do {                                                                                                                 \
		if (large) HMRM_LAUNCH_LIN_SHAPE(LAYOUT, HMRM_LIN_CTAS_LARGE);                                                   \
		else HMRM_LAUNCH_LIN_SHAPE(LAYOUT, HMRM_LIN_CTAS);                                                               \
	} while (0)
	if (c->layout == HMRM_LAYOUT_TILE4) HMRM_LAUNCH_LIN(kLayoutTile4);
	else if (c->layout == HMRM_LAYOUT_ZORDER) HMRM_LAUNCH_LIN(kLayoutZOrder);
	else HMRM_LAUNCH_LIN(kLayoutRowMajor);
#undef HMRM_LAUNCH_LIN
#undef HMRM_LAUNCH_LIN_SHAPE
	return HMRM_OK;
}

// Zeroes slot ls's tile-queue counter and (unless acc_slot >= 0) statistics block on `stream`.
int reset_slot(hmrm_ctx *c, LaunchSlot &slot, int acc_slot, cudaStream_t stream) {
	if (acc_slot >= 0) HMRM_CUDA(c, cudaMemsetAsync(slot.d_tile_counter, 0, sizeof(unsigned int), stream));
	else if (!c->knobs.reset_kernel) {
		HMRM_CUDA(c, cudaMemsetAsync(slot.d_tile_counter, 0, sizeof(unsigned int), stream));
		HMRM_CUDA(c, cudaMemsetAsync(slot.d_stats, 0, sizeof(DeviceStats), stream));
	}
	else {
		// experiment (HMRM_RESET_KERNEL): one tiny kernel instead of the two memsets.  Measured: 0.4411 vs 0.4365 ms per
		// flythrough4k frame, 0.2268 vs 0.2286 ms per 8K band frame at N = 8 — nothing in it; a kernel needs a CTA slot
		// that the previous frame's persistent CTAs still hold, the memsets do not
		k_reset_slot<<<1, 32, 0, stream>>>(slot.d_tile_counter, (unsigned int *)slot.d_stats);
		HMRM_CUDA(c, cudaGetLastError());
	}
	return HMRM_OK;
}

// Enqueue one frame on `stream`, writing the frame's pixel format into d_out (any alignment).  acc_slot >= 0: a later
// sub-frame of a motion-blurred frame whose first sub-frame used launch slot acc_slot (on the same stream).  Its
// statistics add into that slot's block (no reset), the slot's ev_end moves past this kernel, and hmrm_get_stats then
// reports that slot: the sums over the sub-frames, timed from the first one's start to the last one's end.
int enqueue_render(hmrm_ctx *c, const hmrm_frame *f, uint32_t *d_out, cudaStream_t stream, bool timed,
                   int acc_slot = -1) {
	int row_begin = 0, row_end = 0;
	int rc = validate_frame(c, f, &row_begin, &row_end);
	if (rc) return rc;
	HMRM_CUDA(c, cudaSetDevice(c->device));
	const int W = f->screen_width, H = f->screen_height;
	if ((rc = ensure_tables(c, W, H)) != HMRM_OK) return rc;

	int ls = 0;
	if ((rc = take_slot(c, acc_slot, &ls)) != HMRM_OK) return rc;
	LaunchSlot &slot = c->slots[ls];

	const PlaneConst pc = build_plane(*f);

	RenderParams P;
	frame_params(c, f, pc, &P);
	P.row_begin = row_begin;
	P.row_end = row_end;
	P.cycle = f->cycle;
	P.period = f->cycle_period;
	const int tile_rows = (row_end - row_begin + 3) / 4;
	if (f->band_count > 1) {
		// interleaved bands: sky rows are almost free and terrain rows are not, so contiguous bands balance badly
		P.tile_y_first = f->band_index;
		P.tile_y_step = f->band_count;
		P.tiles_y = tile_rows > f->band_index ? (tile_rows - f->band_index + f->band_count - 1) / f->band_count : 0;
	}
	else {
		P.tile_y_first = 0;
		P.tile_y_step = 1;
		P.tiles_y = tile_rows;
	}

	if (f->projection == HMRM_SPHERICAL) {
		const size_t need = (size_t)(2 * W + 2 * H);
		if (need > slot.sph_cap) {
			if (slot.sph_host) cudaFreeHost(slot.sph_host);
			cudaFree(slot.d_sph);
			slot.sph_host = NULL;
			slot.d_sph = NULL;
			slot.sph_cap = 0;
			HMRM_CUDA(c, cudaMallocHost(&slot.sph_host, need * 8));
			HMRM_CUDA(c, cudaMalloc(&slot.d_sph, need * 8));
			slot.sph_cap = need;
		}
		fill_spherical_tables(pc, W, H, c->wtab, c->htab, &c->sph);
		std::memcpy(slot.sph_host, c->sph.data(), need * 8);
		HMRM_CUDA(c, cudaMemcpyAsync(slot.d_sph, slot.sph_host, need * 8, cudaMemcpyHostToDevice, stream));
		P.cos_ha = slot.d_sph;
		P.sin_ha = slot.d_sph + W;
		P.sin_va = slot.d_sph + 2 * W;
		P.cos_va = slot.d_sph + 2 * W + H;
	}

	// tile-row schedule (row_schedule), cached per launch slot
	if (f->projection != HMRM_ORTHOGRAPHIC && P.tiles_y > 1 && !c->knobs.no_row_order) {
		const double key[8] = {(double)f->projection, (double)W, (double)H, f->vang, f->hfov, (double)row_begin,
		                       (double)(P.tile_y_first * 65536 + P.tile_y_step), (double)P.tiles_y};
		if (!slot.row_key_valid || std::memcmp(key, slot.row_key, sizeof key) != 0) {
			std::vector<int> order((size_t)P.tiles_y);
			std::vector<std::pair<double, int> > cost;
			row_schedule(pc, H, row_begin, P.tile_y_first, P.tile_y_step, P.tiles_y, order.data(), &slot.row_sky_first, &cost);
			if (P.tiles_y > slot.row_cap) {
				cudaFree(slot.d_row_order);
				slot.d_row_order = NULL;
				slot.row_cap = 0;
				HMRM_CUDA(c, cudaMalloc(&slot.d_row_order, (size_t)P.tiles_y * sizeof(int)));
				slot.row_cap = P.tiles_y;
			}
			// pageable source: the copy is staged before the call returns; ordered before this slot's kernel
			HMRM_CUDA(c, cudaMemcpyAsync(slot.d_row_order, order.data(), (size_t)P.tiles_y * sizeof(int),
			                             cudaMemcpyHostToDevice, stream));
			HMRM_CUDA(c, cudaStreamSynchronize(stream));
			std::memcpy(slot.row_key, key, sizeof key);
			slot.row_key_valid = true;
		}
		P.row_order = slot.d_row_order;
		// (only when the camera is above the terrain: from below, rows that look up are the expensive ones)
		if (P.cam[2] > std::fmax(P.c0[2], P.c1[2]) && !c->knobs.no_batch)
			P.batch_from_tile = (unsigned)slot.row_sky_first * (unsigned)P.tiles_x;
		if (c->knobs.debug_sched)
			std::fprintf(stderr, "sched: tiles_y %d sky_first %d batch_from %u n_tiles %d\n", P.tiles_y, slot.row_sky_first,
			             P.batch_from_tile, P.tiles_x * P.tiles_y);
	}

	P.fb = d_out;
	// hmrm_render_device and the peer calls take any caller pointer: word stores only where they are aligned
	P.fb_unaligned = ((uintptr_t)d_out & 3u) != 0u ? 1 : 0;
	P.rgb_words = (W % 4) == 0 && !P.fb_unaligned ? 1 : 0;

	const bool want_stats = (f->flags & HMRM_FLAG_STATS) != 0;
	const bool want_steps = (f->flags & HMRM_FLAG_STEP_INDEX) != 0;
	const bool want_dump = (f->flags & HMRM_FLAG_RAY_DUMP) != 0;
	// per-launch-slot outputs: the slot's previous kernel has finished (ev_end above), so growing them is safe while
	// other frames of this context are still in flight on other streams
	if (want_steps) {
		const size_t need = (size_t)W * (size_t)H;
		if (need > slot.step_cap) {
			cudaFree(slot.d_step_index);
			slot.d_step_index = NULL;
			slot.step_cap = 0;
			HMRM_CUDA(c, cudaMalloc(&slot.d_step_index, need * 4));
			slot.step_cap = need;
		}
		HMRM_CUDA(c, cudaMemsetAsync(slot.d_step_index, 0xFD, need * 4, stream));   // -3 = not rendered... bytes FD
		P.step_index = slot.d_step_index;
	}
	if (want_dump) {
		const size_t need = (size_t)W * (size_t)H;
		if (need > slot.dump_cap) {
			cudaFree(slot.d_ray_dump);
			slot.d_ray_dump = NULL;
			slot.dump_cap = 0;
			HMRM_CUDA(c, cudaMalloc(&slot.d_ray_dump, need * 80));
			slot.dump_cap = need;
		}
		HMRM_CUDA(c, cudaMemsetAsync(slot.d_ray_dump, 0xFF, need * 80, stream));    // NaN = not rendered
		P.ray_dump = slot.d_ray_dump;
	}
	P.stats = acc_slot >= 0 ? c->slots[acc_slot].d_stats : slot.d_stats;
	P.tile_counter = slot.d_tile_counter;
	if ((rc = reset_slot(c, slot, acc_slot, stream)) != HMRM_OK) return rc;

	int traversal = f->traversal;
	if (traversal == HMRM_TRAVERSAL_AUTO) traversal = c->skip_ready ? HMRM_TRAVERSAL_SKIP : HMRM_TRAVERSAL_BRUTE;
	if (traversal != HMRM_TRAVERSAL_BRUTE && traversal != HMRM_TRAVERSAL_SKIP && traversal != HMRM_TRAVERSAL_SKIP_FP64 &&
	    traversal != HMRM_TRAVERSAL_PACK)
		return fail(c, HMRM_ERR_INVALID, "unknown traversal %d", f->traversal);
	if (traversal != HMRM_TRAVERSAL_BRUTE) {
		if (!c->skip_ready)
			return fail(c, HMRM_ERR_STATE, "the height range could not be quantised; use HMRM_TRAVERSAL_BRUTE");
		skip_params(c, f, &P);
		if (P.fx_bits < 1 || !std::isfinite(P.fx_scale)) traversal = HMRM_TRAVERSAL_BRUTE;
	}

	const int n_tiles = P.tiles_x * P.tiles_y;
	const int warps_per_block = 8;
	int blocks = c->num_sms * 4;   // brute and FP64 skip kernels: persistent CTAs, 4 x 256 threads per SM (lin, pack: below)
	const int max_useful = (n_tiles + warps_per_block - 1) / warps_per_block;
	if (blocks > max_useful) blocks = max_useful;
	if (blocks < 1) blocks = 1;

	(void)timed;
	HMRM_CUDA(c, cudaEventRecord(slot.ev_begin, stream));
	if (traversal == HMRM_TRAVERSAL_SKIP) {
		if ((rc = launch_lin<false>(c, P, want_stats || want_steps || want_dump, stream)) != HMRM_OK) return rc;
	}
	else if (traversal == HMRM_TRAVERSAL_PACK) {
		const bool stats_kernel = want_stats || want_steps || want_dump;
		const int lin_warps = HMRM_LIN_THREADS / 32;
		int lin_blocks = c->num_sms * HMRM_PACK_CTAS;
		if (lin_blocks > (n_tiles + lin_warps - 1) / lin_warps) lin_blocks = (n_tiles + lin_warps - 1) / lin_warps;
		if (lin_blocks < 1) lin_blocks = 1;
#define HMRM_LAUNCH_PACK(LAYOUT)                                                                              \
		do {                                                                                                  \
			if (stats_kernel) k2_render_pack<true, LAYOUT><<<lin_blocks, HMRM_LIN_THREADS, 0, stream>>>(P);   \
			else k2_render_pack<false, LAYOUT><<<lin_blocks, HMRM_LIN_THREADS, 0, stream>>>(P);               \
		} while (0)
		if (c->layout == HMRM_LAYOUT_TILE4) HMRM_LAUNCH_PACK(kLayoutTile4);
		else if (c->layout == HMRM_LAYOUT_ZORDER) HMRM_LAUNCH_PACK(kLayoutZOrder);
		else HMRM_LAUNCH_PACK(kLayoutRowMajor);
#undef HMRM_LAUNCH_PACK
	}
	else if (traversal == HMRM_TRAVERSAL_SKIP_FP64) {
		if (want_stats || want_steps || want_dump) k2_render_skip<true><<<blocks, warps_per_block * 32, 0, stream>>>(P);
		else k2_render_skip<false><<<blocks, warps_per_block * 32, 0, stream>>>(P);
	}
	else {
		if (want_stats || want_dump) k2_render_brute<true><<<blocks, warps_per_block * 32, 0, stream>>>(P);
		else k2_render_brute<false><<<blocks, warps_per_block * 32, 0, stream>>>(P);
	}
	HMRM_CUDA(c, cudaGetLastError());
	HMRM_CUDA(c, cudaEventRecord(slot.ev_end, stream));
	slot.used = true;
	c->launch_last = ls;
	if (acc_slot >= 0) {
		HMRM_CUDA(c, cudaEventRecord(c->slots[acc_slot].ev_end, stream));
		c->launch_last = acc_slot;
	}

	c->last_stream = stream;
	c->last_had_stats = want_stats;
	c->last_had_step_index = want_steps;
	c->last_had_ray_dump = want_dump;
	c->timing_valid = timed;
	c->last_w = W;
	c->last_h = H;
	return HMRM_OK;
}

// ---- supersampled and motion-blurred frames (K5, csrc/k5_downsample.cuh) -------------------------------------------
int supersample_of(const hmrm_frame *f) {
	return (int)((f->flags & HMRM_FLAG_SUPERSAMPLE_MASK) >> HMRM_FLAG_SUPERSAMPLE_SHIFT) + 1;
}

// The refusals of frames that can only be whole frames: supersampled, motion-blurred and encoded ones; kind names the
// frames in the messages.
int check_whole_frame(hmrm_ctx *c, const hmrm_frame *f, const char *kind) {
	if (f->cycle_period != 1 || f->cycle != 0)
		return fail(c, HMRM_ERR_INVALID, "%s frames are whole frames: cycle_period 1", kind);
	if (f->band_count > 1) return fail(c, HMRM_ERR_INVALID, "%s frames are whole frames: band_count <= 1", kind);
	if (f->row_begin != 0 || (f->row_end != 0 && f->row_end != f->screen_height))
		return fail(c, HMRM_ERR_INVALID, "%s frames are whole frames: row_begin 0, row_end 0 or screen_height", kind);
	if (f->flags & (HMRM_FLAG_STEP_INDEX | HMRM_FLAG_RAY_DUMP))
		return fail(c, HMRM_ERR_INVALID, "%s frames do not record step indices or ray dumps", kind);
	return HMRM_OK;
}

// The supersample field of a frame for the entry points that accept it, s = 1..4, and the context's motion blur: frames
// with s > 1 or blur are whole frames only.
int check_supersample(hmrm_ctx *c, const hmrm_frame *f) {
	const int s = supersample_of(f);
	if (s > 4) return fail(c, HMRM_ERR_INVALID, "supersample factor %d: the field (flags bits 8-11) holds s - 1 <= 3", s);
	if (s == 1 && c->blur_n == 0) return HMRM_OK;
	if (s > 1 && ((long long)s * f->screen_width > 65536 || (long long)s * f->screen_height > 65536))
		return fail(c, HMRM_ERR_INVALID, "supersample %d of %dx%d: the sub-frame is larger than 65536 per axis", s,
		            f->screen_width, f->screen_height);
	return check_whole_frame(c, f, c->blur_n ? "motion-blurred" : "supersampled");
}

void set_camera(hmrm_frame *f, const hmrm_camera &cam) {
	f->cam_pos[0] = cam.cam_pos[0];
	f->cam_pos[1] = cam.cam_pos[1];
	f->cam_pos[2] = cam.cam_pos[2];
	f->hang = cam.hang;
	f->vang = cam.vang;
}

// K5 over `planes` sub-frame planes in phase `phase` (kK5First and kK5Middle always reduce kDownMaxPlanes planes)
template <int S, int G>
void launch_k5_planes(int phase, bool rgb8, dim3 grid, cudaStream_t st, const uint32_t *sub, size_t plane, int W, int H,
                      uint8_t *out, uint2 *acc, uint32_t n) {
	if (phase == kK5Only && rgb8) k5_downsample<S, 3, G, kK5Only><<<grid, kDownThreads, 0, st>>>(sub, W, H, out, plane);
	else if (phase == kK5Only) k5_downsample<S, 4, G, kK5Only><<<grid, kDownThreads, 0, st>>>(sub, W, H, out, plane);
	else if (phase == kK5First)
		k5_downsample<S, 4, kDownMaxPlanes, kK5First><<<grid, kDownThreads, 0, st>>>(sub, W, H, out, plane, acc);
	else if (phase == kK5Middle)
		k5_downsample<S, 4, kDownMaxPlanes, kK5Middle><<<grid, kDownThreads, 0, st>>>(sub, W, H, out, plane, acc);
	else if (rgb8) k5_downsample<S, 3, G, kK5Last><<<grid, kDownThreads, 0, st>>>(sub, W, H, out, plane, acc, n);
	else k5_downsample<S, 4, G, kK5Last><<<grid, kDownThreads, 0, st>>>(sub, W, H, out, plane, acc, n);
}

template <int S>
void launch_k5(int planes, int phase, bool rgb8, dim3 grid, cudaStream_t st, const uint32_t *sub, size_t plane, int W,
               int H, uint8_t *out, uint2 *acc, uint32_t n) {
	if (planes == 1) launch_k5_planes<S, 1>(phase, rgb8, grid, st, sub, plane, W, H, out, acc, n);
	else if (planes == 2) launch_k5_planes<S, 2>(phase, rgb8, grid, st, sub, plane, W, H, out, acc, n);
	else if (planes == 3) launch_k5_planes<S, 3>(phase, rgb8, grid, st, sub, plane, W, H, out, acc, n);
	else launch_k5_planes<S, 4>(phase, rgb8, grid, st, sub, plane, W, H, out, acc, n);
}

// Enqueue one whole frame on `stream` into d_out in the frame's pixel format.  Without supersampling or blur this is
// enqueue_render.  Otherwise its n sub-frames (n = 1 without blur: the frame's own camera) are rendered at sW x sH into
// the planes of one sub-frame scratch, kDownMaxPlanes at a time, and K5 reduces each group into d_out, or through the
// scratch's accumulator when n > kDownMaxPlanes, all on the same stream.
int enqueue_frame(hmrm_ctx *c, const hmrm_frame *f, uint32_t *d_out, cudaStream_t stream) {
	if (int rc = check_supersample(c, f)) return rc;
	const int s = supersample_of(f);
	const int n = c->blur_n > 0 ? c->blur_n : 1;
	hmrm_frame sf = *f;
	if (c->blur_n == 1) set_camera(&sf, c->blur_cams[0]);
	if (s == 1 && n == 1) return enqueue_render(c, &sf, d_out, stream, true);
	const int W = f->screen_width, H = f->screen_height;
	sf.screen_width = s * W;
	sf.screen_height = s * H;
	sf.pixel_format = HMRM_PIXEL_RGBA8;
	sf.flags &= ~HMRM_FLAG_SUPERSAMPLE_MASK;
	sf.row_begin = sf.row_end = 0;
	// every sub-frame is checked before any of them is enqueued
	for (int j = 0; j < n; ++j) {
		if (c->blur_n > 1) set_camera(&sf, c->blur_cams[j]);
		int row_begin = 0, row_end = 0;
		if (int rc = validate_frame(c, &sf, &row_begin, &row_end)) return rc;
	}
	HMRM_CUDA(c, cudaSetDevice(c->device));

	// take a scratch; wait (host side) for the filter that read it kSubFrames such frames ago
	SubFrame &b = c->sub[c->sub_next];
	c->sub_next = (c->sub_next + 1) % kSubFrames;
	if (b.used) HMRM_CUDA(c, cudaEventSynchronize(b.ev_read));
	const int G = std::min(n, kDownMaxPlanes);
	const size_t plane = (size_t)sf.screen_width * (size_t)sf.screen_height;     // words
	if (int rc = grow(c, &b.d, &b.cap, plane * 4 * (size_t)G)) return rc;
	if (int rc = grow(c, &b.acc, &b.acc_cap, n > G ? (size_t)W * (size_t)H * sizeof(uint2) : 0)) return rc;
	const dim3 grid((unsigned)(((W + kDownStrip - 1) / kDownStrip + kDownThreads - 1) / kDownThreads), (unsigned)H);
	uint8_t *out = (uint8_t *)d_out;
	const bool rgb8 = f->pixel_format == HMRM_PIXEL_RGB8;
	const uint32_t divisor = (uint32_t)(n * s * s);
	int acc_slot = -1;
	for (int j = 0; j < n; ++j) {
		// a plane is rendered again only after the K5 launch that read it, which precedes it on this stream
		if (c->blur_n > 1) set_camera(&sf, c->blur_cams[j]);
		if (int rc = enqueue_render(c, &sf, b.d + (size_t)(j % G) * plane, stream, true, acc_slot)) return rc;
		if (j == 0) acc_slot = c->launch_last;
		if (j % G != G - 1 && j != n - 1) continue;
		const int planes = j % G + 1;
		const int phase = n == G ? kK5Only : j < G ? kK5First : j == n - 1 ? kK5Last : kK5Middle;
		if (s == 1) launch_k5<1>(planes, phase, rgb8, grid, stream, b.d, plane, W, H, out, b.acc, divisor);
		else if (s == 2) launch_k5<2>(planes, phase, rgb8, grid, stream, b.d, plane, W, H, out, b.acc, divisor);
		else if (s == 3) launch_k5<3>(planes, phase, rgb8, grid, stream, b.d, plane, W, H, out, b.acc, divisor);
		else launch_k5<4>(planes, phase, rgb8, grid, stream, b.d, plane, W, H, out, b.acc, divisor);
		HMRM_CUDA(c, cudaGetLastError());
	}
	HMRM_CUDA(c, cudaEventRecord(b.ev_read, stream));
	b.used = true;
	return HMRM_OK;
}

// D2H of what one launch of `f` rendered: its row band [rb, re), or with band_count > 1 only the tile rows of that band
// (several ranks may fill one shared, registered host frame, each over its own PCIe link): one strided copy + the
// ragged last tile row.  Enqueued on copy_stream.
int enqueue_copy_out(hmrm_ctx *c, const hmrm_frame *f, const uint32_t *fb, uint8_t *rgba_out, cudaMemcpyKind kind,
                     cudaStream_t copy_stream) {
	int rb = f->row_begin, re = f->row_end;
	if (rb == 0 && re == 0) re = f->screen_height;
	const size_t row_bytes = (size_t)f->screen_width * (f->pixel_format == HMRM_PIXEL_RGB8 ? 3 : 4);
	if (f->band_count > 1) {
		const int tile_rows = (re - rb + 3) / 4;
		const int owned = tile_rows > f->band_index ? (tile_rows - f->band_index + f->band_count - 1) / f->band_count : 0;
		if (owned > 0) {
			const int last_tile = f->band_index + (owned - 1) * f->band_count;
			const int last_rows = (re - rb) - last_tile * 4 < 4 ? (re - rb) - last_tile * 4 : 4;
			const int full = last_rows == 4 ? owned : owned - 1;
			const size_t first = (size_t)(rb + f->band_index * 4) * row_bytes;
			const size_t pitch = (size_t)f->band_count * 4 * row_bytes;
			if (full > 0)
				HMRM_CUDA(c, cudaMemcpy2DAsync(rgba_out + first, pitch, (const uint8_t *)fb + first, pitch, 4 * row_bytes,
				                               (size_t)full, kind, copy_stream));
			if (full < owned) {
				const size_t at = (size_t)(rb + last_tile * 4) * row_bytes;
				HMRM_CUDA(c, cudaMemcpyAsync(rgba_out + at, (const uint8_t *)fb + at, (size_t)last_rows * row_bytes, kind,
				                             copy_stream));
			}
		}
	}
	else {
		HMRM_CUDA(c, cudaMemcpyAsync(rgba_out + (size_t)rb * row_bytes, (const uint8_t *)fb + (size_t)rb * row_bytes,
		                             (size_t)(re - rb) * row_bytes, kind, copy_stream));
	}
	return HMRM_OK;
}

// ---- peer-frame synchronisation words: stream memory operations (default) or one-thread kernels ------------------
// The waits and writes of csrc/peer_sync.cuh's protocol as cuStreamWaitValue32 / cuStreamWriteValue32, executed by the
// GPU's front end.  A one-thread kernel needs a free CTA slot, and the persistent render kernels of the frames in
// flight hold every slot of the device until their tail: each kernel of the protocol then waits for the next render
// kernel to drain.  The memory operations need no SM.  (They have no timeout: a missing peer leaves the stream
// blocked — cudaStreamQuery stays cudaErrorNotReady — instead of raising the error word.)
typedef CUresult (*StreamValueFn)(CUstream, CUdeviceptr, cuuint32_t, unsigned int);
struct MemOps {
	StreamValueFn wait32, write32;   // both NULL: the driver does not have them
};

MemOps lookup_memops() {
	MemOps m = {NULL, NULL};
	void *w = NULL, *x = NULL;
	cudaDriverEntryPointQueryResult qw, qx;
	const cudaError_t e1 = cudaGetDriverEntryPoint("cuStreamWaitValue32", &w, cudaEnableDefault, &qw);
	const cudaError_t e2 = cudaGetDriverEntryPoint("cuStreamWriteValue32", &x, cudaEnableDefault, &qx);
	if (e1 == cudaSuccess && e2 == cudaSuccess && qw == cudaDriverEntryPointSuccess && qx == cudaDriverEntryPointSuccess && w && x) {
		m.wait32 = (StreamValueFn)w;
		m.write32 = (StreamValueFn)x;
	}
	else cudaGetLastError();
	return m;
}

const MemOps &memops() {
	static const MemOps m = lookup_memops();   // looked up once (thread-safe), after a device has been selected
	return m;
}

bool probe_memops() { return memops().wait32 != NULL; }

int load_memops(hmrm_ctx *c) {
	if (!probe_memops()) return fail(c, HMRM_ERR_CUDA, "HMRM_PEER_SYNC=memops: the driver has no stream memory operations");
	return HMRM_OK;
}

int peer_wait_word(hmrm_ctx *c, unsigned int *word, unsigned int target, unsigned int *error, cudaStream_t s) {
	if (c->knobs.peer_memops) {
		if (int rc = load_memops(c)) return rc;
		const CUresult r = memops().wait32((CUstream)s, (CUdeviceptr)(uintptr_t)word, target, CU_STREAM_WAIT_VALUE_GEQ);
		if (r != CUDA_SUCCESS) return fail(c, HMRM_ERR_CUDA, "cuStreamWaitValue32 failed (%d)", (int)r);
		return HMRM_OK;
	}
	k_peer_spin<<<1, 1, 0, s>>>(word, target, error, c->knobs.peer_timeout_ns);
	HMRM_CUDA(c, cudaGetLastError());
	return HMRM_OK;
}

int peer_write_word(hmrm_ctx *c, unsigned int *word, unsigned int value, cudaStream_t s) {
	if (int rc = load_memops(c)) return rc;
	// default flags: a memory barrier orders everything the stream did before (peer stores, the frame copy) ahead of it
	const CUresult r = memops().write32((CUstream)s, (CUdeviceptr)(uintptr_t)word, value, CU_STREAM_WRITE_VALUE_DEFAULT);
	if (r != CUDA_SUCCESS) return fail(c, HMRM_ERR_CUDA, "cuStreamWriteValue32 failed (%d)", (int)r);
	return HMRM_OK;
}

// this rank's bands of use `use` are in the root's frame
int peer_arrive(hmrm_ctx *c, PeerCtrl *ctrl, const hmrm_frame *f, unsigned int use, cudaStream_t s) {
	if (c->knobs.peer_memops) {
		const int r = f->band_count > 1 ? f->band_index : 0;
		if (r < 0 || r > 30) return fail(c, HMRM_ERR_INVALID, "peer frame: band_index %d out of range", r);
		return peer_write_word(c, &ctrl->arrived_by[r], use, s);
	}
	k_peer_signal<<<1, 1, 0, s>>>(&ctrl->arrived);
	HMRM_CUDA(c, cudaGetLastError());
	return HMRM_OK;
}

// ---- encoder scratch of the ring slots ------------------------------------------------------------------------------
// One buffer per slot serves K3, K4 and K6 alike.  Two frames of one slot are ordered on one stream (the copy stream, or
// c->stream after drain for the one-shot calls), and each encoder writes every scratch byte it reads within its frame,
// so what an earlier frame of another format left there is never read.
int ensure_slot_scratch(hmrm_ctx *c, int slot, size_t need) {
	if (need <= c->scratch_cap[slot]) return HMRM_OK;
	// the slot's previous frame may still be encoding from, or copying out of, the buffer about to be replaced
	if (c->copy_pending[slot]) HMRM_CUDA(c, cudaEventSynchronize(c->ev_copied[slot]));
	return grow(c, &c->d_scratch[slot], &c->scratch_cap[slot], need);
}

// Lays pieces out back to back from `base`, each on a 256-byte boundary (K3's gather reads uint4 words of the staged
// pieces, K6 int16 / uint32 arrays); `bytes` is what they take.  From base 0 it only counts.
struct Carve {
	uintptr_t base;
	size_t bytes;
	template <class T>
	T *take(unsigned long long n) {
		T *p = (T *)(base + bytes);
		bytes += ((size_t)n * sizeof(T) + 255) & ~(size_t)255;
		return p;
	}
};

// ---- PNG frames (K3, csrc/k3_png.cuh) ------------------------------------------------------------------------------
// K3's pieces of a slot's scratch: filtered stream, staged chunks, signature / IHDR / tail chunks, per-segment sizes /
// Adler-32 partials, piece offsets
struct PngPieces {
	uint8_t *filt, *stage, *meta;
	PngSegInfo *info;
	unsigned long long *offsets;
	size_t bytes;
};

PngPieces png_pieces(const PngShape &s, uint8_t *scratch) {
	Carve k = {(uintptr_t)scratch, 0};
	PngPieces p;
	p.filt = k.take<uint8_t>(s.total);
	p.stage = k.take<uint8_t>((unsigned long long)s.nseg * kPngStageStride);
	p.meta = k.take<uint8_t>(kPngMetaBytes);
	p.info = k.take<PngSegInfo>((unsigned long long)s.nseg);
	p.offsets = k.take<unsigned long long>((unsigned long long)s.nseg + 3);
	p.bytes = k.bytes;
	return p;
}

// The address the device writes `p` through: device memory of the context's device as it is, pinned / registered host
// memory through its mapping.  Pageable memory is refused with a status (the device cannot write it).
int device_view(hmrm_ctx *c, void *p, const char *what, void **dev) {
	cudaPointerAttributes a;
	const cudaError_t e = cudaPointerGetAttributes(&a, p);
	if (e != cudaSuccess) {
		cudaGetLastError();
		return fail(c, HMRM_ERR_INVALID, "%s: %s", what, cudaGetErrorString(e));
	}
	if (a.type == cudaMemoryTypeDevice) {
		if (a.device != c->device)
			return fail(c, HMRM_ERR_INVALID, "%s is memory of device %d, not of the context's device %d", what, a.device,
			            c->device);
		*dev = p;
		return HMRM_OK;
	}
	if (a.type == cudaMemoryTypeHost && a.devicePointer) {
		*dev = a.devicePointer;
		return HMRM_OK;
	}
	return fail(c, HMRM_ERR_INVALID, "%s must be pinned or registered host memory, or device memory of device %d", what,
	            c->device);
}

// validates the file destination `out` / capacity / size word `bytes` of an encoded file (fmt "png" | "jpeg") whose
// worst-case size is `bound`, and resolves their device addresses
int file_outputs(hmrm_ctx *c, const char *fmt, unsigned long long bound, uint8_t *out, size_t capacity, uint64_t *bytes,
                 uint8_t **d_out, unsigned long long **d_size) {
	if (!out || !bytes) return fail(c, HMRM_ERR_INVALID, "%s_out and %s_bytes must not be NULL", fmt, fmt);
	if ((uintptr_t)bytes % 8 != 0) return fail(c, HMRM_ERR_INVALID, "%s_bytes must be 8-byte aligned", fmt);
	if ((unsigned long long)capacity < bound)
		return fail(c, HMRM_ERR_INVALID, "capacity %zu is below hmrm_%s_bound = %llu", capacity, fmt, bound);
	HMRM_CUDA(c, cudaSetDevice(c->device));
	void *o = NULL, *z = NULL;
	char what[32];
	std::snprintf(what, sizeof what, "%s_out", fmt);
	if (int rc = device_view(c, out, what, &o)) return rc;
	std::snprintf(what, sizeof what, "%s_bytes", fmt);
	if (int rc = device_view(c, bytes, what, &z)) return rc;
	*d_out = (uint8_t *)o;
	*d_size = (unsigned long long *)z;
	return HMRM_OK;
}

// Enqueue the four K3 launches on `st`: d_img [H][W][C] -> PNG file at d_dst, its size at d_size.
int enqueue_png(hmrm_ctx *c, uint8_t *scratch, const uint8_t *d_img, int W, int H, int C, uint8_t *d_dst,
                unsigned long long *d_size, cudaStream_t st) {
	PngShape s{};
	png_shape(W, H, C, &s);
	const PngPieces p = png_pieces(s, scratch);
	k3_png_filter<<<H, 256, 0, st>>>(d_img, (int)s.row_bytes, C, p.filt);
	// the byte one row up is a candidate distance while deflate can reach it
	const int row_dist = s.row_bytes + 1 <= 32768ull ? (int)(s.row_bytes + 1) : 0;
	k3_png_deflate<<<(s.nseg + kPngDeflateWarps - 1) / kPngDeflateWarps, kPngDeflateWarps * 32, 0, st>>>(
		p.filt, s.total, s.nseg, C, row_dist, p.stage, p.info);
	k3_png_finish<<<1, 1024, 0, st>>>(p.info, s.nseg, s.total, W, H, C, p.offsets, p.meta);
	const unsigned long long words = png_bound(s) / 16 + 2;
	const int blocks = (int)std::min((words + 255) / 256, (unsigned long long)c->num_sms * 16ull);
	k3_png_gather<<<blocks, 256, 0, st>>>(p.offsets, s.nseg + 2, p.meta, p.meta + kPngMetaTail, p.stage, kPngStageStride,
	                                      d_dst, d_size);
	HMRM_CUDA(c, cudaGetLastError());
	return HMRM_OK;
}

// ---- YUV frames (K4, csrc/k4_yuv.cuh) ------------------------------------------------------------------------------
// validates matrix / out / capacity for a W x H frame
int yuv_output(hmrm_ctx *c, int W, int H, int32_t matrix, uint8_t *out, size_t capacity) {
	if (matrix != HMRM_YUV_BT601 && matrix != HMRM_YUV_BT709) return fail(c, HMRM_ERR_INVALID, "unknown YUV matrix %d", matrix);
	if (!out) return fail(c, HMRM_ERR_INVALID, "out is NULL");
	const unsigned long long need = yuv420_bytes(W, H);
	if ((unsigned long long)capacity < need)
		return fail(c, HMRM_ERR_INVALID, "capacity %zu is below hmrm_yuv420_bytes = %llu", capacity, need);
	HMRM_CUDA(c, cudaSetDevice(c->device));
	void *unused = NULL;
	return device_view(c, out, "out", &unused);
}

// Enqueue K4 on `st`: d_img [H][W][C] -> I420 planes in the slot's scratch, then one copy of them to `out` (host or
// device memory).
int enqueue_yuv(hmrm_ctx *c, uint8_t *scratch, const uint8_t *d_img, int W, int H, int C, int32_t matrix, uint8_t *out,
                cudaStream_t st) {
	const size_t bytes = (size_t)yuv420_bytes(W, H);
	const dim3 grid((unsigned)(((W + 7) / 8 + kYuvThreads - 1) / kYuvThreads), (unsigned)((H + 1) / 2));
	if (C == 4) k4_yuv420<4><<<grid, kYuvThreads, 0, st>>>(d_img, W, H, kYuvCoef[matrix], scratch);
	else k4_yuv420<3><<<grid, kYuvThreads, 0, st>>>(d_img, W, H, kYuvCoef[matrix], scratch);
	HMRM_CUDA(c, cudaGetLastError());
	HMRM_CUDA(c, cudaMemcpyAsync(out, scratch, bytes, cudaMemcpyDefault, st));
	return HMRM_OK;
}

// The refusals every whole-frame encoder shares (hmrm_render_png_async, _yuv420_async, _jpeg_async); kind names the
// frames in the messages.
int check_encoded_frame(hmrm_ctx *c, const hmrm_frame *f, const char *kind) {
	if (!f) return fail(c, HMRM_ERR_INVALID, "frame is NULL");
	if (int rc = check_supersample(c, f)) return rc;
	if (int rc = check_whole_frame(c, f, kind)) return rc;
	if (f->pixel_format != HMRM_PIXEL_RGBA8 && f->pixel_format != HMRM_PIXEL_RGB8)
		return fail(c, HMRM_ERR_INVALID, "unknown pixel_format %d", (int)f->pixel_format);
	if (f->screen_width < 2 || f->screen_height < 2 || f->screen_width > 65536 || f->screen_height > 65536)
		return fail(c, HMRM_ERR_INVALID, "resolution %dx%d outside [2,65536]", f->screen_width, f->screen_height);
	return HMRM_OK;
}

// ---- JPEG frames (K6, csrc/k6_jpeg.cuh) ----------------------------------------------------------------------------
// K6's pieces of a slot's scratch: quantised coefficients, AC bit counts and bit offsets per block, the rows' bit buffers
// and stuffed pieces, header / EOI, row sizes, piece offsets
struct JpegPieces {
	int16_t *coef;
	uint16_t *acbits;
	uint32_t *boff, *rowbits;
	uint8_t *stage, *meta;
	unsigned long long *rowsize, *offsets;
	size_t bytes;
};

JpegPieces jpeg_pieces(const JpegShape &s, uint8_t *scratch) {
	Carve k = {(uintptr_t)scratch, 0};
	JpegPieces p;
	p.coef = k.take<int16_t>(s.blocks * 64);
	p.acbits = k.take<uint16_t>(s.blocks);
	p.boff = k.take<uint32_t>(s.blocks);
	p.rowbits = k.take<uint32_t>(s.row_words * (unsigned long long)s.mcuy);
	p.stage = k.take<uint8_t>(s.row_stride * (unsigned long long)s.mcuy);
	p.meta = k.take<uint8_t>(kJpegMetaBytes);
	p.rowsize = k.take<unsigned long long>((unsigned long long)s.mcuy);
	p.offsets = k.take<unsigned long long>((unsigned long long)s.mcuy + 3);
	p.bytes = k.bytes;
	return p;
}

int jpeg_params(hmrm_ctx *c, int32_t quality, int32_t chroma) {
	if (quality < 1 || quality > 100) return fail(c, HMRM_ERR_INVALID, "JPEG quality %d outside [1,100]", quality);
	if (chroma != HMRM_JPEG_420 && chroma != HMRM_JPEG_444) return fail(c, HMRM_ERR_INVALID, "unknown JPEG chroma %d", chroma);
	return HMRM_OK;
}

// Enqueue the K6 launches and K3's gather on `st`: d_img [H][W][C] -> JPEG file at d_dst, its size at d_size.
int enqueue_jpeg(hmrm_ctx *c, uint8_t *scratch, const uint8_t *d_img, int W, int H, int C, int quality, int chroma,
                 uint8_t *d_dst, unsigned long long *d_size, cudaStream_t st) {
	JpegShape s{};
	jpeg_shape(W, H, chroma == HMRM_JPEG_420, &s);
	const JpegPieces p = jpeg_pieces(s, scratch);
	const int tile_mcus = kJpegTileBlocks / s.bpm;
	const dim3 grid((unsigned)((s.mcux + tile_mcus - 1) / tile_mcus), (unsigned)s.mcuy);
	const JpegQuant q = jpeg_quant(quality);
	if (C == 4 && s.s420) k6_jpeg_blocks<4, true><<<grid, kJpegBlockThreads, 0, st>>>(d_img, W, H, s.mcux, q, p.coef, p.acbits);
	else if (C == 4) k6_jpeg_blocks<4, false><<<grid, kJpegBlockThreads, 0, st>>>(d_img, W, H, s.mcux, q, p.coef, p.acbits);
	else if (s.s420) k6_jpeg_blocks<3, true><<<grid, kJpegBlockThreads, 0, st>>>(d_img, W, H, s.mcux, q, p.coef, p.acbits);
	else k6_jpeg_blocks<3, false><<<grid, kJpegBlockThreads, 0, st>>>(d_img, W, H, s.mcux, q, p.coef, p.acbits);
	k6_jpeg_rows<<<s.mcuy, kJpegRowThreads, 0, st>>>(p.coef, p.acbits, s.mcux, s.bpm, s.mcuy, p.boff, p.rowbits,
	                                                 s.row_words, p.stage, s.row_stride, p.rowsize);
	k6_jpeg_finish<<<1, 1024, 0, st>>>(p.rowsize, s.mcuy, jpeg_header(s, quality), p.offsets, p.meta);
	const unsigned long long words = jpeg_bound(s) / 16 + 2;
	const int blocks = (int)std::min((words + 255) / 256, (unsigned long long)c->num_sms * 16ull);
	k3_png_gather<<<blocks, 256, 0, st>>>(p.offsets, s.mcuy + 2, p.meta, p.meta + kJpegMetaTail, p.stage, s.row_stride,
	                                      d_dst, d_size);
	HMRM_CUDA(c, cudaGetLastError());
	return HMRM_OK;
}

// ---- the output stage, the frame ring and the one-shot encoders -----------------------------------------------------
// Where a finished [H][W][C] image goes.  PNG, JPEG and YUV work in `scratch` bytes of a ring slot's scratch.
struct Output {
	enum Kind { RAW, PNG, JPEG, YUV } kind;
	uint8_t *dst;                  // RAW, YUV: the caller's memory, written by the copy engine; PNG, JPEG: the device
	                               // address of the file destination (file_outputs)
	unsigned long long *size;      // PNG, JPEG: the device address of the file's size word
	size_t scratch;
	const hmrm_frame *frame;       // RAW: the frame whose row band, or band of band_count, is copied out
	int quality, chroma;           // JPEG
	int matrix;                    // YUV
};

// Enqueue the output stage of the image d_img on `st`, with ring slot `slot`'s scratch
int enqueue_output(hmrm_ctx *c, const Output &o, int slot, const uint8_t *d_img, int W, int H, int C, cudaStream_t st) {
	uint8_t *scratch = c->d_scratch[slot];
	switch (o.kind) {
	case Output::RAW: return enqueue_copy_out(c, o.frame, (const uint32_t *)d_img, o.dst, cudaMemcpyDeviceToHost, st);
	case Output::PNG: return enqueue_png(c, scratch, d_img, W, H, C, o.dst, o.size, st);
	case Output::JPEG: return enqueue_jpeg(c, scratch, d_img, W, H, C, o.quality, o.chroma, o.dst, o.size, st);
	case Output::YUV: return enqueue_yuv(c, scratch, d_img, W, H, C, o.matrix, o.dst, st);
	}
	return fail(c, HMRM_ERR_INVALID, "unknown output kind %d", (int)o.kind);
}

// The frame ring, the one owner of its protocol: every frame of hmrm_render_async, _png_async, _jpeg_async and
// _yuv420_async is rendered into a ring buffer on the buffer's compute stream, and its output stage runs on the copy
// stream.  Whole frames (cycle_period 1) rotate through kFrameRing device buffers so that the output stage of frame n
// overlaps the kernels of frames n+1 and n+2; the progressive interleave (cycle_period > 1) accumulates in the one
// persistent buffer.  Each buffer has its own compute stream, so the kernel of the next frame starts filling SMs as the
// CTAs of this one run out of tiles (a handful of grazing tiles take ~50x the mean: the tail of a frame leaves most SMs
// idle).
int enqueue_ring(hmrm_ctx *c, const hmrm_frame *f, const Output &o) {
	int rc = ensure_framebuffer(c, f->screen_width, f->screen_height, f->pixel_format);
	if (rc) return rc;
	const bool whole = f->cycle_period == 1 && (f->flags & (HMRM_FLAG_STEP_INDEX | HMRM_FLAG_RAY_DUMP)) == 0;
	const int slot = whole ? (c->slot + 1) % kFrameRing : 0;
	if ((rc = ensure_slot_scratch(c, slot, o.scratch)) != HMRM_OK) return rc;
	uint32_t *fb = c->d_fb[slot];
	cudaStream_t cs = c->ring_stream[slot];
	// nothing may be written into this buffer (by the kernel, or by the copy below) while an earlier frame's output
	// stage still reads it
	if (c->copy_pending[slot]) HMRM_CUDA(c, cudaStreamWaitEvent(cs, c->ev_copied[slot], 0));
	if (!whole) {
		// progressive frames and step-index captures are ordered after everything else
		for (int i = 1; i < kFrameRing; ++i) HMRM_CUDA(c, cudaStreamSynchronize(c->ring_stream[i]));
		if (f->cycle_period != 1 && c->slot != 0) {
			// the newest picture lives in another buffer of the ring: a progressive frame must land on top of it
			HMRM_CUDA(c, cudaMemcpyAsync(c->d_fb[0], c->d_fb[c->slot], (size_t)c->fb_w * (size_t)c->fb_h * 4,
			                             cudaMemcpyDeviceToDevice, cs));
		}
	}
	// (Rendering a frame that finds the pipeline idle as four interleaved bands, each copied out as soon as its kernel
	// is done, was measured: four launches mean four tails, the stream turns kernel-bound and stays "idle", 0.59 ->
	// 0.63 ms per frame.  Frames stay whole.)
	if ((rc = enqueue_frame(c, f, fb, cs)) != HMRM_OK) return rc;
	HMRM_CUDA(c, cudaEventRecord(c->ev_rendered[slot], cs));
	HMRM_CUDA(c, cudaStreamWaitEvent(c->copy_stream, c->ev_rendered[slot], 0));
	const int C = f->pixel_format == HMRM_PIXEL_RGB8 ? 3 : 4;
	rc = enqueue_output(c, o, slot, (const uint8_t *)fb, f->screen_width, f->screen_height, C, c->copy_stream);
	if (rc) return rc;
	HMRM_CUDA(c, cudaEventRecord(c->ev_copied[slot], c->copy_stream));
	c->copy_pending[slot] = true;
	c->slot = slot;
	return HMRM_OK;
}

// The caller's pixels in the context's staging buffer, copied on c->stream.  The context must be drained: the buffer
// may be replaced.
int stage_pixels(hmrm_ctx *c, const uint8_t *pixels, size_t bytes) {
	if (int rc = grow(c, &c->d_pixels, &c->pixels_cap, bytes)) return rc;
	HMRM_CUDA(c, cudaMemcpyAsync(c->d_pixels, pixels, bytes, cudaMemcpyDefault, c->stream));
	return HMRM_OK;
}

// hmrm_encode_png, _jpeg and hmrm_convert_yuv420: synchronous.  Whatever the context has in flight finishes first, then
// ring slot 0's scratch is free for the output stage of the caller's [H][W][C] pixels on c->stream.
int encode_staged(hmrm_ctx *c, const Output &o, const uint8_t *pixels, int W, int H, int C) {
	int rc = drain(c);
	if (rc) return rc;
	if ((rc = stage_pixels(c, pixels, (size_t)W * (size_t)H * (size_t)C)) != HMRM_OK) return rc;
	if ((rc = ensure_slot_scratch(c, 0, o.scratch)) != HMRM_OK) return rc;
	if ((rc = enqueue_output(c, o, 0, c->d_pixels, W, H, C, c->stream)) != HMRM_OK) return rc;
	HMRM_CUDA(c, cudaStreamSynchronize(c->stream));
	return HMRM_OK;
}

// ---- batches of views (hmrm_render_views, k2_render_lin<..., kViews = true>) ---------------------------------------
const int kMaxViews = 65536;                 // a schedule entry holds the view in 16 bits
const long long kMaxViewTiles = 1LL << 26;   // tile_row_col's float quotient is exact below 2^26 tiles

// The refusals of hmrm_render_views and hmrm_render_views_device; nothing is enqueued before they pass.
int check_views(hmrm_ctx *c, const hmrm_frame *f, const hmrm_camera *cams, int n, const void *out) {
	if (!f) return fail(c, HMRM_ERR_INVALID, "frame is NULL");
	if (!cams) return fail(c, HMRM_ERR_INVALID, "cams is NULL");
	if (!out) return fail(c, HMRM_ERR_INVALID, "output is NULL");
	if (n < 1 || n > kMaxViews) return fail(c, HMRM_ERR_INVALID, "%d views outside [1,%d]", n, kMaxViews);
	if (c->blur_n > 0) return fail(c, HMRM_ERR_INVALID, "views are single frames: no motion blur");
	if (supersample_of(f) != 1) return fail(c, HMRM_ERR_INVALID, "views are single frames: no supersampling");
	if (int rc = check_whole_frame(c, f, "view")) return rc;
	if (f->traversal != HMRM_TRAVERSAL_AUTO && f->traversal != HMRM_TRAVERSAL_SKIP)
		return fail(c, HMRM_ERR_INVALID, "views take HMRM_TRAVERSAL_AUTO or HMRM_TRAVERSAL_SKIP, not %d", f->traversal);
	for (int j = 0; j < n; ++j) {
		if (!finite3(cams[j].cam_pos) || !std::isfinite(cams[j].hang) || !std::isfinite(cams[j].vang))
			return fail(c, HMRM_ERR_INVALID, "camera %d of the views is not finite", j);
	}
	hmrm_frame sf = *f;
	set_camera(&sf, cams[0]);
	int row_begin = 0, row_end = 0;
	if (int rc = validate_frame(c, &sf, &row_begin, &row_end)) return rc;
	const long long tiles = (long long)n * ((f->screen_width + 7) / 8) * ((f->screen_height + 3) / 4);
	if (tiles > kMaxViewTiles)
		return fail(c, HMRM_ERR_INVALID, "%d views of %dx%d are %lld tiles of 8x4 pixels, more than 2^26", n,
		            f->screen_width, f->screen_height, tiles);
	if (!c->skip_ready) return fail(c, HMRM_ERR_STATE, "the height range could not be quantised; use HMRM_TRAVERSAL_BRUTE");
	RenderParams P;
	skip_params(c, f, &P);
	if (P.fx_bits < 1 || !std::isfinite(P.fx_scale))
		return fail(c, HMRM_ERR_INVALID, "grid_width %g is too small for the skip traversal; views have no FP64 fallback",
		            f->grid_width);
	return HMRM_OK;
}

// A launch slot's pieces of a batch: the view records, the schedule and (spherical) each view's tables, back to back
// from `base`; from base 0 they are only counted.
struct ViewPieces {
	ViewConst *rec;
	uint32_t *rows;
	double *sph;
	size_t bytes;
};

ViewPieces view_pieces(uintptr_t base, int n, int rows, size_t sph) {
	Carve k = {base, 0};
	ViewPieces p;
	p.rec = k.take<ViewConst>((unsigned long long)n);
	p.rows = k.take<uint32_t>((unsigned long long)rows);
	p.sph = k.take<double>(sph);
	p.bytes = k.bytes;
	return p;
}

// Enqueue n views of f (check_views has passed) on `stream` into d_out, view j at byte j * W * H * C.  The records,
// schedule and spherical tables are written into the slot's pinned staging and go to the device in one copy.
int enqueue_views(hmrm_ctx *c, const hmrm_frame *f, const hmrm_camera *cams, int n, uint8_t *d_out, cudaStream_t stream) {
	HMRM_CUDA(c, cudaSetDevice(c->device));
	const int W = f->screen_width, H = f->screen_height;
	int rc = ensure_tables(c, W, H);
	if (rc) return rc;
	int ls = 0;
	if ((rc = take_slot(c, -1, &ls)) != HMRM_OK) return rc;
	LaunchSlot &slot = c->slots[ls];

	const int ty_view = (H + 3) / 4;             // tile rows of one view
	const int rows = n * ty_view;
	const bool spherical = f->projection == HMRM_SPHERICAL;
	const size_t sph_view = spherical ? (size_t)(2 * W + 2 * H) : 0;
	const size_t need = view_pieces(0, n, rows, sph_view * (size_t)n).bytes;
	if (need > slot.view_cap) {
		if (slot.view_host) cudaFreeHost(slot.view_host);
		cudaFree(slot.d_view);
		slot.view_host = NULL;
		slot.d_view = NULL;
		slot.view_cap = 0;
		HMRM_CUDA(c, cudaMallocHost(&slot.view_host, need));
		HMRM_CUDA(c, cudaMalloc(&slot.d_view, need));
		slot.view_cap = need;
	}
	const ViewPieces h = view_pieces((uintptr_t)slot.view_host, n, rows, sph_view * (size_t)n);
	const ViewPieces d = view_pieces((uintptr_t)slot.d_view, n, rows, sph_view * (size_t)n);

	hmrm_frame sf = *f;
	set_camera(&sf, cams[0]);
	RenderParams P;
	frame_params(c, &sf, build_plane(sf), &P);
	skip_params(c, &sf, &P);

	// Per view: its record and its tables.
	for (int j = 0; j < n; ++j) {
		set_camera(&sf, cams[j]);
		const PlaneConst pc = build_plane(sf);
		ViewConst &v = h.rec[j];
		const Vec3 *src[5] = {&pc.cam, &pc.ul, &pc.pr, &pc.pd, &pc.look};
		double *dst[5] = {v.cam, v.ul, v.pr, v.pd, v.look};
		for (int i = 0; i < 5; ++i) {
			dst[i][0] = src[i]->x;
			dst[i][1] = src[i]->y;
			dst[i][2] = src[i]->z;
		}
		v.cos_ha = v.sin_ha = v.sin_va = v.cos_va = NULL;
		if (spherical) {
			fill_spherical_tables(pc, W, H, c->wtab, c->htab, &c->sph);
			std::memcpy(h.sph + (size_t)j * sph_view, c->sph.data(), sph_view * 8);
			const double *t = d.sph + (size_t)j * sph_view;
			v.cos_ha = t;
			v.sin_ha = t + W;
			v.sin_va = t + 2 * W;
			v.cos_va = t + 2 * W + H;
		}
	}
	// Per view: its tile rows costliest first (row_schedule), orders[view_order[j] * ty_view ...], of which the first
	// sky[j] march terrain and the rest look above the horizon from above the box.  The order depends on vang and not on
	// hang or position, so views with one vang share it: the views are sorted by vang once (O(n log n)) and each run of
	// equal vang gets one schedule.
	const bool ordered = f->projection != HMRM_ORTHOGRAPHIC && ty_view > 1 && !c->knobs.no_row_order;
	std::vector<int> view_order((size_t)n, -1), sky((size_t)n, ty_view);
	std::vector<int> orders, identity((size_t)ty_view);
	for (int t = 0; t < ty_view; ++t) identity[(size_t)t] = t;
	if (ordered) {
		std::vector<int> by_vang((size_t)n), order_sky;
		for (int j = 0; j < n; ++j) by_vang[(size_t)j] = j;
		std::sort(by_vang.begin(), by_vang.end(), [&](int a, int b) {
			return cams[a].vang < cams[b].vang || (cams[a].vang == cams[b].vang && a < b);
		});
		std::vector<std::pair<double, int> > cost;
		const double box_top = std::fmax(P.c0[2], P.c1[2]);
		for (int i = 0; i < n; ++i) {
			const int j = by_vang[(size_t)i];
			if (i == 0 || cams[j].vang != cams[by_vang[(size_t)i - 1]].vang) {
				set_camera(&sf, cams[j]);
				orders.resize(orders.size() + (size_t)ty_view);
				order_sky.push_back(0);
				row_schedule(build_plane(sf), H, 0, 0, 1, ty_view, orders.data() + orders.size() - (size_t)ty_view,
				             &order_sky.back(), &cost);
			}
			const int g = (int)order_sky.size() - 1;
			view_order[(size_t)j] = g;
			// (only when the camera is above the terrain: from below, rows that look up are the expensive ones)
			if (cams[j].cam_pos[2] > box_top && !c->knobs.no_batch) sky[(size_t)j] = order_sky[(size_t)g];
		}
	}
	// Global schedule, rank-major: the costliest terrain row of every view, then the second costliest of every view,
	// ...; then every view's sky rows, grabbed sky_batch tiles at a time.  (HMRM_VIEWS_VIEW_MAJOR: view by view.)
	auto row_of = [&](int j, int r) -> uint32_t {
		const int g = view_order[(size_t)j];
		const int t = g < 0 ? identity[(size_t)r] : orders[(size_t)g * (size_t)ty_view + (size_t)r];
		return ((uint32_t)j << 14) | (uint32_t)t;
	};
	size_t at = 0;
	if (c->knobs.views_view_major) {
		for (int j = 0; j < n; ++j)
			for (int r = 0; r < sky[(size_t)j]; ++r) h.rows[at++] = row_of(j, r);
	}
	else {
		for (int r = 0; r < ty_view; ++r)
			for (int j = 0; j < n; ++j)
				if (r < sky[(size_t)j]) h.rows[at++] = row_of(j, r);
	}
	if (ordered) P.batch_from_tile = (unsigned)at * (unsigned)P.tiles_x;
	for (int j = 0; j < n; ++j)
		for (int r = sky[(size_t)j]; r < ty_view; ++r) h.rows[at++] = row_of(j, r);
	HMRM_CUDA(c, cudaMemcpyAsync(slot.d_view, slot.view_host, need, cudaMemcpyHostToDevice, stream));

	P.row_begin = 0;
	P.row_end = H;
	P.cycle = 0;
	P.period = 1;
	P.tile_y_first = 0;
	P.tile_y_step = 1;
	P.tiles_y = rows;
	P.view_rows = d.rows;
	P.views = d.rec;
	P.n_views = n;
	P.view_bytes = (unsigned long long)W * (unsigned long long)H * (f->pixel_format == HMRM_PIXEL_RGB8 ? 3ULL : 4ULL);
	P.fb = (uint32_t *)d_out;                    // (each view's alignment is decided in the kernel)
	P.stats = slot.d_stats;
	P.tile_counter = slot.d_tile_counter;
	if ((rc = reset_slot(c, slot, -1, stream)) != HMRM_OK) return rc;
	const bool want_stats = (f->flags & HMRM_FLAG_STATS) != 0;
	HMRM_CUDA(c, cudaEventRecord(slot.ev_begin, stream));
	if ((rc = launch_lin<true>(c, P, want_stats, stream)) != HMRM_OK) return rc;
	HMRM_CUDA(c, cudaGetLastError());
	HMRM_CUDA(c, cudaEventRecord(slot.ev_end, stream));
	slot.used = true;
	c->launch_last = ls;
	c->last_stream = stream;
	c->last_had_stats = want_stats;
	c->last_had_step_index = false;
	c->last_had_ray_dump = false;
	c->timing_valid = true;
	c->last_w = W;
	c->last_h = H;
	return HMRM_OK;
}

} // namespace

extern "C" {

int hmrm_abi_version(void) { return HMRM_ABI_VERSION; }

int hmrm_device_count(void) {
	int n = 0;
	if (cudaGetDeviceCount(&n) != cudaSuccess) return 0;
	return n;
}

const char *hmrm_last_error(const hmrm_ctx *ctx) { return ctx ? ctx->err.c_str() : g_create_error.c_str(); }

int hmrm_create(int device, hmrm_ctx **out) {
	if (!out) return fail(NULL, HMRM_ERR_INVALID, "out is NULL");
	*out = NULL;
	int n = 0;
	cudaError_t e = cudaGetDeviceCount(&n);
	if (e != cudaSuccess || n == 0)
		return fail(NULL, HMRM_ERR_CUDA, "no CUDA device available (%s); this library has no CPU path",
		            e != cudaSuccess ? cudaGetErrorString(e) : "device count 0");
	if (device < 0 || device >= n) return fail(NULL, HMRM_ERR_INVALID, "device %d not in [0,%d)", device, n);
	HMRM_CUDA(NULL, cudaSetDevice(device));
	cudaDeviceProp prop;
	HMRM_CUDA(NULL, cudaGetDeviceProperties(&prop, device));
	if (prop.major < 10)
		return fail(NULL, HMRM_ERR_CUDA, "device %d is sm_%d%d; this library is built for sm_100a only", device,
		            prop.major, prop.minor);

	if (const char *g = std::getenv("HMRM_L2_FETCH_GRANULARITY")) {
		// experiment knob: bytes the L2 fetches from HBM per miss (32 / 64 / 128; a hint, device-wide)
		cudaDeviceSetLimit(cudaLimitMaxL2FetchGranularity, (size_t)std::atoi(g));
	}
	hmrm_ctx *c = new hmrm_ctx();
	c->device = device;
	{
		// experiment knobs: the environment is read here and nowhere else
		Knobs &k = c->knobs;
		const char *e;
		k.no_row_order = std::getenv("HMRM_NO_ROW_ORDER") != NULL;
		k.reset_kernel = std::getenv("HMRM_RESET_KERNEL") != NULL;
		// peer-frame protocol: stream memory operations when the driver has them (measured at N = 8: 0.2006 ms per 8K
		// band frame against 0.2181 ms with the one-thread kernels), HMRM_PEER_SYNC=kernels / memops forces one
		e = std::getenv("HMRM_PEER_SYNC");
		if (e && std::strcmp(e, "kernels") == 0) k.peer_memops = false;
		else if (e && std::strcmp(e, "memops") == 0) k.peer_memops = true;     // an error at first use if unavailable
		else k.peer_memops = probe_memops();
		k.no_batch = std::getenv("HMRM_NO_BATCH") != NULL;
		k.debug_sched = std::getenv("HMRM_DEBUG_SCHED") != NULL;
		k.views_view_major = std::getenv("HMRM_VIEWS_VIEW_MAJOR") != NULL;
		k.lmin_bias = (e = std::getenv("HMRM_LMIN_BIAS")) ? std::atoi(e) : 0;
		k.lstride = (e = std::getenv("HMRM_LSTRIDE")) ? std::atoi(e) : 1;
		k.lstart = (e = std::getenv("HMRM_LSTART")) ? std::atoi(e) : 6;
		k.sky_batch = (e = std::getenv("HMRM_SKY_BATCH")) ? std::atoi(e) : 8;
		if (k.sky_batch < 1) k.sky_batch = 1;
		k.cell_exit = (e = std::getenv("HMRM_CELL_EXIT")) ? (float)std::atof(e) : 8.0f;
		k.climb = (e = std::getenv("HMRM_CLIMB")) ? (float)std::atof(e) : 4.0f;
		k.zq_shrink_set = (e = std::getenv("HMRM_ZQ_RANGE_SHRINK")) != NULL;
		k.zq_shrink = e ? std::atof(e) : 1.0;
		k.peer_timeout_ns = (unsigned long long)((e = std::getenv("HMRM_PEER_TIMEOUT_MS")) ? std::atof(e) : 5000.0) * 1000000ULL;
		c->layout_wanted = HMRM_LAYOUT_DEFAULT;
		if ((e = std::getenv("HMRM_LAYOUT")) != NULL) {
			if (!std::strcmp(e, "rowmajor")) c->layout_wanted = HMRM_LAYOUT_ROWMAJOR;
			else if (!std::strcmp(e, "tile4")) c->layout_wanted = HMRM_LAYOUT_TILE4;
			else if (!std::strcmp(e, "zorder")) c->layout_wanted = HMRM_LAYOUT_ZORDER;
		}
		c->layout = c->layout_wanted;
	}
	c->d_k1_counter = NULL;
	c->num_sms = prop.multiProcessorCount;
	c->stream = NULL;
	for (int i = 0; i < kFrameRing; ++i) c->ring_stream[i] = NULL;
	c->last_stream = NULL;
	c->map_w = c->map_h = 0;
	c->d_rgb = NULL;
	c->height_bits = 8;
	c->d_color = NULL;
	c->d_surf = NULL;
	c->d_max_bits = NULL;
	c->maps_set = c->heights_set = false;
	c->lum[0] = 0.299;
	c->lum[1] = 0.587;
	c->lum[2] = 0.114;
	c->min_height = 0.0;
	c->max_height = 10.0;
	c->max_surf = c->min_surf = 0.0;
	c->d_mip = NULL;
	c->d_dil = NULL;
	c->mip_levels = 0;
	c->zq_scale = 1.0;
	c->zq_offset = HMRM_MAGIC;
	c->skip_ready = false;
	c->tab_w = c->tab_h = 0;
	c->d_wtab = c->d_htab = NULL;
	std::memset(c->slots, 0, sizeof c->slots);
	for (int i = 0; i < kFrameRing; ++i) {
		c->d_fb[i] = NULL;
		c->copy_pending[i] = false;
		c->ev_rendered[i] = c->ev_copied[i] = NULL;
	}
	c->fb_w = c->fb_h = 0;
	c->copy_stream = NULL;
	c->slot = 0;
	c->fb_format = HMRM_PIXEL_RGBA8;
	std::memset(c->d_scratch, 0, sizeof c->d_scratch);
	std::memset(c->scratch_cap, 0, sizeof c->scratch_cap);
	c->d_pixels = NULL;
	c->pixels_cap = 0;
	c->d_views = NULL;
	c->views_cap = 0;
	std::memset(c->sub, 0, sizeof c->sub);
	c->sub_next = 0;
	c->blur_n = 0;

	c->launch_next = c->launch_last = 0;
	c->last_had_stats = c->last_had_step_index = c->last_had_ray_dump = c->timing_valid = false;
	c->last_w = c->last_h = 0;
	c->last_stream = NULL;

	cudaError_t err = cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking);
	if (err == cudaSuccess) err = cudaStreamCreateWithFlags(&c->copy_stream, cudaStreamNonBlocking);
	c->ring_stream[0] = c->stream;
	for (int i = 0; i < kFrameRing && err == cudaSuccess; ++i) {
		err = cudaEventCreateWithFlags(&c->ev_rendered[i], cudaEventDisableTiming);
		if (err == cudaSuccess) err = cudaEventCreateWithFlags(&c->ev_copied[i], cudaEventDisableTiming);
		if (err == cudaSuccess && i > 0) err = cudaStreamCreateWithFlags(&c->ring_stream[i], cudaStreamNonBlocking);
	}
	for (int i = 0; i < kLaunchSlots && err == cudaSuccess; ++i) {
		err = cudaEventCreate(&c->slots[i].ev_begin);
		if (err == cudaSuccess) err = cudaEventCreate(&c->slots[i].ev_end);
		if (err == cudaSuccess) err = cudaMalloc(&c->slots[i].d_stats, sizeof(DeviceStats));
		if (err == cudaSuccess) err = cudaMalloc(&c->slots[i].d_tile_counter, 256);
	}
	for (int i = 0; i < kSubFrames && err == cudaSuccess; ++i)
		err = cudaEventCreateWithFlags(&c->sub[i].ev_read, cudaEventDisableTiming);
	if (err == cudaSuccess) err = cudaMalloc(&c->d_max_bits, 32);
	if (err == cudaSuccess) err = cudaMalloc(&c->d_k1_counter, 256);
	if (err == cudaSuccess) err = cudaMemset(c->d_k1_counter, 0, 256);
	if (err != cudaSuccess) {
		fail(NULL, HMRM_ERR_CUDA, "context setup failed: %s", cudaGetErrorString(err));
		hmrm_destroy(c);
		return HMRM_ERR_CUDA;
	}
	*out = c;
	return HMRM_OK;
}

void hmrm_destroy(hmrm_ctx *c) {
	if (!c) return;
	cudaSetDevice(c->device);
	for (int i = 0; i < kFrameRing; ++i) {
		if (c->ring_stream[i]) cudaStreamSynchronize(c->ring_stream[i]);
	}
	free_maps(c);
	cudaFree(c->d_max_bits);
	cudaFree(c->d_k1_counter);
	cudaFree(c->d_wtab);
	cudaFree(c->d_htab);

	if (c->copy_stream) cudaStreamSynchronize(c->copy_stream);
	cudaFree(c->d_pixels);
	cudaFree(c->d_views);
	for (int i = 0; i < kFrameRing; ++i) {
		cudaFree(c->d_scratch[i]);
		cudaFree(c->d_fb[i]);
		if (c->ev_rendered[i]) cudaEventDestroy(c->ev_rendered[i]);
		if (c->ev_copied[i]) cudaEventDestroy(c->ev_copied[i]);
	}
	if (c->copy_stream) cudaStreamDestroy(c->copy_stream);
	for (int i = 0; i < kSubFrames; ++i) {
		SubFrame &b = c->sub[i];
		if (b.used) cudaEventSynchronize(b.ev_read);      // a filter on a caller's stream may still read it
		cudaFree(b.d);
		cudaFree(b.acc);
		if (b.ev_read) cudaEventDestroy(b.ev_read);
	}
	for (int i = 0; i < kLaunchSlots; ++i) {
		LaunchSlot &sl = c->slots[i];
		cudaFree(sl.d_step_index);
		cudaFree(sl.d_ray_dump);
		cudaFree(sl.d_stats);
		cudaFree(sl.d_tile_counter);
		cudaFree(sl.d_sph);
		cudaFree(sl.d_row_order);
		if (sl.sph_host) cudaFreeHost(sl.sph_host);
		cudaFree(sl.d_view);
		if (sl.view_host) cudaFreeHost(sl.view_host);
		if (sl.ev_begin) cudaEventDestroy(sl.ev_begin);
		if (sl.ev_end) cudaEventDestroy(sl.ev_end);
	}
	for (int i = 0; i < kFrameRing; ++i) {
		if (c->ring_stream[i]) cudaStreamDestroy(c->ring_stream[i]);
	}
	delete c;
}

namespace {

// hmrm_set_maps* : height (RGB8, or u16 with bits 16) and colormap from host or device memory
int upload_maps(hmrm_ctx *c, const void *height, const void *color_rgba8, int32_t w, int32_t h, int bits,
                cudaMemcpyKind kind) {
	if (!height || !color_rgba8) return fail(c, HMRM_ERR_INVALID, "map pointers must not be NULL");
	int rc = alloc_maps(c, w, h);
	if (rc) return rc;
	const size_t n = (size_t)w * (size_t)h;
	HMRM_CUDA(c, cudaMemcpyAsync(c->d_rgb, height, n * (bits == 16 ? 2 : 3), kind, c->stream));
	HMRM_CUDA(c, cudaMemcpyAsync(c->d_color, color_rgba8, n * 4, kind, c->stream));
	HMRM_CUDA(c, cudaStreamSynchronize(c->stream));
	c->height_bits = bits;
	c->maps_set = true;
	return HMRM_OK;
}

} // namespace

int hmrm_set_maps(hmrm_ctx *c, const uint8_t *height_rgb8, const uint8_t *color_rgba8, int32_t w, int32_t h) {
	if (!c) return HMRM_ERR_INVALID;
	return upload_maps(c, height_rgb8, color_rgba8, w, h, 8, cudaMemcpyHostToDevice);
}

int hmrm_set_maps_device(hmrm_ctx *c, const void *d_rgb8, const void *d_rgba8, int32_t w, int32_t h) {
	if (!c) return HMRM_ERR_INVALID;
	return upload_maps(c, d_rgb8, d_rgba8, w, h, 8, cudaMemcpyDeviceToDevice);
}

int hmrm_set_maps16(hmrm_ctx *c, const uint16_t *height, const uint8_t *color_rgba8, int32_t w, int32_t h) {
	if (!c) return HMRM_ERR_INVALID;
	return upload_maps(c, height, color_rgba8, w, h, 16, cudaMemcpyHostToDevice);
}

int hmrm_set_maps16_device(hmrm_ctx *c, const void *d_height, const void *d_rgba8, int32_t w, int32_t h) {
	if (!c) return HMRM_ERR_INVALID;
	return upload_maps(c, d_height, d_rgba8, w, h, 16, cudaMemcpyDeviceToDevice);
}

int hmrm_synth_maps(hmrm_ctx *c, uint32_t log2n, uint32_t seed) {
	if (!c) return HMRM_ERR_INVALID;
	if (log2n < 4 || log2n > 15) return fail(c, HMRM_ERR_INVALID, "log2n %u outside [4,15]", log2n);
	const int32_t n = (int32_t)(1u << log2n);
	int rc = alloc_maps(c, n, n);
	if (rc) return rc;
	k_synth_maps<<<c->num_sms * 8, 256, 0, c->stream>>>(log2n, seed, c->d_rgb, c->d_color);
	HMRM_CUDA(c, cudaGetLastError());
	HMRM_CUDA(c, cudaStreamSynchronize(c->stream));
	c->height_bits = 8;
	c->maps_set = true;
	return HMRM_OK;
}

int hmrm_synth_maps16(hmrm_ctx *c, uint32_t log2n, uint32_t seed) {
	if (!c) return HMRM_ERR_INVALID;
	if (log2n < 4 || log2n > 15) return fail(c, HMRM_ERR_INVALID, "log2n %u outside [4,15]", log2n);
	const int32_t n = (int32_t)(1u << log2n);
	int rc = alloc_maps(c, n, n);
	if (rc) return rc;
	k_synth_maps16<<<c->num_sms * 8, 256, 0, c->stream>>>(log2n, seed, (uint16_t *)c->d_rgb, c->d_color);
	HMRM_CUDA(c, cudaGetLastError());
	HMRM_CUDA(c, cudaStreamSynchronize(c->stream));
	c->height_bits = 16;
	c->maps_set = true;
	return HMRM_OK;
}

int hmrm_get_maps(hmrm_ctx *c, uint8_t *height_rgb8, uint8_t *color_rgba8) {
	if (!c) return HMRM_ERR_INVALID;
	if (!c->maps_set) return fail(c, HMRM_ERR_STATE, "maps not set");
	if (height_rgb8 && c->height_bits == 16)
		return fail(c, HMRM_ERR_STATE, "the height map is 16-bit (hmrm_set_maps16): it has no RGB8 plane; pass NULL");
	HMRM_CUDA(c, cudaSetDevice(c->device));
	const size_t n = (size_t)c->map_w * (size_t)c->map_h;
	if (height_rgb8) HMRM_CUDA(c, cudaMemcpyAsync(height_rgb8, c->d_rgb, n * 3, cudaMemcpyDeviceToHost, c->stream));
	if (color_rgba8) HMRM_CUDA(c, cudaMemcpyAsync(color_rgba8, c->d_color, n * 4, cudaMemcpyDeviceToHost, c->stream));
	HMRM_CUDA(c, cudaStreamSynchronize(c->stream));
	return HMRM_OK;
}

int hmrm_update_heightmap(hmrm_ctx *c, const double lum[3], double min_height, double max_height) {
	if (!c) return HMRM_ERR_INVALID;
	if (!c->maps_set) return fail(c, HMRM_ERR_STATE, "hmrm_set_maps has not been called");
	if (!lum || !finite3(lum) || !std::isfinite(min_height) || !std::isfinite(max_height))
		return fail(c, HMRM_ERR_INVALID, "lum, min_height and max_height must be finite");
	HMRM_CUDA(c, cudaSetDevice(c->device));
	if (int rc = drain(c)) return rc;
	PrepassParams q;
	q.lum_r = lum[0];
	q.lum_g = lum[1];
	q.lum_b = lum[2];
	q.min_height = min_height;
	q.span = max_height - min_height;
	const long long n = (long long)c->map_w * c->map_h;
	// (1) range of surf from a sample of the rows (at most ~1 M cells): only the quantiser's resolution depends on it
	const unsigned long long init_bits[3] = {0ULL, ~0ULL, 0ULL};
	HMRM_CUDA(c, cudaMemcpyAsync(c->d_max_bits, init_bits, sizeof init_bits, cudaMemcpyHostToDevice, c->stream));
	int row_stride = (int)((n + (1LL << 20) - 1) / (1LL << 20));
	if (row_stride < 1) row_stride = 1;
	// the same rows for either input, so equivalent 8- and 16-bit maps get the same quantiser
	const bool grey16 = c->height_bits == 16;
	const uint16_t *h16 = (const uint16_t *)c->d_rgb;
	if (grey16)
		k1_range<<<c->num_sms * 8, 256, 0, c->stream>>>(Grey16Cells{h16}, c->map_w, c->map_h, row_stride, q,
		                                                 c->d_max_bits, c->d_max_bits + 1);
	else
		k1_range<<<c->num_sms * 8, 256, 0, c->stream>>>(Rgb8Cells{c->d_rgb}, c->map_w, c->map_h, row_stride, q,
		                                                 c->d_max_bits, c->d_max_bits + 1);
	HMRM_CUDA(c, cudaGetLastError());
	unsigned long long bits[3] = {0ULL, 0ULL, 0ULL};
	HMRM_CUDA(c, cudaMemcpyAsync(bits, c->d_max_bits, 16, cudaMemcpyDeviceToHost, c->stream));
	HMRM_CUDA(c, cudaStreamSynchronize(c->stream));
	c->max_surf = from_ordered_bits(bits[0]);
	c->min_surf = from_ordered_bits(bits[1]);

	// Zq: sampled surf range [min_surf, max_surf] -> [2000, 63000] of the 16-bit scale; values outside clamp (and tie)
	if (c->knobs.zq_shrink_set) {
		// test hook: pretend the sampled range was (much) too narrow, so that most values clamp and tie
		const double f = c->knobs.zq_shrink, mid = 0.5 * (c->max_surf + c->min_surf), half = 0.5 * (c->max_surf - c->min_surf);
		c->min_surf = mid - f * half;
		c->max_surf = mid + f * half;
	}
	const double range = c->max_surf - c->min_surf;
	c->zq_scale = (range > 0.0 && std::isfinite(range) && std::isfinite(61000.0 / range)) ? 61000.0 / range : 1.0;
	c->zq_offset = HMRM_MAGIC + (2000.0 - c->min_surf * c->zq_scale);

	// layout of the pyramid the traversal reads (pyramid_layout.cuh); the buffer was sized for any of them
	c->layout = c->layout_wanted;
	layout_pyramid(c, c->layout);

	// (2) fused build of surf, level 0 and the plain max-mip levels 1, 2; (3) plain levels >= 3 in one launch;
	// (4) the 3x3 dilation of every level >= 1, written in the traversal's layout, in one launch
	{
		uint16_t *plain1 = c->mip_levels > 1 ? c->d_dil : NULL;
		uint16_t *plain2 = c->mip_levels > 2 ? c->d_dil + c->plain_offset[2] : NULL;
		if (plain1 && grey16) {
			k1_build16<<<c->num_sms * 8, 256, 0, c->stream>>>(h16, c->map_w, c->map_h, q, c->zq_scale, c->zq_offset,
			                                                   c->d_surf, c->d_mip, c->layout,
			                                                   pyr_level_pitch(c->layout, c->map_w), plain1, c->mip_w[1],
			                                                   plain2, c->mip_levels > 2 ? c->mip_w[2] : 0);
		}
		else if (plain1) {
			k1_build<<<c->num_sms * 8, 256, 0, c->stream>>>(c->d_rgb, c->map_w, c->map_h, q, c->zq_scale, c->zq_offset,
			                                                 c->d_surf, c->d_mip, c->layout,
			                                                 pyr_level_pitch(c->layout, c->map_w), plain1, c->mip_w[1], plain2,
			                                                 c->mip_levels > 2 ? c->mip_w[2] : 0);
		}
		else {
			// 1x1 map: no pyramid
			if (grey16) k1_prepass<<<1, 32, 0, c->stream>>>(Grey16Cells{h16}, n, q, c->d_surf, NULL, NULL, NULL);
			else k1_prepass<<<1, 32, 0, c->stream>>>(Rgb8Cells{c->d_rgb}, n, q, c->d_surf, NULL, NULL, NULL);
			k1_quantise<<<1, 32, 0, c->stream>>>(c->d_surf, n, c->zq_scale, c->zq_offset, c->d_mip,
			                                     (unsigned int *)(c->d_max_bits + 2));
		}
		HMRM_CUDA(c, cudaGetLastError());
	}
	if (c->mip_levels > 3) {
		MipJob job;
		std::memset(&job, 0, sizeof job);
		job.n_levels = c->mip_levels;
		for (int l = 0; l < c->mip_levels; ++l) {
			job.w[l] = c->mip_w[l];
			job.h[l] = c->mip_h[l];
			job.plain_off[l] = (unsigned)c->plain_offset[l];
		}
		const int regions = ((c->mip_w[2] + 127) / 128) * ((c->mip_h[2] + 127) / 128);
		k1_mip_upper<<<regions, 256, 0, c->stream>>>(c->d_dil, job, c->d_k1_counter);
		HMRM_CUDA(c, cudaGetLastError());
	}
	if (c->mip_levels > 1) {
		DilateJob job;
		std::memset(&job, 0, sizeof job);
		job.n_levels = c->mip_levels;
		job.layout = c->layout;
		unsigned long long items = 0;
		job.first_item[0] = job.first_item[1] = 0;
		for (int l = 0; l < c->mip_levels; ++l) {
			job.w[l] = c->mip_w[l];
			job.h[l] = c->mip_h[l];
			job.plain_off[l] = (unsigned)c->plain_offset[l];
			job.dst_off[l] = (unsigned)c->mip_offset[l];
			job.dst_pitch[l] = pyr_level_pitch(c->layout, c->mip_w[l]);
			if (l >= 1) {
				job.first_item[l] = items;
				items += (unsigned long long)((c->mip_w[l] + 3) / 4) * (unsigned long long)((c->mip_h[l] + 3) / 4);
			}
			job.first_item[l + 1] = items;
		}
		unsigned long long want = (items + 255) / 256;
		const unsigned long long cap_blocks = (unsigned long long)c->num_sms * 16ULL;
		const int blocks = (int)std::max(1ULL, std::min(want, cap_blocks));
		k1_dilate_levels<<<blocks, 256, 0, c->stream>>>(c->d_dil, c->d_mip, job);
		HMRM_CUDA(c, cudaGetLastError());
	}
	HMRM_CUDA(c, cudaStreamSynchronize(c->stream));
	c->skip_ready = std::isfinite(c->zq_offset) && std::isfinite(c->zq_scale) && c->zq_scale > 0.0;
	c->lum[0] = lum[0];
	c->lum[1] = lum[1];
	c->lum[2] = lum[2];
	c->min_height = min_height;
	c->max_height = max_height;
	c->heights_set = true;
	return HMRM_OK;
}

int hmrm_get_heights(hmrm_ctx *c, double *heights) {
	if (!c) return HMRM_ERR_INVALID;
	if (!heights) return fail(c, HMRM_ERR_INVALID, "heights is NULL");
	if (!c->heights_set) return fail(c, HMRM_ERR_STATE, "hmrm_update_heightmap has not been called");
	HMRM_CUDA(c, cudaSetDevice(c->device));
	const long long n = (long long)c->map_w * c->map_h;
	double *d_tmp = NULL;
	HMRM_CUDA(c, cudaMalloc(&d_tmp, (size_t)n * 8));
	PrepassParams q;
	q.lum_r = c->lum[0];
	q.lum_g = c->lum[1];
	q.lum_b = c->lum[2];
	q.min_height = c->min_height;
	q.span = c->max_height - c->min_height;
	if (c->height_bits == 16)
		k1_prepass<<<c->num_sms * 8, 256, 0, c->stream>>>(Grey16Cells{(const uint16_t *)c->d_rgb}, n, q, NULL, d_tmp, NULL, NULL);
	else
		k1_prepass<<<c->num_sms * 8, 256, 0, c->stream>>>(Rgb8Cells{c->d_rgb}, n, q, NULL, d_tmp, NULL, NULL);
	cudaError_t e = cudaGetLastError();
	if (e == cudaSuccess) e = cudaMemcpyAsync(heights, d_tmp, (size_t)n * 8, cudaMemcpyDeviceToHost, c->stream);
	if (e == cudaSuccess) e = cudaStreamSynchronize(c->stream);
	cudaFree(d_tmp);
	if (e != cudaSuccess) return fail(c, HMRM_ERR_CUDA, "hmrm_get_heights: %s", cudaGetErrorString(e));
	return HMRM_OK;
}

void hmrm_frame_defaults(hmrm_frame *f) {
	if (!f) return;
	std::memset(f, 0, sizeof *f);
	f->projection = HMRM_PERSPECTIVE;     // main/hmap.cpp:107
	f->screen_width = 800;                // :31
	f->screen_height = 600;               // :32
	f->precision = HMRM_FP64_EXACT;
	f->cam_pos[0] = -5.0;                 // :75
	f->cam_pos[1] = 5.0;
	f->cam_pos[2] = 0.0;
	f->hang = -M_PI / 4.0;                // :80
	f->vang = M_PI / 2.0;                 // :85
	f->hfov = M_PI / 2.0;                 // :35
	f->grid_width = 0.05;                 // :65
	f->step_dist = 5.0 * 0.05;            // :68
	f->ortho_width = 2.0 * 0.05;          // :98
	f->cycle = 0;
	f->cycle_period = 1;                  // the reference's default is 47 (:71); 1 renders a whole frame
	f->traversal = HMRM_TRAVERSAL_AUTO;
}

int hmrm_render_device(hmrm_ctx *c, const hmrm_frame *f, void *d_rgba_out, void *stream) {
	if (!c) return HMRM_ERR_INVALID;
	if (!d_rgba_out) return fail(c, HMRM_ERR_INVALID, "d_rgba_out is NULL");
	if (!f) return fail(c, HMRM_ERR_INVALID, "frame is NULL");
	return enqueue_frame(c, f, (uint32_t *)d_rgba_out, stream ? (cudaStream_t)stream : c->stream);
}

int hmrm_render_views_device(hmrm_ctx *c, const hmrm_frame *f, const hmrm_camera *cams, int32_t n, void *d_out,
                             void *stream) {
	if (!c) return HMRM_ERR_INVALID;
	if (int rc = check_views(c, f, cams, n, d_out)) return rc;
	return enqueue_views(c, f, cams, n, (uint8_t *)d_out, stream ? (cudaStream_t)stream : c->stream);
}

int hmrm_render_views(hmrm_ctx *c, const hmrm_frame *f, const hmrm_camera *cams, int32_t n, uint8_t *out) {
	if (!c) return HMRM_ERR_INVALID;
	if (int rc = check_views(c, f, cams, n, out)) return rc;
	HMRM_CUDA(c, cudaSetDevice(c->device));
	const size_t bytes = (size_t)n * (size_t)f->screen_width * (size_t)f->screen_height *
	                     (f->pixel_format == HMRM_PIXEL_RGB8 ? 3 : 4);
	// the buffer is idle: the call that used it last synchronised before it returned
	if (int rc = grow(c, &c->d_views, &c->views_cap, bytes)) return rc;
	if (int rc = enqueue_views(c, f, cams, n, c->d_views, c->stream)) return rc;
	HMRM_CUDA(c, cudaMemcpyAsync(out, c->d_views, bytes, cudaMemcpyDefault, c->stream));
	HMRM_CUDA(c, cudaStreamSynchronize(c->stream));
	return HMRM_OK;
}

int hmrm_render_async(hmrm_ctx *c, const hmrm_frame *f, uint8_t *rgba_out) {
	if (!c) return HMRM_ERR_INVALID;
	if (!f) return fail(c, HMRM_ERR_INVALID, "frame is NULL");
	if (!rgba_out) return fail(c, HMRM_ERR_INVALID, "rgba_out is NULL");
	if (int rc = check_supersample(c, f)) return rc;
	if (f->screen_width < 2 || f->screen_height < 2 || f->screen_width > 65536 || f->screen_height > 65536)
		return fail(c, HMRM_ERR_INVALID, "resolution %dx%d outside [2,65536]", f->screen_width, f->screen_height);
	HMRM_CUDA(c, cudaSetDevice(c->device));
	if (f->pixel_format != HMRM_PIXEL_RGBA8 && f->pixel_format != HMRM_PIXEL_RGB8)
		return fail(c, HMRM_ERR_INVALID, "unknown pixel_format %d", (int)f->pixel_format);
	Output o = {Output::RAW, rgba_out};
	o.frame = f;
	return enqueue_ring(c, f, o);
}

int hmrm_wait_pending(hmrm_ctx *c, int max_pending) {
	if (!c) return HMRM_ERR_INVALID;
	HMRM_CUDA(c, cudaSetDevice(c->device));
	if (max_pending >= 1) {
		// let the max_pending most recent frames stay in flight; the ones before them must be on the host
		for (int age = kFrameRing - 1; age >= max_pending; --age) {
			const int older = (c->slot + kFrameRing - age) % kFrameRing;
			if (c->copy_pending[older]) {
				HMRM_CUDA(c, cudaEventSynchronize(c->ev_copied[older]));
				c->copy_pending[older] = false;
			}
		}
		return HMRM_OK;
	}
	for (int i = 0; i < kFrameRing; ++i) HMRM_CUDA(c, cudaStreamSynchronize(c->ring_stream[i]));
	HMRM_CUDA(c, cudaStreamSynchronize(c->copy_stream));
	for (int i = 0; i < kFrameRing; ++i) c->copy_pending[i] = false;
	return HMRM_OK;
}

int hmrm_wait(hmrm_ctx *c) { return hmrm_wait_pending(c, 0); }

int hmrm_render(hmrm_ctx *c, const hmrm_frame *f, uint8_t *rgba_out) {
	int rc = hmrm_render_async(c, f, rgba_out);
	if (rc) return rc;
	return hmrm_wait(c);
}

size_t hmrm_png_bound(int32_t width, int32_t height, int32_t channels) {
	PngShape s;
	if (!png_shape(width, height, channels, &s)) return 0;
	return (size_t)png_bound(s);
}

int hmrm_render_png_async(hmrm_ctx *c, const hmrm_frame *f, uint8_t *png_out, size_t capacity, uint64_t *png_bytes) {
	if (!c) return HMRM_ERR_INVALID;
	if (int rc = check_encoded_frame(c, f, "PNG")) return rc;
	PngShape s{};
	png_shape(f->screen_width, f->screen_height, f->pixel_format == HMRM_PIXEL_RGB8 ? 3 : 4, &s);
	Output o = {Output::PNG};
	if (int rc = file_outputs(c, "png", png_bound(s), png_out, capacity, png_bytes, &o.dst, &o.size)) return rc;
	o.scratch = png_pieces(s, NULL).bytes;
	return enqueue_ring(c, f, o);
}

int hmrm_encode_png(hmrm_ctx *c, const uint8_t *pixels, int32_t width, int32_t height, int32_t channels,
                    uint8_t *png_out, size_t capacity, uint64_t *png_bytes) {
	if (!c) return HMRM_ERR_INVALID;
	if (!pixels) return fail(c, HMRM_ERR_INVALID, "pixels is NULL");
	PngShape s;
	if (!png_shape(width, height, channels, &s))
		return fail(c, HMRM_ERR_INVALID, "image %dx%dx%d: need 1 <= width, height <= 65536 and 3 or 4 channels", width,
		            height, channels);
	Output o = {Output::PNG};
	if (int rc = file_outputs(c, "png", png_bound(s), png_out, capacity, png_bytes, &o.dst, &o.size)) return rc;
	o.scratch = png_pieces(s, NULL).bytes;
	return encode_staged(c, o, pixels, width, height, channels);
}

size_t hmrm_jpeg_bound(int32_t width, int32_t height, int32_t chroma) {
	JpegShape s;
	if ((chroma != HMRM_JPEG_420 && chroma != HMRM_JPEG_444) || !jpeg_shape(width, height, chroma == HMRM_JPEG_420, &s))
		return 0;
	return (size_t)jpeg_bound(s);
}

int hmrm_render_jpeg_async(hmrm_ctx *c, const hmrm_frame *f, int32_t quality, int32_t chroma, uint8_t *jpeg_out,
                           size_t capacity, uint64_t *jpeg_bytes) {
	if (!c) return HMRM_ERR_INVALID;
	if (int rc = check_encoded_frame(c, f, "JPEG")) return rc;
	if (int rc = jpeg_params(c, quality, chroma)) return rc;
	JpegShape s;
	if (!jpeg_shape(f->screen_width, f->screen_height, chroma == HMRM_JPEG_420, &s))
		return fail(c, HMRM_ERR_INVALID, "resolution %dx%d: a JPEG frame is at most 65535 pixels per axis",
		            f->screen_width, f->screen_height);
	Output o = {Output::JPEG};
	if (int rc = file_outputs(c, "jpeg", jpeg_bound(s), jpeg_out, capacity, jpeg_bytes, &o.dst, &o.size)) return rc;
	o.scratch = jpeg_pieces(s, NULL).bytes;
	o.quality = quality;
	o.chroma = chroma;
	return enqueue_ring(c, f, o);
}

int hmrm_encode_jpeg(hmrm_ctx *c, const uint8_t *pixels, int32_t width, int32_t height, int32_t channels,
                     int32_t quality, int32_t chroma, uint8_t *jpeg_out, size_t capacity, uint64_t *jpeg_bytes) {
	if (!c) return HMRM_ERR_INVALID;
	if (!pixels) return fail(c, HMRM_ERR_INVALID, "pixels is NULL");
	if (int rc = jpeg_params(c, quality, chroma)) return rc;
	JpegShape s;
	if (!jpeg_shape(width, height, chroma == HMRM_JPEG_420, &s) || (channels != 3 && channels != 4))
		return fail(c, HMRM_ERR_INVALID, "image %dx%dx%d: need 1 <= width, height <= 65535 and 3 or 4 channels", width,
		            height, channels);
	Output o = {Output::JPEG};
	if (int rc = file_outputs(c, "jpeg", jpeg_bound(s), jpeg_out, capacity, jpeg_bytes, &o.dst, &o.size)) return rc;
	o.scratch = jpeg_pieces(s, NULL).bytes;
	o.quality = quality;
	o.chroma = chroma;
	return encode_staged(c, o, pixels, width, height, channels);
}

size_t hmrm_yuv420_bytes(int32_t width, int32_t height) { return (size_t)yuv420_bytes(width, height); }

int hmrm_render_yuv420_async(hmrm_ctx *c, const hmrm_frame *f, int32_t matrix, uint8_t *out, size_t capacity) {
	if (!c) return HMRM_ERR_INVALID;
	if (int rc = check_encoded_frame(c, f, "YUV")) return rc;
	if (int rc = yuv_output(c, f->screen_width, f->screen_height, matrix, out, capacity)) return rc;
	Output o = {Output::YUV, out};
	o.scratch = (size_t)yuv420_bytes(f->screen_width, f->screen_height);
	o.matrix = matrix;
	return enqueue_ring(c, f, o);
}

int hmrm_convert_yuv420(hmrm_ctx *c, const uint8_t *pixels, int32_t width, int32_t height, int32_t channels,
                        int32_t matrix, uint8_t *out, size_t capacity) {
	if (!c) return HMRM_ERR_INVALID;
	if (!pixels) return fail(c, HMRM_ERR_INVALID, "pixels is NULL");
	if (yuv420_bytes(width, height) == 0 || (channels != 3 && channels != 4))
		return fail(c, HMRM_ERR_INVALID, "image %dx%dx%d: need 1 <= width, height <= 65536 and 3 or 4 channels", width,
		            height, channels);
	if (int rc = yuv_output(c, width, height, matrix, out, capacity)) return rc;
	Output o = {Output::YUV, out};
	o.scratch = (size_t)yuv420_bytes(width, height);
	o.matrix = matrix;
	return encode_staged(c, o, pixels, width, height, channels);
}

int hmrm_get_stats(hmrm_ctx *c, hmrm_stats *out) {
	if (!c) return HMRM_ERR_INVALID;
	if (!out) return fail(c, HMRM_ERR_INVALID, "out is NULL");
	HMRM_CUDA(c, cudaSetDevice(c->device));
	HMRM_CUDA(c, cudaStreamSynchronize(c->last_stream ? c->last_stream : c->stream));
	std::memset(out, 0, sizeof *out);
	DeviceStats ds;
	HMRM_CUDA(c, cudaMemcpy(&ds, c->slots[c->launch_last].d_stats, sizeof ds, cudaMemcpyDeviceToHost));
	if (c->last_had_stats) {
		out->rays = (int64_t)ds.rays;
		out->box_hits = (int64_t)ds.box_hits;
		out->surf_hits = (int64_t)ds.surf_hits;
		out->steps = (int64_t)ds.steps;
		out->fetches = (int64_t)ds.fetches;
		out->max_steps = (int64_t)ds.max_steps;
	}
	out->status = (int32_t)ds.status;
	if (c->timing_valid) {
		float ms = 0.f;
		if (cudaEventElapsedTime(&ms, c->slots[c->launch_last].ev_begin, c->slots[c->launch_last].ev_end) == cudaSuccess)
			out->kernel_ms = ms;
	}
	return HMRM_OK;
}

int hmrm_get_debug_counters(hmrm_ctx *c, int64_t out[12]) {
	if (!c || !out) return HMRM_ERR_INVALID;
	HMRM_CUDA(c, cudaSetDevice(c->device));
	HMRM_CUDA(c, cudaStreamSynchronize(c->last_stream ? c->last_stream : c->stream));
	DeviceStats ds;
	HMRM_CUDA(c, cudaMemcpy(&ds, c->slots[c->launch_last].d_stats, sizeof ds, cudaMemcpyDeviceToHost));
	for (int i = 0; i < 12; ++i) out[i] = (int64_t)ds.dbg[i];
	return HMRM_OK;
}

int hmrm_get_step_index(hmrm_ctx *c, int32_t *step_index) {
	if (!c) return HMRM_ERR_INVALID;
	if (!step_index) return fail(c, HMRM_ERR_INVALID, "step_index is NULL");
	if (!c->last_had_step_index) return fail(c, HMRM_ERR_STATE, "last render did not set HMRM_FLAG_STEP_INDEX");
	HMRM_CUDA(c, cudaSetDevice(c->device));
	HMRM_CUDA(c, cudaStreamSynchronize(c->last_stream ? c->last_stream : c->stream));
	HMRM_CUDA(c, cudaMemcpy(step_index, c->slots[c->launch_last].d_step_index, (size_t)c->last_w * (size_t)c->last_h * 4,
	                        cudaMemcpyDeviceToHost));
	return HMRM_OK;
}

int hmrm_get_ray_dump(hmrm_ctx *c, double *out) {
	if (!c) return HMRM_ERR_INVALID;
	if (!out) return fail(c, HMRM_ERR_INVALID, "out is NULL");
	if (!c->last_had_ray_dump) return fail(c, HMRM_ERR_STATE, "last render did not set HMRM_FLAG_RAY_DUMP");
	HMRM_CUDA(c, cudaSetDevice(c->device));
	HMRM_CUDA(c, cudaStreamSynchronize(c->last_stream ? c->last_stream : c->stream));
	HMRM_CUDA(c, cudaMemcpy(out, c->slots[c->launch_last].d_ray_dump, (size_t)c->last_w * (size_t)c->last_h * 80,
	                        cudaMemcpyDeviceToHost));
	return HMRM_OK;
}

int hmrm_set_layout(hmrm_ctx *c, int layout) {
	if (!c) return HMRM_ERR_INVALID;
	if (layout != HMRM_LAYOUT_ROWMAJOR && layout != HMRM_LAYOUT_TILE4 && layout != HMRM_LAYOUT_ZORDER)
		return fail(c, HMRM_ERR_INVALID, "unknown layout %d", layout);
	HMRM_CUDA(c, cudaSetDevice(c->device));
	if (int rc = drain(c)) return rc;
	if (layout != c->layout) c->heights_set = false;      // the pyramid must be rebuilt: hmrm_update_heightmap
	c->layout_wanted = layout;
	return HMRM_OK;
}

int hmrm_get_layout(hmrm_ctx *c) { return c ? c->layout_wanted : -1; }

int hmrm_set_motion_blur(hmrm_ctx *c, const hmrm_camera *cams, int32_t n) {
	if (!c) return HMRM_ERR_INVALID;
	if (n < 0 || n > kBlurMax) return fail(c, HMRM_ERR_INVALID, "motion blur of %d sub-frames outside [0,%d]", n, kBlurMax);
	if (n > 0 && !cams) return fail(c, HMRM_ERR_INVALID, "cams is NULL");
	// frames already enqueued keep the cameras they were enqueued with: they are copied into each frame's launches
	if (n > 0) std::memcpy(c->blur_cams, cams, (size_t)n * sizeof(hmrm_camera));
	c->blur_n = n;
	return HMRM_OK;
}

int hmrm_debug_aabb(hmrm_ctx *c, int32_t n, const double *rays, const double *boxes, double *out) {
	if (!c) return HMRM_ERR_INVALID;
	if (n < 1 || !rays || !boxes || !out) return fail(c, HMRM_ERR_INVALID, "hmrm_debug_aabb: bad arguments");
	HMRM_CUDA(c, cudaSetDevice(c->device));
	double *d = NULL;
	HMRM_CUDA(c, cudaMalloc(&d, (size_t)n * 17 * sizeof(double)));
	cudaError_t e = cudaMemcpy(d, rays, (size_t)n * 6 * sizeof(double), cudaMemcpyHostToDevice);
	if (e == cudaSuccess) e = cudaMemcpy(d + (size_t)n * 6, boxes, (size_t)n * 6 * sizeof(double), cudaMemcpyHostToDevice);
	if (e == cudaSuccess) {
		k_debug_aabb<<<(n + 127) / 128, 128, 0, c->stream>>>(n, d, d + (size_t)n * 6, d + (size_t)n * 12);
		e = cudaGetLastError();
	}
	if (e == cudaSuccess) e = cudaStreamSynchronize(c->stream);
	if (e == cudaSuccess) e = cudaMemcpy(out, d + (size_t)n * 12, (size_t)n * 5 * sizeof(double), cudaMemcpyDeviceToHost);
	cudaFree(d);
	if (e != cudaSuccess) return fail(c, HMRM_ERR_CUDA, "hmrm_debug_aabb: %s", cudaGetErrorString(e));
	return HMRM_OK;
}

double hmrm_deg2rad(double degrees) { return deg2rad(degrees); }

void hmrm_camera_basis(double hang, double vang, double look[3], double up[3]) {
	Vec3 l, u;
	camera_basis(hang, vang, &l, &u);
	look[0] = l.x; look[1] = l.y; look[2] = l.z;
	up[0] = u.x; up[1] = u.y; up[2] = u.z;
}

int hmrm_get_ray(const hmrm_frame *f, double w, double h, double pos[3], double dir[3]) {
	if (!f || !pos || !dir) return HMRM_ERR_INVALID;
	if (f->projection < HMRM_PERSPECTIVE || f->projection > HMRM_ORTHOGRAPHIC) return HMRM_ERR_INVALID;
	const PlaneConst pc = build_plane(*f);
	Vec3 p, d;
	plane_ray(pc, w, h, &p, &d);
	pos[0] = p.x; pos[1] = p.y; pos[2] = p.z;
	dir[0] = d.x; dir[1] = d.y; dir[2] = d.z;
	return HMRM_OK;
}

int hmrm_host_alloc(void **ptr, size_t bytes) {
	if (!ptr) return HMRM_ERR_INVALID;
	*ptr = NULL;
	cudaError_t e = cudaMallocHost(ptr, bytes);
	if (e != cudaSuccess) return fail(NULL, HMRM_ERR_CUDA, "cudaMallocHost(%zu) failed: %s", bytes, cudaGetErrorString(e));
	return HMRM_OK;
}

int hmrm_host_alloc_flags(void **ptr, size_t bytes, uint32_t flags) {
	if (!ptr || (flags & ~(uint32_t)HMRM_HOST_WRITE_COMBINED)) return HMRM_ERR_INVALID;
	*ptr = NULL;
	const unsigned cf = cudaHostAllocPortable | ((flags & HMRM_HOST_WRITE_COMBINED) ? cudaHostAllocWriteCombined : 0u);
	cudaError_t e = cudaHostAlloc(ptr, bytes, cf);
	if (e != cudaSuccess) return fail(NULL, HMRM_ERR_CUDA, "cudaHostAlloc(%zu, %u) failed: %s", bytes, cf, cudaGetErrorString(e));
	return HMRM_OK;
}

void hmrm_host_free(void *ptr) {
	if (ptr) cudaFreeHost(ptr);
}

int hmrm_host_register(void *ptr, size_t bytes) {
	if (!ptr || bytes == 0) return HMRM_ERR_INVALID;
	cudaError_t e = cudaHostRegister(ptr, bytes, cudaHostRegisterPortable);
	if (e != cudaSuccess) return fail(NULL, HMRM_ERR_CUDA, "cudaHostRegister(%zu) failed: %s", bytes, cudaGetErrorString(e));
	return HMRM_OK;
}

int hmrm_host_unregister(void *ptr) {
	if (!ptr) return HMRM_ERR_INVALID;
	cudaError_t e = cudaHostUnregister(ptr);
	if (e != cudaSuccess) return fail(NULL, HMRM_ERR_CUDA, "cudaHostUnregister failed: %s", cudaGetErrorString(e));
	return HMRM_OK;
}

int hmrm_device_alloc(hmrm_ctx *c, size_t bytes, void **dptr) {
	if (!c || !dptr || bytes == 0) return c ? fail(c, HMRM_ERR_INVALID, "hmrm_device_alloc: bad arguments") : HMRM_ERR_INVALID;
	*dptr = NULL;
	HMRM_CUDA(c, cudaSetDevice(c->device));
	HMRM_CUDA(c, cudaMalloc(dptr, bytes));
	HMRM_CUDA(c, cudaMemset(*dptr, 0, bytes));
	HMRM_CUDA(c, cudaDeviceSynchronize());
	return HMRM_OK;
}

int hmrm_device_free(hmrm_ctx *c, void *dptr) {
	if (!c) return HMRM_ERR_INVALID;
	HMRM_CUDA(c, cudaSetDevice(c->device));
	if (int rc = drain(c)) return rc;
	if (dptr) HMRM_CUDA(c, cudaFree(dptr));
	return HMRM_OK;
}

int hmrm_ipc_export(hmrm_ctx *c, void *dptr, uint8_t handle[HMRM_IPC_HANDLE_BYTES]) {
	if (!c || !dptr || !handle) return c ? fail(c, HMRM_ERR_INVALID, "hmrm_ipc_export: bad arguments") : HMRM_ERR_INVALID;
	static_assert(sizeof(cudaIpcMemHandle_t) == HMRM_IPC_HANDLE_BYTES, "CUDA IPC handle size");
	HMRM_CUDA(c, cudaSetDevice(c->device));
	cudaIpcMemHandle_t h;
	HMRM_CUDA(c, cudaIpcGetMemHandle(&h, dptr));
	std::memcpy(handle, &h, sizeof h);
	return HMRM_OK;
}

int hmrm_ipc_open(hmrm_ctx *c, const uint8_t handle[HMRM_IPC_HANDLE_BYTES], void **dptr) {
	if (!c || !dptr || !handle) return c ? fail(c, HMRM_ERR_INVALID, "hmrm_ipc_open: bad arguments") : HMRM_ERR_INVALID;
	*dptr = NULL;
	HMRM_CUDA(c, cudaSetDevice(c->device));
	cudaIpcMemHandle_t h;
	std::memcpy(&h, handle, sizeof h);
	// maps the exporting device's memory into this process and enables peer access to it (NVLink / NVSwitch)
	HMRM_CUDA(c, cudaIpcOpenMemHandle(dptr, h, cudaIpcMemLazyEnablePeerAccess));
	return HMRM_OK;
}

int hmrm_render_peer(hmrm_ctx *c, const hmrm_frame *f, void *d_frame, void *d_ctrl, uint32_t use, void *stream) {
	if (!c) return HMRM_ERR_INVALID;
	if (!d_frame || !d_ctrl || use == 0u) return fail(c, HMRM_ERR_INVALID, "hmrm_render_peer: bad arguments");
	if (f && (supersample_of(f) != 1 || c->blur_n > 0))
		return fail(c, HMRM_ERR_INVALID, "peer frames are band-split: no supersampling or motion blur");
	HMRM_CUDA(c, cudaSetDevice(c->device));
	cudaStream_t s = stream ? (cudaStream_t)stream : c->stream;
	PeerCtrl *ctrl = (PeerCtrl *)d_ctrl;
	// the buffer may be overwritten once the root has read its previous use
	int rc = peer_wait_word(c, &ctrl->released, use - 1u, &ctrl->error, s);
	if (rc) return rc;
	rc = enqueue_render(c, f, (uint32_t *)d_frame, s, true);
	if (rc) return rc;
	return peer_arrive(c, ctrl, f, use, s);
}

int hmrm_render_peer_staged(hmrm_ctx *c, const hmrm_frame *f, void *d_stage, void *d_frame, void *d_ctrl, uint32_t use,
                            void *stream) {
	if (!c) return HMRM_ERR_INVALID;
	if (!d_stage || !d_frame || !d_ctrl || use == 0u) return fail(c, HMRM_ERR_INVALID, "hmrm_render_peer_staged: bad arguments");
	if (f && (supersample_of(f) != 1 || c->blur_n > 0))
		return fail(c, HMRM_ERR_INVALID, "peer frames are band-split: no supersampling or motion blur");
	HMRM_CUDA(c, cudaSetDevice(c->device));
	cudaStream_t s = stream ? (cudaStream_t)stream : c->stream;
	PeerCtrl *ctrl = (PeerCtrl *)d_ctrl;
	// render into this device's own staging frame (ordinary stores), ...
	int rc = enqueue_render(c, f, (uint32_t *)d_stage, s, true);
	if (rc) return rc;
	// ... then, once the root has read the previous use of the shared buffer, push this rank's tile rows over NVLink
	// with the copy engine: large transfers instead of the kernel's 24- or 32-byte row pieces
	rc = peer_wait_word(c, &ctrl->released, use - 1u, &ctrl->error, s);
	if (rc) return rc;
	rc = enqueue_copy_out(c, f, (const uint32_t *)d_stage, (uint8_t *)d_frame, cudaMemcpyDeviceToDevice, s);
	if (rc) return rc;
	return peer_arrive(c, ctrl, f, use, s);
}

int hmrm_peer_wait(hmrm_ctx *c, void *d_ctrl, uint32_t use, int32_t ranks, void *stream) {
	if (!c) return HMRM_ERR_INVALID;
	if (!d_ctrl || use == 0u || ranks < 1 || ranks > 31) return fail(c, HMRM_ERR_INVALID, "hmrm_peer_wait: bad arguments");
	HMRM_CUDA(c, cudaSetDevice(c->device));
	PeerCtrl *ctrl = (PeerCtrl *)d_ctrl;
	cudaStream_t s = stream ? (cudaStream_t)stream : c->stream;
	if (c->knobs.peer_memops) {
		for (int r = 0; r < ranks; ++r)
			if (int rc = peer_wait_word(c, &ctrl->arrived_by[r], use, &ctrl->error, s)) return rc;
		return HMRM_OK;
	}
	return peer_wait_word(c, &ctrl->arrived, use * (uint32_t)ranks, &ctrl->error, s);
}

int hmrm_peer_release(hmrm_ctx *c, void *d_ctrl, uint32_t use, void *stream) {
	if (!c) return HMRM_ERR_INVALID;
	if (!d_ctrl) return fail(c, HMRM_ERR_INVALID, "hmrm_peer_release: bad arguments");
	HMRM_CUDA(c, cudaSetDevice(c->device));
	cudaStream_t s = stream ? (cudaStream_t)stream : c->stream;
	if (c->knobs.peer_memops) return peer_write_word(c, &((PeerCtrl *)d_ctrl)->released, use, s);
	k_peer_release<<<1, 1, 0, s>>>(&((PeerCtrl *)d_ctrl)->released, use);
	HMRM_CUDA(c, cudaGetLastError());
	return HMRM_OK;
}

int hmrm_peer_status(hmrm_ctx *c, void *d_ctrl, uint32_t out[3]) {
	if (!c) return HMRM_ERR_INVALID;
	if (!d_ctrl || !out) return fail(c, HMRM_ERR_INVALID, "hmrm_peer_status: bad arguments");
	HMRM_CUDA(c, cudaSetDevice(c->device));
	PeerCtrl h;
	HMRM_CUDA(c, cudaMemcpy(&h, d_ctrl, sizeof h, cudaMemcpyDeviceToHost));
	out[0] = h.arrived;
	out[1] = h.released;
	out[2] = h.error;
	return HMRM_OK;
}

int hmrm_peer_sync_mode(const hmrm_ctx *c) {
	if (!c) return -HMRM_ERR_INVALID;
	return c->knobs.peer_memops ? HMRM_PEER_SYNC_MEMOPS : HMRM_PEER_SYNC_KERNELS;
}

int hmrm_ipc_close(hmrm_ctx *c, void *dptr) {
	if (!c) return HMRM_ERR_INVALID;
	HMRM_CUDA(c, cudaSetDevice(c->device));
	if (int rc = drain(c)) return rc;
	if (dptr) HMRM_CUDA(c, cudaIpcCloseMemHandle(dptr));
	return HMRM_OK;
}

} // extern "C"
