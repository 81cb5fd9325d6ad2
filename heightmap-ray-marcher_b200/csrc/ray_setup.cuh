// Per-pixel front end shared by the render kernels: ray generation for the three
// projections, AABB slab entry, miss shading, pixel store.
//
// Arithmetic contract (operation order = rounding order), reference lines:
//   Perspective::GetRay   src/Perspective.cpp:25-32
//   Spherical::GetRay     src/Spherical.cpp:17-31 (trig factors come from host tables)
//   Orthographic::GetRay  src/Orthographic.cpp:19-25
//   distance/intersection src/AABB.cpp:30-77
//   miss shading          main/hmap.cpp:1041-1057
//   SetPixel              main/hmap.cpp:139-154
#ifndef HMRM_RAY_SETUP_CUH
#define HMRM_RAY_SETUP_CUH

#include "device_math.cuh"
#include "render_params.h"

namespace hmrm {

struct Ray {
	double ox, oy, oz;
	double dx, dy, dz;
};

__device__ __forceinline__ Ray generate_ray(const RenderParams &P, int px, int py) {
	Ray r;
	if (P.projection == 2) {
		const double sv = __ldg(P.sin_va + py);
		r.ox = P.cam[0]; r.oy = P.cam[1]; r.oz = P.cam[2];
		r.dx = fmul(sv, __ldg(P.cos_ha + px));
		r.dy = fmul(sv, __ldg(P.sin_ha + px));
		r.dz = __ldg(P.cos_va + py);
		return r;
	}
	const double w = __ldg(P.wtab + px);
	const double h = __ldg(P.htab + py);
	// (upper_left + w * plane_right) + h * plane_down
	const double qx = fadd(fadd(P.ul[0], fmul(w, P.pr[0])), fmul(h, P.pd[0]));
	const double qy = fadd(fadd(P.ul[1], fmul(w, P.pr[1])), fmul(h, P.pd[1]));
	const double qz = fadd(fadd(P.ul[2], fmul(w, P.pr[2])), fmul(h, P.pd[2]));
	if (P.projection == 1) {
		const double vx = fsub(qx, P.cam[0]);
		const double vy = fsub(qy, P.cam[1]);
		const double vz = fsub(qz, P.cam[2]);
		// glm::normalize: v * (1 / sqrt(dot(v, v))), dot = (x*x + y*y) + z*z
		const double len2 = fadd(fadd(fmul(vx, vx), fmul(vy, vy)), fmul(vz, vz));
		const double inv = frcp(fsqrt(len2));
		r.ox = P.cam[0]; r.oy = P.cam[1]; r.oz = P.cam[2];
		r.dx = fmul(vx, inv);
		r.dy = fmul(vy, inv);
		r.dz = fmul(vz, inv);
	}
	else {
		r.ox = qx; r.oy = qy; r.oz = qz;
		r.dx = P.look[0]; r.dy = P.look[1]; r.dz = P.look[2];
	}
	return r;
}

// One axis of the slab test; returns false when the ray misses (src/AABB.cpp:58-73).
__device__ __forceinline__ bool slab_axis(double c0, double c1, double o, double d, double &lo, double &hi) {
	double t_near = fdiv(fsub(c0, o), d);
	double t_far = fdiv(fsub(c1, o), d);
	if (t_near > t_far) {
		const double t = t_near;
		t_near = t_far;
		t_far = t;
	}
	if (t_far < lo || t_near > hi) return false;
	if (t_near > lo) lo = t_near;
	if (t_far < hi) hi = t_far;
	return true;
}

// distance() + intersection() (src/AABB.cpp:30-77): `dist` is what distance() returns (+inf when a slab test fails
// or lo > hi, else the entry distance lo); true and the entry point when 0 <= dist < inf.
__device__ __forceinline__ bool box_entry_at(const double *c0, const double *c1, const Ray &r, double &ex, double &ey,
                                             double &ez, double &dist) {
	const double inf = __longlong_as_double(0x7FF0000000000000LL);
	double lo = -inf, hi = inf;
	dist = inf;
	if (!slab_axis(c0[0], c1[0], r.ox, r.dx, lo, hi)) return false;
	if (!slab_axis(c0[1], c1[1], r.oy, r.dy, lo, hi)) return false;
	if (!slab_axis(c0[2], c1[2], r.oz, r.dz, lo, hi)) return false;
	if (lo > hi) return false;
	dist = lo;
	if (lo == inf) return false;
	if (lo < 0.0) return false;
	ex = fadd(r.ox, fmul(lo, r.dx));
	ey = fadd(r.oy, fmul(lo, r.dy));
	ez = fadd(r.oz, fmul(lo, r.dz));
	return true;
}

// A ray that starts outside one slab of the box and points away from it on that axis cannot enter: both of that
// axis' quotients (c - o) / d are then strictly negative (never NaN: numerator and denominator are non-zero), so
// distance() either bails out with +inf or returns lo <= hi < 0 and intersection() rejects d < 0 (src/AABB.cpp:36-39,
// :69-76).  Decided exactly, without the six divides — every ray above the horizon of a camera above the terrain.
__device__ __forceinline__ bool certain_miss(const RenderParams &P, const Ray &r) {
	return (r.ox > P.bmax[0] && r.dx > 0.0) || (r.ox < P.bmin[0] && r.dx < 0.0) ||
	       (r.oy > P.bmax[1] && r.dy > 0.0) || (r.oy < P.bmin[1] && r.dy < 0.0) ||
	       (r.oz > P.bmax[2] && r.dz > 0.0) || (r.oz < P.bmin[2] && r.dz < 0.0);
}

// `dist` is only meaningful when the slab test ran (always when P.ray_dump is set).
__device__ __forceinline__ bool box_entry(const RenderParams &P, const Ray &r, double &ex, double &ey, double &ez, double &dist) {
#ifndef HMRM_EXP_NO_EARLYOUT
	if (!P.ray_dump && certain_miss(P, r)) {
		dist = __longlong_as_double(0x7FF0000000000000LL);
		return false;
	}
#endif
	return box_entry_at(P.c0, P.c1, r, ex, ey, ez, dist);
}

__device__ __forceinline__ uint32_t sky_channel(double v) {
	if (v < 0.0) v = 0.0;
	else if (v > 255.0) v = 255.0;
	return (uint32_t)__double2uint_rd(v);   // (Uint8)floor(v), v in [0,255]
}

// colour of a ray that hit nothing (main/hmap.cpp:1041-1057); alpha 255
__device__ __forceinline__ uint32_t miss_colour(const RenderParams &P, double dz) {
	if (dz > 0.0) {
		const double zz = fmul(dz, dz);   // std::pow(z, 2) == z*z under -std=c++98
		const uint32_t r = sky_channel(fadd(fmul(220.0, zz), (double)P.bg[0]));
		const uint32_t g = sky_channel(fadd(fmul(240.0, zz), (double)P.bg[1]));
		const uint32_t b = sky_channel(fadd(fmul(255.0, dz), (double)P.bg[2]));
		return r | (g << 8) | (b << 16) | 0xFF000000u;
	}
	return P.bg_rgba;
}

// colour of a terrain hit (main/hmap.cpp:1018-1031): alpha-0 texels draw the background colour
__device__ __forceinline__ uint32_t hit_colour(const RenderParams &P, uint32_t texel) {
	return ((texel >> 24) == 0u) ? P.bg_rgba : (texel | 0xFF000000u);
}

// HMRM_FLAG_RAY_DUMP: the device's own intermediates of this pixel, for bit-pattern comparison with the reference's
// GetRay / distance / intersection (src/Perspective.cpp:25-32, src/AABB.cpp:30-77): frames are blind to ulp errors.
// Record = pos[3], dir[3], distance() as the reference returns it, entry[3] (zeros when intersection() is false).
__device__ __noinline__ void dump_ray(const RenderParams &P, int px, int py, const Ray &r, bool entered, double lo,
                                      double ex, double ey, double ez) {
	double *o = P.ray_dump + ((size_t)py * (size_t)P.W + (size_t)px) * 10;
	o[0] = r.ox; o[1] = r.oy; o[2] = r.oz;
	o[3] = r.dx; o[4] = r.dy; o[5] = r.dz;
	o[6] = lo;
	o[7] = entered ? ex : 0.0;
	o[8] = entered ? ey : 0.0;
	o[9] = entered ? ez : 0.0;
}

// RGBA8 pixel `at` (index into [H][W]): one 32-bit store, or four byte stores into a destination that is not 4-byte
// aligned (hmrm_render_device and the peer calls accept any device pointer).
__device__ __forceinline__ void store_rgba8(const RenderParams &P, size_t at, uint32_t rgba) {
	if (!P.fb_unaligned) {
		P.fb[at] = rgba;
		return;
	}
	uint8_t *o = (uint8_t *)P.fb + at * 4;
	o[0] = (uint8_t)rgba;
	o[1] = (uint8_t)(rgba >> 8);
	o[2] = (uint8_t)(rgba >> 16);
	o[3] = (uint8_t)(rgba >> 24);
}

// SetPixel (main/hmap.cpp:139-154).  Called by the whole warp (8x4-pixel tile, lane = 8 * row + column); `active`
// lanes own a pixel of this frame.  RGBA8: one 32-bit store per pixel, A = 255.  RGB8 (HMRM_PIXEL_RGB8: the alpha
// byte is always 255 in the reference, so it is dead weight on PCIe / NVLink): a tile row is 24 contiguous bytes;
// when all 8 pixels of the row are written and rows are 4-byte aligned, lanes 0..5 of the row assemble them as six
// 32-bit words from their neighbours' colours (two shuffles), otherwise every lane stores its 3 bytes.
__device__ __forceinline__ void store_pixel(const RenderParams &P, int px, int py, bool active, uint32_t rgba) {
	if (P.pixel_format == 0) {
		if (active) store_rgba8(P, HMRM_CHECKED(P, (size_t)py * (size_t)P.W + (size_t)px, (size_t)P.W * (size_t)P.H), rgba);
		return;
	}
	const int lane = threadIdx.x & 31, i = lane & 7;
	const unsigned full = __ballot_sync(0xFFFFFFFFu, active);
	const bool row_full = ((full >> (lane & 24)) & 0xFFu) == 0xFFu && P.rgb_words;
	const int a = (i * 4) / 3;                         // first pixel contributing to word i (i < 6): 0 1 2 4 5 6
	const uint32_t A = __shfl_sync(0xFFFFFFFFu, rgba, (lane & 24) | min(a, 7)) & 0xFFFFFFu;
	const uint32_t B = __shfl_sync(0xFFFFFFFFu, rgba, (lane & 24) | min(a + 1, 7)) & 0xFFFFFFu;
	uint8_t *fb8 = (uint8_t *)P.fb;
	if (row_full) {
		if (i < 6) {
			const int sh = 8 * ((i * 4) % 3);
			const uint32_t word = (A >> sh) | (B << (24 - sh));
			const size_t at = ((size_t)py * (size_t)P.W + (size_t)(px & ~7)) * 3;   // multiple of 4 (W % 4 == 0, fb aligned)
			*(uint32_t *)(fb8 + HMRM_CHECKED(P, at + (size_t)i * 4, (size_t)P.W * (size_t)P.H * 3)) = word;
		}
	}
	else if (active) {
		uint8_t *o = fb8 + HMRM_CHECKED(P, ((size_t)py * (size_t)P.W + (size_t)px) * 3, (size_t)P.W * (size_t)P.H * 3);
		o[0] = (uint8_t)rgba;
		o[1] = (uint8_t)(rgba >> 8);
		o[2] = (uint8_t)(rgba >> 16);
	}
}

} // namespace hmrm

#endif
