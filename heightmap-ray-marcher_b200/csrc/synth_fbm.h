/* Synthetic terrain generator: integer-only value-noise fBm.
 *
 * Shared by the test oracle (plain C, CPU) and by the CUDA library (device
 * kernel), which is why it is a header of `static inline` functions with no
 * floating point at all: every platform produces the same bytes, so a map
 * generated on the GPU box can be rendered by the CPU oracle and vice versa.
 *
 * The reference ships no maps (its README images are external links), so the
 * benchmark inputs named in BASELINE.json ("synthetic fBm heightmaps of the
 * named sizes") are defined here, following SURVEY.md §8(d): base lattice 4,
 * lacunarity 2, gain 1/2, octaves = log2(N) - 2 (finest lattice N/2),
 * smoothstep interpolation, seed 1234, height written as grey RGB (R=G=B),
 * colormap = RGBA ramp of the same field with one centred N/64 square of
 * alpha 0 (exercises main/hmap.cpp:1020 of the reference).  The min-max
 * normalisation of the survey is replaced by a fixed contrast stretch
 * (15 %..85 % of the theoretical range) so no global reduction is needed.
 */
#ifndef HMRM_SYNTH_FBM_H
#define HMRM_SYNTH_FBM_H

#include <stdint.h>

#if defined(__CUDACC__)
#define HMRM_SYNTH_FN __host__ __device__ static inline
#else
#define HMRM_SYNTH_FN static inline
#endif

/* 16-bit lattice value from an integer avalanche hash. */
HMRM_SYNTH_FN uint32_t hmrm_synth_lattice(uint32_t ix, uint32_t iy, uint32_t octave, uint32_t seed) {
	uint32_t h = seed * 0x9E3779B1u + octave * 0x85EBCA77u;
	h ^= ix * 0xC2B2AE3Du;
	h = (h << 15) | (h >> 17);
	h ^= iy * 0x27D4EB2Fu;
	h ^= h >> 16;
	h *= 0x7FEB352Du;
	h ^= h >> 15;
	h *= 0x846CA68Bu;
	h ^= h >> 16;
	return h & 0xFFFFu;
}

/* smoothstep(t) = t*t*(3-2t) on 16.16 fixed point, t in [0,65536). */
HMRM_SYNTH_FN uint32_t hmrm_synth_smooth(uint32_t t16) {
	uint64_t t2 = ((uint64_t)t16 * t16) >> 16;
	return (uint32_t)((t2 * (uint64_t)(196608u - 2u * t16)) >> 16);
}

/* fBm sum at pixel (x,y) of a 2^log2n square map, and the same sum for the all-ones lattice in *top. */
HMRM_SYNTH_FN uint32_t hmrm_synth_acc(uint32_t x, uint32_t y, uint32_t log2n, uint32_t seed, uint32_t *top_out) {
	const uint32_t octaves = log2n - 2u;
	uint32_t acc = 0u;   /* sum of (16-bit value << 8) >> octave */
	uint32_t top = 0u;   /* the same sum for the all-ones lattice */
	for (uint32_t o = 0u; o < octaves; ++o) {
		const uint32_t shift = log2n - 2u - o;          /* lattice cell = 2^shift pixels */
		const uint32_t mask = (1u << shift) - 1u;
		const uint32_t cx = x >> shift, cy = y >> shift;
		const uint32_t sx = hmrm_synth_smooth((x & mask) << (16u - shift));
		const uint32_t sy = hmrm_synth_smooth((y & mask) << (16u - shift));
		const uint32_t v00 = hmrm_synth_lattice(cx, cy, o, seed);
		const uint32_t v10 = hmrm_synth_lattice(cx + 1u, cy, o, seed);
		const uint32_t v01 = hmrm_synth_lattice(cx, cy + 1u, o, seed);
		const uint32_t v11 = hmrm_synth_lattice(cx + 1u, cy + 1u, o, seed);
		const uint32_t a = (v00 * (65536u - sx) + v10 * sx) >> 16;
		const uint32_t b = (v01 * (65536u - sx) + v11 * sx) >> 16;
		const uint32_t v = (a * (65536u - sy) + b * sy) >> 16;
		acc += (v << 8) >> o;
		top += (65535u << 8) >> o;
	}
	*top_out = top;
	return acc;
}

/* Height sample in [0,255] at pixel (x,y) of a 2^log2n square map. */
HMRM_SYNTH_FN uint32_t hmrm_synth_height(uint32_t x, uint32_t y, uint32_t log2n, uint32_t seed) {
	uint32_t top;
	const uint32_t acc = hmrm_synth_acc(x, y, log2n, seed, &top);
	/* contrast stretch [15 %, 85 %] of the range -> [0,255], clamped */
	const uint64_t lo = ((uint64_t)top * 15u) / 100u;
	const uint64_t hi = ((uint64_t)top * 85u) / 100u;
	if ((uint64_t)acc <= lo) return 0u;
	if ((uint64_t)acc >= hi) return 255u;
	return (uint32_t)((((uint64_t)acc - lo) * 255u) / (hi - lo));
}

/* The same field on the 16-bit scale, [0,65535]: the same stretch with 65535 for 255 (hmrm_synth_maps16). */
HMRM_SYNTH_FN uint32_t hmrm_synth_height16(uint32_t x, uint32_t y, uint32_t log2n, uint32_t seed) {
	uint32_t top;
	const uint32_t acc = hmrm_synth_acc(x, y, log2n, seed, &top);
	const uint64_t lo = ((uint64_t)top * 15u) / 100u;
	const uint64_t hi = ((uint64_t)top * 85u) / 100u;
	if ((uint64_t)acc <= lo) return 0u;
	if ((uint64_t)acc >= hi) return 65535u;
	return (uint32_t)((((uint64_t)acc - lo) * 65535u) / (hi - lo));
}

/* Colormap texel for height sample v at pixel (x,y) of an n*n map: RGBA. */
HMRM_SYNTH_FN uint32_t hmrm_synth_color(uint32_t v, uint32_t x, uint32_t y, uint32_t n) {
	uint32_t r, g, b, a = 255u;
	if (v < 64u) {            /* water: dark to light blue */
		r = 10u + v / 2u;  g = 40u + v;  b = 120u + 2u * v;
	} else if (v < 144u) {    /* lowland: green */
		const uint32_t t = v - 64u;
		r = 40u + t;  g = 120u + t / 2u;  b = 40u + t / 4u;
	} else if (v < 208u) {    /* highland: brown */
		const uint32_t t = v - 144u;
		r = 120u + t;  g = 100u + t / 2u;  b = 60u + t / 2u;
	} else {                  /* snow */
		const uint32_t t = v - 208u;
		r = 200u + t;  g = 200u + t;  b = 210u + (t * 45u) / 47u;
	}
	/* one centred n/64 square (at least 1 texel) of alpha 0 */
	uint32_t half = n / 128u;
	const uint32_t c = n / 2u;
	if (half == 0u) half = 1u;
	if (x >= c - half && x < c + half && y >= c - half && y < c + half) a = 0u;
	if (r > 255u) r = 255u;
	if (g > 255u) g = 255u;
	if (b > 255u) b = 255u;
	return r | (g << 8) | (b << 16) | (a << 24);   /* little-endian RGBA bytes */
}

#endif
