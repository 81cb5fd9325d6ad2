/* TEST INFRASTRUCTURE — not product code.
 *
 * CPU statement of the 16-bit height definition (include/hmrm.h, hmrm_set_maps16): the reference's UpdateHeightmap
 * (main/hmap.cpp:171-191) with 255 replaced by 65535, for one sample x used as R = G = B.  Every operation is one
 * IEEE-754 binary64 operation in the order written, compiled without FMA contraction (-ffp-contract=off), as
 * oracle/hmap_oracle.c is.  Also the synthetic 16-bit map of hmrm_synth_maps16 on the CPU.  Loaded by
 * tests/height16_lib.py.
 *
 * It lives beside the tests rather than in oracle/: the oracle restates the unmodified reference and is pinned against
 * it, and the reference has no 16-bit path.  This statement is pinned to the oracle instead, through the widened-grey
 * identity (x = 257 v8, unit lum: bit-identical heights, tests/test_height16.py).  Renders over 16-bit maps use the
 * oracle's own oracle_render over these heights.
 */
#include <stdint.h>
#include <stddef.h>

#include "../heightmap-ray-marcher_b200/csrc/synth_fbm.h"

void h16_update_heightmap(const uint16_t *samples, int64_t num_pixels, double lum_r, double lum_g, double lum_b,
                          double min_height, double max_height, double *heights) {
	const double span = max_height - min_height;
#pragma omp parallel for schedule(static)
	for (int64_t p = 0; p < num_pixels; ++p) {
		const double x = (double)samples[p];
		double v = (lum_r * x + lum_g * x) + lum_b * x;
		if (v < 0.0) v = 0.0;
		else if (v > 65535.0) v = 65535.0;
		heights[p] = (v / 65535.0) * span + min_height;
	}
}

/* height [n][n] (hmrm_synth_height16) and the RGBA8 colormap of hmrm_synth_maps [n][n][4]; either may be NULL */
void h16_synth_maps16(uint32_t log2n, uint32_t seed, uint16_t *height, uint8_t *color_rgba8) {
	const uint32_t n = 1u << log2n;
#pragma omp parallel for schedule(static)
	for (int64_t y = 0; y < (int64_t)n; ++y) {
		for (uint32_t x = 0; x < n; ++x) {
			const size_t p = (size_t)y * n + x;
			if (height) height[p] = (uint16_t)hmrm_synth_height16(x, (uint32_t)y, log2n, seed);
			if (color_rgba8) {
				const uint32_t v = hmrm_synth_height(x, (uint32_t)y, log2n, seed);
				const uint32_t c = hmrm_synth_color(v, x, (uint32_t)y, n);
				color_rgba8[4 * p + 0] = (uint8_t)(c & 255u);
				color_rgba8[4 * p + 1] = (uint8_t)((c >> 8) & 255u);
				color_rgba8[4 * p + 2] = (uint8_t)((c >> 16) & 255u);
				color_rgba8[4 * p + 3] = (uint8_t)(c >> 24);
			}
		}
	}
}
