// K5: box filter of a supersampled frame (HMRM_FLAG_SUPERSAMPLE; hmrm_render*, hmrm_render_device).
//
// The exact definition is in include/hmrm.h.  The sub-frame is the RGBA8 render of the same camera at sW x sH; output
// pixel (px, py) is the rounded mean of its s x s subsamples, channel by channel, with alpha 255.  One launch,
// k5_downsample<S, C>: each thread owns a strip of 4 output pixels of one row (S sub-rows of 4S subsamples), reads every
// subsample once, sums in integers and divides by the compile-time S*S.  When a whole strip's sub-rows start on a
// 16-byte boundary ((S*W) % 4 == 0) each sub-row is S 16-byte loads; the last strip of a row that has fewer than 4 pixels
// and sub-rows of other widths take the scalar path, which only touches subsamples of pixels inside the frame.  Output
// is RGBA8 (C = 4) or packed RGB8 (C = 3): one 16-byte store, or three 4-byte words, when W % 4 == 0 and the destination
// is 16-byte aligned, else bytes.
#pragma once

#include <cstdint>

namespace hmrm {

constexpr int kDownThreads = 128;
constexpr int kDownStrip = 4;      // output pixels per thread

// grid: x over ceil(W/4) strips, y over H rows.  sub: RGBA8 [S*H][S*W]; out: [H][W][C]
template <int S, int C>
__global__ void __launch_bounds__(kDownThreads) k5_downsample(const uint32_t *__restrict__ sub, int W, int H,
                                                              uint8_t *__restrict__ out) {
	const int x0 = (blockIdx.x * kDownThreads + threadIdx.x) * kDownStrip;
	if (x0 >= W) return;
	const int y = blockIdx.y;
	const size_t sw = (size_t)W * S;
	const bool whole = x0 + kDownStrip <= W;

	// per output pixel: R, G, B sums over its S x S subsamples (at most 16 * 255)
	uint32_t sr[kDownStrip] = {0u, 0u, 0u, 0u}, sg[kDownStrip] = {0u, 0u, 0u, 0u}, sb[kDownStrip] = {0u, 0u, 0u, 0u};
	if (whole && ((S * W) & 3) == 0) {
		#pragma unroll
		for (int j = 0; j < S; ++j) {
			const uint4 *row = (const uint4 *)(sub + (size_t)(S * y + j) * sw + (size_t)S * x0);
			#pragma unroll
			for (int q = 0; q < S; ++q) {
				const uint4 v = __ldg(row + q);
				const uint32_t w[4] = {v.x, v.y, v.z, v.w};
				#pragma unroll
				for (int k = 0; k < 4; ++k) {
					const int p = (4 * q + k) / S;      // output pixel of subsample 4q + k of the strip's sub-row
					sr[p] += w[k] & 255u;
					sg[p] += (w[k] >> 8) & 255u;
					sb[p] += (w[k] >> 16) & 255u;
				}
			}
		}
	}
	else {
		#pragma unroll
		for (int j = 0; j < S; ++j) {
			const uint32_t *row = sub + (size_t)(S * y + j) * sw + (size_t)S * x0;
			#pragma unroll
			for (int p = 0; p < kDownStrip; ++p) {
				if (x0 + p >= W) break;
				#pragma unroll
				for (int i = 0; i < S; ++i) {
					const uint32_t w = __ldg(row + S * p + i);
					sr[p] += w & 255u;
					sg[p] += (w >> 8) & 255u;
					sb[p] += (w >> 16) & 255u;
				}
			}
		}
	}

	constexpr uint32_t n = S * S, half = n / 2;
	uint8_t px[kDownStrip * C];
	#pragma unroll
	for (int p = 0; p < kDownStrip; ++p) {
		px[C * p + 0] = (uint8_t)((sr[p] + half) / n);
		px[C * p + 1] = (uint8_t)((sg[p] + half) / n);
		px[C * p + 2] = (uint8_t)((sb[p] + half) / n);
		if (C == 4) px[C * p + 3] = 255u;
	}
	uint8_t *dst = out + ((size_t)y * (size_t)W + (size_t)x0) * C;
	if (whole && (W & 3) == 0 && ((uintptr_t)out & 15) == 0) {
		uint32_t wd[C];
		#pragma unroll
		for (int k = 0; k < C; ++k)
			wd[k] = (uint32_t)px[4 * k] | ((uint32_t)px[4 * k + 1] << 8) | ((uint32_t)px[4 * k + 2] << 16) |
			        ((uint32_t)px[4 * k + 3] << 24);
		if constexpr (C == 4) *(uint4 *)dst = make_uint4(wd[0], wd[1], wd[2], wd[3]);
		else {
			#pragma unroll
			for (int k = 0; k < C; ++k) ((uint32_t *)dst)[k] = wd[k];
		}
	}
	else {
		#pragma unroll
		for (int p = 0; p < kDownStrip; ++p) {
			if (x0 + p >= W) break;
			#pragma unroll
			for (int k = 0; k < C; ++k) dst[C * p + k] = px[C * p + k];
		}
	}
}

} // namespace hmrm
