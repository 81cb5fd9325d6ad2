// K5: box filter of supersampled and motion-blurred frames (HMRM_FLAG_SUPERSAMPLE, hmrm_set_motion_blur; hmrm_render*,
// hmrm_render_device).
//
// The exact definitions are in include/hmrm.h.  A sub-frame is the RGBA8 render of one camera at sW x sH; output pixel
// (px, py) is the rounded mean, channel by channel, of its s x s subsamples in every sub-frame of the frame, with alpha
// 255.  k5_downsample<S, C, G, P> reduces G sub-frame planes per launch: each thread owns a strip of 4 output pixels of
// one row (S sub-rows of 4S subsamples per plane), reads every subsample once and sums in integers.  A frame of n
// sub-frames takes ceil(n / G) launches: P = kK5Only when one launch covers all of them (divides by the compile-time
// G*S*S), else kK5First writes the per-pixel sums to a uint16 accumulator, kK5Middle adds into it and kK5Last adds,
// divides by the runtime n*S*S and writes the pixels.  The sums never exceed 16 * 16 * 255 = 65280.  A supersampled frame
// without blur is G = 1, kK5Only.  When a whole strip's sub-rows start on a 16-byte boundary ((S*W) % 4 == 0) each sub-row
// is S 16-byte loads; the last strip of a row that has fewer than 4 pixels and sub-rows of other widths take the scalar
// path, which only touches subsamples of pixels inside the frame.  Output is RGBA8 (C = 4) or packed RGB8 (C = 3): one
// 16-byte store, or three 4-byte words, when W % 4 == 0 and the destination is 16-byte aligned, else bytes.
#pragma once

#include <cstdint>

namespace hmrm {

constexpr int kDownThreads = 128;
constexpr int kDownStrip = 4;      // output pixels per thread
constexpr int kDownMaxPlanes = 4;  // largest G

enum K5Phase { kK5Only, kK5First, kK5Middle, kK5Last };

// grid: x over ceil(W/4) strips, y over H rows.  sub: G RGBA8 planes [S*H][S*W], `plane` words apart; out: [H][W][C]
// (kK5Only, kK5Last); acc: [H][W] of (R | G << 16, B) sums (kK5First writes it, kK5Middle and kK5Last read it); n: the
// divisor of kK5Last
template <int S, int C, int G = 1, int P = kK5Only>
__global__ void __launch_bounds__(kDownThreads) k5_downsample(const uint32_t *__restrict__ sub, int W, int H,
                                                              uint8_t *__restrict__ out, size_t plane = 0,
                                                              uint2 *__restrict__ acc = nullptr, uint32_t n = 0) {
	static_assert(G >= 1 && G <= kDownMaxPlanes && (P == kK5Only || P == kK5Last || C == 4), "K5 instantiation");
	const int x0 = (blockIdx.x * kDownThreads + threadIdx.x) * kDownStrip;
	if (x0 >= W) return;
	const int y = blockIdx.y;
	const size_t sw = (size_t)W * S;
	const bool whole = x0 + kDownStrip <= W;

	// per output pixel: R, G, B sums over its S x S subsamples in the G planes (and the accumulator)
	uint32_t sr[kDownStrip] = {0u, 0u, 0u, 0u}, sg[kDownStrip] = {0u, 0u, 0u, 0u}, sb[kDownStrip] = {0u, 0u, 0u, 0u};
	#pragma unroll
	for (int g = 0; g < G; ++g) {
		const uint32_t *src = sub + (size_t)g * plane;
		if (whole && ((S * W) & 3) == 0) {
			#pragma unroll
			for (int j = 0; j < S; ++j) {
				const uint4 *row = (const uint4 *)(src + (size_t)(S * y + j) * sw + (size_t)S * x0);
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
				const uint32_t *row = src + (size_t)(S * y + j) * sw + (size_t)S * x0;
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
	}
	const size_t at = (size_t)y * (size_t)W + (size_t)x0;
	if constexpr (P == kK5Middle || P == kK5Last) {
		#pragma unroll
		for (int p = 0; p < kDownStrip; ++p) {
			if (x0 + p >= W) break;
			const uint2 a = acc[at + p];
			sr[p] += a.x & 0xFFFFu;
			sg[p] += a.x >> 16;
			sb[p] += a.y;
		}
	}
	if constexpr (P == kK5First || P == kK5Middle) {
		#pragma unroll
		for (int p = 0; p < kDownStrip; ++p) {
			if (x0 + p >= W) break;
			acc[at + p] = make_uint2(sr[p] | (sg[p] << 16), sb[p]);
		}
		return;
	}

	const uint32_t d = P == kK5Only ? (uint32_t)(G * S * S) : n, half = d / 2;
	uint8_t px[kDownStrip * C];
	#pragma unroll
	for (int p = 0; p < kDownStrip; ++p) {
		px[C * p + 0] = (uint8_t)((sr[p] + half) / d);
		px[C * p + 1] = (uint8_t)((sg[p] + half) / d);
		px[C * p + 2] = (uint8_t)((sb[p] + half) / d);
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
