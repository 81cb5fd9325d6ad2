// K4: RGB -> limited-range 4:2:0 YCbCr planes on the device (hmrm_render_yuv420_async, hmrm_convert_yuv420).
//
// The exact integer definition is in include/hmrm.h.  One launch, k4_yuv420<C>: each thread owns a strip of 2 rows x 8
// columns of the [H][W][C] frame (C = 4: RGBA8, alpha ignored; C = 3: packed RGB8) and writes its 16 Y bytes and the
// 4 Cb + 4 Cr bytes of the strip's 2x2 blocks.  When W is a multiple of 8 every strip is whole and aligned: RGBA8 rows
// are read as 2 x 16-byte words per row, RGB8 rows as 3 x 8-byte words (24 bytes = 8 pixels), Y is stored as 8-byte
// words and each chroma row piece as one 4-byte word.  Other widths take the clamped byte path, which also covers odd
// sizes; an odd last row is read twice (the clamp) and its second Y row is not stored.
#pragma once

#include <cstdint>

namespace hmrm {

struct YuvCoef {
	int y[3], cb[3], cr[3];     // R, G, B weights, 2^-14 fixed point
};

// the table of include/hmrm.h, indexed by HMRM_YUV_BT601 / HMRM_YUV_BT709
constexpr YuvCoef kYuvCoef[2] = {
	{{4207, 8260, 1604}, {-2428, -4768, 7196}, {7196, -6026, -1170}},
	{{2991, 10064, 1016}, {-1649, -5547, 7196}, {7196, -6536, -660}},
};

// W*H + 2*ceil(W/2)*ceil(H/2); 0 outside [1, 65536] per axis
inline unsigned long long yuv420_bytes(int W, int H) {
	if (W < 1 || H < 1 || W > 65536 || H > 65536) return 0ull;
	const unsigned long long cw = (unsigned long long)(W + 1) / 2, ch = (unsigned long long)(H + 1) / 2;
	return (unsigned long long)W * (unsigned long long)H + 2ull * cw * ch;
}

constexpr int kYuvThreads = 128;

// byte k of a little-endian word array (k is a compile-time constant after unrolling)
__device__ __forceinline__ int yuv_byte(const uint32_t *w, int k) { return (int)((w[k >> 2] >> (8 * (k & 3))) & 255u); }

// grid: x over ceil(W/8) strips, y over ceil(H/2) row pairs.  planes: Y, then Cb, then Cr (I420, no padding)
template <int C>
__global__ void __launch_bounds__(kYuvThreads) k4_yuv420(const uint8_t *__restrict__ img, int W, int H, YuvCoef k,
                                                        uint8_t *__restrict__ planes) {
	const int x0 = (blockIdx.x * kYuvThreads + threadIdx.x) * 8;
	if (x0 >= W) return;
	const int i = blockIdx.y;
	const int rows[2] = {2 * i, min(2 * i + 1, H - 1)};
	const int cw = (W + 1) >> 1;
	const size_t ysize = (size_t)W * (size_t)H, csize = (size_t)cw * (size_t)((H + 1) >> 1);
	const bool whole = (W & 7) == 0;

	int r[2][8], g[2][8], b[2][8];
	if (whole) {
		#pragma unroll
		for (int h = 0; h < 2; ++h) {
			const uint8_t *src = img + ((size_t)rows[h] * (size_t)W + (size_t)x0) * C;
			uint32_t w[2 * C];
			if (C == 4) {
				const uint4 a = __ldg((const uint4 *)src), c = __ldg((const uint4 *)src + 1);
				w[0] = a.x; w[1] = a.y; w[2] = a.z; w[3] = a.w;
				w[4] = c.x; w[5] = c.y; w[6] = c.z; w[7] = c.w;
			}
			else {
				#pragma unroll
				for (int q = 0; q < 3; ++q) {
					const uint2 a = __ldg((const uint2 *)src + q);
					w[2 * q] = a.x;
					w[2 * q + 1] = a.y;
				}
			}
			#pragma unroll
			for (int p = 0; p < 8; ++p) {
				r[h][p] = yuv_byte(w, p * C + 0);
				g[h][p] = yuv_byte(w, p * C + 1);
				b[h][p] = yuv_byte(w, p * C + 2);
			}
		}
	}
	else {
		#pragma unroll
		for (int h = 0; h < 2; ++h) {
			const uint8_t *row = img + (size_t)rows[h] * (size_t)W * C;
			#pragma unroll
			for (int p = 0; p < 8; ++p) {
				const uint8_t *px = row + (size_t)min(x0 + p, W - 1) * C;
				r[h][p] = px[0];
				g[h][p] = px[1];
				b[h][p] = px[2];
			}
		}
	}

	// luma
	#pragma unroll
	for (int h = 0; h < 2; ++h) {
		if (h == 1 && 2 * i + 1 >= H) break;
		uint32_t packed[2] = {0u, 0u};
		#pragma unroll
		for (int p = 0; p < 8; ++p) {
			const int y = ((k.y[0] * r[h][p] + k.y[1] * g[h][p] + k.y[2] * b[h][p] + (1 << 13)) >> 14) + 16;
			packed[p >> 2] |= (uint32_t)y << (8 * (p & 3));
		}
		uint8_t *dst = planes + (size_t)rows[h] * (size_t)W + (size_t)x0;
		if (whole) *(uint2 *)dst = make_uint2(packed[0], packed[1]);
		else {
			#pragma unroll
			for (int p = 0; p < 8; ++p)
				if (x0 + p < W) dst[p] = (uint8_t)(packed[p >> 2] >> (8 * (p & 3)));
		}
	}

	// chroma of the strip's four 2x2 blocks
	uint32_t cbw = 0u, crw = 0u;
	#pragma unroll
	for (int m = 0; m < 4; ++m) {
		const int sr = r[0][2 * m] + r[0][2 * m + 1] + r[1][2 * m] + r[1][2 * m + 1];
		const int sg = g[0][2 * m] + g[0][2 * m + 1] + g[1][2 * m] + g[1][2 * m + 1];
		const int sb = b[0][2 * m] + b[0][2 * m + 1] + b[1][2 * m] + b[1][2 * m + 1];
		const int cb = ((k.cb[0] * sr + k.cb[1] * sg + k.cb[2] * sb + (1 << 15)) >> 16) + 128;
		const int cr = ((k.cr[0] * sr + k.cr[1] * sg + k.cr[2] * sb + (1 << 15)) >> 16) + 128;
		cbw |= (uint32_t)cb << (8 * m);
		crw |= (uint32_t)cr << (8 * m);
	}
	const size_t at = (size_t)i * (size_t)cw + (size_t)(x0 >> 1);
	uint8_t *dcb = planes + ysize + at, *dcr = planes + ysize + csize + at;
	if (whole) {
		*(uint32_t *)dcb = cbw;
		*(uint32_t *)dcr = crw;
	}
	else {
		#pragma unroll
		for (int m = 0; m < 4; ++m)
			if ((x0 >> 1) + m < cw) {
				dcb[m] = (uint8_t)(cbw >> (8 * m));
				dcr[m] = (uint8_t)(crw >> (8 * m));
			}
	}
}

} // namespace hmrm
