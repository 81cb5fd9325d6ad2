// K6: baseline JPEG encoding on the device (hmrm_render_jpeg_async, hmrm_encode_jpeg).
//
// The file is defined to the byte in include/hmrm.h: libjpeg-turbo's baseline file with the Annex K tables, IJG
// quality scaling, 4:2:0 or 4:4:4, and one restart interval per MCU row.  Every 8x8 block is transformed, quantised
// and sized on its own; blocks are linked only by prefix sums (DC predictor, bit offsets, 0xFF stuffing), so the
// encoder is three launches plus K3's gather, all on one stream:
//   k6_jpeg_blocks  one CTA per strip of 48 blocks (8 MCUs of 4:2:0 = 128 x 16 pixels, or 16 MCUs of 4:4:4 = 128 x 8):
//                   the frame's pixels (clamped at the edges, which is libjpeg's edge replication) become Y / Cb / Cr
//                   in shared memory, 4:2:0 chroma with libjpeg's 1, 2, 1, 2 bias; then 8 threads per block run
//                   jfdctint's two passes (a row each, then a column each) and quantise; the block's coefficients are
//                   stored in zig-zag order with the number of bits its AC codes take;
//   k6_jpeg_rows    one CTA per MCU row (= restart interval): DC differences and block bit lengths, a CTA scan into
//                   bit offsets (32 bits: a row is at most 4096 MCUs x 6 blocks x 1660 bits < 2^32), every block's
//                   codes ORed into the row's bit buffer by 8 threads at once (each writes the codes of 8 zig-zag
//                   positions at its own offset), the padding 1-bits, then 0xFF stuffing by a chunked CTA scan into the
//                   row's staging piece, which ends with the row's RST marker;
//   k6_jpeg_finish  one CTA: 64-bit scan of the row piece sizes into file offsets, the header (built on the host: it
//                   depends only on the size, quality and chroma mode) and EOI into the meta buffer;
//   k3_png_gather   writes the pieces (header, rows, EOI) to the destination with aligned 16-byte stores.
#pragma once

#include <cstdint>
#include <cstring>

namespace hmrm {

constexpr int kJpegHeadBytes = 629;         // SOI .. SOS, the bytes before the entropy-coded data
constexpr int kJpegMetaTail = 640;          // offset of EOI inside the meta buffer
constexpr int kJpegMetaBytes = 656;
constexpr int kJpegTileBlocks = 48;         // blocks per k6_jpeg_blocks CTA
constexpr int kJpegBlockThreads = kJpegTileBlocks * 8;
constexpr int kJpegRowThreads = 1024;
constexpr int kJpegMaxBlockBits = 1660;     // DC 11 + 11, 63 AC positions x (16 + 10): see hmrm_jpeg_bound

// Annex K.3 Huffman tables: code counts per length 1..16, then the symbols
constexpr uint8_t kJpegDcLumaBits[16] = {0, 1, 5, 1, 1, 1, 1, 1, 1, 0, 0, 0, 0, 0, 0, 0};
constexpr uint8_t kJpegDcChromaBits[16] = {0, 3, 1, 1, 1, 1, 1, 1, 1, 1, 1, 0, 0, 0, 0, 0};
constexpr uint8_t kJpegDcVals[12] = {0, 1, 2, 3, 4, 5, 6, 7, 8, 9, 10, 11};
constexpr uint8_t kJpegAcLumaBits[16] = {0, 2, 1, 3, 3, 2, 4, 3, 5, 5, 4, 4, 0, 0, 1, 0x7d};
constexpr uint8_t kJpegAcLumaVals[162] = {
	0x01, 0x02, 0x03, 0x00, 0x04, 0x11, 0x05, 0x12, 0x21, 0x31, 0x41, 0x06, 0x13, 0x51, 0x61, 0x07, 0x22, 0x71, 0x14,
	0x32, 0x81, 0x91, 0xa1, 0x08, 0x23, 0x42, 0xb1, 0xc1, 0x15, 0x52, 0xd1, 0xf0, 0x24, 0x33, 0x62, 0x72, 0x82, 0x09,
	0x0a, 0x16, 0x17, 0x18, 0x19, 0x1a, 0x25, 0x26, 0x27, 0x28, 0x29, 0x2a, 0x34, 0x35, 0x36, 0x37, 0x38, 0x39, 0x3a,
	0x43, 0x44, 0x45, 0x46, 0x47, 0x48, 0x49, 0x4a, 0x53, 0x54, 0x55, 0x56, 0x57, 0x58, 0x59, 0x5a, 0x63, 0x64, 0x65,
	0x66, 0x67, 0x68, 0x69, 0x6a, 0x73, 0x74, 0x75, 0x76, 0x77, 0x78, 0x79, 0x7a, 0x83, 0x84, 0x85, 0x86, 0x87, 0x88,
	0x89, 0x8a, 0x92, 0x93, 0x94, 0x95, 0x96, 0x97, 0x98, 0x99, 0x9a, 0xa2, 0xa3, 0xa4, 0xa5, 0xa6, 0xa7, 0xa8, 0xa9,
	0xaa, 0xb2, 0xb3, 0xb4, 0xb5, 0xb6, 0xb7, 0xb8, 0xb9, 0xba, 0xc2, 0xc3, 0xc4, 0xc5, 0xc6, 0xc7, 0xc8, 0xc9, 0xca,
	0xd2, 0xd3, 0xd4, 0xd5, 0xd6, 0xd7, 0xd8, 0xd9, 0xda, 0xe1, 0xe2, 0xe3, 0xe4, 0xe5, 0xe6, 0xe7, 0xe8, 0xe9, 0xea,
	0xf1, 0xf2, 0xf3, 0xf4, 0xf5, 0xf6, 0xf7, 0xf8, 0xf9, 0xfa};
constexpr uint8_t kJpegAcChromaBits[16] = {0, 2, 1, 2, 4, 4, 3, 4, 7, 5, 4, 4, 0, 1, 2, 0x77};
constexpr uint8_t kJpegAcChromaVals[162] = {
	0x00, 0x01, 0x02, 0x03, 0x11, 0x04, 0x05, 0x21, 0x31, 0x06, 0x12, 0x41, 0x51, 0x07, 0x61, 0x71, 0x13, 0x22, 0x32,
	0x81, 0x08, 0x14, 0x42, 0x91, 0xa1, 0xb1, 0xc1, 0x09, 0x23, 0x33, 0x52, 0xf0, 0x15, 0x62, 0x72, 0xd1, 0x0a, 0x16,
	0x24, 0x34, 0xe1, 0x25, 0xf1, 0x17, 0x18, 0x19, 0x1a, 0x26, 0x27, 0x28, 0x29, 0x2a, 0x35, 0x36, 0x37, 0x38, 0x39,
	0x3a, 0x43, 0x44, 0x45, 0x46, 0x47, 0x48, 0x49, 0x4a, 0x53, 0x54, 0x55, 0x56, 0x57, 0x58, 0x59, 0x5a, 0x63, 0x64,
	0x65, 0x66, 0x67, 0x68, 0x69, 0x6a, 0x73, 0x74, 0x75, 0x76, 0x77, 0x78, 0x79, 0x7a, 0x82, 0x83, 0x84, 0x85, 0x86,
	0x87, 0x88, 0x89, 0x8a, 0x92, 0x93, 0x94, 0x95, 0x96, 0x97, 0x98, 0x99, 0x9a, 0xa2, 0xa3, 0xa4, 0xa5, 0xa6, 0xa7,
	0xa8, 0xa9, 0xaa, 0xb2, 0xb3, 0xb4, 0xb5, 0xb6, 0xb7, 0xb8, 0xb9, 0xba, 0xc2, 0xc3, 0xc4, 0xc5, 0xc6, 0xc7, 0xc8,
	0xc9, 0xca, 0xd2, 0xd3, 0xd4, 0xd5, 0xd6, 0xd7, 0xd8, 0xd9, 0xda, 0xe2, 0xe3, 0xe4, 0xe5, 0xe6, 0xe7, 0xe8, 0xe9,
	0xea, 0xf2, 0xf3, 0xf4, 0xf5, 0xf6, 0xf7, 0xf8, 0xf9, 0xfa};

// Annex K.1 quantisation tables, natural order
constexpr uint8_t kJpegLumaQuant[64] = {16, 11, 10, 16, 24, 40, 51, 61, 12, 12, 14, 19, 26, 58, 60, 55,
                                        14, 13, 16, 24, 40, 57, 69, 56, 14, 17, 22, 29, 51, 87, 80, 62,
                                        18, 22, 37, 56, 68, 109, 103, 77, 24, 35, 55, 64, 81, 104, 113, 92,
                                        49, 64, 78, 87, 103, 121, 120, 101, 72, 92, 95, 98, 112, 100, 103, 99};
constexpr uint8_t kJpegChromaQuant[64] = {17, 18, 24, 47, 99, 99, 99, 99, 18, 21, 26, 66, 99, 99, 99, 99,
                                          24, 26, 56, 99, 99, 99, 99, 99, 47, 66, 99, 99, 99, 99, 99, 99,
                                          99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99,
                                          99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99};
// zig-zag position -> natural index
constexpr uint8_t kJpegZigzag[64] = {0, 1, 8, 16, 9, 2, 3, 10, 17, 24, 32, 25, 18, 11, 4, 5,
                                     12, 19, 26, 33, 40, 48, 41, 34, 27, 20, 13, 6, 7, 14, 21, 28,
                                     35, 42, 49, 56, 57, 50, 43, 36, 29, 22, 15, 23, 30, 37, 44, 51,
                                     58, 59, 52, 45, 38, 31, 39, 46, 53, 60, 61, 54, 47, 55, 62, 63};

// Device tables: canonical Huffman codes, (length << 16) | code by symbol ([0] DC luma, [1] AC luma, [2] DC chroma,
// [3] AC chroma), and the zig-zag position of each natural index
struct JpegCodes {
	uint32_t t[4][256];
	uint8_t zpos[64];
};

constexpr JpegCodes jpeg_make_codes() {
	JpegCodes r{};
	const uint8_t *bits[4] = {kJpegDcLumaBits, kJpegAcLumaBits, kJpegDcChromaBits, kJpegAcChromaBits};
	const uint8_t *vals[4] = {kJpegDcVals, kJpegAcLumaVals, kJpegDcVals, kJpegAcChromaVals};
	for (int k = 0; k < 4; ++k) {
		uint32_t code = 0;
		int n = 0;
		for (int len = 1; len <= 16; ++len) {
			for (int i = 0; i < bits[k][len - 1]; ++i) r.t[k][vals[k][n++]] = ((uint32_t)len << 16) | code++;
			code <<= 1;
		}
	}
	for (int k = 0; k < 64; ++k) r.zpos[kJpegZigzag[k]] = (uint8_t)k;
	return r;
}

__device__ const JpegCodes kJpegCodesDev = jpeg_make_codes();

// Per frame: the divisor of every coefficient as the exact reciprocal below, natural order, [0] luma, [1] chroma.
// A coefficient c against table entry t is (|c| + 4t) / (8t), truncated, with c's sign (libjpeg's quantiser).  With
// a = |c| + 4t, d = 8t and m = ceil(2^32 / d), umulhi(a, m) = floor(a / d) whenever a d < 2^32: writing a = q d + r,
// a m / 2^32 = q + r / d + a e / (d 2^32) with e = m d - 2^32 < d, and r / d + a e / (d 2^32) < (d - 1) / d + a / 2^32,
// which is below 1 when a < 2^32 / d.  Here |c| <= 8192 (jfdctint's output is 8x the DCT, |DCT| <= 1024), so a < 2^14
// and d <= 2040 < 2^11.  tests/test_jpeg_model.py also checks it for every |c| <= 2^15 and every t.
struct JpegQuant {
	uint32_t recip[2][64];
	uint16_t half[2][64];       // 4t
};

inline int jpeg_quant_entry(int base, int quality) {
	const int s = quality < 50 ? 5000 / quality : 200 - 2 * quality;
	const int v = (base * s + 50) / 100;
	return v < 1 ? 1 : v > 255 ? 255 : v;
}

inline JpegQuant jpeg_quant(int quality) {
	JpegQuant q;
	for (int i = 0; i < 64; ++i)
		for (int k = 0; k < 2; ++k) {
			const uint32_t t = (uint32_t)jpeg_quant_entry(k ? kJpegChromaQuant[i] : kJpegLumaQuant[i], quality);
			q.recip[k][i] = (uint32_t)((0x100000000ull + 8u * t - 1u) / (8u * t));
			q.half[k][i] = (uint16_t)(4u * t);
		}
	return q;
}

// host arithmetic shared by hmrm_jpeg_bound and the launches
struct JpegShape {
	int W, H, s420;             // s420: 4:2:0
	int mcux, mcuy, bpm;        // MCUs per row, MCU rows, blocks per MCU (6 | 3)
	unsigned long long blocks;  // mcux * mcuy * bpm, dummies included
	unsigned long long row_words;   // uint32 words of one row's bit buffer
	unsigned long long row_stride;  // bytes of one row's staging piece: 415 per block + 4, rounded up to 16
};

inline bool jpeg_shape(long long W, long long H, int s420, JpegShape *out) {
	if (W < 1 || H < 1 || W > 65535 || H > 65535) return false;
	const int m = s420 ? 16 : 8;
	out->W = (int)W;
	out->H = (int)H;
	out->s420 = s420;
	out->mcux = (int)((W + m - 1) / m);
	out->mcuy = (int)((H + m - 1) / m);
	out->bpm = s420 ? 6 : 3;
	out->blocks = (unsigned long long)out->mcux * (unsigned long long)out->mcuy * (unsigned long long)out->bpm;
	const unsigned long long bpr = (unsigned long long)out->mcux * (unsigned long long)out->bpm;
	out->row_words = (bpr * kJpegMaxBlockBits + 31ull) / 32ull + 1ull;
	out->row_stride = (415ull * bpr + 4ull + 15ull) & ~15ull;
	return true;
}

// SOI + EOI + per block 1660 bits, 0xFF stuffing at most doubling the bytes; per row the padding byte (stuffed: 2) and
// the marker (2).  A row of b blocks codes at most ceil(1660 b / 8) <= 207.5 b + 1 bytes with its padding, stuffed
// <= 415 b + 2, plus 2 for RST.  So 631 + 415 B + 4 R.
inline unsigned long long jpeg_bound(const JpegShape &s) {
	return 631ull + 415ull * s.blocks + 4ull * (unsigned long long)s.mcuy;
}

// The 629 bytes before the entropy-coded data (include/hmrm.h, step 5)
struct JpegHeader {
	uint8_t b[kJpegHeadBytes];
};

inline JpegHeader jpeg_header(const JpegShape &s, int quality) {
	JpegHeader h;
	uint8_t *p = h.b;
	auto put = [&p](std::initializer_list<int> v) {
		for (int x : v) *p++ = (uint8_t)x;
	};
	put({0xFF, 0xD8, 0xFF, 0xE0, 0x00, 0x10, 'J', 'F', 'I', 'F', 0x00, 0x01, 0x01, 0x00, 0x00, 0x01, 0x00, 0x01, 0x00,
	     0x00});
	for (int t = 0; t < 2; ++t) {
		put({0xFF, 0xDB, 0x00, 0x43, t});
		for (int k = 0; k < 64; ++k)
			*p++ = (uint8_t)jpeg_quant_entry(t ? kJpegChromaQuant[kJpegZigzag[k]] : kJpegLumaQuant[kJpegZigzag[k]],
			                                 quality);
	}
	const int samp = s.s420 ? 0x22 : 0x11;
	put({0xFF, 0xC0, 0x00, 0x11, 0x08, s.H >> 8, s.H & 255, s.W >> 8, s.W & 255, 3, 1, samp, 0, 2, 0x11, 1, 3, 0x11, 1});
	const uint8_t *bits[4] = {kJpegDcLumaBits, kJpegAcLumaBits, kJpegDcChromaBits, kJpegAcChromaBits};
	const uint8_t *vals[4] = {kJpegDcVals, kJpegAcLumaVals, kJpegDcVals, kJpegAcChromaVals};
	const int nvals[4] = {12, 162, 12, 162}, cls[4] = {0x00, 0x10, 0x01, 0x11};
	for (int k = 0; k < 4; ++k) {
		const int len = 19 + nvals[k];
		put({0xFF, 0xC4, len >> 8, len & 255, cls[k]});
		std::memcpy(p, bits[k], 16);
		p += 16;
		std::memcpy(p, vals[k], (size_t)nvals[k]);
		p += nvals[k];
	}
	put({0xFF, 0xDD, 0x00, 0x04, s.mcux >> 8, s.mcux & 255});
	put({0xFF, 0xDA, 0x00, 0x0C, 0x03, 0x01, 0x00, 0x02, 0x11, 0x03, 0x11, 0x00, 0x3F, 0x00});
	return h;
}

// ---- jfdctint (libjpeg's "islow"): CONST_BITS 13, PASS1_BITS 2 ----
// Every intermediate is a linear form of the 64 level-shifted samples (|x| <= 128) plus pass 1's rounding; the largest
// one is below 2^23.4 in pass 1 and 2^28.4 in pass 2 (tests/test_jpeg_model.py computes both), so 32 bits suffice.
__device__ __forceinline__ void jpeg_fdct8(const int (&v)[8], int (&o)[8], bool pass1) {
	const int t0 = v[0] + v[7], t7 = v[0] - v[7], t1 = v[1] + v[6], t6 = v[1] - v[6];
	const int t2 = v[2] + v[5], t5 = v[2] - v[5], t3 = v[3] + v[4], t4 = v[3] - v[4];
	const int t10 = t0 + t3, t13 = t0 - t3, t11 = t1 + t2, t12 = t1 - t2;
	const int sh = pass1 ? 11 : 15;
	const int rnd = 1 << (sh - 1);
	if (pass1) {
		o[0] = (t10 + t11) * 4;
		o[4] = (t10 - t11) * 4;
	}
	else {
		o[0] = (t10 + t11 + 2) >> 2;
		o[4] = (t10 - t11 + 2) >> 2;
	}
	const int z1 = (t12 + t13) * 4433;
	o[2] = (z1 + t13 * 6270 + rnd) >> sh;
	o[6] = (z1 - t12 * 15137 + rnd) >> sh;
	const int z5 = (t4 + t6 + t5 + t7) * 9633;
	const int a4 = t4 * 2446, a5 = t5 * 16819, a6 = t6 * 25172, a7 = t7 * 12299;
	const int y1 = (t4 + t7) * -7373, y2 = (t5 + t6) * -20995;
	const int y3 = (t4 + t6) * -16069 + z5, y4 = (t5 + t7) * -3196 + z5;
	o[7] = (a4 + y1 + y3 + rnd) >> sh;
	o[5] = (a5 + y2 + y4 + rnd) >> sh;
	o[3] = (a6 + y2 + y3 + rnd) >> sh;
	o[1] = (a7 + y1 + y4 + rnd) >> sh;
}

// number of significant bits of |v| (JPEG's SSSS)
__device__ __forceinline__ int jpeg_nbits(int v) { return v ? 32 - __clz(v < 0 ? -v : v) : 0; }

// the (len << 16 | code) bits of the AC codes a block's zig-zag positions 8l .. 8l + 7 take, l = lane & 7; `mask` has
// bit k set for every nonzero AC coefficient k >= 1 of the block.  The lane holding the last nonzero one (lane 0 when
// there is none) also codes EOB, unless that coefficient is position 63.
template <bool EMIT, class Put>
__device__ __forceinline__ int jpeg_ac_codes(const int (&c)[8], int l, unsigned long long mask, const uint32_t *ac,
                                             Put &&put) {
	int bits = 0;
	#pragma unroll
	for (int j = 0; j < 8; ++j) {
		const int k = 8 * l + j;
		if (!((mask >> k) & 1ull)) continue;
		const unsigned long long below = mask & ((1ull << k) - 1ull);
		const int prev = below ? 63 - __clzll((long long)below) : 0;
		int run = k - prev - 1;
		for (; run > 15; run -= 16) {
			const uint32_t e = ac[0xF0];
			bits += (int)(e >> 16);
			if (EMIT) put(e & 0xFFFFu, (int)(e >> 16));
		}
		const int v = c[j], s = jpeg_nbits(v);
		const uint32_t e = ac[(run << 4) | s];
		bits += (int)(e >> 16) + s;
		if (EMIT) {
			put(e & 0xFFFFu, (int)(e >> 16));
			put((uint32_t)(v < 0 ? v - 1 : v) & ((1u << s) - 1u), s);
		}
	}
	const int last = mask ? 63 - __clzll((long long)mask) : 0;
	if (last < 63 && (last >> 3) == l) {
		const uint32_t e = ac[0];
		bits += (int)(e >> 16);
		if (EMIT) put(e & 0xFFFFu, (int)(e >> 16));
	}
	return bits;
}

// bit mask of the nonzero AC coefficients of a block whose zig-zag positions 8l .. 8l + 7 this lane holds; the 8
// lanes of a block are aligned groups of 8 in the warp
__device__ __forceinline__ unsigned long long jpeg_ac_mask(const int (&c)[8], int l) {
	unsigned m = 0u;
	#pragma unroll
	for (int j = 0; j < 8; ++j) m |= (c[j] != 0 ? 1u : 0u) << j;
	unsigned long long mask = (unsigned long long)m << (8 * l);
	#pragma unroll
	for (int o = 1; o < 8; o <<= 1) mask |= __shfl_xor_sync(0xffffffffu, mask, o);
	return mask & ~1ull;
}

__device__ __forceinline__ void jpeg_unpack(const uint4 w, int (&c)[8]) {
	const uint32_t u[4] = {w.x, w.y, w.z, w.w};
	#pragma unroll
	for (int j = 0; j < 8; ++j) c[j] = (int)(int16_t)(uint16_t)(u[j >> 1] >> (16 * (j & 1)));
}

template <int C>
__device__ __forceinline__ void jpeg_pixel(const uint8_t *__restrict__ img, int W, int x, int y, int &r, int &g,
                                           int &b) {
	const size_t i = (size_t)y * (size_t)W + (size_t)x;
	if (C == 4) {
		const uint32_t p = __ldg((const uint32_t *)img + i);
		r = (int)(p & 255u);
		g = (int)((p >> 8) & 255u);
		b = (int)((p >> 16) & 255u);
	}
	else {
		r = __ldg(img + 3 * i);
		g = __ldg(img + 3 * i + 1);
		b = __ldg(img + 3 * i + 2);
	}
}

__device__ __forceinline__ int jpeg_y(int r, int g, int b) { return (19595 * r + 38470 * g + 7471 * b + 32768) >> 16; }
__device__ __forceinline__ int jpeg_cb(int r, int g, int b) {
	return (-11059 * r - 21709 * g + 32768 * b + 8421375) >> 16;
}
__device__ __forceinline__ int jpeg_cr(int r, int g, int b) {
	return (32768 * r - 27439 * g - 5329 * b + 8421375) >> 16;
}

// grid: x over strips of kTileMcus MCUs, y over MCU rows.  coef: [blocks][64] int16 in zig-zag order, blocks in coding
// order (MCU by MCU; Y0 Y1 Y2 Y3 Cb Cr or Y Cb Cr); acbits: bits of each block's AC codes, EOB included.
template <int C, bool S420>
__global__ void __launch_bounds__(kJpegBlockThreads) k6_jpeg_blocks(const uint8_t *__restrict__ img, int W, int H,
                                                                    int mcux, JpegQuant quant, int16_t *__restrict__ coef,
                                                                    uint16_t *__restrict__ acbits) {
	constexpr int kBpm = S420 ? 6 : 3;
	constexpr int kTileMcus = kJpegTileBlocks / kBpm;
	constexpr int kRows = S420 ? 16 : 8;           // pixel rows of the strip; it is 128 pixels wide
	__shared__ int16_t plane[3072];                // 4:2:0: Y [16][128], Cb [8][64], Cr [8][64]; 4:4:4: [3][8][128]
	__shared__ int work[kJpegTileBlocks][64];      // pass 1 output, natural order
	__shared__ __align__(16) int16_t zz[kJpegTileBlocks][64];
	__shared__ uint32_t recip[2][64];
	__shared__ uint16_t half[2][64];
	__shared__ uint8_t zpos[64];                   // natural index -> zig-zag position
	__shared__ uint32_t ac_codes[2][256];
	const int t = threadIdx.x;
	if (t < 128) {
		recip[t >> 6][t & 63] = quant.recip[t >> 6][t & 63];
		half[t >> 6][t & 63] = quant.half[t >> 6][t & 63];
	}
	if (t < 64) zpos[t] = kJpegCodesDev.zpos[t];
	for (int i = t; i < 512; i += blockDim.x) ac_codes[i >> 8][i & 255] = kJpegCodesDev.t[(i >> 8) ? 3 : 1][i & 255];

	const int x0 = blockIdx.x * 128, y0 = blockIdx.y * kRows;
	if (S420) {
		const int ch = (H + 1) >> 1;
		for (int i = t; i < 512; i += blockDim.x) {    // one 2x2 quad each: 4 luma samples, 1 Cb, 1 Cr
			const int qx = i & 63, qy = i >> 6;
			const int xa = min(x0 + 2 * qx, W - 1), xb = min(x0 + 2 * qx + 1, W - 1);
			const int ya = min(y0 + 2 * qy, H - 1), yb = min(y0 + 2 * qy + 1, H - 1);
			int r[4], g[4], b[4];
			jpeg_pixel<C>(img, W, xa, ya, r[0], g[0], b[0]);
			jpeg_pixel<C>(img, W, xb, ya, r[1], g[1], b[1]);
			jpeg_pixel<C>(img, W, xa, yb, r[2], g[2], b[2]);
			jpeg_pixel<C>(img, W, xb, yb, r[3], g[3], b[3]);
			#pragma unroll
			for (int k = 0; k < 4; ++k) plane[(2 * qy + (k >> 1)) * 128 + 2 * qx + (k & 1)] = (int16_t)jpeg_y(r[k], g[k], b[k]);
			// chroma rows: an odd last source row is duplicated, then the last chroma row is replicated downwards,
			// which below the frame is not the luma rows' clamp
			const int cy = min(blockIdx.y * 8 + qy, ch - 1);
			const int r0 = 2 * cy, r1 = min(2 * cy + 1, H - 1);
			if (r0 != ya || r1 != yb) {
				jpeg_pixel<C>(img, W, xa, r0, r[0], g[0], b[0]);
				jpeg_pixel<C>(img, W, xb, r0, r[1], g[1], b[1]);
				jpeg_pixel<C>(img, W, xa, r1, r[2], g[2], b[2]);
				jpeg_pixel<C>(img, W, xb, r1, r[3], g[3], b[3]);
			}
			int scb = 0, scr = 0;
			#pragma unroll
			for (int k = 0; k < 4; ++k) {
				scb += jpeg_cb(r[k], g[k], b[k]);
				scr += jpeg_cr(r[k], g[k], b[k]);
			}
			const int bias = 1 + (qx & 1);
			plane[2048 + qy * 64 + qx] = (int16_t)((scb + bias) >> 2);
			plane[2560 + qy * 64 + qx] = (int16_t)((scr + bias) >> 2);
		}
	}
	else {
		for (int i = t; i < 1024; i += blockDim.x) {
			const int px = i & 127, py = i >> 7;
			int r, g, b;
			jpeg_pixel<C>(img, W, min(x0 + px, W - 1), min(y0 + py, H - 1), r, g, b);
			plane[i] = (int16_t)jpeg_y(r, g, b);
			plane[1024 + i] = (int16_t)jpeg_cb(r, g, b);
			plane[2048 + i] = (int16_t)jpeg_cr(r, g, b);
		}
	}
	__syncthreads();

	const int blk = t >> 3, l = t & 7;
	const int m = blk / kBpm, k = blk % kBpm;
	const int comp = S420 ? (k < 4 ? 0 : k - 3) : k;
	int base, stride;
	if (S420 && k < 4) {
		base = (k >> 1) * 8 * 128 + (2 * m + (k & 1)) * 8;
		stride = 128;
	}
	else if (S420) {
		base = 2048 + (k - 4) * 512 + m * 8;
		stride = 64;
	}
	else {
		base = k * 1024 + m * 8;
		stride = 128;
	}
	{   // pass 1: row l of the block
		int v[8], o[8];
		#pragma unroll
		for (int j = 0; j < 8; ++j) v[j] = plane[base + l * stride + j] - 128;
		jpeg_fdct8(v, o, true);
		#pragma unroll
		for (int j = 0; j < 8; ++j) work[blk][l * 8 + j] = o[j];
	}
	__syncthreads();
	{   // pass 2: column l, then quantisation into zig-zag order
		int v[8], o[8];
		#pragma unroll
		for (int j = 0; j < 8; ++j) v[j] = work[blk][j * 8 + l];
		jpeg_fdct8(v, o, false);
		const int tq = comp ? 1 : 0;
		#pragma unroll
		for (int u = 0; u < 8; ++u) {
			const int n = u * 8 + l;
			const int c = o[u];
			const int q = (int)__umulhi((uint32_t)(abs(c) + half[tq][n]), recip[tq][n]);
			zz[blk][zpos[n]] = (int16_t)(c < 0 ? -q : q);
		}
	}
	__syncthreads();

	const int mx = blockIdx.x * kTileMcus + m;
	// 4:2:0 luma blocks outside ceil(W/8) x ceil(H/8) are libjpeg's dummy blocks: AC 0, DC copied from the block to the
	// left, or, in a bottom dummy row, from the last block of the MCU's row above
	int src = blk;
	bool dummy = false;
	if (S420 && k < 4) {
		const int wb = (W + 7) >> 3, hb = (H + 7) >> 3;
		const int bx = 2 * mx + (k & 1), by = 2 * blockIdx.y + (k >> 1);
		if (by >= hb) {
			dummy = true;
			src = blk - k + (2 * mx + 1 < wb ? 1 : 0);
		}
		else if (bx >= wb) {
			dummy = true;
			src = blk - 1;
		}
	}
	int c[8];
	jpeg_unpack(*(const uint4 *)&zz[blk][8 * l], c);
	if (dummy) {
		#pragma unroll
		for (int j = 0; j < 8; ++j) c[j] = 0;
		if (l == 0) c[0] = zz[src][0];
	}
	const unsigned long long mask = jpeg_ac_mask(c, l);
	int bits = jpeg_ac_codes<false>(c, l, mask, ac_codes[comp ? 1 : 0], [](uint32_t, int) {});
	#pragma unroll
	for (int o = 1; o < 8; o <<= 1) bits += __shfl_xor_sync(0xffffffffu, bits, o);
	if (mx >= mcux) return;
	const unsigned long long g = ((unsigned long long)blockIdx.y * (unsigned long long)mcux + (unsigned long long)mx) * kBpm +
	                             (unsigned long long)k;
	uint4 w;
	w.x = (uint32_t)(uint16_t)c[0] | ((uint32_t)(uint16_t)c[1] << 16);
	w.y = (uint32_t)(uint16_t)c[2] | ((uint32_t)(uint16_t)c[3] << 16);
	w.z = (uint32_t)(uint16_t)c[4] | ((uint32_t)(uint16_t)c[5] << 16);
	w.w = (uint32_t)(uint16_t)c[6] | ((uint32_t)(uint16_t)c[7] << 16);
	*(uint4 *)(coef + g * 64 + 8 * l) = w;
	if (l == 0) acbits[g] = (uint16_t)bits;
}

// MSB-first bit writer over a zeroed word array whose bytes are in stream order; words it shares with other writers are
// ORed, so any number of writers may fill one array
struct JpegBitWriter {
	uint32_t *words;
	uint32_t w;
	unsigned long long acc;     // bits from the top; the first (start & 31) are another writer's (zeros here)
	int n;
	__device__ JpegBitWriter(uint32_t *base, uint32_t start) : words(base), w(start >> 5), acc(0ull), n((int)(start & 31u)) {}
	__device__ __forceinline__ void operator()(uint32_t v, int len) {   // len <= 27
		if (len == 0) return;
		acc |= (unsigned long long)v << (64 - n - len);
		n += len;
		if (n >= 32) {
			atomicOr(words + w, __byte_perm((uint32_t)(acc >> 32), 0u, 0x0123));
			++w;
			acc <<= 32;
			n -= 32;
		}
	}
	__device__ __forceinline__ void flush() {
		if (n > 0) atomicOr(words + w, __byte_perm((uint32_t)(acc >> 32), 0u, 0x0123));
	}
};

// exclusive scan of one value per thread over the CTA; *total receives the sum
template <class T>
__device__ __forceinline__ T jpeg_cta_scan(T v, T *total) {
	__shared__ T warp_sum[33];   // exclusive prefix of each warp, then the total
	const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5, nw = (int)(blockDim.x >> 5);
	T incl = v;
	#pragma unroll
	for (int o = 1; o < 32; o <<= 1) {
		const T u = __shfl_up_sync(0xffffffffu, incl, o);
		if (lane >= o) incl += u;
	}
	__syncthreads();             // warp_sum may still be read by a previous call
	if (lane == 31) warp_sum[wid] = incl;
	__syncthreads();
	if (wid == 0) {
		const T s = lane < nw ? warp_sum[lane] : (T)0;
		T x = s;
		#pragma unroll
		for (int o = 1; o < 32; o <<= 1) {
			const T u = __shfl_up_sync(0xffffffffu, x, o);
			if (lane >= o) x += u;
		}
		warp_sum[lane] = x - s;
		if (lane == 31) warp_sum[32] = x;
	}
	__syncthreads();
	*total = warp_sum[32];
	return warp_sum[wid] + incl - v;
}

// one CTA per MCU row.  boff: scratch, bit offset of each block inside its row.  rowbits: [mcuy][row_words] bit buffers,
// stage: [mcuy][row_stride] stuffed rows with their RST marker, rowsize: bytes of each staged row.
__global__ void __launch_bounds__(kJpegRowThreads) k6_jpeg_rows(const int16_t *__restrict__ coef,
                                                               const uint16_t *__restrict__ acbits, int mcux, int bpm,
                                                               int mcuy, uint32_t *__restrict__ boff,
                                                               uint32_t *__restrict__ rowbits,
                                                               unsigned long long row_words,
                                                               uint8_t *__restrict__ stage,
                                                               unsigned long long row_stride,
                                                               unsigned long long *__restrict__ rowsize) {
	__shared__ uint32_t codes[4][256];
	__shared__ unsigned wff[32];
	const int t = threadIdx.x, row = blockIdx.x;
	for (int i = t; i < 1024; i += blockDim.x) codes[i >> 8][i & 255] = kJpegCodesDev.t[i >> 8][i & 255];
	__syncthreads();
	const int nblk = mcux * bpm;
	const int16_t *rc = coef + (unsigned long long)row * (unsigned long long)nblk * 64ull;
	const uint16_t *rac = acbits + (unsigned long long)row * (unsigned long long)nblk;
	uint32_t *rbo = boff + (unsigned long long)row * (unsigned long long)nblk;
	uint32_t *bitsbuf = rowbits + (unsigned long long)row * row_words;
	// component (0 luma, 1 chroma) and DC difference of block b of the row; each component's predictor starts at 0
	auto comp_of = [bpm](int b) {
		const int k = b % bpm;
		return bpm == 6 ? (k < 4 ? 0 : 1) : (k ? 1 : 0);
	};
	auto dc_diff = [&](int b) {
		const int k = b % bpm;
		int p = b - bpm + (bpm == 6 && k == 0 ? 3 : 0);           // the same component's block of the previous MCU
		if (bpm == 6 && k > 0 && k < 4) p = b - 1;
		return (int)rc[(size_t)b * 64] - (b >= bpm || (bpm == 6 && k > 0 && k < 4) ? (int)rc[(size_t)p * 64] : 0);
	};
	auto dc_bits = [&](int b) {
		const int s = jpeg_nbits(dc_diff(b));
		return (uint32_t)(codes[comp_of(b) ? 2 : 0][s] >> 16) + (uint32_t)s;
	};

	// block bit lengths -> offsets: each thread takes a contiguous run of blocks
	const int per = (nblk + (int)blockDim.x - 1) / (int)blockDim.x;
	const int b0 = min(t * per, nblk), b1 = min(b0 + per, nblk);
	uint32_t sum = 0;
	for (int b = b0; b < b1; ++b) sum += dc_bits(b) + rac[b];
	uint32_t total_bits;
	uint32_t off = jpeg_cta_scan<uint32_t>(sum, &total_bits);
	for (int b = b0; b < b1; ++b) {
		rbo[b] = off;
		off += dc_bits(b) + rac[b];
	}
	const uint32_t nwords = (total_bits + 31u) >> 5;
	for (uint32_t i = t; i < nwords; i += blockDim.x) bitsbuf[i] = 0u;
	__syncthreads();

	// the codes, 8 threads per block; whole groups of 8 stay in the loop for the shuffles
	const int l = t & 7, groups = (int)blockDim.x >> 3;
	for (int g0 = 0; g0 < nblk; g0 += groups) {
		const int b = g0 + (t >> 3);
		const bool live = b < nblk;
		const int bb = live ? b : nblk - 1;
		const int comp = comp_of(bb);
		int c[8];
		jpeg_unpack(*(const uint4 *)(rc + (size_t)bb * 64 + 8 * l), c);
		const unsigned long long mask = jpeg_ac_mask(c, l);
		const uint32_t *ac = codes[comp ? 3 : 1];
		int bits = jpeg_ac_codes<false>(c, l, mask, ac, [](uint32_t, int) {});
		int diff = 0, s = 0;
		uint32_t dc = 0u;
		if (l == 0) {
			diff = dc_diff(bb);
			s = jpeg_nbits(diff);
			dc = codes[comp ? 2 : 0][s];
			bits += (int)(dc >> 16) + s;
		}
		int before = bits;
		#pragma unroll
		for (int o = 1; o < 8; o <<= 1) {
			const int u = __shfl_up_sync(0xffffffffu, before, o, 8);
			if (l >= o) before += u;
		}
		if (live) {
			JpegBitWriter put(bitsbuf, rbo[bb] + (uint32_t)(before - bits));
			if (l == 0) {
				put(dc & 0xFFFFu, (int)(dc >> 16));
				put((uint32_t)(diff < 0 ? diff - 1 : diff) & ((1u << s) - 1u), s);
			}
			jpeg_ac_codes<true>(c, l, mask, ac, put);
			put.flush();
		}
	}
	__syncthreads();
	if (t == 0 && (total_bits & 7u)) {   // pad the last byte with 1-bits
		const uint32_t p = total_bits >> 3;
		uint8_t *bytes = (uint8_t *)bitsbuf;
		bytes[p] |= (uint8_t)(0xFFu >> (total_bits & 7u));
	}
	__syncthreads();

	// 0xFF stuffing, blockDim.x bytes per step
	const uint32_t nbytes = (total_bits + 7u) >> 3;
	const uint8_t *src = (const uint8_t *)bitsbuf;
	uint8_t *dst = stage + (unsigned long long)row * row_stride;
	const int lane = t & 31, wid = t >> 5, nw = (int)(blockDim.x >> 5);
	uint32_t stuffed = 0;   // 0x00 bytes inserted before this step
	for (uint32_t c0 = 0; c0 < nbytes; c0 += blockDim.x) {
		const uint32_t i = c0 + (uint32_t)t;
		const uint8_t v = i < nbytes ? src[i] : 0;
		const bool ff = i < nbytes && v == 0xFF;
		const unsigned bal = __ballot_sync(0xffffffffu, ff);
		if (lane == 0) wff[wid] = (unsigned)__popc(bal);
		__syncthreads();
		unsigned before = (unsigned)__popc(bal & ((1u << lane) - 1u)), step = 0;
		for (int w = 0; w < nw; ++w) {
			const unsigned n = wff[w];
			if (w < wid) before += n;
			step += n;
		}
		if (i < nbytes) {
			const uint32_t at = i + stuffed + before;
			dst[at] = v;
			if (ff) dst[at + 1] = 0x00;
		}
		stuffed += step;
		__syncthreads();
	}
	if (t == 0) {
		uint32_t n = nbytes + stuffed;
		if (row < mcuy - 1) {
			dst[n] = 0xFF;
			dst[n + 1] = (uint8_t)(0xD0 + (row & 7));
			n += 2;
		}
		rowsize[row] = n;
	}
}

// one CTA of 1024 threads.  offsets[0..mcuy+2]: piece 0 = the header, pieces 1..mcuy = the rows, piece mcuy + 1 = EOI;
// offsets[mcuy + 2] = file size
__global__ void __launch_bounds__(1024) k6_jpeg_finish(const unsigned long long *__restrict__ rowsize, int mcuy,
                                                       JpegHeader head, unsigned long long *__restrict__ offsets,
                                                       uint8_t *__restrict__ meta) {
	const int t = threadIdx.x, per = (mcuy + (int)blockDim.x - 1) / (int)blockDim.x;
	const int i0 = min(t * per, mcuy), i1 = min(i0 + per, mcuy);
	unsigned long long sum = 0;
	for (int i = i0; i < i1; ++i) sum += rowsize[i];
	unsigned long long total;
	unsigned long long off = kJpegHeadBytes + jpeg_cta_scan<unsigned long long>(sum, &total);
	for (int i = i0; i < i1; ++i) {
		offsets[1 + i] = off;
		off += rowsize[i];
	}
	if (t == 0) {
		offsets[0] = 0;
		offsets[mcuy + 1] = kJpegHeadBytes + total;
		offsets[mcuy + 2] = kJpegHeadBytes + total + 2;
		meta[kJpegMetaTail] = 0xFF;
		meta[kJpegMetaTail + 1] = 0xD9;
	}
	for (int i = t; i < kJpegHeadBytes; i += blockDim.x) meta[i] = head.b[i];
}

} // namespace hmrm
