// K1 — one-shot height prepass (replaces UpdateHeightmap, main/hmap.cpp:171-191).
//
//   v      = clamp((lum_r*R + lum_g*G) + lum_b*B, 0, 255)
//   height = (v / 255) * (max_height - min_height) + min_height            (:187-188)
//   surf   = height + min_height     <- what the march compares against     (:1016, hmap_c0.z = min_height)
//
// The reference keeps `height` and adds min_height again at every march step;
// K1 stores `surf` (same two roundings, done once per cell) plus the global
// maximum of surf, which bounds every terrain sample from above.
//
// 16-bit maps (hmrm_set_maps16) have one sample x per cell, used as R = G = B, and 65535 in place of 255:
//   v      = clamp((lum_r*x + lum_g*x) + lum_b*x, 0, 65535)
//   height = (v / 65535) * (max_height - min_height) + min_height
// k1_range / k1_prepass take either input through a cell reader (Rgb8Cells, Grey16Cells); k1_build16 shares k1_build's
// block body.
#ifndef HMRM_K1_PREPASS_CUH
#define HMRM_K1_PREPASS_CUH

#include "device_math.cuh"
#include "pyramid_layout.cuh"

namespace hmrm {

struct PrepassParams {
	double lum_r, lum_g, lum_b;
	double min_height;
	double span;          // fl(max_height - min_height)
};

// exact u8 / u16 -> double without the quarter-rate I2F: (2^52 + n) - 2^52
__device__ __forceinline__ double byte_to_double(uint32_t n) {
	return fsub(__hiloint2double(0x43300000, (int)n), 4503599627370496.0);
}

__device__ __forceinline__ double height_of(const PrepassParams &q, uint32_t r, uint32_t g, uint32_t b) {
	double v = fadd(fadd(fmul(q.lum_r, byte_to_double(r)), fmul(q.lum_g, byte_to_double(g))),
	                fmul(q.lum_b, byte_to_double(b)));
	if (v < 0.0) v = 0.0;
	else if (v > 255.0) v = 255.0;
	return fadd(fmul(fdiv(v, 255.0), q.span), q.min_height);
}

// the same for one 16-bit sample x (R = G = B = x) on the 0..65535 scale
__device__ __forceinline__ double height16_of(const PrepassParams &q, uint32_t x) {
	const double d = byte_to_double(x);
	double v = fadd(fadd(fmul(q.lum_r, d), fmul(q.lum_g, d)), fmul(q.lum_b, d));
	if (v < 0.0) v = 0.0;
	else if (v > 65535.0) v = 65535.0;
	return fadd(fmul(fdiv(v, 65535.0), q.span), q.min_height);
}

// cell readers: the height of cell p of the map ([h][w] row-major)
struct Rgb8Cells {
	const uint8_t *__restrict__ rgb8;          // [n][3]
	__device__ __forceinline__ double height(const PrepassParams &q, long long p) const {
		const uint8_t *px = rgb8 + 3 * p;
		return height_of(q, px[0], px[1], px[2]);
	}
};
struct Grey16Cells {
	const uint16_t *__restrict__ h16;          // [n]
	__device__ __forceinline__ double height(const PrepassParams &q, long long p) const { return height16_of(q, h16[p]); }
};

// order-preserving map double -> uint64 so that atomicMax works on FP64 values
__device__ __forceinline__ unsigned long long ordered_bits(double v) {
	const unsigned long long b = (unsigned long long)__double_as_longlong(v);
	return (b & 0x8000000000000000ULL) ? ~b : (b | 0x8000000000000000ULL);
}
__host__ __device__ inline double from_ordered_bits(unsigned long long o) {
	const unsigned long long b = (o & 0x8000000000000000ULL) ? (o & 0x7FFFFFFFFFFFFFFFULL) : ~o;
	double v;
#if defined(__CUDA_ARCH__)
	v = __longlong_as_double((long long)b);
#else
	__builtin_memcpy(&v, &b, sizeof v);
#endif
	return v;
}

// cells: Rgb8Cells | Grey16Cells over [n] cells; surf: [n] (may be NULL); heights: [n] (may be NULL, parity checks only)
template <class Cells>
__global__ void __launch_bounds__(256) k1_prepass(Cells cells, long long n, PrepassParams q,
                                                  double *__restrict__ surf, double *__restrict__ heights,
                                                  unsigned long long *__restrict__ max_surf_bits,
                                                  unsigned long long *__restrict__ min_surf_bits) {
	unsigned long long local_max = 0ULL, local_min = ~0ULL;
	const long long stride = (long long)gridDim.x * blockDim.x;
	for (long long p = (long long)blockIdx.x * blockDim.x + threadIdx.x; p < n; p += stride) {
		const double h = cells.height(q, p);
		if (heights) heights[p] = h;
		const double s = fadd(h, q.min_height);
		if (surf) surf[p] = s;
		const unsigned long long ob = ordered_bits(s);
		if (ob > local_max) local_max = ob;
		if (ob < local_min) local_min = ob;
	}
	if (max_surf_bits) {
		for (int off = 16; off > 0; off >>= 1) {
			const unsigned long long o = __shfl_xor_sync(0xFFFFFFFFu, local_max, off);
			if (o > local_max) local_max = o;
		}
		if ((threadIdx.x & 31) == 0 && local_max != 0ULL) atomicMax(max_surf_bits, local_max);
	}
	if (min_surf_bits) {
		for (int off = 16; off > 0; off >>= 1) {
			const unsigned long long o = __shfl_xor_sync(0xFFFFFFFFu, local_min, off);
			if (o < local_min) local_min = o;
		}
		if ((threadIdx.x & 31) == 0 && local_min != ~0ULL) atomicMin(min_surf_bits, local_min);
	}
}

// ---- conservative fixed-point view of the surface (used by the skip traversal) -------------
//
// Zq(v) = low 32 bits of fma(v, zq_scale, zq_offset) where zq_offset = 1.5*2^52 + c: the classic
// magic-number conversion, one DFMA instead of a quarter-rate F2I.  Zq is monotone non-decreasing
// in v (zq_scale > 0, rounding is monotone), and K1 and K2 evaluate the very same instruction, so
//     Zq(z) > Zq(surf)  =>  z > surf   (the march's test `z < surf` is false)
//     Zq(z) < Zq(surf)  =>  z < surf   (hit)
// with no error analysis; only Zq(z) == Zq(surf) needs the FP64 surf value.
#define HMRM_MAGIC 6755399441055744.0   /* 1.5 * 2^52 */

// low word of (magic + n) is n for |n| < 2^31; the high word tells whether that held
__device__ __forceinline__ bool magic_decode(double t, int &v) {
	const int hi = __double2hiint(t);
	v = __double2loint(t);
	return (hi == 0x43380000 && v >= 0) || (hi == 0x4337FFFF && v < 0);
}

__device__ __forceinline__ int zq_of(double z, double zq_scale, double zq_offset) {
	int v;
	const double t = __fma_rn(z, zq_scale, zq_offset);
	if (magic_decode(t, v)) return v;
	return (t > HMRM_MAGIC) ? INT_MAX : INT_MIN;   // far above / far below every surface value (NaN: below)
}

// Zq clamped to 16 bits.  Clamping keeps Zq monotone (weakly), so the two implications above survive as long as
// BOTH sides are clamped: values beyond the range simply tie and fall back to the FP64 comparison.  That makes any
// choice of scale/offset safe — the range is only estimated from a sample of the map (k1_range).
__device__ __forceinline__ int zq16(double z, double zq_scale, double zq_offset) {
	return min(max(zq_of(z, zq_scale, zq_offset), 0), 65535);
}

// min / max of surf over every `row_stride`-th row (order-preserving bit patterns, atomics)
template <class Cells>
__global__ void __launch_bounds__(256) k1_range(Cells cells, int w, int h, int row_stride,
                                                PrepassParams q, unsigned long long *__restrict__ max_bits,
                                                unsigned long long *__restrict__ min_bits) {
	unsigned long long local_max = 0ULL, local_min = ~0ULL;
	const int rows = (h + row_stride - 1) / row_stride;
	const long long n = (long long)rows * w;
	const long long stride = (long long)gridDim.x * blockDim.x;
	for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
		const int x = (int)(i % w);
		const long long y = (i / w) * row_stride;
		const unsigned long long ob = ordered_bits(fadd(cells.height(q, y * w + x), q.min_height));
		if (ob > local_max) local_max = ob;
		if (ob < local_min) local_min = ob;
	}
	for (int off = 16; off > 0; off >>= 1) {
		const unsigned long long a = __shfl_xor_sync(0xFFFFFFFFu, local_max, off);
		const unsigned long long b = __shfl_xor_sync(0xFFFFFFFFu, local_min, off);
		if (a > local_max) local_max = a;
		if (b < local_min) local_min = b;
	}
	if ((threadIdx.x & 31) == 0) {
		if (local_max != 0ULL) atomicMax(max_bits, local_max);
		if (local_min != ~0ULL) atomicMin(min_bits, local_min);
	}
}

// Fused build: one thread owns a 4x4 block of cells.  Reads the map once, writes surf (FP64), level 0 (Zq16 per cell)
// and the plain max-mip levels 1 and 2 of that block.  HBM-bound: 3 B (RGB8) or 2 B (16-bit) in, 8 + 2 + 0.5 + 0.125 B
// out per cell.  `Rows` turns four cells of one row into their surf and Zq16 values (Rgb8Rows, Grey16Rows).
template <class Rows>
__device__ __forceinline__ void k1_build_blocks(const Rows &rows, int w, int h, double *__restrict__ surf,
                                                uint16_t *__restrict__ lv0, int layout, unsigned pitch0,
                                                uint16_t *__restrict__ plain1, int w1, uint16_t *__restrict__ plain2,
                                                int w2) {
	const int tiles_x = (w + 3) / 4, tiles_y = (h + 3) / 4;
	const long long n_tiles = (long long)tiles_x * tiles_y;
	const long long stride = (long long)gridDim.x * blockDim.x;
	const bool vec = (w & 3) == 0;     // rows are 4-byte aligned in rgb8, 8-byte in the 16-bit plane and lv0, 32-byte in surf
	for (long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x; t < n_tiles; t += stride) {
		const int bx = (int)(t % tiles_x), by = (int)(t / tiles_x);
		const int x0 = bx * 4, y0 = by * 4;
		int m1[2][2] = {{0, 0}, {0, 0}};
		// tiled layouts: this thread's 4x4 cells are one 32-byte sector of level 0 (pyramid_layout.cuh)
		const bool sector_store = vec && layout != kLayoutRowMajor;
		uint2 zrow[4] = {{0u, 0u}, {0u, 0u}, {0u, 0u}, {0u, 0u}};
#pragma unroll
		for (int j = 0; j < 4; ++j) {
			const int y = y0 + j;
			if (y >= h) break;
			const size_t row = (size_t)y * (size_t)w + (size_t)x0;
			int valid = min(4, w - x0);
			double s[4];
			int zq[4];
			rows.load(row, valid, vec, s, zq);
#pragma unroll
			for (int i = 0; i < 4; ++i) {
				if (i < valid) m1[j >> 1][i >> 1] = max(m1[j >> 1][i >> 1], zq[i]);
			}
			if (vec) {
				double2 *sp = (double2 *)(surf + row);
				sp[0] = make_double2(s[0], s[1]);
				sp[1] = make_double2(s[2], s[3]);
				const uint2 packed = make_uint2((unsigned)zq[0] | ((unsigned)zq[1] << 16), (unsigned)zq[2] | ((unsigned)zq[3] << 16));
				if (sector_store) zrow[j] = packed;
				else *(uint2 *)(lv0 + row) = packed;
			}
			else {
				for (int i = 0; i < valid; ++i) {
					surf[row + i] = s[i];
					lv0[pyr_index_rt(layout, (unsigned)(x0 + i), (unsigned)y, pitch0)] = (uint16_t)zq[i];
				}
			}
		}
		if (sector_store) {
			uint4 *sp = (uint4 *)(lv0 + pyr_index_rt(layout, (unsigned)x0, (unsigned)y0, pitch0));
			sp[0] = make_uint4(zrow[0].x, zrow[0].y, zrow[1].x, zrow[1].y);
			sp[1] = make_uint4(zrow[2].x, zrow[2].y, zrow[3].x, zrow[3].y);
		}
		// plain level 1: 2x2 texels of this block (those that exist), level 2: one texel
		const int h1 = (h + 1) / 2;
		int m2 = 0;
		for (int j = 0; j < 2; ++j) {
			for (int i = 0; i < 2; ++i) {
				const int tx = bx * 2 + i, ty = by * 2 + j;
				if (tx < w1 && ty < h1) plain1[(size_t)ty * w1 + tx] = (uint16_t)m1[j][i];
				m2 = max(m2, m1[j][i]);
			}
		}
		if (plain2) plain2[(size_t)by * w2 + bx] = (uint16_t)m2;
	}
}

// RGB8 rows: three 4-byte words per row when w % 4 == 0, else single cells (clamped to the last valid one)
struct Rgb8Rows {
	const uint8_t *__restrict__ rgb8;
	PrepassParams q;
	double zq_scale, zq_offset;
	const double *s_grey;
	const unsigned short *z_grey;
	__device__ __forceinline__ void load(size_t row, int valid, bool vec, double s[4], int zq[4]) const {
		uint32_t r[4], g[4], b[4];
		if (vec) {
			const uint32_t *p = (const uint32_t *)(rgb8 + 3 * row);
			const uint32_t a0 = __ldg(p), a1 = __ldg(p + 1), a2 = __ldg(p + 2);
			r[0] = a0 & 255u; g[0] = (a0 >> 8) & 255u; b[0] = (a0 >> 16) & 255u;
			r[1] = a0 >> 24; g[1] = a1 & 255u; b[1] = (a1 >> 8) & 255u;
			r[2] = (a1 >> 16) & 255u; g[2] = a1 >> 24; b[2] = a2 & 255u;
			r[3] = (a2 >> 8) & 255u; g[3] = (a2 >> 16) & 255u; b[3] = a2 >> 24;
		}
		else {
			for (int i = 0; i < 4; ++i) {
				const bool in = i < valid;
				const uint8_t *p = rgb8 + 3 * (row + (in ? i : 0));
				r[i] = p[0]; g[i] = p[1]; b[i] = p[2];
			}
		}
		const bool grey = r[0] == g[0] && g[0] == b[0] && r[1] == g[1] && g[1] == b[1] &&
		                  r[2] == g[2] && g[2] == b[2] && r[3] == g[3] && g[3] == b[3];
		if (grey) {
#pragma unroll
			for (int i = 0; i < 4; ++i) {
				s[i] = s_grey[r[i]];
				zq[i] = (int)z_grey[r[i]];
			}
		}
		else {
#pragma unroll
			for (int i = 0; i < 4; ++i) {
				s[i] = fadd(height_of(q, r[i], g[i], b[i]), q.min_height);
				zq[i] = zq16(s[i], zq_scale, zq_offset);
			}
		}
	}
};

__global__ void __launch_bounds__(256) k1_build(const uint8_t *__restrict__ rgb8, int w, int h, PrepassParams q,
                                                double zq_scale, double zq_offset, double *__restrict__ surf,
                                                uint16_t *__restrict__ lv0, int layout, unsigned pitch0,
                                                uint16_t *__restrict__ plain1, int w1,
                                                uint16_t *__restrict__ plain2, int w2) {
	// Grey cells (R == G == B: every greyscale image after stb's channel replication, vendor/stb_image.h:1758) take
	// their height from a 256-entry table built by the same expressions: bit-identical, and it removes the IEEE divide
	// and ~60 other instructions per cell, which is what bounds this kernel (ncu: issue-active 66 %, DRAM 62 %).
	__shared__ double s_grey[256];
	__shared__ unsigned short z_grey[256];
	for (int v = threadIdx.x; v < 256; v += blockDim.x) {
		const double sv = fadd(height_of(q, (uint32_t)v, (uint32_t)v, (uint32_t)v), q.min_height);
		s_grey[v] = sv;
		z_grey[v] = (unsigned short)zq16(sv, zq_scale, zq_offset);
	}
	__syncthreads();
	const Rgb8Rows rows = {rgb8, q, zq_scale, zq_offset, s_grey, z_grey};
	k1_build_blocks(rows, w, h, surf, lv0, layout, pitch0, plain1, w1, plain2, w2);
}

// ---- 16-bit maps ------------------------------------------------------------------------------------------
//
// Every 16-bit cell is grey, so the height is a function of the sample alone; but a 65536-entry table of surf and Zq16
// does not fit shared memory, and gathering from it in L2 measured slower than the arithmetic: 1.10 ms (two tables,
// 8 + 2 B) and 1.12 ms (one 16 B table) against 0.78 ms for the divide per cell, at 16384^2
// (profiles/r06_k1_16_table_variants.txt).
// 16-bit rows: one 8-byte word per row when w % 4 == 0, else single samples (clamped to the last valid one)
struct Grey16Rows {
	const uint16_t *__restrict__ h16;
	PrepassParams q;
	double zq_scale, zq_offset;
	__device__ __forceinline__ void load(size_t row, int valid, bool vec, double s[4], int zq[4]) const {
		uint32_t x[4];
		if (vec) {
			const uint2 a = __ldg((const uint2 *)(h16 + row));
			x[0] = a.x & 0xFFFFu; x[1] = a.x >> 16; x[2] = a.y & 0xFFFFu; x[3] = a.y >> 16;
		}
		else {
#pragma unroll
			for (int i = 0; i < 4; ++i) x[i] = __ldg(h16 + row + (i < valid ? i : 0));
		}
#pragma unroll
		for (int i = 0; i < 4; ++i) {
			s[i] = fadd(height16_of(q, x[i]), q.min_height);
			zq[i] = zq16(s[i], zq_scale, zq_offset);
		}
	}
};

__global__ void __launch_bounds__(256) k1_build16(const uint16_t *__restrict__ h16, int w, int h, PrepassParams q,
                                                  double zq_scale, double zq_offset, double *__restrict__ surf,
                                                  uint16_t *__restrict__ lv0, int layout, unsigned pitch0,
                                                  uint16_t *__restrict__ plain1, int w1,
                                                  uint16_t *__restrict__ plain2, int w2) {
	const Grey16Rows rows = {h16, q, zq_scale, zq_offset};
	k1_build_blocks(rows, w, h, surf, lv0, layout, pitch0, plain1, w1, plain2, w2);
}

// q0[p] = Zq(surf[p]); flags an error if a value does not fit 16 bits (cannot happen with the host's scale)
__global__ void __launch_bounds__(256) k1_quantise(const double *__restrict__ surf, long long n, double zq_scale,
                                                   double zq_offset, uint16_t *__restrict__ q0,
                                                   unsigned int *__restrict__ error_flag) {
	const long long stride = (long long)gridDim.x * blockDim.x;
	for (long long p = (long long)blockIdx.x * blockDim.x + threadIdx.x; p < n; p += stride) {
		(void)error_flag;
		q0[p] = (uint16_t)zq16(surf[p], zq_scale, zq_offset);
	}
}

// ---- plain max-mip levels >= 3 in ONE launch --------------------------------------------------------------
//
// Level l texel (X, Y) = max of level l-1 texels (2X, 2Y) .. (2X+1, 2Y+1), clipped at the edges.  A CTA owns a
// 128 x 128 region of plain level 2 and reduces it in shared memory to its 64 x 64 texels of level 3, 32 x 32 of
// level 4, ... 1 texel of level 9 (region edges are multiples of 2^7, so the texels of those levels nest inside
// regions).  The last CTA to finish (global counter) reduces the few remaining levels (>= 10, at most 64 x 64
// texels of input) on its own.  Heights are unsigned, so missing texels are 0 and every reduction is a plain max.
struct MipJob {
	int n_levels;                 // levels 0 .. n_levels-1 exist
	int w[16], h[16];
	unsigned plain_off[16];       // element offset of plain level l inside the scratch (l >= 1)
};

__global__ void __launch_bounds__(256) k1_mip_upper(uint16_t *__restrict__ plain, MipJob job, unsigned int *done_counter) {
	__shared__ unsigned short s_a[64 * 64];
	__shared__ unsigned short s_b[32 * 32];
	__shared__ bool s_last;
	const int w2 = job.w[2], h2 = job.h[2];
	const int regions_x = (w2 + 127) / 128;
	const int rx = (int)(blockIdx.x % (unsigned)regions_x), ry = (int)(blockIdx.x / (unsigned)regions_x);
	const uint16_t *p2 = plain + job.plain_off[2];
	// level 3 of this region from plain level 2 (global)
	for (int t = threadIdx.x; t < 64 * 64; t += blockDim.x) {
		const int lx = t & 63, ly = t >> 6;
		const int x0 = rx * 128 + 2 * lx, y0 = ry * 128 + 2 * ly;
		unsigned m = 0u;
		if (y0 < h2) {
			if (x0 < w2) m = __ldg(p2 + (size_t)y0 * w2 + x0);
			if (x0 + 1 < w2) m = max(m, (unsigned)__ldg(p2 + (size_t)y0 * w2 + x0 + 1));
		}
		if (y0 + 1 < h2) {
			if (x0 < w2) m = max(m, (unsigned)__ldg(p2 + (size_t)(y0 + 1) * w2 + x0));
			if (x0 + 1 < w2) m = max(m, (unsigned)__ldg(p2 + (size_t)(y0 + 1) * w2 + x0 + 1));
		}
		s_a[t] = (unsigned short)m;
		const int X = rx * 64 + lx, Y = ry * 64 + ly;
		if (job.n_levels > 3 && X < job.w[3] && Y < job.h[3]) plain[job.plain_off[3] + (size_t)Y * job.w[3] + X] = (uint16_t)m;
	}
	__syncthreads();
	// levels 4 .. 9 inside shared memory, ping-pong between the two arrays
	unsigned short *src = s_a, *dst = s_b;
	int side = 64;
	for (int l = 4; l <= 9 && l < job.n_levels; ++l) {
		const int half = side >> 1;
		for (int t = threadIdx.x; t < half * half; t += blockDim.x) {
			const int lx = t % half, ly = t / half;
			const unsigned a = src[(2 * ly) * side + 2 * lx], b = src[(2 * ly) * side + 2 * lx + 1];
			const unsigned c = src[(2 * ly + 1) * side + 2 * lx], d = src[(2 * ly + 1) * side + 2 * lx + 1];
			const unsigned m = max(max(a, b), max(c, d));
			dst[ly * half + lx] = (unsigned short)m;
			const int X = rx * half + lx, Y = ry * half + ly;
			if (X < job.w[l] && Y < job.h[l]) plain[job.plain_off[l] + (size_t)Y * job.w[l] + X] = (uint16_t)m;
		}
		__syncthreads();
		unsigned short *tmp = src; src = dst; dst = tmp;
		side = half;
	}
	if (job.n_levels <= 10) return;
	// the remaining levels: by the last CTA to arrive
	__threadfence();
	__syncthreads();
	if (threadIdx.x == 0) s_last = atomicAdd(done_counter, 1u) == gridDim.x - 1u;
	__syncthreads();
	if (!s_last) return;
	__threadfence();
	for (int l = 10; l < job.n_levels; ++l) {
		const int sw = job.w[l - 1], sh = job.h[l - 1], dw = job.w[l], dh = job.h[l];
		const uint16_t *below = plain + job.plain_off[l - 1];
		for (int t = threadIdx.x; t < dw * dh; t += blockDim.x) {
			const int x = t % dw, y = t / dw;
			const int x0 = 2 * x, y0 = 2 * y;
			const int x1 = (x0 + 1 < sw) ? x0 + 1 : x0, y1 = (y0 + 1 < sh) ? y0 + 1 : y0;
			const unsigned a = __ldcg(below + (size_t)y0 * sw + x0), b = __ldcg(below + (size_t)y0 * sw + x1);
			const unsigned c = __ldcg(below + (size_t)y1 * sw + x0), d = __ldcg(below + (size_t)y1 * sw + x1);
			plain[job.plain_off[l] + t] = (uint16_t)max(max(a, b), max(c, d));
		}
		__threadfence();
		__syncthreads();
	}
	if (threadIdx.x == 0) *done_counter = 0u;
}

// ---- 3x3 dilation of every level >= 1 in ONE launch, written in the traversal's layout ---------------------
//
// dst(l)[y][x] = max of plain(l) over the 3x3 neighbourhood (clipped): a sample that clears dst clears the block it
// is in AND the eight blocks around it, so a jump may run on into the neighbouring blocks instead of stopping at an
// edge.
struct DilateJob {
	int n_levels;
	int layout;
	int w[16], h[16];
	unsigned plain_off[16];       // source: plain level l in the scratch (row-major)
	unsigned dst_off[16];         // destination: level l in the pyramid the traversal reads
	unsigned dst_pitch[16];
	unsigned long long first_item[17];   // work items of level l are [first_item[l], first_item[l+1]); level 0 has none
};

__global__ void __launch_bounds__(256) k1_dilate_levels(const uint16_t *__restrict__ plain, uint16_t *__restrict__ pyr, DilateJob job) {
	// Work item = a 4 x 4 block of outputs: six input rows (two of halo), each one 8-byte load plus its two horizontal
	// neighbours, give the sixteen 3x3 maxima; in the tiled layouts the block is one 32-byte sector of the destination.
	const unsigned long long total = job.first_item[job.n_levels];
	const unsigned long long stride = (unsigned long long)gridDim.x * blockDim.x;
	for (unsigned long long item = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x; item < total; item += stride) {
		int l = 1;
		while (l + 1 < job.n_levels && item >= job.first_item[l + 1]) l += 1;
		const int w = job.w[l], h = job.h[l];
		const unsigned wq = (unsigned)(w + 3) / 4u;
		const unsigned t = (unsigned)(item - job.first_item[l]);          // < 2^26 items per level
		const int xq = (int)(t % wq), yq = (int)(t / wq);
		const int x = xq * 4, y = yq * 4;
		const uint16_t *src = plain + job.plain_off[l];
		const bool vec = (w & 3) == 0;
		// All loads are issued unconditionally from clamped addresses and masked afterwards: with a branch per row the
		// six rows were fetched one after the other (12 bytes in flight per thread, 1.8 TB/s); this way the eighteen
		// loads of a block are independent.
		unsigned hmax[6][4];           // per input row y-1 .. y+4: horizontal 3-max of the four columns
		uint2 vrow[6];
		unsigned lft[6], rgt[6];
		const int xl = max(x - 1, 0), xr = min(x + 4, w - 1);
#pragma unroll
		for (int r = 0; r < 6; ++r) {
			const int yy = min(max(y - 1 + r, 0), h - 1);
			const uint16_t *row = src + (size_t)yy * w;
			if (vec) vrow[r] = __ldg((const uint2 *)(row + x));
			else {
				const unsigned c0 = __ldg(row + x), c1 = __ldg(row + min(x + 1, w - 1));
				const unsigned c2 = __ldg(row + min(x + 2, w - 1)), c3 = __ldg(row + min(x + 3, w - 1));
				vrow[r] = make_uint2(c0 | (c1 << 16), c2 | (c3 << 16));
			}
			lft[r] = __ldg(row + xl);
			rgt[r] = __ldg(row + xr);
		}
#pragma unroll
		for (int r = 0; r < 6; ++r) {
			const int yy = y - 1 + r;
			const bool row_in = yy >= 0 && yy < h;
			unsigned c0 = vrow[r].x & 0xFFFFu, c1 = vrow[r].x >> 16, c2 = vrow[r].y & 0xFFFFu, c3 = vrow[r].y >> 16;
			unsigned l_ = lft[r], r_ = rgt[r];
			// texels outside the level count as 0 (heights are unsigned)
			if (!row_in) c0 = c1 = c2 = c3 = l_ = r_ = 0u;
			if (x + 1 >= w) c1 = 0u;
			if (x + 2 >= w) c2 = 0u;
			if (x + 3 >= w) c3 = 0u;
			if (x == 0) l_ = 0u;
			if (x + 4 >= w) r_ = 0u;
			hmax[r][0] = max(l_, max(c0, c1));
			hmax[r][1] = max(c0, max(c1, c2));
			hmax[r][2] = max(c1, max(c2, c3));
			hmax[r][3] = max(c2, max(c3, r_));
		}
		uint16_t *dst = pyr + job.dst_off[l];
		uint2 rows[4];
#pragma unroll
		for (int r = 0; r < 4; ++r) {
			const unsigned o0 = max(hmax[r][0], max(hmax[r + 1][0], hmax[r + 2][0]));
			const unsigned o1 = max(hmax[r][1], max(hmax[r + 1][1], hmax[r + 2][1]));
			const unsigned o2 = max(hmax[r][2], max(hmax[r + 1][2], hmax[r + 2][2]));
			const unsigned o3 = max(hmax[r][3], max(hmax[r + 1][3], hmax[r + 2][3]));
			rows[r] = make_uint2(o0 | (o1 << 16), o2 | (o3 << 16));
		}
		if (job.layout != kLayoutRowMajor) {
			// one sector: rows of the block are consecutive (the level's allocation is padded to whole sectors)
			uint4 *sp = (uint4 *)(dst + pyr_index_rt(job.layout, (unsigned)x, (unsigned)y, job.dst_pitch[l]));
			sp[0] = make_uint4(rows[0].x, rows[0].y, rows[1].x, rows[1].y);
			sp[1] = make_uint4(rows[2].x, rows[2].y, rows[3].x, rows[3].y);
		}
		else {
#pragma unroll
			for (int r = 0; r < 4; ++r) {
				if (y + r >= h) break;
				uint16_t *d = dst + (size_t)(y + r) * w + x;
				if (vec) *(uint2 *)d = rows[r];
				else {
					d[0] = (uint16_t)(rows[r].x & 0xFFFFu);
					if (x + 1 < w) d[1] = (uint16_t)(rows[r].x >> 16);
					if (x + 2 < w) d[2] = (uint16_t)(rows[r].y & 0xFFFFu);
					if (x + 3 < w) d[3] = (uint16_t)(rows[r].y >> 16);
				}
			}
		}
	}
}

} // namespace hmrm

#endif
