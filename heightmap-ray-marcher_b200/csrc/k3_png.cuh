// K3: PNG encoding on the device (hmrm_render_png_async, hmrm_encode_png).
//
// A frame [H][W][C] (C = 4: colour type 6, C = 3: colour type 2; 8 bit, no interlace) becomes a complete PNG file in
// four launches, all on one stream:
//   k3_png_filter   one CTA per row: the PNG filter (None / Sub / Up / Average / Paeth) with the smallest sum of
//                   |signed residual| (the PNG specification's heuristic), written with its filter byte to the filtered
//                   stream (H * (W*C + 1) bytes);
//   k3_png_deflate  one warp per kPngSeg-byte segment of the filtered stream: greedy LZ77 over three candidate distances
//                   (1, C, and W*C + 1 = the same byte one row up, while that is <= 32768), coded as one fixed-Huffman
//                   block closed by the sync-flush idiom (EOB, empty stored block), or as one stored block when that is
//                   not larger.  Either way the segment ends byte-aligned, so segments concatenate as they are.  Each
//                   segment is its own IDAT chunk, CRC-32 included, staged at a fixed stride; the first one carries the
//                   zlib header 78 01.  The warp also sums the segment's Adler-32 partials;
//   k3_png_finish   one CTA: exclusive scan of the chunk sizes, Adler-32 of the whole stream from the partials, the
//                   constant signature / IHDR and the last IDAT (final empty fixed block 03 00 + Adler-32) + IEND;
//   k3_png_gather   output-driven: each thread assembles one aligned 16-byte word of the file (binary search of the
//                   piece offsets) and stores it, so the stores stay aligned and coalesced even when the destination is
//                   pinned host memory written over PCIe; it also stores the file size.  K6 (JPEG) writes its files
//                   with it too: any file made of a head piece, pieces at a fixed stride and a tail piece.
// A segment may match back across its start (never before byte 0 of the stream) but never past its end, and a match is
// at most 258 bytes: the block decodes with any inflate.
#pragma once

#include <cstdint>

namespace hmrm {

constexpr int kPngSeg = 4096;                      // bytes of the filtered stream per segment (one IDAT chunk each)
constexpr int kPngStageStride = kPngSeg + 64;      // staging bytes per segment: chunk head 8, zlib 2, stored 5, CRC 4
constexpr int kPngDeflateWarps = 4;
constexpr int kPngMaskWords = kPngSeg / 32 + 4;   // + zero words read past the segment's end
constexpr int kPngHeadBytes = 33;                  // signature + IHDR chunk
constexpr int kPngTailBytes = 30;                  // last IDAT chunk (6 data bytes) + IEND chunk
constexpr int kPngMetaTail = 64;                   // offset of the tail piece inside the meta buffer
constexpr int kPngMetaBytes = 256;

struct PngSegInfo {
	uint32_t chunk_bytes;       // length + type + data + CRC
	uint32_t adler_a;           // sum of the segment's bytes mod 65521
	uint64_t adler_b;           // sum of (n - j) * byte_j mod 65521
};

__device__ __forceinline__ unsigned png_absres(int v) {
	const unsigned r = (unsigned)v & 255u;
	return r < 128u ? r : 256u - r;
}

__device__ __forceinline__ int png_paeth(int a, int b, int c) {
	const int p = a + b - c;
	const int pa = abs(p - a), pb = abs(p - b), pc = abs(p - c);
	if (pa <= pb && pa <= pc) return a;
	if (pb <= pc) return b;
	return c;
}

__device__ __forceinline__ int png_residual(int type, int x, int a, int b, int c) {
	switch (type) {
	case 1: return x - a;
	case 2: return x - b;
	case 3: return x - ((a + b) >> 1);
	case 4: return x - png_paeth(a, b, c);
	default: return x;
	}
}

// one CTA per image row
__global__ void __launch_bounds__(256) k3_png_filter(const uint8_t *__restrict__ img, int row_bytes, int bpp,
                                                     uint8_t *__restrict__ filt) {
	const int y = blockIdx.x;
	const uint8_t *cur = img + (size_t)y * (size_t)row_bytes;
	const uint8_t *prv = y > 0 ? cur - row_bytes : NULL;
	unsigned s[5] = {0u, 0u, 0u, 0u, 0u};
	for (int i = threadIdx.x; i < row_bytes; i += blockDim.x) {
		const int x = cur[i], a = i >= bpp ? cur[i - bpp] : 0, b = prv ? prv[i] : 0, c = (prv && i >= bpp) ? prv[i - bpp] : 0;
		s[0] += png_absres(x);
		s[1] += png_absres(x - a);
		s[2] += png_absres(x - b);
		s[3] += png_absres(x - ((a + b) >> 1));
		s[4] += png_absres(x - png_paeth(a, b, c));
	}
	__shared__ unsigned part[8][5];
	__shared__ int best;
	for (int k = 0; k < 5; ++k) {
		unsigned v = s[k];
		for (int o = 16; o > 0; o >>= 1) v += __shfl_down_sync(0xffffffffu, v, o);
		if ((threadIdx.x & 31) == 0) part[threadIdx.x >> 5][k] = v;
	}
	__syncthreads();
	if (threadIdx.x == 0) {
		unsigned tot[5] = {0u, 0u, 0u, 0u, 0u};
		for (int w = 0; w < (int)(blockDim.x >> 5); ++w)
			for (int k = 0; k < 5; ++k) tot[k] += part[w][k];
		int t = 0;
		for (int k = 1; k < 5; ++k)
			if (tot[k] < tot[t]) t = k;
		best = t;
	}
	__syncthreads();
	const int t = best;
	uint8_t *out = filt + (size_t)y * (size_t)(row_bytes + 1);
	if (threadIdx.x == 0) out[0] = (uint8_t)t;
	for (int i = threadIdx.x; i < row_bytes; i += blockDim.x) {
		const int x = cur[i], a = i >= bpp ? cur[i - bpp] : 0, b = prv ? prv[i] : 0, c = (prv && i >= bpp) ? prv[i - bpp] : 0;
		out[1 + i] = (uint8_t)png_residual(t, x, a, b, c);
	}
}

// ---- CRC-32 (reflected 0xEDB88320), combined across lanes as zlib's crc32_combine does ----
__device__ __forceinline__ uint32_t png_multmodp(uint32_t a, uint32_t b) {   // a != 0
	uint32_t m = 1u << 31, p = 0u;
	for (;;) {
		if (a & m) {
			p ^= b;
			if ((a & (m - 1u)) == 0u) break;
		}
		m >>= 1;
		b = (b & 1u) ? (b >> 1) ^ 0xEDB88320u : b >> 1;
	}
	return p;
}

// x^(8 n) mod P from the table of x^(2^k)
__device__ __forceinline__ uint32_t png_x8nmodp(uint32_t n, const uint32_t *x2n) {
	uint32_t p = 1u << 31;
	int k = 3;
	while (n) {
		if (n & 1u) p = png_multmodp(x2n[k & 31], p);
		n >>= 1;
		k += 1;
	}
	return p;
}

__device__ __forceinline__ uint32_t png_crc_bytes(const uint8_t *p, int n) {   // plain bitwise, for the small chunks
	uint32_t c = 0xFFFFFFFFu;
	for (int i = 0; i < n; ++i) {
		c ^= p[i];
		for (int k = 0; k < 8; ++k) c = (c & 1u) ? (c >> 1) ^ 0xEDB88320u : c >> 1;
	}
	return ~c;
}

__device__ __forceinline__ void png_put_bits(uint32_t *buf, uint32_t bitpos, uint32_t value, int nbits) {
	const uint32_t w = bitpos >> 5, o = bitpos & 31u;
	atomicOr(&buf[w], value << o);
	if (o + (uint32_t)nbits > 32u) atomicOr(&buf[w + 1], value >> (32u - o));
}

__device__ __forceinline__ uint32_t png_rev(uint32_t code, int len) { return __brev(code) >> (32 - len); }

// 64 bits of a bit array from bit o on
__device__ __forceinline__ unsigned long long png_bits64(const uint32_t *m, int o) {
	const int w = o >> 5, b = o & 31;
	const unsigned long long lo = (unsigned long long)m[w] | ((unsigned long long)m[w + 1] << 32);
	return b ? (lo >> b) | ((unsigned long long)m[w + 2] << (64 - b)) : lo;
}

// one warp per segment
__global__ void __launch_bounds__(kPngDeflateWarps * 32) k3_png_deflate(const uint8_t *__restrict__ filt,
                                                                        unsigned long long total, int nseg, int bpp,
                                                                        int row_dist, uint8_t *__restrict__ stage,
                                                                        PngSegInfo *__restrict__ info) {
	__shared__ uint32_t crc_tab[256];
	__shared__ uint32_t x2n[32];
	__shared__ __align__(16) uint32_t sbuf[kPngDeflateWarps][kPngStageStride / 4];
	__shared__ __align__(16) uint8_t sseg[kPngDeflateWarps][kPngSeg];          // the segment's bytes
	__shared__ uint32_t smask[kPngDeflateWarps][3][kPngMaskWords];              // equality bits per candidate distance
	for (int i = threadIdx.x; i < 256; i += blockDim.x) {
		uint32_t c = (uint32_t)i;
		for (int k = 0; k < 8; ++k) c = (c & 1u) ? (c >> 1) ^ 0xEDB88320u : c >> 1;
		crc_tab[i] = c;
	}
	if (threadIdx.x == 0) {
		uint32_t p = 1u << 30;   // x^1
		x2n[0] = p;
		for (int n = 1; n < 32; ++n) x2n[n] = p = png_multmodp(p, p);
	}
	__syncthreads();

	const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
	const int s = blockIdx.x * kPngDeflateWarps + warp;
	if (s >= nseg) return;
	const unsigned long long s0 = (unsigned long long)s * kPngSeg;
	const int n = (int)(total - s0 < (unsigned long long)kPngSeg ? total - s0 : (unsigned long long)kPngSeg);
	const unsigned long long s1 = s0 + (unsigned long long)n;
	uint32_t *buf = sbuf[warp];
	uint8_t *bb = (uint8_t *)buf;
	for (int i = lane; i < kPngStageStride / 4; i += 32) buf[i] = 0u;
	__syncwarp();
	const int data_start = s == 0 ? 10 : 8;
	if (lane == 0) {
		bb[4] = 'I'; bb[5] = 'D'; bb[6] = 'A'; bb[7] = 'T';
		if (s == 0) { bb[8] = 0x78; bb[9] = 0x01; }
	}
	__syncwarp();

	// ---- fixed-Huffman attempt; abandoned as soon as it cannot beat the stored block ----
	const unsigned long long dist[3] = {1ull, (unsigned long long)bpp, (unsigned long long)row_dist};   // 0: unused
	const uint32_t limit = (uint32_t)(data_start + 1 + n) * 8u;   // + EOB / stored header bits, + 00 00 FF FF
	uint32_t bp = (uint32_t)data_start * 8u;
	if (lane == 0) png_put_bits(buf, bp, 2u, 3);   // BFINAL 0, BTYPE 01
	bp += 3;
	bool coded = true;
	// Parallel pre-pass: the segment's bytes, and bit p of mask[di] = "byte p equals the byte dist[di] before it" (never
	// before byte 0 of the stream; 0 past the segment's end).  The serial parse below then reads shared memory only.
	uint8_t *seg = sseg[warp];
	uint32_t(*mask)[kPngMaskWords] = smask[warp];
#pragma unroll 4
	for (int w = 0; w < kPngMaskWords; ++w) {
		const unsigned long long p = s0 + (unsigned long long)(32 * w + lane);
		const bool in = p < s1;
		const int x = in ? filt[p] : 0;
		if (in) seg[32 * w + lane] = (uint8_t)x;
#pragma unroll
		for (int di = 0; di < 3; ++di) {
			const unsigned long long d = dist[di];
			const unsigned m = __ballot_sync(0xffffffffu, in && d && p >= d && filt[p - d] == x);
			if (lane == 0) mask[di][w] = m;
		}
	}
	__syncwarp();
	int o = 0;   // parse position inside the segment
	while (o < n) {
		const int x0 = o + lane < n ? seg[o + lane] : 0;
		unsigned long long E[3], M = 0;
#pragma unroll
		for (int di = 0; di < 3; ++di) {
			E[di] = png_bits64(mask[di], o);
			M |= E[di] & (E[di] >> 1) & (E[di] >> 2);
		}
		M &= 0xFFFFFFFFull;
		int nlit = M ? __ffsll((long long)M) - 1 : (n - o < 32 ? n - o : 32);
		if (nlit > 0) {
			const bool lit = lane < nlit, nine = lit && x0 >= 144;
			const unsigned b9 = __ballot_sync(0xffffffffu, nine);
			const uint32_t bits = 8u * (uint32_t)nlit + (uint32_t)__popc(b9);
			if (bp + bits + 10u > limit) { coded = false; break; }
			if (lit) {
				const uint32_t off = 8u * (uint32_t)lane + (uint32_t)__popc(b9 & ((1u << lane) - 1u));
				if (nine) png_put_bits(buf, bp + off, png_rev(0x190u + (uint32_t)(x0 - 144), 9), 9);
				else png_put_bits(buf, bp + off, png_rev(0x30u + (uint32_t)x0, 8), 8);
			}
			bp += bits;
			o += nlit;
			continue;
		}
		// a match starts at o: the longest of the candidate distances (the first on a tie)
		int best_len = 0;
		unsigned long long best_d = 1;
#pragma unroll
		for (int di = 0; di < 3; ++di) {
			if ((E[di] & 7ull) != 7ull) continue;
			int len = E[di] == ~0ull ? 64 : __ffsll((long long)~E[di]) - 1;
			if (len == 64) {
				while (len < 258) {   // all bits set so far: o + len <= n, and mask bits past n are 0
					const uint32_t m = (uint32_t)png_bits64(mask[di], o + len);
					const int k = m == 0xffffffffu ? 32 : __ffs(~m) - 1;
					len += k;
					if (k < 32) break;
				}
			}
			if (len > 258) len = 258;
			if (len > best_len) { best_len = len; best_d = dist[di]; }
		}
		// length symbol 257..285 with its extra bits, distance code 0..29 with its extra bits
		uint32_t sym, ne = 0, ev = 0;
		if (best_len == 258) sym = 285;
		else if (best_len <= 10) sym = 257u + (uint32_t)(best_len - 3);
		else {
			const uint32_t l = (uint32_t)(best_len - 3);
			ne = 31u - __clz(l) - 2u;
			sym = 257u + 4u * (ne + 1u) + ((l >> ne) & 3u);
			ev = l & ((1u << ne) - 1u);
		}
		const uint32_t dd = (uint32_t)best_d - 1u;
		uint32_t dc, de = 0, dv = 0;
		if (dd < 4u) dc = dd;
		else {
			de = 31u - __clz(dd) - 1u;
			dc = 2u * (de + 1u) + ((dd >> de) & 1u);
			dv = dd & ((1u << de) - 1u);
		}
		const int hl = sym < 280u ? 7 : 8;
		const uint32_t hc = sym < 280u ? sym - 256u : 0xC0u + (sym - 280u);
		const uint32_t bits = (uint32_t)hl + ne + 5u + de;
		if (bp + bits + 10u > limit) { coded = false; break; }
		if (lane == 0) {
			const uint32_t v = png_rev(hc, hl) | (ev << hl) | (png_rev(dc, 5) << (hl + ne)) | (dv << (hl + ne + 5u));
			png_put_bits(buf, bp, v, (int)bits);
		}
		bp += bits;
		o += best_len;
	}
	__syncwarp();
	int payload_end;
	if (coded) {
		bp += 10u;   // EOB (7 zero bits) + the empty stored block's header (3 zero bits)
		const int bytes = (int)((bp + 7u) >> 3);
		if (lane == 0) { bb[bytes + 2] = 0xFF; bb[bytes + 3] = 0xFF; }
		payload_end = bytes + 4;
	}
	else {
		for (int i = data_start + lane; i < data_start + 5 + n; i += 32) {
			uint8_t v;
			const int k = i - data_start;
			if (k == 0) v = 0x00;                                  // BFINAL 0, BTYPE 00
			else if (k == 1) v = (uint8_t)(n & 255);
			else if (k == 2) v = (uint8_t)(n >> 8);
			else if (k == 3) v = (uint8_t)(~n & 255);
			else if (k == 4) v = (uint8_t)((~n >> 8) & 255);
			else v = seg[k - 5];
			bb[i] = v;
		}
		payload_end = data_start + 5 + n;
	}
	__syncwarp();

	// ---- chunk length and CRC-32 over type + data ----
	const int crc_len = payload_end - 4;
	const int per = (crc_len + 31) / 32;
	const int lo = 4 + lane * per, hi = min(4 + (lane + 1) * per, payload_end);
	uint32_t c = 0xFFFFFFFFu;
	for (int i = lo; i < hi; ++i) c = crc_tab[(c ^ bb[i]) & 255u] ^ (c >> 8);
	c = lo < hi ? ~c : 0u;
	if (lo < hi && hi < payload_end) c = png_multmodp(png_x8nmodp((uint32_t)(payload_end - hi), x2n), c);
	for (int o = 16; o > 0; o >>= 1) c ^= __shfl_xor_sync(0xffffffffu, c, o);
	const uint32_t len = (uint32_t)(payload_end - 8);
	__syncwarp();
	if (lane == 0) {
		bb[0] = (uint8_t)(len >> 24); bb[1] = (uint8_t)(len >> 16); bb[2] = (uint8_t)(len >> 8); bb[3] = (uint8_t)len;
		bb[payload_end + 0] = (uint8_t)(c >> 24);
		bb[payload_end + 1] = (uint8_t)(c >> 16);
		bb[payload_end + 2] = (uint8_t)(c >> 8);
		bb[payload_end + 3] = (uint8_t)c;
	}

	// ---- Adler-32 partials of the segment's bytes ----
	unsigned long long a = 0, b = 0;
	for (int j = lane; j < n; j += 32) {
		const unsigned long long x = seg[j];
		a += x;
		b += (unsigned long long)(n - j) * x;
	}
	for (int o = 16; o > 0; o >>= 1) {
		a += __shfl_xor_sync(0xffffffffu, a, o);
		b += __shfl_xor_sync(0xffffffffu, b, o);
	}
	__syncwarp();

	const int chunk = payload_end + 4;
	uint4 *dst = (uint4 *)(stage + (size_t)s * kPngStageStride);
	const uint4 *src = (const uint4 *)buf;
	for (int i = lane; i < (chunk + 15) / 16; i += 32) dst[i] = src[i];
	if (lane == 0) {
		PngSegInfo si;
		si.chunk_bytes = (uint32_t)chunk;
		si.adler_a = (uint32_t)(a % 65521ull);
		si.adler_b = b % 65521ull;
		info[s] = si;
	}
}

__device__ __forceinline__ void png_be32(uint8_t *p, uint32_t v) {
	p[0] = (uint8_t)(v >> 24); p[1] = (uint8_t)(v >> 16); p[2] = (uint8_t)(v >> 8); p[3] = (uint8_t)v;
}

// one CTA of 1024 threads.  offsets[0..nseg+2]: piece 0 = signature + IHDR, pieces 1..nseg = the segments' chunks,
// piece nseg + 1 = last IDAT + IEND; offsets[nseg + 2] = file size
__global__ void __launch_bounds__(1024) k3_png_finish(const PngSegInfo *__restrict__ info, int nseg,
                                                      unsigned long long total, int width, int height, int channels,
                                                      unsigned long long *__restrict__ offsets, uint8_t *__restrict__ meta) {
	__shared__ unsigned long long wsum[32];
	__shared__ unsigned long long wa[32], wb[32];
	const int t = threadIdx.x, per = (nseg + (int)blockDim.x - 1) / (int)blockDim.x;
	const int i0 = min(t * per, nseg), i1 = min(i0 + per, nseg);
	unsigned long long sum = 0, A = 0, B = 0;
	for (int i = i0; i < i1; ++i) {
		const PngSegInfo si = info[i];
		sum += si.chunk_bytes;
		const unsigned long long o = (unsigned long long)i * kPngSeg;
		const unsigned long long nn = total - o < (unsigned long long)kPngSeg ? total - o : (unsigned long long)kPngSeg;
		A += si.adler_a;
		B = (B + si.adler_b + ((total - o - nn) % 65521ull) * si.adler_a) % 65521ull;
	}
	A %= 65521ull;
	// block exclusive scan of `sum`, block sums of A and B
	const int lane = t & 31, w = t >> 5;
	unsigned long long incl = sum;
	for (int o = 1; o < 32; o <<= 1) {
		const unsigned long long v = __shfl_up_sync(0xffffffffu, incl, o);
		if (lane >= o) incl += v;
	}
	unsigned long long ra = A, rb = B;
	for (int o = 16; o > 0; o >>= 1) {
		ra += __shfl_xor_sync(0xffffffffu, ra, o);
		rb += __shfl_xor_sync(0xffffffffu, rb, o);
	}
	if (lane == 31) wsum[w] = incl;
	if (lane == 0) { wa[w] = ra; wb[w] = rb; }
	__syncthreads();
	if (w == 0) {
		const int nw = (int)(blockDim.x >> 5);
		unsigned long long v = lane < nw ? wsum[lane] : 0ull, x = v;
		for (int o = 1; o < 32; o <<= 1) {
			const unsigned long long u = __shfl_up_sync(0xffffffffu, x, o);
			if (lane >= o) x += u;
		}
		wsum[lane] = x - v;   // exclusive prefix of the warps
		unsigned long long sa = lane < nw ? wa[lane] : 0ull, sb = lane < nw ? wb[lane] : 0ull;
		for (int o = 16; o > 0; o >>= 1) {
			sa += __shfl_xor_sync(0xffffffffu, sa, o);
			sb += __shfl_xor_sync(0xffffffffu, sb, o);
		}
		if (lane == 0) { wa[0] = sa; wb[0] = sb; }
	}
	__syncthreads();
	unsigned long long off = kPngHeadBytes + wsum[w] + incl - sum;
	for (int i = i0; i < i1; ++i) {
		offsets[1 + i] = off;
		off += info[i].chunk_bytes;
	}
	if (t == (int)blockDim.x - 1) {
		offsets[0] = 0;
		offsets[nseg + 1] = off;
		offsets[nseg + 2] = off + kPngTailBytes;
	}
	if (t == 0) {
		static const uint8_t sig[8] = {137, 80, 78, 71, 13, 10, 26, 10};
		for (int k = 0; k < 8; ++k) meta[k] = sig[k];
		uint8_t *ih = meta + 8;
		png_be32(ih, 13u);
		ih[4] = 'I'; ih[5] = 'H'; ih[6] = 'D'; ih[7] = 'R';
		png_be32(ih + 8, (uint32_t)width);
		png_be32(ih + 12, (uint32_t)height);
		ih[16] = 8;
		ih[17] = channels == 4 ? 6 : 2;
		ih[18] = ih[19] = ih[20] = 0;
		png_be32(ih + 21, png_crc_bytes(ih + 4, 17));
		const uint32_t a32 = (uint32_t)((1ull + wa[0]) % 65521ull);
		const uint32_t b32 = (uint32_t)((total % 65521ull + wb[0]) % 65521ull);
		uint8_t *tl = meta + kPngMetaTail;
		png_be32(tl, 6u);
		tl[4] = 'I'; tl[5] = 'D'; tl[6] = 'A'; tl[7] = 'T';
		tl[8] = 0x03; tl[9] = 0x00;                      // BFINAL 1, fixed block, EOB
		png_be32(tl + 10, (b32 << 16) | a32);
		png_be32(tl + 14, png_crc_bytes(tl + 4, 10));
		static const uint8_t iend[12] = {0, 0, 0, 0, 'I', 'E', 'N', 'D', 0xAE, 0x42, 0x60, 0x82};
		for (int k = 0; k < 12; ++k) tl[18 + k] = iend[k];
	}
}

// piece 0 is `first`, piece npieces - 1 is `last`, piece i between them starts at stage + (i - 1) * stride
__device__ __forceinline__ const uint8_t *png_piece(int i, int npieces, const uint8_t *first, const uint8_t *last,
                                                    const uint8_t *stage, unsigned long long stride) {
	if (i == 0) return first;
	if (i == npieces - 1) return last;
	return stage + (unsigned long long)(i - 1) * stride;
}

// Each thread writes the bytes of one 16-byte-aligned word of the destination (word -1: the bytes before the first
// aligned address).  Grid-stride; offsets[0..npieces]: where each piece starts in the file, then the file size.
__global__ void __launch_bounds__(256) k3_png_gather(const unsigned long long *__restrict__ offsets, int npieces,
                                                     const uint8_t *__restrict__ first, const uint8_t *__restrict__ final_piece,
                                                     const uint8_t *__restrict__ stage, unsigned long long piece_stride,
                                                     uint8_t *dst, unsigned long long *size_out) {
	const unsigned long long total = offsets[npieces];
	const unsigned long long head = (16u - ((uintptr_t)dst & 15u)) & 15u;
	const long long last = total > head ? (long long)((total - head + 15) / 16) - 1 : -1;
	const long long stride = (long long)gridDim.x * blockDim.x;
	const long long gid = (long long)blockIdx.x * blockDim.x + threadIdx.x;
	if (gid == 0) *size_out = total;
	for (long long w = gid - 1; w <= last; w += stride) {
		const long long lo_s = (long long)head + 16 * w;
		const unsigned long long lo = lo_s < 0 ? 0ull : (unsigned long long)lo_s;
		const unsigned long long hi_u = (unsigned long long)(lo_s + 16);
		const unsigned long long hi = hi_u < total ? hi_u : total;
		if (lo >= hi) continue;
		// piece containing lo: the last i with offsets[i] <= lo
		int a = 0, b = npieces - 1;
		while (a < b) {
			const int m = (a + b + 1) >> 1;
			if (offsets[m] <= lo) a = m;
			else b = m - 1;
		}
		int i = a;
		unsigned long long end = offsets[i + 1];
		const uint8_t *src = png_piece(i, npieces, first, final_piece, stage, piece_stride) - offsets[i];
		const bool whole = hi - lo == 16 && lo_s >= 0;
		unsigned long long w0 = 0, w1 = 0;
		for (unsigned long long k = lo; k < hi; ++k) {
			while (k >= end) {
				i += 1;
				src = png_piece(i, npieces, first, final_piece, stage, piece_stride) - offsets[i];
				end = offsets[i + 1];
			}
			const unsigned long long v = src[k];
			const unsigned j = (unsigned)(k - lo);
			if (!whole) dst[k] = (uint8_t)v;
			else if (j < 8) w0 |= v << (8 * j);
			else w1 |= v << (8 * (j - 8));
		}
		if (whole) {
			uint4 word;
			word.x = (uint32_t)w0;
			word.y = (uint32_t)(w0 >> 32);
			word.z = (uint32_t)w1;
			word.w = (uint32_t)(w1 >> 32);
			*(uint4 *)(dst + lo) = word;
		}
	}
}

// host arithmetic shared by hmrm_png_bound and the launches
struct PngShape {
	unsigned long long row_bytes, total;   // filtered stream: H rows of (1 + row_bytes)
	int nseg;
};

inline bool png_shape(long long width, long long height, long long channels, PngShape *out) {
	if (width < 1 || height < 1 || width > 65536 || height > 65536 || (channels != 3 && channels != 4)) return false;
	out->row_bytes = (unsigned long long)(width * channels);
	out->total = (unsigned long long)height * (out->row_bytes + 1ull);
	out->nseg = (int)((out->total + kPngSeg - 1) / kPngSeg);
	return true;
}

// signature + IHDR + zlib header + every segment stored (chunk 12 + block header 5) + last IDAT + IEND
inline unsigned long long png_bound(const PngShape &s) {
	return (unsigned long long)kPngHeadBytes + 2ull + s.total + 17ull * (unsigned long long)s.nseg + kPngTailBytes;
}

} // namespace hmrm
