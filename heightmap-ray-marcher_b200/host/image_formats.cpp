// BMP, GIF (first frame), PSD, TGA and binary PNM ingest: decoded to the pixels stb_image v2.27 returns for the same
// file (vendor/stb_image.h: stbi__bmp_load :5467, stbi__gif_load :6970, stbi__psd_load :6048, stbi__tga_load :5792,
// stbi__pnm_load :7428), which is what the reference's config loader hands to the renderer (main/hmap.cpp:320-321,
// :341-342).  Independent implementations of each format's decoded-pixel contract, including the corners that are
// stb's own: BMP alpha that is all zero reads as opaque; a GIF's undrawn first-frame pixels take the background entry
// in B,G,R order while transparent ones stay 0; PSD's un-matting in float; TGA 15/16-bit (r*255)/31; 16-bit PNM
// samples narrowed to the byte stb's little-endian reading keeps.
#include "image_internal.hpp"

#include <cstdlib>
#include <cstring>

namespace hmrm_host {
namespace {

// bounds-checked little/big-endian reader over the file bytes; reads past the end give 0 (as stb's do)
struct Reader {
	const std::vector<uint8_t> &f;
	size_t pos;
	explicit Reader(const std::vector<uint8_t> &file) : f(file), pos(0) {}
	int u8() { return pos < f.size() ? f[pos++] : (++pos, 0); }
	int le16() { const int a = u8(); return a | (u8() << 8); }
	uint32_t le32() { const uint32_t a = (uint32_t)le16(); return a | ((uint32_t)le16() << 16); }
	int be16() { const int a = u8(); return (a << 8) | u8(); }
	uint32_t be32() { const uint32_t a = (uint32_t)be16(); return (a << 16) | (uint32_t)be16(); }
	void skip(long n) { if (n > 0) pos += (size_t)n; }
	bool eof() const { return pos >= f.size(); }
};

bool fail(std::string *error, const char *why) { *error = why; return false; }

// ---------------------------------------------------------------------------------------------
// BMP
// ---------------------------------------------------------------------------------------------
int high_bit(uint32_t z) {
	int n = -1;
	while (z) { ++n; z >>= 1; }
	return n;
}
int bit_count(uint32_t z) {
	int n = 0;
	while (z) { n += (int)(z & 1u); z >>= 1; }
	return n;
}
// an arbitrarily placed `bits`-wide field of v, widened to 8 bits by replication of its pattern
int field_to_byte(uint32_t v, int shift, int bits) {
	static const uint32_t mul[9] = {0, 0xFF, 0x55, 0x49, 0x11, 0x21, 0x41, 0x81, 0x01};
	static const int shr[9] = {0, 0, 0, 1, 0, 2, 4, 6, 0};
	if (shift < 0) v <<= -shift;
	else v >>= shift;
	v >>= (8 - bits);
	return (int)((v * mul[bits]) >> shr[bits]);
}

} // namespace

bool looks_like_bmp(const std::vector<uint8_t> &file) {
	if (file.size() < 18 || file[0] != 'B' || file[1] != 'M') return false;
	const uint32_t hsz = (uint32_t)file[14] | ((uint32_t)file[15] << 8) | ((uint32_t)file[16] << 16) | ((uint32_t)file[17] << 24);
	return hsz == 12 || hsz == 40 || hsz == 56 || hsz == 108 || hsz == 124;
}

bool decode_bmp(const std::vector<uint8_t> &file, Decoded *out, std::string *error) {
	Reader s(file);
	if (s.u8() != 'B' || s.u8() != 'M') return fail(error, "not BMP");
	s.le32(); s.le16(); s.le16();
	const int offset = (int)s.le32();
	const int hsz = (int)s.le32();
	uint32_t mr = 0, mg = 0, mb = 0, ma = 0, all_a = 255;
	int extra_read = 14;
	if (offset < 0) return fail(error, "bad BMP");
	if (hsz != 12 && hsz != 40 && hsz != 56 && hsz != 108 && hsz != 124) return fail(error, "BMP type not supported: unknown");
	int w, hraw;
	if (hsz == 12) { w = s.le16(); hraw = s.le16(); }
	else { w = (int)s.le32(); hraw = (int)s.le32(); }
	if (s.le16() != 1) return fail(error, "bad BMP");
	const int bpp = s.le16();
	auto default_masks = [&](int compress) {
		if (compress != 0) return;
		if (bpp == 16) { mr = 31u << 10; mg = 31u << 5; mb = 31u; }
		else if (bpp == 32) { mr = 0xFFu << 16; mg = 0xFFu << 8; mb = 0xFFu; ma = 0xFFu << 24; all_a = 0; }
		else mr = mg = mb = ma = 0;
	};
	if (hsz != 12) {
		const int compress = (int)s.le32();
		if (compress == 1 || compress == 2) return fail(error, "BMP type not supported: RLE");
		if (compress >= 4) return fail(error, "BMP type not supported: unsupported compression");
		if (compress == 3 && bpp != 16 && bpp != 32) return fail(error, "bad BMP");
		s.le32(); s.le32(); s.le32(); s.le32(); s.le32();
		if (hsz == 40 || hsz == 56) {
			if (hsz == 56) { s.le32(); s.le32(); s.le32(); s.le32(); }
			if (bpp == 16 || bpp == 32) {
				if (compress == 0) default_masks(compress);
				else if (compress == 3) {
					mr = s.le32(); mg = s.le32(); mb = s.le32();
					extra_read += 12;
					if (mr == mg && mg == mb) return fail(error, "bad BMP");
				}
				else return fail(error, "bad BMP");
			}
		}
		else {
			mr = s.le32(); mg = s.le32(); mb = s.le32(); ma = s.le32();
			if (compress != 3) default_masks(compress);
			s.le32();
			for (int i = 0; i < 12; ++i) s.le32();
			if (hsz == 124) { s.le32(); s.le32(); s.le32(); s.le32(); }
		}
	}
	const bool flip = hraw > 0;
	const int h = std::abs(hraw);
	if (w <= 0 || h <= 0 || w > (1 << 24) || h > (1 << 24) || (long long)w * h > (1LL << 28)) return fail(error, "bad BMP size");
	int psize = 0;
	if (hsz == 12) { if (bpp < 24) psize = (offset - extra_read - 24) / 3; }
	else if (bpp < 16) psize = (offset - extra_read - hsz) >> 2;
	if (psize == 0 && offset != (int)s.pos) return fail(error, "bad offset");

	out->w = w;
	out->h = h;
	out->channels = 4;
	out->px.assign((size_t)w * (size_t)h * 4, 0);
	uint8_t *o = out->px.data();
	size_t z = 0;
	if (bpp < 16) {
		if (psize == 0 || psize > 256) return fail(error, "Corrupt BMP (palette)");
		uint8_t pal[256][3];
		for (int i = 0; i < psize; ++i) {
			pal[i][2] = (uint8_t)s.u8(); pal[i][1] = (uint8_t)s.u8(); pal[i][0] = (uint8_t)s.u8();
			if (hsz != 12) s.u8();
		}
		s.skip(offset - extra_read - hsz - psize * (hsz == 12 ? 3 : 4));
		int width;
		if (bpp == 1) width = (w + 7) >> 3;
		else if (bpp == 4) width = (w + 1) >> 1;
		else if (bpp == 8) width = w;
		else return fail(error, "bad bpp");
		const int pad = (-width) & 3;
		for (int j = 0; j < h; ++j) {
			int v = 0, have = 0;
			for (int i = 0; i < w; ++i) {
				int color;
				if (bpp == 8) color = s.u8();
				else if (bpp == 4) {
					if (!have) { v = s.u8(); have = 2; }
					color = have == 2 ? v >> 4 : v & 15;
					--have;
				}
				else {
					if (!have) { v = s.u8(); have = 8; }
					color = (v >> (have - 1)) & 1;
					--have;
				}
				// (indices beyond the palette read stb's uninitialised stack: not reproducible — rejected)
				if (color >= psize) return fail(error, "BMP palette index out of range");
				o[z++] = pal[color][0]; o[z++] = pal[color][1]; o[z++] = pal[color][2]; o[z++] = 255;
			}
			s.skip(pad);
		}
		all_a = 255;
	}
	else {
		s.skip(offset - extra_read - hsz);
		int width = 0;
		if (bpp == 24) width = 3 * w;
		else if (bpp == 16) width = 2 * w;
		const int pad = (-width) & 3;
		int easy = 0;
		if (bpp == 24) easy = 1;
		else if (bpp == 32 && mb == 0xFF && mg == 0xFF00 && mr == 0x00FF0000 && ma == 0xFF000000) easy = 2;
		else if (bpp != 16 && bpp != 32) return fail(error, "bad bpp");
		int rs = 0, gs = 0, bs = 0, as = 0, rc = 0, gc = 0, bc = 0, ac = 0;
		if (!easy) {
			if (!mr || !mg || !mb) return fail(error, "bad masks");
			rs = high_bit(mr) - 7; rc = bit_count(mr);
			gs = high_bit(mg) - 7; gc = bit_count(mg);
			bs = high_bit(mb) - 7; bc = bit_count(mb);
			as = high_bit(ma) - 7; ac = bit_count(ma);
			if (rc > 8 || gc > 8 || bc > 8 || ac > 8) return fail(error, "bad masks");
		}
		for (int j = 0; j < h; ++j) {
			for (int i = 0; i < w; ++i) {
				uint32_t a;
				if (easy) {
					o[z + 2] = (uint8_t)s.u8(); o[z + 1] = (uint8_t)s.u8(); o[z] = (uint8_t)s.u8();
					a = easy == 2 ? (uint32_t)s.u8() : 255u;
				}
				else {
					const uint32_t v = bpp == 16 ? (uint32_t)s.le16() : s.le32();
					o[z] = (uint8_t)field_to_byte(v & mr, rs, rc);
					o[z + 1] = (uint8_t)field_to_byte(v & mg, gs, gc);
					o[z + 2] = (uint8_t)field_to_byte(v & mb, bs, bc);
					a = ma ? (uint32_t)field_to_byte(v & ma, as, ac) : 255u;
				}
				all_a |= a;
				o[z + 3] = (uint8_t)a;
				z += 4;
			}
			s.skip(pad);
		}
	}
	if (all_a == 0) {
		for (size_t i = 3; i < out->px.size(); i += 4) o[i] = 255;      // an alpha channel of zeros means "no alpha"
	}
	if (flip) {
		const size_t stride = (size_t)w * 4;
		std::vector<uint8_t> tmp(stride);
		for (int j = 0; j < h / 2; ++j) {
			uint8_t *a = o + (size_t)j * stride, *b = o + (size_t)(h - 1 - j) * stride;
			std::memcpy(tmp.data(), a, stride);
			std::memcpy(a, b, stride);
			std::memcpy(b, tmp.data(), stride);
		}
	}
	return true;
}

// ---------------------------------------------------------------------------------------------
// GIF: the first frame, composited as stb does
// ---------------------------------------------------------------------------------------------
namespace {

struct GifState {
	int w, h;
	std::vector<uint8_t> out;       // RGBA
	std::vector<uint8_t> drawn;     // per pixel: touched by the raster (transparent pixels included)
	const uint8_t (*table)[4];      // B, G, R, A entries
	int start_x, start_y, max_x, max_y, cur_x, cur_y, step, parse, line;
	struct Code { int16_t prefix; uint8_t first, suffix; } codes[8192];
};

void gif_emit(GifState &g, int code) {
	// the chain is stored last-to-first: walk it with an explicit stack
	static thread_local uint16_t stack[8192];
	int n = 0;
	for (int c = code; c >= 0 && n < 8192; c = g.codes[c].prefix) stack[n++] = (uint16_t)c;
	while (n > 0) {
		const int c = stack[--n];
		if (g.cur_y >= g.max_y) return;
		const int idx = g.cur_x + g.cur_y;
		g.drawn[(size_t)idx / 4] = 1;
		const uint8_t *e = g.table[g.codes[c].suffix];
		if (e[3] > 128) {
			uint8_t *p = &g.out[(size_t)idx];
			p[0] = e[2]; p[1] = e[1]; p[2] = e[0]; p[3] = e[3];
		}
		g.cur_x += 4;
		if (g.cur_x >= g.max_x) {
			g.cur_x = g.start_x;
			g.cur_y += g.step;
			while (g.cur_y >= g.max_y && g.parse > 0) {
				g.step = (1 << g.parse) * g.line;
				g.cur_y = g.start_y + (g.step >> 1);
				--g.parse;
			}
		}
	}
}

bool gif_raster(Reader &s, GifState &g, std::string *error) {
	const int lzw_cs = s.u8();
	if (lzw_cs > 12) return fail(error, "Corrupt GIF (code size)");
	const int clear = 1 << lzw_cs;
	bool first = true;
	int codesize = lzw_cs + 1, codemask = (1 << codesize) - 1, bits = 0, valid = 0;
	for (int i = 0; i < clear; ++i) { g.codes[i].prefix = -1; g.codes[i].first = (uint8_t)i; g.codes[i].suffix = (uint8_t)i; }
	int avail = clear + 2, oldcode = -1, len = 0;
	for (;;) {
		if (valid < codesize) {
			if (len == 0) {
				len = s.u8();
				if (len == 0) return true;
			}
			--len;
			bits |= s.u8() << valid;
			valid += 8;
			if (s.pos > s.f.size() + 16) return fail(error, "truncated GIF");
			continue;
		}
		const int code = bits & codemask;
		bits >>= codesize;
		valid -= codesize;
		if (code == clear) {
			codesize = lzw_cs + 1;
			codemask = (1 << codesize) - 1;
			avail = clear + 2;
			oldcode = -1;
			first = false;
		}
		else if (code == clear + 1) {
			s.skip(len);
			while ((len = s.u8()) > 0) s.skip(len);
			return true;
		}
		else if (code <= avail) {
			if (first) return fail(error, "no clear code");
			if (oldcode >= 0) {
				if (avail + 1 > 8192) return fail(error, "too many codes");
				GifState::Code &p = g.codes[avail++];
				p.prefix = (int16_t)oldcode;
				p.first = g.codes[oldcode].first;
				p.suffix = (code == avail) ? p.first : g.codes[code].first;
			}
			else if (code == avail) return fail(error, "illegal code in raster");
			gif_emit(g, code);
			if ((avail & codemask) == 0 && avail <= 0x0FFF) {
				codesize++;
				codemask = (1 << codesize) - 1;
			}
			oldcode = code;
		}
		else return fail(error, "illegal code in raster");
	}
}

} // namespace

bool decode_gif(const std::vector<uint8_t> &file, Decoded *out, std::string *error) {
	Reader s(file);
	if (s.u8() != 'G' || s.u8() != 'I' || s.u8() != 'F' || s.u8() != '8') return fail(error, "not GIF");
	const int version = s.u8();
	if ((version != '7' && version != '9') || s.u8() != 'a') return fail(error, "not GIF");
	GifState *g = new GifState();
	struct Guard { GifState *p; ~Guard() { delete p; } } guard = {g};
	g->w = s.le16();
	g->h = s.le16();
	const int flags = s.u8();
	const int bgindex = s.u8();
	s.u8();
	if (g->w <= 0 || g->h <= 0) return fail(error, "bad GIF size");
	static thread_local uint8_t pal[256][4], lpal[256][4];
	std::memset(pal, 0, sizeof pal);
	auto read_table = [&](uint8_t t[256][4], int n, int transparent) {
		for (int i = 0; i < n; ++i) {
			t[i][2] = (uint8_t)s.u8(); t[i][1] = (uint8_t)s.u8(); t[i][0] = (uint8_t)s.u8();
			t[i][3] = transparent == i ? 0 : 255;
		}
	};
	if (flags & 0x80) read_table(pal, 2 << (flags & 7), -1);
	const size_t pcount = (size_t)g->w * (size_t)g->h;
	g->out.assign(pcount * 4, 0);
	g->drawn.assign(pcount, 0);
	int transparent = -1, eflags = 0;
	for (;;) {
		if (s.eof()) return fail(error, "truncated GIF");
		const int tag = s.u8();
		if (tag == 0x2C) {
			const int x = s.le16(), y = s.le16(), w = s.le16(), h = s.le16();
			if (x + w > g->w || y + h > g->h) return fail(error, "bad Image Descriptor");
			g->line = g->w * 4;
			g->start_x = x * 4;
			g->start_y = y * g->line;
			g->max_x = g->start_x + w * 4;
			g->max_y = g->start_y + h * g->line;
			g->cur_x = g->start_x;
			g->cur_y = w == 0 ? g->max_y : g->start_y;
			const int lflags = s.u8();
			if (lflags & 0x40) { g->step = 8 * g->line; g->parse = 3; }
			else { g->step = g->line; g->parse = 0; }
			if (lflags & 0x80) {
				read_table(lpal, 2 << (lflags & 7), (eflags & 1) ? transparent : -1);
				g->table = lpal;
			}
			else if (flags & 0x80) g->table = pal;
			else return fail(error, "missing color table");
			if (!gif_raster(s, *g, error)) return false;
			if (bgindex > 0) {
				// undrawn pixels of the first frame take the background entry, bytes as stored (B, G, R), opaque
				for (size_t i = 0; i < pcount; ++i) {
					if (!g->drawn[i]) {
						g->out[i * 4] = pal[bgindex][0]; g->out[i * 4 + 1] = pal[bgindex][1];
						g->out[i * 4 + 2] = pal[bgindex][2]; g->out[i * 4 + 3] = 255;
					}
				}
			}
			out->w = g->w;
			out->h = g->h;
			out->channels = 4;
			out->px.swap(g->out);
			return true;
		}
		else if (tag == 0x21) {
			const int ext = s.u8();
			int len;
			if (ext == 0xF9) {
				len = s.u8();
				if (len == 4) {
					eflags = s.u8();
					s.le16();
					if (transparent >= 0) pal[transparent][3] = 255;
					if (eflags & 1) {
						transparent = s.u8();
						pal[transparent][3] = 0;
					}
					else { s.skip(1); transparent = -1; }
				}
				else { s.skip(len); continue; }
			}
			while ((len = s.u8()) != 0) {
				s.skip(len);
				if (s.eof()) return fail(error, "truncated GIF");
			}
		}
		else if (tag == 0x3B) return fail(error, "GIF has no image");
		else return fail(error, "unknown code");
	}
}

// ---------------------------------------------------------------------------------------------
// PSD: the composited RGB(A) image, 8 or 16 bit, raw or RLE
// ---------------------------------------------------------------------------------------------
bool decode_psd(const std::vector<uint8_t> &file, Decoded *out, std::string *error) {
	Reader s(file);
	if (s.be32() != 0x38425053u) return fail(error, "not PSD");
	if (s.be16() != 1) return fail(error, "Unsupported version of PSD image");
	s.skip(6);
	const int channels = s.be16();
	if (channels < 0 || channels > 16) return fail(error, "Unsupported number of channels in PSD image");
	const int h = (int)s.be32(), w = (int)s.be32();
	const int depth = s.be16();
	if (depth != 8 && depth != 16) return fail(error, "PSD bit depth is not 8 or 16 bit");
	if (s.be16() != 3) return fail(error, "PSD is not in RGB color format");
	s.skip((long)s.be32());
	s.skip((long)s.be32());
	s.skip((long)s.be32());
	const int compression = s.be16();
	if (compression > 1) return fail(error, "PSD has an unknown compression format");
	if (w <= 0 || h <= 0 || (long long)w * h > (1LL << 28)) return fail(error, "bad PSD size");
	const size_t n = (size_t)w * (size_t)h;
	out->w = w;
	out->h = h;
	out->channels = 4;
	out->px.assign(n * 4, 0);
	uint8_t *o = out->px.data();
	if (compression) s.skip((long)h * channels * 2);
	for (int c = 0; c < 4; ++c) {
		uint8_t *p = o + c;
		if (c >= channels) {
			for (size_t i = 0; i < n; ++i, p += 4) *p = c == 3 ? 255 : 0;
		}
		else if (compression) {
			size_t count = 0;
			while (count < n) {
				if (s.eof()) return fail(error, "bad RLE data");
				int len = s.u8();
				if (len == 128) continue;
				if (len < 128) {
					++len;
					if ((size_t)len > n - count) return fail(error, "bad RLE data");
					count += (size_t)len;
					while (len--) { *p = (uint8_t)s.u8(); p += 4; }
				}
				else {
					len = 257 - len;
					if ((size_t)len > n - count) return fail(error, "bad RLE data");
					const uint8_t v = (uint8_t)s.u8();
					count += (size_t)len;
					while (len--) { *p = v; p += 4; }
				}
			}
		}
		else if (depth == 16) {
			for (size_t i = 0; i < n; ++i, p += 4) *p = (uint8_t)(s.be16() >> 8);
		}
		else {
			for (size_t i = 0; i < n; ++i, p += 4) *p = (uint8_t)s.u8();
		}
	}
	if (channels >= 4) {
		// colours are stored matted against white: undo it where the pixel is partly transparent
		for (size_t i = 0; i < n; ++i) {
			uint8_t *px = o + 4 * i;
			if (px[3] != 0 && px[3] != 255) {
				const float a = px[3] / 255.0f;
				const float ra = 1.0f / a;
				const float inv_a = 255.0f * (1 - ra);
				px[0] = (unsigned char)(px[0] * ra + inv_a);
				px[1] = (unsigned char)(px[1] * ra + inv_a);
				px[2] = (unsigned char)(px[2] * ra + inv_a);
			}
		}
	}
	return true;
}

// ---------------------------------------------------------------------------------------------
// TGA: true colour 15/16/24/32 bit, grey 8 / grey+alpha 16, colour-mapped with 8- or 16-bit indices; raw or RLE
// ---------------------------------------------------------------------------------------------
namespace {

int tga_components(int bits, bool grey, bool *rgb16) {
	*rgb16 = false;
	switch (bits) {
	case 8: return 1;
	case 16: if (grey) return 2;   // fall through
	case 15: *rgb16 = true; return 3;
	case 24: return 3;
	case 32: return 4;
	default: return 0;
	}
}

void tga_rgb16(Reader &s, uint8_t *o) {
	const int px = s.le16();
	o[0] = (uint8_t)((((px >> 10) & 31) * 255) / 31);
	o[1] = (uint8_t)((((px >> 5) & 31) * 255) / 31);
	o[2] = (uint8_t)(((px & 31) * 255) / 31);
}

} // namespace

bool looks_like_tga(const std::vector<uint8_t> &file) {
	Reader s(file);
	s.u8();
	const int color_type = s.u8();
	if (color_type > 1) return false;
	int sz = s.u8();
	if (color_type == 1) {
		if (sz != 1 && sz != 9) return false;
		s.skip(4);
		sz = s.u8();
		if (sz != 8 && sz != 15 && sz != 16 && sz != 24 && sz != 32) return false;
		s.skip(4);
	}
	else {
		if (sz != 2 && sz != 3 && sz != 10 && sz != 11) return false;
		s.skip(9);
	}
	if (s.le16() < 1) return false;
	if (s.le16() < 1) return false;
	sz = s.u8();
	if (color_type == 1 && sz != 8 && sz != 16) return false;
	if (sz != 8 && sz != 15 && sz != 16 && sz != 24 && sz != 32) return false;
	return s.pos <= file.size();
}

bool decode_tga(const std::vector<uint8_t> &file, Decoded *out, std::string *error) {
	Reader s(file);
	const int id_len = s.u8(), indexed = s.u8();
	int type = s.u8();
	const int pal_start = s.le16(), pal_len = s.le16(), pal_bits = s.u8();
	s.le16(); s.le16();
	const int w = s.le16(), h = s.le16(), bpp = s.u8();
	const int desc = s.u8();
	bool rle = false;
	if (type >= 8) { type -= 8; rle = true; }
	const bool bottom_up = ((desc >> 5) & 1) == 0;
	bool rgb16 = false;
	const int comp = indexed ? tga_components(pal_bits, false, &rgb16) : tga_components(bpp, type == 3, &rgb16);
	if (!comp) return fail(error, "Can't find out TGA pixelformat");
	if (w <= 0 || h <= 0) return fail(error, "bad TGA size");
	out->w = w;
	out->h = h;
	out->channels = comp;
	const size_t npx = (size_t)w * (size_t)h;
	out->px.assign(npx * (size_t)comp, 0);
	uint8_t *data = out->px.data();
	s.skip(id_len);
	std::vector<uint8_t> palette;
	if (indexed) {
		if (pal_len == 0) return fail(error, "bad palette");
		s.skip(pal_start);
		palette.assign((size_t)pal_len * (size_t)comp, 0);
		if (rgb16) {
			for (int i = 0; i < pal_len; ++i) tga_rgb16(s, &palette[(size_t)i * 3]);
		}
		else {
			if (s.pos + palette.size() > file.size()) return fail(error, "bad palette");
			for (size_t i = 0; i < palette.size(); ++i) palette[i] = (uint8_t)s.u8();
		}
	}
	uint8_t raw[4] = {0, 0, 0, 0};
	int run = 0;
	bool repeating = false, read_next = true;
	for (size_t i = 0; i < npx; ++i) {
		if (rle) {
			if (run == 0) {
				const int cmd = s.u8();
				run = 1 + (cmd & 127);
				repeating = (cmd >> 7) != 0;
				read_next = true;
			}
			else if (!repeating) read_next = true;
		}
		else read_next = true;
		if (read_next) {
			if (s.pos > file.size() + 8) return fail(error, "truncated TGA data");
			if (indexed) {
				int idx = bpp == 8 ? s.u8() : s.le16();
				if (idx >= pal_len) idx = 0;
				for (int j = 0; j < comp; ++j) raw[j] = palette[(size_t)idx * (size_t)comp + (size_t)j];
			}
			else if (rgb16) tga_rgb16(s, raw);
			else {
				for (int j = 0; j < comp; ++j) raw[j] = (uint8_t)s.u8();
			}
			read_next = false;
		}
		for (int j = 0; j < comp; ++j) data[i * (size_t)comp + (size_t)j] = raw[j];
		--run;
	}
	if (bottom_up) {
		const size_t stride = (size_t)w * (size_t)comp;
		std::vector<uint8_t> tmp(stride);
		for (int j = 0; j * 2 < h; ++j) {
			uint8_t *a = data + (size_t)j * stride, *b = data + (size_t)(h - 1 - j) * stride;
			if (a == b) continue;
			std::memcpy(tmp.data(), a, stride);
			std::memcpy(a, b, stride);
			std::memcpy(b, tmp.data(), stride);
		}
	}
	if (comp >= 3 && !rgb16) {
		for (size_t i = 0; i < npx; ++i) {           // stored B, G, R
			uint8_t *p = data + i * (size_t)comp;
			const uint8_t t = p[0];
			p[0] = p[2];
			p[2] = t;
		}
	}
	return true;
}

// ---------------------------------------------------------------------------------------------
// binary PNM (P5 / P6), maxval up to 65535
// ---------------------------------------------------------------------------------------------
bool decode_pnm(const std::vector<uint8_t> &file, int want_channels, Decoded *out, std::string *error) {
	Reader s(file);
	if (s.u8() != 'P') return fail(error, "not PNM");
	const int t = s.u8();
	if (t != '5' && t != '6') return fail(error, "not PNM");
	const int comp = t == '6' ? 3 : 1;
	int c = s.u8();
	auto is_space = [](int ch) { return ch == ' ' || ch == '\t' || ch == '\n' || ch == '\v' || ch == '\f' || ch == '\r'; };
	auto skip_ws = [&]() {
		for (;;) {
			while (!s.eof() && is_space(c)) c = s.u8();
			if (s.eof() || c != '#') break;
			while (!s.eof() && c != '\n' && c != '\r') c = s.u8();
		}
	};
	auto integer = [&]() {
		long v = 0;
		while (!s.eof() && c >= '0' && c <= '9') {
			v = v * 10 + (c - '0');
			if (v > (1L << 30)) v = (1L << 30);
			c = s.u8();
		}
		return (int)v;
	};
	skip_ws();
	const int w = integer();
	skip_ws();
	const int h = integer();
	skip_ws();
	const int maxv = integer();
	if (maxv > 65535) return fail(error, "PPM image supports only 8-bit and 16-bit images");
	if (w <= 0 || h <= 0 || (long long)w * h > (1LL << 28)) return fail(error, "bad PNM size");
	const int bytes = maxv > 255 ? 2 : 1;
	const size_t need = (size_t)w * (size_t)h * (size_t)comp * (size_t)bytes;
	if (file.size() < s.pos || file.size() - s.pos < need) return fail(error, "truncated PNM data");
	out->w = w;
	out->h = h;
	out->channels = comp;
	if (bytes == 1) {
		out->px.assign(file.begin() + (long)s.pos, file.begin() + (long)(s.pos + need));
		return true;
	}
	// 16-bit samples.  stb 2.27 reads the big-endian samples into host (little-endian) 16-bit words and narrows with
	// >> 8, i.e. it keeps the SECOND byte of every sample; and when the channel count has to change it runs its 8-bit
	// converter over the 16-bit buffer and then reads past its end (vendor/stb_image.h:7449-7453, :1202-1206) —
	// undefined pixels that cannot be reproduced.  Only the well-defined case is accepted.
	if (out->keep16) {
		out->channels16 = comp;
		out->px16.resize((size_t)w * (size_t)h * (size_t)comp);
		for (size_t i = 0; i < out->px16.size(); ++i)
			out->px16[i] = (uint16_t)((file[s.pos + 2 * i] << 8) | file[s.pos + 2 * i + 1]);
		return true;
	}
	if (want_channels != comp) return fail(error, "16-bit PNM whose channel count must change: stb_image 2.27 reads out of bounds here (undefined pixels)");
	out->px.resize((size_t)w * (size_t)h * (size_t)comp);
	for (size_t i = 0; i < out->px.size(); ++i) out->px[i] = file[s.pos + 2 * i + 1];
	return true;
}

} // namespace hmrm_host
