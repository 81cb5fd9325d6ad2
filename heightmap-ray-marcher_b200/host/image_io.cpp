// See image_io.hpp.  PNG / PNM / TGA decode to the pixel values stb_image v2.27 would return.
#include "image_internal.hpp"

#include <zlib.h>

#include <cstdio>
#include <cstring>
#include <string>

namespace hmrm_host {
namespace {

bool read_file(const std::string &path, std::vector<uint8_t> *data) {
	FILE *f = std::fopen(path.c_str(), "rb");
	if (!f) return false;
	std::fseek(f, 0, SEEK_END);
	const long n = std::ftell(f);
	std::fseek(f, 0, SEEK_SET);
	if (n < 0) {
		std::fclose(f);
		return false;
	}
	data->resize((size_t)n);
	const size_t got = n ? std::fread(data->data(), 1, (size_t)n, f) : 0;
	std::fclose(f);
	return got == (size_t)n;
}

uint32_t be32(const uint8_t *p) { return ((uint32_t)p[0] << 24) | ((uint32_t)p[1] << 16) | ((uint32_t)p[2] << 8) | p[3]; }

} // namespace

// stbi__convert_format semantics for 8-bit data
void convert_channels(const Decoded &d, int want, Image *out) {
	out->width = d.w;
	out->height = d.h;
	out->channels = want;
	const size_t n = (size_t)d.w * (size_t)d.h;
	out->pixels.resize(n * (size_t)want);
	const uint8_t *s = d.px.data();
	uint8_t *t = out->pixels.data();
	for (size_t i = 0; i < n; ++i, s += d.channels, t += want) {
		uint8_t r, g, b, a = 255;
		switch (d.channels) {
		case 1: r = g = b = s[0]; break;
		case 2: r = g = b = s[0]; a = s[1]; break;
		case 3: r = s[0]; g = s[1]; b = s[2]; break;
		default: r = s[0]; g = s[1]; b = s[2]; a = s[3]; break;
		}
		t[0] = r;
		t[1] = g;
		t[2] = b;
		if (want == 4) t[3] = a;
	}
}

// ---------------------------------------------------------------------------------------------
// PNG
// ---------------------------------------------------------------------------------------------
namespace {

int paeth(int a, int b, int c) {
	const int p = a + b - c;
	const int pa = p > a ? p - a : a - p, pb = p > b ? p - b : b - p, pc = p > c ? p - c : c - p;
	if (pa <= pb && pa <= pc) return a;
	if (pb <= pc) return b;
	return c;
}

// Reverse the PNG filters of one (sub)image in place.  `raw` holds rows of (1 + stride) bytes.
bool unfilter(uint8_t *raw, int rows, size_t stride, int bpp, std::string *error) {
	std::vector<uint8_t> zero(stride, 0);
	const uint8_t *prev = zero.data();
	for (int y = 0; y < rows; ++y) {
		uint8_t *line = raw + (size_t)y * (stride + 1);
		const int ft = line[0];
		uint8_t *cur = line + 1;
		for (size_t i = 0; i < stride; ++i) {
			const int a = i >= (size_t)bpp ? cur[i - bpp] : 0;
			const int b = prev[i];
			const int c = i >= (size_t)bpp ? prev[i - bpp] : 0;
			int v = cur[i];
			switch (ft) {
			case 0: break;
			case 1: v += a; break;
			case 2: v += b; break;
			case 3: v += (a + b) >> 1; break;
			case 4: v += paeth(a, b, c); break;
			default: *error = "bad PNG filter type"; return false;
			}
			cur[i] = (uint8_t)v;
		}
		prev = cur;
	}
	return true;
}

} // namespace

bool decode_png(const std::vector<uint8_t> &file, Decoded *out, std::string *error) {
	static const uint8_t sig[8] = {137, 80, 78, 71, 13, 10, 26, 10};
	if (file.size() < 8 || std::memcmp(file.data(), sig, 8) != 0) { *error = "not a PNG"; return false; }
	size_t pos = 8;
	uint32_t w = 0, h = 0;
	int depth = 0, color = 0, interlace = 0;
	std::vector<uint8_t> idat, palette, trns;
	bool have_ihdr = false, done = false;
	while (!done && pos + 8 <= file.size()) {
		const uint32_t len = be32(&file[pos]);
		const uint32_t type = be32(&file[pos + 4]);
		pos += 8;
		if (pos + (size_t)len + 4 > file.size()) { *error = "truncated PNG"; return false; }
		const uint8_t *p = &file[pos];
		switch (type) {
		case 0x49484452: {   // IHDR
			if (len != 13) { *error = "bad IHDR"; return false; }
			w = be32(p); h = be32(p + 4); depth = p[8]; color = p[9]; interlace = p[12];
			if (p[10] != 0 || p[11] != 0 || interlace > 1) { *error = "unsupported PNG method"; return false; }
			have_ihdr = true;
			break;
		}
		case 0x504C5445: palette.assign(p, p + len); break;   // PLTE
		case 0x74524E53: trns.assign(p, p + len); break;      // tRNS
		case 0x49444154: idat.insert(idat.end(), p, p + len); break;   // IDAT
		case 0x49454E44: done = true; break;                   // IEND
		default: break;
		}
		pos += (size_t)len + 4;   // data + CRC (not verified, as in stb_image)
	}
	if (!have_ihdr || w == 0 || h == 0 || w > (1u << 24) || h > (1u << 24)) { *error = "bad PNG header"; return false; }
	int src_n;
	switch (color) {
	case 0: src_n = 1; break;
	case 2: src_n = 3; break;
	case 3: src_n = 1; break;
	case 4: src_n = 2; break;
	case 6: src_n = 4; break;
	default: *error = "bad PNG colour type"; return false;
	}
	if (!(depth == 1 || depth == 2 || depth == 4 || depth == 8 || depth == 16)) { *error = "bad PNG bit depth"; return false; }
	if ((color == 3 && depth == 16) || ((color == 2 || color == 4 || color == 6) && depth < 8)) { *error = "bad PNG depth/colour"; return false; }
	if (color == 3 && palette.empty()) { *error = "PNG palette missing"; return false; }

	// pass geometry (Adam7 or a single pass)
	static const int xo[7] = {0, 4, 0, 2, 0, 1, 0}, yo[7] = {0, 0, 4, 0, 2, 0, 1};
	static const int xs[7] = {8, 8, 4, 4, 2, 2, 1}, ys[7] = {8, 8, 8, 4, 4, 2, 2};
	const int passes = interlace ? 7 : 1;
	const int bits_pp = src_n * depth;
	const int bpp = bits_pp >= 8 ? bits_pp / 8 : 1;
	size_t total = 0;
	size_t pass_off[7], pass_stride[7];
	int pass_w[7], pass_h[7];
	for (int i = 0; i < passes; ++i) {
		pass_w[i] = interlace ? (int)((w - xo[i] + xs[i] - 1) / xs[i]) : (int)w;
		pass_h[i] = interlace ? (int)((h - yo[i] + ys[i] - 1) / ys[i]) : (int)h;
		if ((int)w <= xo[i] && interlace) pass_w[i] = 0;
		if ((int)h <= yo[i] && interlace) pass_h[i] = 0;
		pass_stride[i] = ((size_t)pass_w[i] * (size_t)bits_pp + 7) / 8;
		pass_off[i] = total;
		if (pass_w[i] && pass_h[i]) total += (size_t)pass_h[i] * (pass_stride[i] + 1);
	}

	std::vector<uint8_t> raw(total);
	{
		z_stream zs;
		std::memset(&zs, 0, sizeof zs);
		if (inflateInit(&zs) != Z_OK) { *error = "zlib init failed"; return false; }
		size_t in_pos = 0, out_pos = 0;
		int rc = Z_OK;
		while (rc != Z_STREAM_END && out_pos < total) {
			const size_t in_chunk = idat.size() - in_pos < (1u << 30) ? idat.size() - in_pos : (1u << 30);
			const size_t out_chunk = total - out_pos < (1u << 30) ? total - out_pos : (1u << 30);
			zs.next_in = idat.data() + in_pos;
			zs.avail_in = (uInt)in_chunk;
			zs.next_out = raw.data() + out_pos;
			zs.avail_out = (uInt)out_chunk;
			rc = inflate(&zs, Z_NO_FLUSH);
			in_pos += in_chunk - zs.avail_in;
			out_pos += out_chunk - zs.avail_out;
			if (rc != Z_OK && rc != Z_STREAM_END) break;
			if (in_chunk == 0 && rc == Z_OK) break;
		}
		inflateEnd(&zs);
		if (out_pos < total) { *error = "PNG data too short or corrupt"; return false; }
	}

	// samples at 16 bits per channel (low depths kept unscaled for palette indices / scaled for grey)
	std::vector<uint16_t> smp((size_t)w * h * (size_t)src_n);
	static const int depth_scale[9] = {0, 0xFF, 0x55, 0, 0x11, 0, 0, 0, 0x01};
	for (int pi = 0; pi < passes; ++pi) {
		if (!pass_w[pi] || !pass_h[pi]) continue;
		uint8_t *base = raw.data() + pass_off[pi];
		if (!unfilter(base, pass_h[pi], pass_stride[pi], bpp, error)) return false;
		for (int y = 0; y < pass_h[pi]; ++y) {
			const uint8_t *line = base + (size_t)y * (pass_stride[pi] + 1) + 1;
			const size_t oy = interlace ? (size_t)y * ys[pi] + yo[pi] : (size_t)y;
			for (int x = 0; x < pass_w[pi]; ++x) {
				const size_t ox = interlace ? (size_t)x * xs[pi] + xo[pi] : (size_t)x;
				uint16_t *dst = &smp[(oy * w + ox) * (size_t)src_n];
				for (int c = 0; c < src_n; ++c) {
					const size_t si = (size_t)x * src_n + c;
					if (depth == 16) dst[c] = (uint16_t)((line[2 * si] << 8) | line[2 * si + 1]);
					else if (depth == 8) dst[c] = line[si];
					else {
						const size_t bit = si * (size_t)depth;
						const int v = (line[bit >> 3] >> (8 - depth - (int)(bit & 7))) & ((1 << depth) - 1);
						dst[c] = (uint16_t)(color == 3 ? v : v * depth_scale[depth]);
					}
				}
			}
		}
	}

	const size_t npx = (size_t)w * h;
	out->w = (int)w;
	out->h = (int)h;
	if (out->keep16 && depth == 16) {
		out->px16 = smp;
		out->channels16 = src_n;
	}
	if (color == 3) {
		// palette expansion (stbi__expand_png_palette): RGB, or RGBA when a tRNS chunk exists
		const bool alpha = !trns.empty();
		out->channels = alpha ? 4 : 3;
		out->px.resize(npx * (size_t)out->channels);
		const size_t pal_n = palette.size() / 3;
		for (size_t i = 0; i < npx; ++i) {
			const size_t idx = smp[i];
			uint8_t *t = &out->px[i * (size_t)out->channels];
			if (idx < pal_n) { t[0] = palette[3 * idx]; t[1] = palette[3 * idx + 1]; t[2] = palette[3 * idx + 2]; }
			else { t[0] = t[1] = t[2] = 0; }
			if (alpha) t[3] = idx < trns.size() ? trns[idx] : 255;
		}
		return true;
	}

	// colour-key transparency (stbi__compute_transparency / 16): compared at the file's bit depth
	const bool keyed = !trns.empty() && (color == 0 || color == 2) && trns.size() >= (size_t)(2 * src_n);
	uint16_t key[3] = {0, 0, 0};
	if (keyed) {
		for (int c = 0; c < src_n; ++c) {
			const uint16_t v = (uint16_t)((trns[2 * c] << 8) | trns[2 * c + 1]);
			key[c] = depth == 16 ? v : (uint16_t)((v & 255) * depth_scale[depth]);
		}
	}
	out->channels = src_n + (keyed ? 1 : 0);
	out->px.resize(npx * (size_t)out->channels);
	for (size_t i = 0; i < npx; ++i) {
		const uint16_t *s = &smp[i * (size_t)src_n];
		uint8_t *t = &out->px[i * (size_t)out->channels];
		bool match = keyed;
		for (int c = 0; c < src_n; ++c) {
			t[c] = (uint8_t)(depth == 16 ? (s[c] >> 8) : s[c]);     // stbi__convert_16_to_8
			if (keyed && s[c] != key[c]) match = false;
		}
		if (keyed) t[src_n] = match ? 0 : 255;
	}
	return true;
}

// ---------------------------------------------------------------------------------------------
// binary PNM (P5 / P6, maxval <= 255; samples are taken as they are, like stb_image)
bool load_image(const std::string &path, int want_channels, Image *out, std::string *error) {
	std::vector<uint8_t> file;
	if (want_channels != 3 && want_channels != 4) { *error = "want_channels must be 3 or 4"; return false; }
	if (!read_file(path, &file)) { *error = "cannot read file"; return false; }
	return load_image_memory(file, want_channels, out, error);
}

bool load_image_memory(const std::vector<uint8_t> &file, int want_channels, Image *out, std::string *error) {
	std::string err;
	if (want_channels != 3 && want_channels != 4) { *error = "want_channels must be 3 or 4"; return false; }
	// Format by content, in the order stb tries its loaders (vendor/stb_image.h stbi__load_main :1118-1170):
	// PNG, BMP, GIF, PSD, PIC, JPEG, PNM, HDR, and TGA last because it has no signature.
	Decoded d;
	bool ok;
	const size_t n = file.size();
	if (n >= 8 && file[0] == 137 && file[1] == 'P' && file[2] == 'N' && file[3] == 'G') ok = decode_png(file, &d, &err);
	else if (looks_like_bmp(file)) ok = decode_bmp(file, &d, &err);
	else if (n >= 6 && !std::memcmp(file.data(), "GIF8", 4) && (file[4] == '7' || file[4] == '9') && file[5] == 'a') ok = decode_gif(file, &d, &err);
	else if (n >= 4 && !std::memcmp(file.data(), "8BPS", 4)) ok = decode_psd(file, &d, &err);
	else if (looks_like_pic(file)) ok = decode_pic(file, &d, &err);
	else if (n >= 2 && file[0] == 0xFF && file[1] == 0xD8) {
		if (!decode_jpeg(file, want_channels, out, &err)) { *error = err; return false; }
		return true;
	}
	else if (n >= 2 && file[0] == 'P' && (file[1] == '5' || file[1] == '6')) ok = decode_pnm(file, want_channels, &d, &err);
	else if (looks_like_hdr(file)) ok = decode_hdr(file, &d, &err);
	else if (looks_like_tga(file)) ok = decode_tga(file, &d, &err);
	else { ok = false; err = "unknown image type"; }
	if (!ok) { *error = err; return false; }
	convert_channels(d, want_channels, out);
	return true;
}

bool load_heightmap16(const std::string &path, Image16 *out, std::string *error) {
	std::vector<uint8_t> file;
	if (!read_file(path, &file)) { *error = path + ": cannot read file"; return false; }
	const size_t n = file.size();
	Decoded d;
	d.keep16 = true;
	std::string err;
	bool ok = true;
	bool decoded = false;
	if (n >= 8 && file[0] == 137 && file[1] == 'P' && file[2] == 'N' && file[3] == 'G') ok = decoded = decode_png(file, &d, &err);
	else if (n >= 2 && file[0] == 'P' && (file[1] == '5' || file[1] == '6')) ok = decoded = decode_pnm(file, 1, &d, &err);
	if (!ok) { *error = path + ": " + err; return false; }
	const size_t npx = (size_t)d.w * (size_t)d.h;
	out->samples.resize(npx);
	if (!d.px16.empty()) {
		// 16-bit samples as the file stores them: grey (+ alpha, dropped), or RGB(A) whose three channels agree
		const int cn = d.channels16;
		for (size_t i = 0; i < npx; ++i) {
			const uint16_t *t = &d.px16[i * (size_t)cn];
			if (cn >= 3 && (t[0] != t[1] || t[1] != t[2])) {
				*error = path + ": 16-bit heightmap is not grey (R, G and B differ at pixel " + std::to_string(i % (size_t)d.w) +
				         ", " + std::to_string(i / (size_t)d.w) + ")";
				return false;
			}
			out->samples[i] = t[0];
		}
		out->width = d.w;
		out->height = d.h;
		return true;
	}
	// everything else through the 8-bit decoder: it must be grey, and each sample v becomes 257 v (= v / 255 of 65535)
	Image img;
	if (decoded) convert_channels(d, 3, &img);
	else if (!load_image_memory(file, 3, &img, &err)) { *error = path + ": " + err; return false; }
	const size_t npx8 = (size_t)img.width * (size_t)img.height;
	out->samples.resize(npx8);
	for (size_t i = 0; i < npx8; ++i) {
		const uint8_t *t = &img.pixels[3 * i];
		if (t[0] != t[1] || t[1] != t[2]) {
			*error = path + ": heightmap is not grey (R, G and B differ at pixel " + std::to_string(i % (size_t)img.width) +
			         ", " + std::to_string(i / (size_t)img.width) + ")";
			return false;
		}
		out->samples[i] = (uint16_t)(t[0] * 257u);
	}
	out->width = img.width;
	out->height = img.height;
	return true;
}

bool write_bytes(const std::string &path, const uint8_t *data, size_t n) {
	FILE *f = std::fopen(path.c_str(), "wb");
	if (!f) return false;
	const bool wrote = n == 0 || std::fwrite(data, 1, n, f) == n;
	return std::fclose(f) == 0 && wrote;
}

} // namespace hmrm_host
