// Internals shared by the image decoders of the hmap host (image_io.cpp, image_formats.cpp, image_jpeg.cpp).
#ifndef HMRM_HOST_IMAGE_INTERNAL_HPP
#define HMRM_HOST_IMAGE_INTERNAL_HPP

#include "image_io.hpp"

namespace hmrm_host {

// A decoded image in its source channel count (1 grey, 2 grey+alpha, 3 RGB, 4 RGBA), 8 bits per sample.
struct Decoded {
	int w, h, channels;
	std::vector<uint8_t> px;
	// set by the caller: also keep the samples of a 16-bit PNG (not palette) or 16-bit PNM in px16 at full precision
	// (load_heightmap16), channels16 per pixel: the file's own channels, without the alpha a tRNS colour key adds to px
	bool keep16;
	int channels16;
	std::vector<uint16_t> px16;
	Decoded() : w(0), h(0), channels(0), keep16(false), channels16(0) {}
};

// stbi__convert_format for 8-bit data (vendor/stb_image.h:1735-1781): grey -> R=G=B, missing alpha -> 255, alpha dropped
void convert_channels(const Decoded &d, int want, Image *out);

// Format decoders: false + message on failure.  Each follows the loader of the same name in vendor/stb_image.h v2.27.
bool decode_png(const std::vector<uint8_t> &file, Decoded *out, std::string *error);
bool decode_pnm(const std::vector<uint8_t> &file, int want_channels, Decoded *out, std::string *error);
bool decode_tga(const std::vector<uint8_t> &file, Decoded *out, std::string *error);
bool decode_bmp(const std::vector<uint8_t> &file, Decoded *out, std::string *error);
bool decode_gif(const std::vector<uint8_t> &file, Decoded *out, std::string *error);
bool decode_psd(const std::vector<uint8_t> &file, Decoded *out, std::string *error);
bool decode_hdr(const std::vector<uint8_t> &file, Decoded *out, std::string *error);   // tone-mapped to 8 bit like stbi_load
bool decode_pic(const std::vector<uint8_t> &file, Decoded *out, std::string *error);
bool decode_jpeg(const std::vector<uint8_t> &file, int want_channels, Image *out, std::string *error);

// Content sniffing in stb's order (stbi__load_main, :1118-1170): tells which loader stb would pick.
bool looks_like_bmp(const std::vector<uint8_t> &file);
bool looks_like_tga(const std::vector<uint8_t> &file);
bool looks_like_hdr(const std::vector<uint8_t> &file);
bool looks_like_pic(const std::vector<uint8_t> &file);

} // namespace hmrm_host

#endif
