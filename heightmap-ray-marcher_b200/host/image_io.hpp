// Image ingest / output for the hmap host.
//
// The reference decodes its maps with stb_image (vendor/stb_image.h v2.27) as
//   heightmap: stbi_load(path, &w, &h, &n, 3)  -> RGB8   (main/hmap.cpp:320-321)
//   colormap : stbi_load(path, &w, &h, &n, 4)  -> RGBA8  (main/hmap.cpp:341-342)
// and writes frames with stbi_write_png(path, w, h, 4, buf, w*4) (main/hmap.cpp:158-160); hmap encodes its frames on
// the device instead (include/hmrm.h: hmrm_render_png_async, hmrm_encode_png) and only writes the files here.
// This is an independent implementation of the same *decoded-pixel contract* — for every file the pixels stb returns,
// byte for byte (tests/golden/images.json holds stb's own output for each flavour):
//   PNG   all colour types and bit depths, tRNS, Adam7                                   image_io.cpp
//   JPEG  baseline and progressive, 1 / 3 / 4 components, any subsampling, restarts      image_jpeg.cpp
//   BMP   1/4/8-bit palette, 16/24/32-bit with bit fields, OS/2 and V4/V5 headers         image_formats.cpp
//   GIF   first frame (interlace, transparency, local colour table, background fill)      image_formats.cpp
//   PSD   composited RGB(A), 8/16 bit, raw or RLE                                          image_formats.cpp
//   TGA   true colour 15/16/24/32, grey, grey+alpha, colour-mapped, raw or RLE            image_formats.cpp
//   PNM   binary P5 / P6, 8 bit, and 16 bit where stb's result is defined                 image_formats.cpp
//   PIC   Softimage: raw, pure and mixed run-length packets, any channel split            image_hdr_pic.cpp
//   HDR   Radiance RGBE, run-length or flat, tone-mapped to 8 bit as stbi_load does       image_hdr_pic.cpp
// The format is recognised from the file's content in stb's order (TGA last: it has no signature), not from its name.
// That is every format stbi_load reads; BMP RLE is refused by stb too.
//
// Conversion rules reproduced (vendor/stb_image.h: stbi__convert_format, stbi__convert_16_to_8,
// stbi__compute_transparency, stbi__expand_png_palette): grey -> R=G=B; missing alpha -> 255;
// 16-bit samples -> high byte; 1/2/4-bit grey scaled by 0xFF/0x55/0x11; palette + tRNS expansion;
// a tRNS colour key makes matching pixels alpha 0; dropping alpha just drops it.
#ifndef HMRM_HOST_IMAGE_IO_HPP
#define HMRM_HOST_IMAGE_IO_HPP

#include <stdint.h>

#include <string>
#include <vector>

namespace hmrm_host {

struct Image {
	int width, height, channels;      // channels as requested (3 or 4)
	std::vector<uint8_t> pixels;      // row-major, top row first
	Image() : width(0), height(0), channels(0) {}
};

// Decode `path` into 8-bit pixels with `want_channels` (3 = RGB, 4 = RGBA).  Returns false and a
// message in `error` on failure.
bool load_image(const std::string &path, int want_channels, Image *out, std::string *error);
// The same on a file already in memory (stbi_load_from_memory's role).
bool load_image_memory(const std::vector<uint8_t> &file, int want_channels, Image *out, std::string *error);

// One 16-bit sample per pixel: a heightmap loaded at full precision (hmrm_set_maps16).
struct Image16 {
	int width, height;
	std::vector<uint16_t> samples;    // row-major, top row first
	Image16() : width(0), height(0) {}
};

// Load a heightmap at 16 bits (hmap --height-bits 16):
//   16-bit PNG, grey or grey + alpha: the samples, alpha dropped;
//   16-bit PNG, RGB or RGBA: accepted only if R = G = B at every pixel (alpha dropped);
//   binary PGM / PPM (P5 / P6) with maxval > 255: the big-endian samples as stored (a PPM only if it is grey);
//   any other file: decoded by load_image to 8-bit RGB, which must be grey (R = G = B everywhere), and widened x257.
// Anything else is refused: false, and a message naming the file in `error`.
bool load_heightmap16(const std::string &path, Image16 *out, std::string *error);

// Write n bytes to `path` (a PNG file the device encoded: hmrm_render_png_async / hmrm_encode_png).  Returns false on
// failure.
bool write_bytes(const std::string &path, const uint8_t *data, size_t n);

} // namespace hmrm_host

#endif
