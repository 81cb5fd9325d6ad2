// hmap — the reference's binary (`./hmap path/to/config.txt`, main/hmap.cpp:526-544) with a headless
// render-to-PNG mode beside the (SDL) loop.  The config grammar is the reference's; the frame body
// main/hmap.cpp:952-1058 is one call into libhmrm.so (include/hmrm.h).  There is no CPU renderer here, and no CPU
// PNG encoder either: every PNG this program writes is filtered, deflated and framed on the device (kernel K3,
// hmrm_render_png_async / hmrm_encode_png), so only compressed bytes cross PCIe and the host only writes files.
//
//   hmap config.txt --headless out.png [--projection 1|2|3] [--precision fp64|fp32]
//                   [--traversal auto|brute|skip] [--gpus N] [--stats-json file]
//   hmap config.txt --script frames.txt [--frames N] [--out-prefix P | --record] [--gpus N] ...
//   hmap config.txt --script frames.txt --video FILE|- [--fps N] [--video-matrix bt601|bt709] ...
//   ... [--supersample 1|2|3|4]                    (anti-aliasing: the box filter of an N x N-times larger frame)
//   ... [--height-bits 8|16]                       (16: heightmaps load at full precision, hmrm_set_maps16)
//   ... [--jpeg Q [--jpeg-chroma 420|444]]         (JPEG files / Motion-JPEG video of quality Q instead of PNG / Y4M)
//   ... [--motion-blur K [--shutter F]]            (--script only: each frame averages K cameras towards the next one)
//   hmap config.txt --parse-only                    (grammar check: echo + validation, no GPU)
//   hmap --decode-image in.png 3|4|h16 out.raw      (image ingest check, no GPU; h16: little-endian u16 samples)
//
// --script: one line of config grammar per frame (what the reference's console accepts, :760-804),
// applied before the frame is rendered — the programmatic animation the reference leaves as a stub
// (:916-926).  Frame n goes to GPU n mod N, which renders and encodes it into one of four pinned PNG buffers it
// rotates; the oldest frame of a device is written to its file when that device needs the buffer again.  --record
// names files as the reference's recorder does (screenshots/hmap_<id>_<n>.png, :1132-1136) and prints its messages.
// --video writes the frames, in script order, as one YUV4MPEG2 stream of limited-range 4:2:0 planes converted on the
// device (kernel K4, hmrm_render_yuv420_async): the raw input every video encoder reads.  "-" is stdout, for a pipe
// into an encoder; the config echo and the messages then go to stderr.
// --headless with --gpus N > 1 assembles the frame's bands in one pinned host frame and device 0 encodes it.
// Projection is not part of the grammar (keys 1/2/3 only, :851-868), hence --projection.
// --supersample N renders every headless, recorded or video frame at N x N rays per pixel and box-filters it on the
// device (HMRM_FLAG_SUPERSAMPLE, kernel K5); the files keep the configured resolution.  Supersampled frames are whole
// frames, so --headless over several devices (tile-row bands) refuses N > 1; --script still deals whole frames to them.
// --height-bits 16 loads every `heightmap` of the config, the script and the console with load_heightmap16 (16-bit PNG
// and PNM samples as stored, grey 8-bit files widened x257) and passes it to hmrm_set_maps16; the default, 8, is the
// reference's RGB8 ingest.
// --jpeg Q (1-100) makes every still a JPEG file encoded on the device (kernel K6, hmrm_render_jpeg_async /
// hmrm_encode_jpeg; 4:2:0 unless --jpeg-chroma 444): --headless writes the path given, --script files end in .jpg.
// With --video it writes Motion-JPEG instead of Y4M: the frames' JPEG files back to back in script order, the stream
// `ffmpeg -f mjpeg -framerate N -i` reads.  Such a stream carries no frame rate or matrix, so --fps and
// --video-matrix are refused with --jpeg.
// --motion-blur K (1-16, --script only) blurs every recorded or video frame over the camera's motion to the next frame
// (hmrm_set_motion_blur, kernel K5).  With c_n the camera after script line n and c_{n+1} the camera of the next rendered
// frame, sub-frame j of frame n uses t = (F * j) / K and c = c_n + t * (c_{n+1} - c_n), per component of cam_pos, hang
// and vang, in doubles and in that order; F is --shutter (0 < F <= 1, default 0.5), the fraction of the frame interval
// the shutter stays open.  Angles are not wrapped: a turn from 350 to 370 degrees blurs over 20 degrees, one from 350
// to 10 over 340.  Line n+1 is applied once frame n's maps are on the devices and its frame is built, so frame n renders
// with exactly its own maps and fields.  The last rendered frame has no successor and is rendered without blur.
// --motion-blur 1 renders exactly the frames without the option.
// Headless frames are complete images: cycle_period is forced to 1 (the reference's own advice, :913).
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <ctime>
#include <deque>
#include <fstream>
#include <iostream>
#include <sstream>
#include <string>
#include <vector>

#include "../../include/hmrm.h"
#include "config.hpp"
#include "image_io.hpp"

using namespace hmrm_host;

#ifdef HMAP_WITH_SDL
namespace hmrm_host {
int run_interactive(Config &cfg, hmrm_ctx *ctx, int precision, int traversal);   // hmap_sdl.cpp
}
#endif

namespace {

struct Options {
	std::string config_path, headless_out, script_path, out_prefix, stats_json, video_path;
	int projection, precision, traversal, gpus, frames, fps, video_matrix, supersample, height_bits;
	int jpeg_quality, jpeg_chroma;   // jpeg_quality 0: PNG stills and Y4M video
	int motion_blur;                 // 0: not given
	double shutter;
	bool record, parse_only, supersample_given, y4m_option_given, jpeg_chroma_given, shutter_given;
	Options() : projection(0), precision(HMRM_FP64_EXACT), traversal(HMRM_TRAVERSAL_AUTO), gpus(1), frames(-1), fps(30),
	            video_matrix(HMRM_YUV_BT709), supersample(1), height_bits(8), jpeg_quality(0), jpeg_chroma(HMRM_JPEG_420),
	            motion_blur(0), shutter(0.5), record(false), parse_only(false), supersample_given(false),
	            y4m_option_given(false), jpeg_chroma_given(false), shutter_given(false) {}
};

void usage_and_exit() {
	std::cerr << "USAGE: hmap.exe path/to/config.txt\n";     // main/hmap.cpp:528
	std::cerr << "       hmap path/to/config.txt --headless out.png [--projection 1|2|3] [--precision fp64|fp32]\n"
	             "            [--traversal auto|brute|skip] [--gpus N] [--script frames.txt [--frames N]\n"
	             "            [--out-prefix P | --record | --video FILE|- [--fps N] [--video-matrix bt601|bt709]]]\n"
	             "            [--supersample 1|2|3|4] [--height-bits 8|16] [--jpeg Q [--jpeg-chroma 420|444]]\n"
	             "            [--motion-blur 1..16 [--shutter F]] [--stats-json file] [--parse-only]\n"
	             "       hmap --decode-image in 3|4|h16 out.raw\n";
	std::exit(1);
}

const int kPngInFlight = 4;   // PNG, JPEG or YUV frames one device may have in flight (the library's frame ring)

struct PngBuffer {
	uint8_t *file;            // pinned, hmrm_png_bound / hmrm_jpeg_bound bytes (Y4M video: hmrm_yuv420_bytes of planes)
	size_t cap;
	uint64_t *bytes;          // pinned: the file size the device writes
	int frame_index;
	PngBuffer() : file(NULL), cap(0), bytes(NULL), frame_index(-1) {}
};

struct Device {
	hmrm_ctx *ctx;
	uint8_t *host_frame;      // pinned RGBA8 (a frame split over several devices)
	size_t host_bytes;
	bool busy;
	PngBuffer png[kPngInFlight];
	int png_head, png_count;  // oldest frame in flight, frames in flight
	bool stats_pending;       // the most recent frame's statistics have not been collected yet
	Device() : ctx(NULL), host_frame(NULL), host_bytes(0), busy(false), png_head(0), png_count(0), stats_pending(false) {}
};

void die_hmrm(hmrm_ctx *ctx, const char *what) {
	std::cerr << "hmap: " << what << ": " << hmrm_last_error(ctx) << "\n";
	std::exit(1);
}

void push_maps(std::vector<Device> &devs, Config &cfg) {
	for (size_t i = 0; i < devs.size(); ++i) {
		if (cfg.maps_changed && cfg.height_bits == 16 &&
		    hmrm_set_maps16(devs[i].ctx, cfg.heightmap16.samples.data(), cfg.colormap.pixels.data(),
		                    cfg.heightmap16.width, cfg.heightmap16.height) != HMRM_OK)
			die_hmrm(devs[i].ctx, "hmrm_set_maps16");
		if (cfg.maps_changed && cfg.height_bits == 8 &&
		    hmrm_set_maps(devs[i].ctx, cfg.heightmap.pixels.data(), cfg.colormap.pixels.data(), cfg.heightmap.width,
		                  cfg.heightmap.height) != HMRM_OK)
			die_hmrm(devs[i].ctx, "hmrm_set_maps");
		if (cfg.maps_changed || cfg.should_update_heightmap) {
			const double lum[3] = {cfg.lum_r, cfg.lum_g, cfg.lum_b};
			if (hmrm_update_heightmap(devs[i].ctx, lum, cfg.min_height, cfg.max_height) != HMRM_OK)
				die_hmrm(devs[i].ctx, "hmrm_update_heightmap");
		}
	}
	cfg.maps_changed = false;
	cfg.should_update_heightmap = false;
}

hmrm_camera camera_of(const Config &cfg) {
	hmrm_camera c;
	c.cam_pos[0] = cfg.cam_pos[0];
	c.cam_pos[1] = cfg.cam_pos[1];
	c.cam_pos[2] = cfg.cam_pos[2];
	c.hang = cfg.hang;
	c.vang = cfg.vang;
	return c;
}

// --motion-blur: sub-frame j of k between cameras a and b (see the header comment)
hmrm_camera blur_camera(const hmrm_camera &a, const hmrm_camera &b, double shutter, int j, int k) {
	const double t = (shutter * j) / k;
	hmrm_camera c;
	for (int i = 0; i < 3; ++i) c.cam_pos[i] = a.cam_pos[i] + t * (b.cam_pos[i] - a.cam_pos[i]);
	c.hang = a.hang + t * (b.hang - a.hang);
	c.vang = a.vang + t * (b.vang - a.vang);
	return c;
}

hmrm_frame make_frame(const Config &cfg, const Options &opt) {
	hmrm_frame f;
	hmrm_frame_defaults(&f);
	f.projection = opt.projection ? opt.projection : cfg.image_plane;
	f.screen_width = cfg.screen_width;
	f.screen_height = cfg.screen_height;
	f.precision = opt.precision;
	f.cam_pos[0] = cfg.cam_pos[0];
	f.cam_pos[1] = cfg.cam_pos[1];
	f.cam_pos[2] = cfg.cam_pos[2];
	f.hang = cfg.hang;
	f.vang = cfg.vang;
	f.hfov = cfg.hfov;
	f.ortho_width = cfg.ortho_width;
	f.grid_width = cfg.grid_width;
	f.step_dist = cfg.step_dist;
	f.bg[0] = cfg.bg_r;
	f.bg[1] = cfg.bg_g;
	f.bg[2] = cfg.bg_b;
	f.cycle = 0;
	f.cycle_period = 1;
	f.traversal = opt.traversal;
	// counting costs per-warp atomics: only when the caller asked for the numbers (the cut-off status is always reported)
	f.flags = opt.stats_json.empty() ? 0u : HMRM_FLAG_STATS;
	f.flags |= HMRM_FLAG_SUPERSAMPLE(opt.supersample);
	return f;
}

void ensure_host_frame(Device &d, size_t bytes) {
	if (d.host_bytes >= bytes) return;
	if (d.host_frame) hmrm_host_free(d.host_frame);
	void *p = NULL;
	if (hmrm_host_alloc(&p, bytes) != HMRM_OK) {
		std::cerr << "hmap: cannot allocate " << bytes << " bytes of pinned host memory\n";
		std::exit(1);
	}
	d.host_frame = (uint8_t *)p;
	d.host_bytes = bytes;
}

void ensure_png_buffer(PngBuffer &b, size_t bytes) {
	if (!b.bytes) {
		void *p = NULL;
		if (hmrm_host_alloc(&p, sizeof(uint64_t)) != HMRM_OK) die_hmrm(NULL, "hmrm_host_alloc");
		b.bytes = (uint64_t *)p;
	}
	if (b.cap >= bytes) return;
	if (b.file) hmrm_host_free(b.file);
	void *p = NULL;
	if (hmrm_host_alloc(&p, bytes) != HMRM_OK) {
		std::cerr << "hmap: cannot allocate " << bytes << " bytes of pinned host memory\n";
		std::exit(1);
	}
	b.file = (uint8_t *)p;
	b.cap = bytes;
}

// worst-case size of the frame's file: JPEG with --jpeg, else PNG
size_t file_bound_of(const hmrm_frame &f, const Options &opt) {
	if (opt.jpeg_quality) return hmrm_jpeg_bound(f.screen_width, f.screen_height, opt.jpeg_chroma);
	return hmrm_png_bound(f.screen_width, f.screen_height, f.pixel_format == HMRM_PIXEL_RGB8 ? 3 : 4);
}

// render f and encode it on the device into b (JPEG with --jpeg, else PNG)
void render_file_async(hmrm_ctx *ctx, const hmrm_frame &f, const Options &opt, PngBuffer &b) {
	if (opt.jpeg_quality) {
		if (hmrm_render_jpeg_async(ctx, &f, opt.jpeg_quality, opt.jpeg_chroma, b.file, b.cap, b.bytes) != HMRM_OK)
			die_hmrm(ctx, "hmrm_render_jpeg_async");
	}
	else if (hmrm_render_png_async(ctx, &f, b.file, b.cap, b.bytes) != HMRM_OK)
		die_hmrm(ctx, "hmrm_render_png_async");
}

struct Totals {
	long long frames, rays, box_hits, surf_hits, steps, fetches, png_bytes, jpeg_bytes, video_bytes;
	double kernel_ms;
	int status;
	Totals() : frames(0), rays(0), box_hits(0), surf_hits(0), steps(0), fetches(0), png_bytes(0), jpeg_bytes(0),
	           video_bytes(0), kernel_ms(0.0), status(0) {}
};

// SavePNG, main/hmap.cpp:157-168: the file's bytes (PNG, or JPEG with --jpeg) come from the device encoder
void save_image(const uint8_t *file, uint64_t bytes, const std::string &path, const Options &opt, Totals &t) {
	if (!write_bytes(path, file, (size_t)bytes)) std::cerr << "Failed to write screenshot to " << path << "\n";
	else {
		(opt.jpeg_quality ? t.jpeg_bytes : t.png_bytes) += (long long)bytes;
		std::cout << "Saved screenshot at " << path << "\n";
	}
}

void collect(Device &d, Totals &t) {
	hmrm_stats st;
	if (hmrm_get_stats(d.ctx, &st) != HMRM_OK) die_hmrm(d.ctx, "hmrm_get_stats");
	t.frames += 1;
	t.rays += st.rays;
	t.box_hits += st.box_hits;
	t.surf_hits += st.surf_hits;
	t.steps += st.steps;
	t.fetches += st.fetches;
	t.kernel_ms += st.kernel_ms;
	t.status |= st.status;
}

int decode_image_mode(int argc, char **argv) {
	if (argc != 5) usage_and_exit();
	std::string why;
	if (std::strcmp(argv[3], "h16") == 0) {
		Image16 img;
		if (!load_heightmap16(argv[2], &img, &why)) {
			std::cerr << "Failed to load image from " << argv[2] << " (" << why << ")\n";
			return 1;
		}
		std::vector<uint8_t> le(img.samples.size() * 2);
		for (size_t i = 0; i < img.samples.size(); ++i) {
			le[2 * i] = (uint8_t)(img.samples[i] & 255u);
			le[2 * i + 1] = (uint8_t)(img.samples[i] >> 8);
		}
		std::ofstream out(argv[4], std::ios::binary);
		out.write((const char *)le.data(), (std::streamsize)le.size());
		std::cout << img.width << " " << img.height << " 1\n";
		return out ? 0 : 1;
	}
	Image img;
	if (!load_image(argv[2], std::atoi(argv[3]), &img, &why)) {
		std::cerr << "Failed to load image from " << argv[2] << " (" << why << ")\n";
		return 1;
	}
	std::ofstream out(argv[4], std::ios::binary);
	out.write((const char *)img.pixels.data(), (std::streamsize)img.pixels.size());
	std::cout << img.width << " " << img.height << " " << img.channels << "\n";
	return out ? 0 : 1;
}

} // namespace

int main(int argc, char **argv) {
	if (argc >= 2 && std::strcmp(argv[1], "--decode-image") == 0) return decode_image_mode(argc, argv);
	if (argc < 2) usage_and_exit();

	Options opt;
	opt.config_path = argv[1];
	for (int i = 2; i < argc; ++i) {
		const std::string a = argv[i];
		const bool has_val = i + 1 < argc;
		if (a == "--headless" && has_val) opt.headless_out = argv[++i];
		else if (a == "--projection" && has_val) opt.projection = std::atoi(argv[++i]);
		else if (a == "--precision" && has_val) {
			const std::string v = argv[++i];
			if (v == "fp64") opt.precision = HMRM_FP64_EXACT;
			else if (v == "fp32") opt.precision = HMRM_FP32_FAST;
			else usage_and_exit();
		}
		else if (a == "--traversal" && has_val) {
			const std::string v = argv[++i];
			opt.traversal = v == "brute" ? HMRM_TRAVERSAL_BRUTE : v == "skip" ? HMRM_TRAVERSAL_SKIP : HMRM_TRAVERSAL_AUTO;
		}
		else if (a == "--gpus" && has_val) opt.gpus = std::atoi(argv[++i]);
		else if (a == "--script" && has_val) opt.script_path = argv[++i];
		else if (a == "--frames" && has_val) opt.frames = std::atoi(argv[++i]);
		else if (a == "--out-prefix" && has_val) opt.out_prefix = argv[++i];
		else if (a == "--record") opt.record = true;
		else if (a == "--stats-json" && has_val) opt.stats_json = argv[++i];
		else if (a == "--parse-only") opt.parse_only = true;
		else if (a == "--video" && has_val) opt.video_path = argv[++i];
		else if (a == "--fps" && has_val) {
			opt.fps = std::atoi(argv[++i]);
			opt.y4m_option_given = true;
		}
		else if (a == "--height-bits" && has_val) {
			const std::string v = argv[++i];
			if (v == "8") opt.height_bits = 8;
			else if (v == "16") opt.height_bits = 16;
			else usage_and_exit();
		}
		else if (a == "--supersample" && has_val) {
			opt.supersample = std::atoi(argv[++i]);
			opt.supersample_given = true;
		}
		else if (a == "--video-matrix" && has_val) {
			const std::string v = argv[++i];
			if (v == "bt601") opt.video_matrix = HMRM_YUV_BT601;
			else if (v == "bt709") opt.video_matrix = HMRM_YUV_BT709;
			else usage_and_exit();
			opt.y4m_option_given = true;
		}
		else if (a == "--jpeg" && has_val) {
			opt.jpeg_quality = std::atoi(argv[++i]);
			if (opt.jpeg_quality < 1 || opt.jpeg_quality > 100) usage_and_exit();
		}
		else if (a == "--motion-blur" && has_val) {
			opt.motion_blur = std::atoi(argv[++i]);
			if (opt.motion_blur < 1 || opt.motion_blur > 16) usage_and_exit();
		}
		else if (a == "--shutter" && has_val) {
			const char *v = argv[++i];
			char *end = NULL;
			opt.shutter = std::strtod(v, &end);
			if (end == v || *end != '\0' || !(opt.shutter > 0.0 && opt.shutter <= 1.0)) usage_and_exit();
			opt.shutter_given = true;
		}
		else if (a == "--jpeg-chroma" && has_val) {
			const std::string v = argv[++i];
			if (v == "420") opt.jpeg_chroma = HMRM_JPEG_420;
			else if (v == "444") opt.jpeg_chroma = HMRM_JPEG_444;
			else usage_and_exit();
			opt.jpeg_chroma_given = true;
		}
		else usage_and_exit();
	}
	if (opt.projection < 0 || opt.projection > 3 || opt.gpus < 1 || opt.fps < 1) usage_and_exit();
	if (opt.supersample < 1 || opt.supersample > 4) usage_and_exit();
	// one frame over several devices is dealt in tile-row bands, which supersampled frames are not
	if (opt.supersample > 1 && !opt.headless_out.empty() && opt.script_path.empty() && opt.gpus > 1) usage_and_exit();
	// motion blur needs the next frame's camera: recordings only
	if (opt.motion_blur && (opt.script_path.empty() || !opt.headless_out.empty())) usage_and_exit();
	if (opt.shutter_given && !opt.motion_blur) usage_and_exit();
	const bool blur = opt.motion_blur > 1;
	const bool video = !opt.video_path.empty();
	if (video && (opt.script_path.empty() || !opt.headless_out.empty() || opt.record || !opt.out_prefix.empty()))
		usage_and_exit();
	if (opt.jpeg_chroma_given && !opt.jpeg_quality) {
		std::cerr << "hmap: --jpeg-chroma chooses the chroma of JPEG files; it needs --jpeg Q\n";
		return 1;
	}
	if (opt.jpeg_quality && opt.y4m_option_given) {
		std::cerr << "hmap: --fps and --video-matrix describe a Y4M stream; with --jpeg the video is Motion-JPEG, which "
		             "carries neither\n";
		return 1;
	}
	// a video on stdout leaves stdout to the stream
	std::ostream &msg = opt.video_path == "-" ? std::cerr : std::cout;

	// main/hmap.cpp:534-544
	std::ifstream input(opt.config_path.c_str());
	if (!input.is_open()) {
		std::cerr << "Failed to open input file: " << opt.config_path << "\n";
		return 1;
	}
	Config cfg;
	cfg.height_bits = opt.height_bits;
	if (consume_config_stream(input, cfg, msg, std::cerr) != PARSE_OK) return 1;
	input.close();
	if (opt.parse_only) return 0;

#ifndef HMAP_WITH_SDL
	if (opt.headless_out.empty() && opt.script_path.empty()) {
		std::cerr << "hmap: this build has no SDL window (SDL2 is not available here); use --headless out.png "
		             "or --script frames.txt\n";
		return 1;
	}
#endif

	const int available = hmrm_device_count();
	if (available < 1) {
		std::cerr << "hmap: no CUDA device; there is no CPU renderer\n";
		return 1;
	}
	// HMAP_DEVICE_LIST=2,3,5 picks the CUDA devices --gpus counts over (a device may be listed more than once: several
	// contexts then share it, which is how the multi-device paths are tested on a one-GPU box)
	std::vector<int> device_ids;
	if (const char *list = std::getenv("HMAP_DEVICE_LIST")) {
		std::stringstream ls(list);
		std::string item;
		while (std::getline(ls, item, ',')) {
			const int id = std::atoi(item.c_str());
			if (id < 0 || id >= available) {
				std::cerr << "hmap: HMAP_DEVICE_LIST names device " << id << " but " << available << " device(s) are present\n";
				return 1;
			}
			device_ids.push_back(id);
		}
	}
	else {
		for (int i = 0; i < available; ++i) device_ids.push_back(i);
	}
	if (opt.gpus > (int)device_ids.size()) {
		std::cerr << "hmap: --gpus " << opt.gpus << " but only " << device_ids.size() << " device(s) present\n";
		return 1;
	}
	std::vector<Device> devs((size_t)opt.gpus);
	for (int i = 0; i < opt.gpus; ++i) {
		if (hmrm_create(device_ids[(size_t)i], &devs[(size_t)i].ctx) != HMRM_OK) die_hmrm(NULL, "hmrm_create");
	}
	cfg.maps_changed = true;
	push_maps(devs, cfg);

#ifdef HMAP_WITH_SDL
	if (opt.headless_out.empty() && opt.script_path.empty()) {
		// the reference's interactive mode: `hmap config.txt`
		if (opt.projection) cfg.image_plane = opt.projection;
		const int rc = run_interactive(cfg, devs[0].ctx, opt.precision, opt.traversal);
		for (size_t i = 0; i < devs.size(); ++i) hmrm_destroy(devs[i].ctx);
		return rc;
	}
#endif

	Totals totals;
	const std::clock_t t_start = std::clock();

	if (opt.script_path.empty()) {
		// ---- one frame; with several GPUs its 4-row tile rows are dealt round-robin to the devices (interleaved:
		// sky rows cost nothing and terrain rows do, so contiguous bands balance badly) ----
		hmrm_frame f = make_frame(cfg, opt);
		PngBuffer &out = devs[0].png[0];
		ensure_png_buffer(out, file_bound_of(f, opt));
		const int G = opt.gpus;
		if (G == 1) {
			render_file_async(devs[0].ctx, f, opt, out);
			if (hmrm_wait(devs[0].ctx) != HMRM_OK) die_hmrm(devs[0].ctx, "hmrm_wait");
			collect(devs[0], totals);
		}
		else {
			const size_t bytes = (size_t)f.screen_width * (size_t)f.screen_height * 4;
			ensure_host_frame(devs[0], bytes);
			for (int g = 0; g < G; ++g) {
				hmrm_frame fb = f;
				fb.band_count = G;
				fb.band_index = g;
				if (g * 4 >= f.screen_height) continue;       // more devices than tile rows
				// every device copies its own tile rows straight into the one pinned host frame
				if (hmrm_render_async(devs[(size_t)g].ctx, &fb, devs[0].host_frame) != HMRM_OK)
					die_hmrm(devs[(size_t)g].ctx, "hmrm_render");
				devs[(size_t)g].busy = true;
			}
			for (int g = 0; g < G; ++g) {
				if (!devs[(size_t)g].busy) continue;
				if (hmrm_wait(devs[(size_t)g].ctx) != HMRM_OK) die_hmrm(devs[(size_t)g].ctx, "hmrm_wait");
				collect(devs[(size_t)g], totals);
				devs[(size_t)g].busy = false;
			}
			if (opt.jpeg_quality) {
				if (hmrm_encode_jpeg(devs[0].ctx, devs[0].host_frame, f.screen_width, f.screen_height, 4, opt.jpeg_quality,
				                     opt.jpeg_chroma, out.file, out.cap, out.bytes) != HMRM_OK)
					die_hmrm(devs[0].ctx, "hmrm_encode_jpeg");
			}
			else if (hmrm_encode_png(devs[0].ctx, devs[0].host_frame, f.screen_width, f.screen_height, 4, out.file,
			                         out.cap, out.bytes) != HMRM_OK)
				die_hmrm(devs[0].ctx, "hmrm_encode_png");
		}
		totals.frames = 1;
		save_image(out.file, *out.bytes, opt.headless_out, opt, totals);
	}
	else {
		// ---- recording: one grammar line per frame, frame n rendered and encoded on GPU n mod N ----
		std::ifstream script(opt.script_path.c_str());
		if (!script.is_open()) {
			std::cerr << "Failed to open input file: " << opt.script_path << "\n";
			return 1;
		}
		std::vector<std::string> lines;
		std::string line;
		while (std::getline(script, line)) {
			if (line.find_first_not_of(" \t\r\n") != std::string::npos) lines.push_back(line);
		}
		int n_frames = opt.frames >= 0 ? opt.frames : (int)lines.size();
		if (opt.record && opt.frames < 0 && lines.empty()) n_frames = cfg.recording_frame_count;
		const std::time_t recording_id = std::time(NULL);      // :879

		const char *ext = opt.jpeg_quality ? ".jpg" : ".png";
		auto frame_path = [&](int n) {
			std::ostringstream ss;
			if (opt.record || opt.out_prefix.empty()) ss << "screenshots/hmap_" << recording_id << "_" << n << ext;   // :1132-1134
			else ss << opt.out_prefix << n << ext;
			return ss.str();
		};
		// statistics are of a context's most recent render: read them before the device gets its next frame (the
		// read waits for that render only, not for its encoding)
		auto collect_pending = [&](Device &d) {
			if (!d.stats_pending) return;
			collect(d, totals);
			d.stats_pending = false;
		};
		// --video: one Y4M (or, with --jpeg, Motion-JPEG) stream; frames leave the devices in script order, through one
		// FIFO of the devices of the frames in flight (each device's own frames are in order in its ring)
		FILE *vf = NULL;
		int video_w = 0, video_h = 0;
		long long video_frames = 0;
		std::deque<int> video_order;
		if (video) {
			vf = opt.video_path == "-" ? stdout : std::fopen(opt.video_path.c_str(), "wb");
			if (!vf) {
				std::cerr << "hmap: cannot open " << opt.video_path << " for writing\n";
				return 1;
			}
		}
		auto video_write = [&](const void *p, size_t n) {
			if (std::fwrite(p, 1, n, vf) != n) {
				std::cerr << "hmap: writing the video to " << opt.video_path << " failed\n";
				std::exit(1);
			}
			totals.video_bytes += (long long)n;
		};
		auto video_header = [&](int w, int h) {
			// C420jpeg: the 2x2 box puts chroma at the centre of the block
			char head[160];
			const int n = std::snprintf(head, sizeof head, "YUV4MPEG2 W%d H%d F%d:1 Ip A1:1 C420jpeg XCOLORRANGE=LIMITED\n",
			                            w, h, opt.fps);
			video_write(head, (size_t)n);
			video_w = w;
			video_h = h;
		};
		// the oldest frame of the device is complete once at most png_count - 1 newer ones are pending
		auto retire_oldest = [&](Device &d) {
			if (hmrm_wait_pending(d.ctx, d.png_count - 1) != HMRM_OK) die_hmrm(d.ctx, "hmrm_wait_pending");
			const PngBuffer &b = d.png[d.png_head];
			if (video && opt.jpeg_quality) {
				video_write(b.file, (size_t)*b.bytes);
				totals.jpeg_bytes += (long long)*b.bytes;
				video_frames += 1;
			}
			else if (video) {
				video_write("FRAME\n", 6);
				video_write(b.file, hmrm_yuv420_bytes(video_w, video_h));
				video_frames += 1;
			}
			else save_image(b.file, *b.bytes, frame_path(b.frame_index), opt, totals);
			d.png_head = (d.png_head + 1) % kPngInFlight;
			d.png_count -= 1;
		};
		auto retire_first_video_frame = [&]() {
			const int g = video_order.front();
			video_order.pop_front();
			retire_oldest(devs[(size_t)g]);
		};
		auto drain_all = [&]() {
			for (size_t i = 0; i < devs.size(); ++i) collect_pending(devs[i]);
			if (video) while (!video_order.empty()) retire_first_video_frame();
			for (size_t i = 0; i < devs.size(); ++i)
				while (devs[i].png_count > 0) retire_oldest(devs[i]);
		};

		auto apply_line = [&](int n) {
			if (n >= (int)lines.size()) return true;
			std::istringstream iss(lines[(size_t)n]);
			return consume_config_stream(iss, cfg, msg, std::cerr) == PARSE_OK;
		};
		bool line_applied = false;      // --motion-blur: line n was applied while frame n - 1 was set up
		for (int n = 0; n < n_frames; ++n) {
			if (!line_applied && !apply_line(n)) return 1;
			line_applied = false;
			if (video && !opt.jpeg_quality && n > 0 && (cfg.screen_width != video_w || cfg.screen_height != video_h)) {
				// the frames before this one stay a valid stream
				drain_all();
				std::fflush(vf);
				if (vf != stdout) std::fclose(vf);
				std::cerr << "hmap: frame " << n << " changes the resolution from " << video_w << "x" << video_h << " to "
				          << cfg.screen_width << "x" << cfg.screen_height << "; a Y4M stream has one frame size\n";
				return 1;
			}
			Device &d = devs[(size_t)(n % opt.gpus)];
			if (video) {
				while (d.png_count == kPngInFlight) retire_first_video_frame();
			}
			else if (d.png_count == kPngInFlight) retire_oldest(d);
			if (cfg.maps_changed || cfg.should_update_heightmap) {
				drain_all();
				push_maps(devs, cfg);
			}
			collect_pending(d);
			const hmrm_frame f = make_frame(cfg, opt);
			if (blur) {
				// the cameras from this frame's towards the next rendered frame's; the last frame is plain
				hmrm_camera cams[16];
				int k = 0;
				if (n + 1 < n_frames) {
					const hmrm_camera from = camera_of(cfg);
					if (!apply_line(n + 1)) return 1;
					line_applied = true;
					const hmrm_camera to = camera_of(cfg);
					for (k = 0; k < opt.motion_blur; ++k) cams[k] = blur_camera(from, to, opt.shutter, k, opt.motion_blur);
				}
				if (hmrm_set_motion_blur(d.ctx, cams, k) != HMRM_OK) die_hmrm(d.ctx, "hmrm_set_motion_blur");
			}
			PngBuffer &b = d.png[(d.png_head + d.png_count) % kPngInFlight];
			if (video && !opt.jpeg_quality) {
				if (n == 0) video_header(f.screen_width, f.screen_height);
				ensure_png_buffer(b, hmrm_yuv420_bytes(f.screen_width, f.screen_height));
				if (hmrm_render_yuv420_async(d.ctx, &f, opt.video_matrix, b.file, b.cap) != HMRM_OK)
					die_hmrm(d.ctx, "hmrm_render_yuv420_async");
			}
			else {
				ensure_png_buffer(b, file_bound_of(f, opt));
				render_file_async(d.ctx, f, opt, b);
			}
			if (video) video_order.push_back(n % opt.gpus);
			b.frame_index = n;
			d.png_count += 1;
			d.stats_pending = true;
		}
		drain_all();
		if (video) {
			if (n_frames <= 0 && !opt.jpeg_quality) video_header(cfg.screen_width, cfg.screen_height);
			if (std::fflush(vf) != 0 || (vf != stdout && std::fclose(vf) != 0)) {
				std::cerr << "hmap: writing the video to " << opt.video_path << " failed\n";
				return 1;
			}
			msg << "Saved video at " << opt.video_path << " (" << video_frames << " frames)\n";
		}
		else std::cout << "Done recording.\n";      // :1142
	}

	if (totals.status & HMRM_ERR_NONTERMINATING)
		std::cerr << "WARNING: some rays can never leave the grid (the reference would hang); they were cut off\n";

	if (!opt.stats_json.empty()) {
		std::ofstream js(opt.stats_json.c_str());
		js << "{\"frames\": " << totals.frames << ", \"rays\": " << totals.rays << ", \"box_hits\": " << totals.box_hits
		   << ", \"surf_hits\": " << totals.surf_hits << ", \"steps\": " << totals.steps << ", \"fetches\": "
		   << totals.fetches << ", \"kernel_ms\": " << totals.kernel_ms << ", \"status\": " << totals.status
		   << ", \"gpus\": " << opt.gpus << ", \"cpu_seconds\": " << (double)(std::clock() - t_start) / CLOCKS_PER_SEC
		   << ", \"png_bytes\": " << totals.png_bytes;
		if (opt.jpeg_quality) js << ", \"jpeg_bytes\": " << totals.jpeg_bytes;
		if (video) js << ", \"video_bytes\": " << totals.video_bytes;
		if (opt.supersample_given) js << ", \"supersample\": " << opt.supersample;
		if (opt.motion_blur) js << ", \"motion_blur\": " << opt.motion_blur << ", \"shutter\": " << opt.shutter;
		js << "}\n";
	}

	for (size_t i = 0; i < devs.size(); ++i) {
		if (devs[i].host_frame) hmrm_host_free(devs[i].host_frame);
		for (int k = 0; k < kPngInFlight; ++k) {
			if (devs[i].png[k].file) hmrm_host_free(devs[i].png[k].file);
			if (devs[i].png[k].bytes) hmrm_host_free(devs[i].png[k].bytes);
		}
		hmrm_destroy(devs[i].ctx);
	}
	return 0;
}
