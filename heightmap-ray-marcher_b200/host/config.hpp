// The reference's configuration state and grammar (main/hmap.cpp:28-112 globals, :309-520 parser),
// kept as the API surface of the `hmap` binary: same identifiers, same arity, same echo lines on
// stdout, same warnings and validation messages on stderr, last value wins.
#ifndef HMRM_HOST_CONFIG_HPP
#define HMRM_HOST_CONFIG_HPP

#include <iosfwd>
#include <string>

#include "image_io.hpp"

namespace hmrm_host {

struct Config {
	// names and defaults follow the reference's globals
	int screen_width, screen_height;          // main/hmap.cpp:31-32
	double hfov;                              // :35  (radians)
	double min_height, max_height;            // :38-39
	double lum_r, lum_g, lum_b;               // :45-47
	std::string heightmap_path, colormap_path;
	double grid_width;                        // :65
	double step_dist;                         // :68
	int cycle_period, cycle;                  // :71-72
	double cam_pos[3];                        // :75
	double hang, vang;                        // :80, :85 (radians)
	double mouse_sens, scroll_sens, move_speed;   // :88-93 (parsed and echoed; only the interactive shell uses them)
	double ortho_width;                       // :98
	int recording_frame_count;                // :102
	int image_plane;                          // :107 (selected by keys 1/2/3 in the reference; --projection here)
	unsigned char bg_r, bg_g, bg_b;           // :110-112

	Image heightmap;                          // RGB8  (stbi_load(...,3), :320-321), with height_bits 8
	Image16 heightmap16;                      // one 16-bit sample per pixel (load_heightmap16), with height_bits 16
	int height_bits;                          // 8 | 16 (hmap --height-bits): the depth the `heightmap` key loads at
	Image colormap;                           // RGBA8 (stbi_load(...,4), :341-342)

	// change tracking for the caller (what must be pushed to the device)
	bool maps_changed;                        // a heightmap or colormap token was consumed
	bool should_update_heightmap;             // :310, :331, :403, :408, :413, :423, :428, :433, :438

	Config();
};

enum ParseStatus {
	PARSE_OK = 0,
	PARSE_FATAL = 1      // the reference calls std::exit(1) here; the message has been written to `err`
};

// ConsumeConfigStream (main/hmap.cpp:309-520): reads `input` to its end, updates `cfg`, echoes to `out`,
// warns / reports to `err`.
ParseStatus consume_config_stream(std::istream &input, Config &cfg, std::ostream &out, std::ostream &err);

// PrintAllOptions (main/hmap.cpp:282-302)
void print_all_options(const Config &cfg, std::ostream &out);

double degrees_to_rads(double degrees);       // :131-133
double rads_to_degrees(double rads);          // :135-137

} // namespace hmrm_host

#endif
