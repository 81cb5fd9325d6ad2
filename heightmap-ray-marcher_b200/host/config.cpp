// See config.hpp.  A table-driven restatement of the reference's option grammar: every identifier of
// main/hmap.cpp:314-485 with the same arity, echo text and side effects.
#include "config.hpp"

#include <cmath>
#include <iostream>
#include <istream>
#include <ostream>

namespace hmrm_host {

double degrees_to_rads(double degrees) { return (degrees / 180.0) * M_PI; }
double rads_to_degrees(double rads) { return (rads / M_PI) * 180.0; }

Config::Config()
	: screen_width(800), screen_height(600), hfov(M_PI / 2.0), min_height(0.0), max_height(10.0), lum_r(0.299),
	  lum_g(0.587), lum_b(0.114), grid_width(0.05), step_dist(5.0 * 0.05), cycle_period(47), cycle(0),
	  hang(-M_PI / 4.0), vang(M_PI / 2.0), mouse_sens(1.0), scroll_sens(1.0), move_speed(0.05),
	  ortho_width(2.0 * 0.05), recording_frame_count(200), image_plane(1), bg_r(0), bg_g(0), bg_b(0),
	  height_bits(8), maps_changed(false), should_update_heightmap(false) {
	cam_pos[0] = -5.0;
	cam_pos[1] = 5.0;
	cam_pos[2] = 0.0;
}

namespace {

// one echo line per option, in the reference's wording (main/hmap.cpp:197-280)
void echo(const Config &c, const std::string &id, std::ostream &o) {
	if (id == "heightmap") o << "heightmap " << c.heightmap_path << "\n";
	else if (id == "colormap") o << "colormap " << c.colormap_path << "\n";
	else if (id == "resolution") o << "resolution " << c.screen_width << " " << c.screen_height << "\n";
	else if (id == "hfov") o << "hfov " << rads_to_degrees(c.hfov) << "\n";
	else if (id == "hang") o << "hang " << rads_to_degrees(c.hang) << "\n";
	else if (id == "vang") o << "vang " << rads_to_degrees(c.vang) << "\n";
	else if (id == "pos") o << "pos " << c.cam_pos[0] << " " << c.cam_pos[1] << " " << c.cam_pos[2] << "\n";
	else if (id == "pos_x") o << "pos_x " << c.cam_pos[0] << "\n";
	else if (id == "pos_y") o << "pos_y " << c.cam_pos[1] << "\n";
	else if (id == "pos_z") o << "pos_z " << c.cam_pos[2] << "\n";
	else if (id == "min_height") o << "min_height " << c.min_height << "\n";
	else if (id == "max_height") o << "max_height " << c.max_height << "\n";
	else if (id == "lum") o << "lum " << c.lum_r << " " << c.lum_g << " " << c.lum_b << "\n";
	else if (id == "lum_r") o << "lum_r " << c.lum_r << "\n";
	else if (id == "lum_g") o << "lum_g " << c.lum_g << "\n";
	else if (id == "lum_b") o << "lum_b " << c.lum_b << "\n";
	else if (id == "grid_width") o << "grid_width " << c.grid_width << "\n";
	else if (id == "ortho_width") o << "ortho_width " << c.ortho_width << "\n";
	else if (id == "step_dist") o << "step_dist " << c.step_dist << "\n";
	else if (id == "bg_color") o << "bg_color " << (int)c.bg_r << " " << (int)c.bg_g << " " << (int)c.bg_b << "\n";
	else if (id == "cycle") o << "cycle " << c.cycle_period << "\n";
	else if (id == "mouse_sens") o << "mouse_sens " << c.mouse_sens << "\n";
	else if (id == "scroll_sens") o << "scroll_sens " << c.scroll_sens << "\n";
	else if (id == "move") o << "move " << c.move_speed << "\n";
	else if (id == "recording_frame_count") o << "recording_frame_count " << c.recording_frame_count << "\n";
}

struct ScalarOption {
	const char *id;
	double Config::*field;
	bool degrees;         // stored in radians, given in degrees (:367-384)
	bool touches_heights; // reruns the height prepass
};

const ScalarOption kScalars[] = {
	{"hfov", &Config::hfov, true, false},
	{"hang", &Config::hang, true, false},
	{"vang", &Config::vang, true, false},
	{"min_height", &Config::min_height, false, true},
	{"max_height", &Config::max_height, false, true},
	{"lum_r", &Config::lum_r, false, true},
	{"lum_g", &Config::lum_g, false, true},
	{"lum_b", &Config::lum_b, false, true},
	{"grid_width", &Config::grid_width, false, false},     // NB: does not touch step_dist / ortho_width (:441-444)
	{"ortho_width", &Config::ortho_width, false, false},
	{"step_dist", &Config::step_dist, false, false},
	{"mouse_sens", &Config::mouse_sens, false, false},
	{"scroll_sens", &Config::scroll_sens, false, false},
	{"move", &Config::move_speed, false, false},
};

bool load_map(const std::string &path, int channels, Image *dst, const char *what, std::ostream &err) {
	std::string why;
	Image img;
	if (!load_image(path, channels, &img, &why)) {
		// main/hmap.cpp:324-329, :345-350
		err << "Failed to load image for " << what << " from " << path << "\n";
		err << "  (" << why << ")\n";
		return false;
	}
	*dst = img;
	return true;
}

} // namespace

void print_all_options(const Config &c, std::ostream &o) {
	static const char *order[] = {"heightmap", "colormap", "resolution", "hfov", "hang", "vang", "pos", "min_height",
	                              "max_height", "lum", "grid_width", "ortho_width", "step_dist", "bg_color", "cycle",
	                              "mouse_sens", "scroll_sens", "move", "recording_frame_count"};
	for (size_t i = 0; i < sizeof order / sizeof order[0]; ++i) echo(c, order[i], o);
}

ParseStatus consume_config_stream(std::istream &input, Config &c, std::ostream &out, std::ostream &err) {
	c.should_update_heightmap = false;
	std::string id;
	while (input >> id) {
		bool handled = false;
		for (size_t i = 0; i < sizeof kScalars / sizeof kScalars[0] && !handled; ++i) {
			if (id != kScalars[i].id) continue;
			// A malformed number stores 0 and ends parsing at the next token read, as in the reference; a missing one (end
			// of the text) leaves the value alone: the reference extracts straight into its global.  (Its three angles
			// go through an uninitialised local, :367-384, and are indeterminate in that case; here they stay as well.)
			double v = c.*(kScalars[i].field);
			if (kScalars[i].degrees) v = rads_to_degrees(v);
			input >> v;
			c.*(kScalars[i].field) = kScalars[i].degrees ? degrees_to_rads(v) : v;
			if (kScalars[i].touches_heights) c.should_update_heightmap = true;
			echo(c, id, out);
			handled = true;
		}
		if (handled) continue;

		if (id == "heightmap") {
			input >> c.heightmap_path;
			if (c.height_bits == 16) {
				std::string why;
				Image16 img;
				if (!load_heightmap16(c.heightmap_path, &img, &why)) {
					err << "Failed to load image for heightmap from " << c.heightmap_path << "\n";
					err << "  (" << why << ")\n";
					return PARSE_FATAL;
				}
				c.heightmap16 = img;
			}
			else if (!load_map(c.heightmap_path, 3, &c.heightmap, "heightmap", err)) return PARSE_FATAL;
			c.should_update_heightmap = true;
			c.maps_changed = true;
			echo(c, id, out);
		}
		else if (id == "colormap") {
			input >> c.colormap_path;
			if (!load_map(c.colormap_path, 4, &c.colormap, "colormap", err)) return PARSE_FATAL;
			c.maps_changed = true;
			echo(c, id, out);
		}
		else if (id == "print") {
			out << "print\n";
			print_all_options(c, out);
		}
		else if (id == "resolution") {
			input >> c.screen_width >> c.screen_height;
			echo(c, id, out);
		}
		else if (id == "pos") {
			input >> c.cam_pos[0] >> c.cam_pos[1] >> c.cam_pos[2];
			echo(c, id, out);
		}
		else if (id == "pos_x" || id == "pos_y" || id == "pos_z") {
			input >> c.cam_pos[id[4] - 'x'];
			echo(c, id, out);
		}
		else if (id == "lum") {
			input >> c.lum_r >> c.lum_g >> c.lum_b;
			c.should_update_heightmap = true;
			echo(c, id, out);
		}
		else if (id == "lum_norm") {
			double r, g, b;
			input >> r >> g >> b;
			const double total = r + g + b;      // :419-422
			c.lum_r = r / total;
			c.lum_g = g / total;
			c.lum_b = b / total;
			c.should_update_heightmap = true;
			echo(c, "lum", out);
		}
		else if (id == "bg_color") {
			// The reference reads into three uninitialised ints (:456-457): when an extraction fails it stores 0 and the
			// components after it are indeterminate there.  Here they keep their current values.
			int r = c.bg_r, g = c.bg_g, b = c.bg_b;
			input >> r >> g >> b;
			c.bg_r = (unsigned char)r;
			c.bg_g = (unsigned char)g;
			c.bg_b = (unsigned char)b;
			echo(c, id, out);
		}
		else if (id == "cycle") {
			input >> c.cycle_period;
			c.cycle = 0;
			echo(c, id, out);
		}
		else if (id == "recording_frame_count") {
			input >> c.recording_frame_count;
			echo(c, id, out);
		}
		else {
			err << "WARNING: Unknown identifier: " << id << "\n";     // :486-488
		}
	}

	// validation, main/hmap.cpp:491-515
	const bool h16 = c.height_bits == 16;
	const int hw = h16 ? c.heightmap16.width : c.heightmap.width, hh = h16 ? c.heightmap16.height : c.heightmap.height;
	if (h16 ? c.heightmap16.samples.empty() : c.heightmap.pixels.empty()) {
		err << "Must specify heightmap in config\n";
		return PARSE_FATAL;
	}
	if (c.colormap.pixels.empty()) {
		err << "Must specify colormap in config\n";
		return PARSE_FATAL;
	}
	if (hw != c.colormap.width || hh != c.colormap.height) {
		err << "heightmap dimensions (" << hw << "x" << hh
		    << ") must match colormap dimensions (" << c.colormap.width << "x" << c.colormap.height << ")\n";
		return PARSE_FATAL;
	}
	return PARSE_OK;
}

} // namespace hmrm_host
