// Interactive shell of `hmap` (only with -DHMAP_WITH_SDL): the reference's SDL application loop
// (main/hmap.cpp:546-1161) around the GPU renderer.  SDL2 / SDL2_ttf are not installable in the build image, so
// the default build leaves this file empty and `hmap` is headless; the tests build it against the scripted fake SDL
// of the test oracle and compare its frames with the unmodified reference driven by the same event script.
//
// What is kept from the reference, event by event (line numbers in main/hmap.cpp):
//   loop top: ticks -> delta (:652-657); look/up/forward/right from hang/vang BEFORE events (:661-685), so console or
//             mouse changes of hang/vang reach Perspective/Orthographic one frame late while Spherical, cam_pos, hfov
//             and ortho_width are read after the events (:952-965) — SURVEY.md D-6
//   events:   quit, resize (:693-713), focus (:714-727), mouse look with vang clamped to [0, pi] (:729-739), wheel zoom
//             of hfov / ortho_width (:740-759), console text (:760-762), keys: Ctrl+Q, `, Backspace, Return (parses the
//             console line with the config grammar), F1, F11, F12 (screenshot of the PREVIOUS frame), 1/2/3, Ctrl+Shift+R
//   movement: W/S/D/A/Space/Q scaled by delta * move (:928-950), only without modifiers and with the console closed
//   render:   cycle = (cycle + 1) % cycle_period (:976), then the frame body — here one hmrm_render call
//   present:  FPS / console overlays (:1060-1125), SDL_UpdateTexture + RenderCopy + RenderPresent (:1082-1127)
//   record:   screenshots/hmap_<id>_<n>.png after each frame, "Done recording." (:1131-1144); screenshots and recorded
//             frames are PNG-encoded on the device (hmrm_encode_png)
#ifdef HMAP_WITH_SDL

#include <SDL2/SDL.h>
#include <SDL2/SDL_ttf.h>

#include <cmath>
#include <cstdlib>
#include <ctime>
#include <iomanip>
#include <iostream>
#include <sstream>
#include <string>
#include <vector>

#include "../../include/hmrm.h"
#include "config.hpp"
#include "image_io.hpp"

namespace hmrm_host {

namespace {

struct Basis {
	double forward[3], right[3];
	double hang, vang;      // the angles look/up are derived from this iteration
};

struct Shell {
	Config &cfg;
	hmrm_ctx *ctx;
	int precision, traversal;

	SDL_Window *window;
	SDL_Renderer *renderer;
	SDL_Texture *texture;
	TTF_Font *font;
	SDL_Surface *fps_surface, *console_surface;
	std::vector<uint8_t> framebuf;
	uint8_t *png_file;       // pinned PNG file of the last screenshot, png_cap bytes
	size_t png_cap;
	uint64_t *png_bytes;     // pinned: its size

	bool quit, show_fps, console_active, recording, fullscreen;
	std::string console_buf;
	std::time_t recording_id;
	int recording_frame_num;
	Uint32 text_timer_ms;

	Shell(Config &c, hmrm_ctx *x, int prec, int trav)
		: cfg(c), ctx(x), precision(prec), traversal(trav), window(NULL), renderer(NULL), texture(NULL), font(NULL),
		  fps_surface(NULL), console_surface(NULL), png_file(NULL), png_cap(0), png_bytes(NULL), quit(false), show_fps(false), console_active(false), recording(false),
		  fullscreen(false), console_buf(" "), recording_id(0), recording_frame_num(0), text_timer_ms(201) {}

	void fatal(const std::string &msg) {
		std::cerr << msg << "\n";
		std::exit(1);
	}

	void push_maps_if_needed() {
		if (cfg.maps_changed && cfg.height_bits == 16 &&
		    hmrm_set_maps16(ctx, cfg.heightmap16.samples.data(), cfg.colormap.pixels.data(), cfg.heightmap16.width,
		                    cfg.heightmap16.height) != HMRM_OK)
			fatal(std::string("hmrm_set_maps16: ") + hmrm_last_error(ctx));
		if (cfg.maps_changed && cfg.height_bits == 8 &&
		    hmrm_set_maps(ctx, cfg.heightmap.pixels.data(), cfg.colormap.pixels.data(), cfg.heightmap.width,
		                  cfg.heightmap.height) != HMRM_OK)
			fatal(std::string("hmrm_set_maps: ") + hmrm_last_error(ctx));
		if (cfg.maps_changed || cfg.should_update_heightmap) {
			const double lum[3] = {cfg.lum_r, cfg.lum_g, cfg.lum_b};
			if (hmrm_update_heightmap(ctx, lum, cfg.min_height, cfg.max_height) != HMRM_OK)
				fatal(std::string("hmrm_update_heightmap: ") + hmrm_last_error(ctx));
		}
		cfg.maps_changed = false;
		cfg.should_update_heightmap = false;
	}

	void recreate_target() {
		framebuf.assign((size_t)cfg.screen_width * (size_t)cfg.screen_height * 4, 0);
		if (texture) SDL_DestroyTexture(texture);
		texture = SDL_CreateTexture(renderer, SDL_PIXELFORMAT_ABGR8888, SDL_TEXTUREACCESS_STREAMING, cfg.screen_width,
		                            cfg.screen_height);
		if (texture == NULL) fatal(std::string("Failed to recreate texture: ") + SDL_GetError());
	}

	void init() {
		if (SDL_Init(SDL_INIT_VIDEO) != 0) fatal(std::string("SDL_Init failed: ") + SDL_GetError());
		if (TTF_Init() != 0) fatal(std::string("TTF_Init failed: ") + TTF_GetError());
		const char font_path[] = "fonts/NotoSansMono-Regular.ttf";
		font = TTF_OpenFont(font_path, 12);
		if (font == NULL) fatal(std::string("Failed to open font at: ") + font_path);
		window = SDL_CreateWindow("Heightmap Ray Marcher", SDL_WINDOWPOS_UNDEFINED, SDL_WINDOWPOS_UNDEFINED,
		                          cfg.screen_width, cfg.screen_height, SDL_WINDOW_RESIZABLE);
		if (window == NULL) fatal(std::string("SDL_CreateWindow failed: ") + SDL_GetError());
		renderer = SDL_CreateRenderer(window, -1, SDL_RENDERER_ACCELERATED);
		if (renderer == NULL) fatal(std::string("Failed to create renderer: ") + SDL_GetError());
		texture = SDL_CreateTexture(renderer, SDL_PIXELFORMAT_ABGR8888, SDL_TEXTUREACCESS_STREAMING, cfg.screen_width,
		                            cfg.screen_height);
		if (texture == NULL) fatal(std::string("Failed to create texture: ") + SDL_GetError());
		framebuf.assign((size_t)cfg.screen_width * (size_t)cfg.screen_height * 4, 0);
	}

	// SavePNG (main/hmap.cpp:157-168): framebuf encoded on the device
	void save_png(const std::string &path) {
		const size_t cap = hmrm_png_bound(cfg.screen_width, cfg.screen_height, 4);
		if (png_cap < cap) {
			// pinned: the device writes the file straight into it
			hmrm_host_free(png_file);
			png_file = NULL;
			png_cap = 0;
			void *p = NULL;
			if (hmrm_host_alloc(&p, cap) != HMRM_OK) fatal(std::string("hmrm_host_alloc: ") + hmrm_last_error(NULL));
			png_file = (uint8_t *)p;
			png_cap = cap;
		}
		if (!png_bytes) {
			void *p = NULL;
			if (hmrm_host_alloc(&p, sizeof(uint64_t)) != HMRM_OK) fatal(std::string("hmrm_host_alloc: ") + hmrm_last_error(NULL));
			png_bytes = (uint64_t *)p;
		}
		if (hmrm_encode_png(ctx, framebuf.data(), cfg.screen_width, cfg.screen_height, 4, png_file, png_cap, png_bytes) !=
		    HMRM_OK)
			fatal(std::string("hmrm_encode_png: ") + hmrm_last_error(ctx));
		if (!write_bytes(path, png_file, (size_t)*png_bytes)) std::cerr << "Failed to write screenshot to " << path << "\n";
		else std::cout << "Saved screenshot at " << path << "\n";
	}

	void run_console_line() {
		const int w0 = cfg.screen_width, h0 = cfg.screen_height;
		std::istringstream iss(console_buf);
		if (consume_config_stream(iss, cfg, std::cout, std::cerr) != PARSE_OK) std::exit(1);
		if (cfg.screen_width != w0 || cfg.screen_height != h0) SDL_SetWindowSize(window, cfg.screen_width, cfg.screen_height);
		push_maps_if_needed();
	}

	void on_key(SDL_Keycode sym, double /*ddelta*/) {
		const SDL_Keymod mod = SDL_GetModState();
		if (sym == SDLK_q) {
			if (mod & KMOD_CTRL) quit = true;
		}
		else if (sym == SDLK_BACKQUOTE) {
			console_active = !console_active;
			if (console_active) console_buf.assign(" ");
		}
		else if (sym == SDLK_BACKSPACE) {
			if (console_active && console_buf.length() > 1) console_buf.erase(console_buf.length() - 1, 1);
		}
		else if (sym == SDLK_RETURN) {
			if (console_active) {
				console_active = false;
				run_console_line();
				console_buf.assign(" ");
			}
		}
		else if (sym == SDLK_F1) show_fps = !show_fps;
		else if (sym == SDLK_F11) {
			if (mod != KMOD_NONE) return;
			fullscreen = !fullscreen;
			SDL_SetWindowFullscreen(window, fullscreen ? SDL_WINDOW_FULLSCREEN_DESKTOP : 0);
		}
		else if (sym == SDLK_F12) {
			if (mod != KMOD_NONE) return;
			const std::time_t seconds = std::time(NULL);
			if (seconds == (std::time_t)(-1)) std::cerr << "Failed to get time for screenshot. Screenshot NOT saved.\n";
			else {
				std::stringstream ss;
				ss << "screenshots/hmap_" << seconds << ".png";
				save_png(ss.str());
			}
		}
		else if (sym == SDLK_1 || sym == SDLK_2 || sym == SDLK_3) {
			if (!console_active) cfg.image_plane = sym == SDLK_1 ? 1 : (sym == SDLK_2 ? 2 : 3);
		}
		else if (sym == SDLK_r) {
			if (!console_active && (mod & KMOD_CTRL) && (mod & KMOD_SHIFT)) {
				if (!recording) {
					recording = true;
					recording_frame_num = 0;
					recording_id = std::time(NULL);
					if (recording_id == (std::time_t)(-1)) {
						std::cerr << "Failed to get time for recording. Recording NOT started.\n";
						recording = false;
					}
				}
				else recording = false;
			}
		}
	}

	void on_event(const SDL_Event &ev, double ddelta) {
		switch (ev.type) {
		case SDL_QUIT: quit = true; break;
		case SDL_WINDOWEVENT:
			if (ev.window.event == SDL_WINDOWEVENT_SIZE_CHANGED) {
				SDL_GetWindowSize(window, &cfg.screen_width, &cfg.screen_height);
				recreate_target();
			}
			else if (ev.window.event == SDL_WINDOWEVENT_FOCUS_GAINED) {
				if (SDL_SetRelativeMouseMode(SDL_TRUE))
					std::cerr << "FOCUS_GAINED SDL_SetRelativeMouseMode failed: " << SDL_GetError() << "\n";
			}
			else if (ev.window.event == SDL_WINDOWEVENT_FOCUS_LOST) {
				if (SDL_SetRelativeMouseMode(SDL_FALSE))
					std::cerr << "FOCUS_LOST SDL_SetRelativeMouseMode failed: " << SDL_GetError() << "\n";
			}
			break;
		case SDL_MOUSEMOTION:
			cfg.hang -= cfg.mouse_sens * 0.00025 * ev.motion.xrel * ddelta;
			cfg.vang += cfg.mouse_sens * 0.00025 * ev.motion.yrel * ddelta;
			if (cfg.vang < 0.0) cfg.vang = 0.0;
			else if (cfg.vang > M_PI) cfg.vang = M_PI;
			break;
		case SDL_MOUSEWHEEL:
			if (cfg.image_plane == 1 || cfg.image_plane == 2) {
				const double new_hfov = cfg.hfov - (cfg.scroll_sens * 0.03 * ev.wheel.y);
				if (new_hfov > 0.0 && new_hfov < M_PI) cfg.hfov = new_hfov;
			}
			else if (cfg.image_plane == 3) {
				const double new_ortho_width = cfg.ortho_width - (cfg.scroll_sens * 0.0075 * ev.wheel.y);
				if (new_ortho_width > 0.0) cfg.ortho_width = new_ortho_width;
			}
			break;
		case SDL_TEXTINPUT:
			if (console_active) console_buf.append(ev.text.text);
			break;
		case SDL_KEYUP: on_key(ev.key.keysym.sym, ddelta); break;
		default: break;
		}
	}

	void move_camera(const Basis &b, double ddelta) {
		const Uint8 *kb = SDL_GetKeyboardState(NULL);
		const SDL_Keymod mod = SDL_GetModState();
		if (console_active || mod != KMOD_NONE) return;
		const double k = ddelta * cfg.move_speed;
		if (kb[SDL_SCANCODE_W]) for (int i = 0; i < 3; ++i) cfg.cam_pos[i] += k * b.forward[i];
		if (kb[SDL_SCANCODE_S]) for (int i = 0; i < 3; ++i) cfg.cam_pos[i] -= k * b.forward[i];
		if (kb[SDL_SCANCODE_D]) for (int i = 0; i < 3; ++i) cfg.cam_pos[i] += k * b.right[i];
		if (kb[SDL_SCANCODE_A]) for (int i = 0; i < 3; ++i) cfg.cam_pos[i] -= k * b.right[i];
		if (kb[SDL_SCANCODE_SPACE]) cfg.cam_pos[2] += k;
		if (kb[SDL_SCANCODE_Q]) cfg.cam_pos[2] -= k;
	}

	void render(const Basis &b) {
		if (cfg.cycle_period <= 0) fatal("cycle must be positive");      // the reference divides by zero here (:976)
		cfg.cycle = (cfg.cycle + 1) % cfg.cycle_period;
		hmrm_frame f;
		hmrm_frame_defaults(&f);
		f.projection = cfg.image_plane;
		f.screen_width = cfg.screen_width;
		f.screen_height = cfg.screen_height;
		f.precision = precision;
		f.traversal = traversal;
		for (int i = 0; i < 3; ++i) f.cam_pos[i] = cfg.cam_pos[i];
		// look/up were computed at the top of the loop; Spherical reads hang/vang itself, after the events
		f.hang = cfg.image_plane == 2 ? cfg.hang : b.hang;
		f.vang = cfg.image_plane == 2 ? cfg.vang : b.vang;
		f.hfov = cfg.hfov;
		f.ortho_width = cfg.ortho_width;
		f.grid_width = cfg.grid_width;
		f.step_dist = cfg.step_dist;
		f.bg[0] = cfg.bg_r;
		f.bg[1] = cfg.bg_g;
		f.bg[2] = cfg.bg_b;
		f.cycle = cfg.cycle;
		f.cycle_period = cfg.cycle_period;
		if (hmrm_render(ctx, &f, framebuf.data()) != HMRM_OK) fatal(std::string("hmrm_render: ") + hmrm_last_error(ctx));
	}

	bool present(double ddelta) {
		if (text_timer_ms >= 200) {
			text_timer_ms = 0;
			SDL_Color fg = {255, 255, 255, 255};
			SDL_Color bg = {0, 0, 0, 255};
			std::stringstream ss;
			ss << "FPS: " << std::fixed << std::setprecision(1) << 1000.0 / ddelta;
			SDL_FreeSurface(fps_surface);
			fps_surface = TTF_RenderUTF8_Shaded(font, ss.str().c_str(), fg, bg);
			const SDL_Color console_bg = {50, 100, 250, 255};
			SDL_FreeSurface(console_surface);
			console_surface = TTF_RenderUTF8_Shaded(font, console_buf.c_str(), fg, console_bg);
		}
		SDL_UpdateTexture(texture, NULL, framebuf.data(), cfg.screen_width * 4);
		SDL_RenderClear(renderer);
		SDL_RenderCopy(renderer, texture, NULL, NULL);
		if (show_fps && fps_surface != NULL) {
			SDL_Texture *t = SDL_CreateTextureFromSurface(renderer, fps_surface);
			if (t == NULL) {
				std::cerr << "Failed to create texture from fps_surface: " << SDL_GetError() << "\n";
				return false;
			}
			SDL_Rect dst = {5, 2, fps_surface->w, fps_surface->h};
			SDL_RenderCopy(renderer, t, NULL, &dst);
			SDL_DestroyTexture(t);
		}
		if (console_active && console_surface != NULL) {
			SDL_Texture *t = SDL_CreateTextureFromSurface(renderer, console_surface);
			if (t == NULL) {
				std::cerr << "Failed to create texture from console_surface: " << SDL_GetError() << "\n";
				return false;
			}
			SDL_Rect dst = {0, cfg.screen_height - console_surface->h - 10, console_surface->w, console_surface->h};
			SDL_RenderCopy(renderer, t, NULL, &dst);
			SDL_DestroyTexture(t);
		}
		SDL_RenderPresent(renderer);
		return true;
	}

	int loop() {
		Uint32 old_time = SDL_GetTicks();
		if (SDL_SetRelativeMouseMode(SDL_TRUE)) fatal(std::string("Initial SDL_SetRelativeMouseMode failed: ") + SDL_GetError());
		while (!quit) {
			const Uint32 new_time = SDL_GetTicks();
			const Uint32 delta = new_time - old_time;
			const double ddelta = (double)delta;
			old_time = new_time;
			text_timer_ms += delta;

			Basis b;
			b.hang = cfg.hang;
			b.vang = cfg.vang;
			b.forward[0] = std::cos(cfg.hang);
			b.forward[1] = std::sin(cfg.hang);
			b.forward[2] = 0.0;
			const double right_hang = cfg.hang - (M_PI / 2.0);
			b.right[0] = std::cos(right_hang);
			b.right[1] = std::sin(right_hang);
			b.right[2] = 0.0;

			SDL_Event ev;
			while (SDL_PollEvent(&ev)) on_event(ev, ddelta);
			move_camera(b, ddelta);
			render(b);
			if (!present(ddelta)) break;

			if (recording) {
				std::stringstream ss;
				ss << "screenshots/hmap_" << recording_id << "_" << recording_frame_num << ".png";
				save_png(ss.str());
				recording_frame_num += 1;
				if (recording_frame_num == cfg.recording_frame_count) {
					recording = false;
					std::cout << "Done recording.\n";
				}
			}
		}
		SDL_DestroyWindow(window);
		SDL_DestroyRenderer(renderer);
		SDL_DestroyTexture(texture);
		SDL_FreeSurface(fps_surface);
		SDL_FreeSurface(console_surface);
		TTF_CloseFont(font);
		TTF_Quit();
		SDL_Quit();
		hmrm_host_free(png_file);
		hmrm_host_free(png_bytes);
		return 0;
	}
};

} // namespace

int run_interactive(Config &cfg, hmrm_ctx *ctx, int precision, int traversal) {
	Shell shell(cfg, ctx, precision, traversal);
	shell.init();
	return shell.loop();
}

} // namespace hmrm_host

#endif // HMAP_WITH_SDL
