// Kernel-side view of one frame: everything K2 needs, passed by value as a
// __grid_constant__ parameter (no constant-memory upload, no per-frame malloc).
#ifndef HMRM_RENDER_PARAMS_H
#define HMRM_RENDER_PARAMS_H

#include <stdint.h>
#include <vector_types.h>

namespace hmrm {

struct DeviceStats {
	unsigned long long rays;
	unsigned long long box_hits;
	unsigned long long surf_hits;
	unsigned long long steps;      // reference-equivalent march steps
	unsigned long long fetches;    // loads actually issued on the march
	unsigned long long max_steps;
	unsigned int status;           // HMRM_ERR_NONTERMINATING if a ray was cut off
	unsigned int pad;
	unsigned long long dbg[12];    // traversal diagnostics (stats mode only), see hmrm_get_debug_counters
};

struct RenderParams {
	// screen
	int projection;
	int W, H;
	int row_begin, row_end;
	int cycle, period;
	int tiles_x, tiles_y;          // 8x4-pixel tiles this launch renders
	float inv_tiles_x;             // slightly less than 1 / tiles_x: tile -> (row, column) without an integer divide
	int tile_y_first, tile_y_step; // launch tile row t is frame tile row tile_y_first + t * tile_y_step (row interleave)
	const int *row_order;          // optional permutation of the launch tile rows: expensive (grazing) rows first
	unsigned batch_from_tile;      // tiles from this queue position on look above the horizon: grabbed sky_batch at a time
	unsigned sky_batch;
	// k2_render_lin: grid extents in fixed-point units (map << fx_bits, <= 2^30) and the same minus twice the margin;
	// host-computed so that the march loop reads them as constant-bank operands
	unsigned lin_grid_x, lin_grid_y, lin_span_x, lin_span_y;
	double inv_gw_up;              // slightly more than 1 / grid_width (host): turns a position bound into a cell-coordinate bound
	float climb_ratio;             // climb a level while the height leaves room for this many times the lateral room
	unsigned long long lv_total;   // u16 elements behind `lv` (bounds checks of the -DHMRM_BOUNDS_CHECK test build)
	// map
	int map_w, map_h;
	// image plane (host-built, frame_setup.h)
	double cam[3], ul[3], pr[3], pd[3], look[3];
	// AABB (main/hmap.cpp:967-974) and march constants
	double c0[3], c1[3];
	double bmin[3], bmax[3];       // the same box as per-axis min / max (c1.y is negative: main/hmap.cpp:971)
	double gw;                     // grid_width
	double nudge;                  // fl(grid_width * 0.01), :998
	double step_dist;
	double max_surf;               // max over cells of fl(height + min_height)
	// tables (device pointers)
	const double *wtab, *htab;     // px/(W-1), py/(H-1)
	const double *cos_ha, *sin_ha, *sin_va, *cos_va;   // spherical only
	// map planes
	const double *surf;            // fl(height + min_height), row-major [map_h][map_w]
	const uint32_t *color;         // RGBA8 little-endian, row-major
	// outputs
	uint32_t *fb;                  // RGBA8 [H][W], or packed RGB8 [H][W][3] (pixel_format 1); any alignment (fb_unaligned)
	int pixel_format;              // HMRM_PIXEL_RGBA8 (0) / HMRM_PIXEL_RGB8 (1)
	int rgb_words;                 // RGB8: rows are 4-byte aligned (W % 4 == 0, fb aligned) -> tile rows go out as 32-bit words
	int32_t *step_index;           // optional [H][W]
	double *ray_dump;              // optional [H][W][10] (HMRM_FLAG_RAY_DUMP, ray_setup.cuh:dump_ray)
	DeviceStats *stats;            // optional
	unsigned int *tile_counter;    // persistent-thread tile queue head
	// ---- skip traversal (k2_render_skip.cuh): fixed-point view of the march ----
	double fx_scale;               // fl(2^fx_bits / grid_width): cell coordinate in 2^-fx_bits cell units
	double zq_scale, zq_offset;    // Zq(z) = low32(fma(z, zq_scale, zq_offset)); same function quantises surf in K1
	int fx_bits;                   // fractional bits of the fixed-point cell coordinate
	int lmin, lstride, ltop;       // mip levels used this frame: lmin, lmin+lstride, ... <= ltop (0 = cell test)
	int lstart;                    // level of a ray's first test
	float cell_exit_scale;         // leave cell-by-cell mode when Zq(z) - q exceeds this many steps of descent
	const uint16_t *lv;            // all levels back to back: level 0 = Zq(surf) per cell, level l >= 1 = max of level 0
	                               // over the 2^l x 2^l block and its eight neighbours; texel order per `layout`
	int layout;                    // pyramid_layout.cuh (the lin kernel takes it as a template parameter)
	uint2 lv_desc[16];             // per level: (element offset into lv, layout's pitch term)
	uint32_t bg_rgba;              // bg colour with alpha 255
	uint8_t bg[3];
	uint8_t fb_unaligned;          // fb is not 4-byte aligned (a caller's device pointer): RGBA8 pixels go out as 4 bytes
};

} // namespace hmrm

// Test build (-DHMRM_BOUNDS_CHECK, tools/bounds_check.sh): every table index of the traversal kernels is validated;
// a bad one sets bit 3 of DeviceStats::status (the parity tests then fail on the status) and reads element 0 instead.
#ifdef HMRM_BOUNDS_CHECK
#define HMRM_CHECKED(P, idx, limit) (((unsigned long long)(idx) < (unsigned long long)(limit)) ? (idx) : (atomicOr(&(P).stats->status, 8u), (idx) * 0))
#else
#define HMRM_CHECKED(P, idx, limit) (idx)
#endif

#endif
