// K2 (packed-lane skip traversal) — the integer-model traversal of k2_render_lin.cuh with the lanes kept busy.
//
// Same contract as every K2 kernel (main/hmap.cpp:978-1058): same framebuffer, same per-pixel first-hit sample
// index, same reference-equivalent step count.  Same exactness argument as k2_render_lin.cuh (facts 1-4): every
// decision is taken from the integer model with its proven margins, or by the reference's own FP64 expressions.
//
// What changes is WHO marches WHAT.  In k2_render_lin a warp owns an 8x4 tile from ray generation to the last pixel:
// its 32 rays end after different numbers of iterations, so the march loop runs with 24 of 32 lanes busy on the 4K
// flythrough and 20 of 32 on the orthographic stress (hmrm_get_debug_counters [6], [8..11]).  Here a ray that enters
// the box is reduced to a 64-byte record — the integer model (three slopes, three offsets), pixel, sample index,
// level, the colour it gets if it leaves the grid — and pushed on a small per-warp stack in shared memory; lanes pop
// records whenever they are idle.  The warp alternates between two fully convergent phases:
//   produce   all 32 lanes set up the 32 pixels of the next tile (ray generation, slab test: the FP64-heavy part),
//             store the pixels that miss the box, push the rest;
//   march     every lane holding a record runs one iteration of the traversal; a lane that finishes shades and
//             stores its pixel and pops the next record.
// When the stack is empty and no more than HMRM_PACK_THRESH lanes are still marching, those lanes push their records
// back (a record is resumable) and the warp produces again, so that set-up never runs under a divergent mask and the
// march never runs with fewer than THRESH + 1 lanes while tiles remain.  No atomics, no barriers: the stack is
// private to the warp.
//
// The exact FP64 anchor of a ray (k2_render_lin keeps it on the stack of every thread: 12.5 M sectors of L2 writes
// per 4K frame) is not stored at all.  A sample that needs the reference's own arithmetic (undecided in the model, or
// the model's window ran out) takes the ray out of the march: a 3-word note (pixel, sample, level / reason) goes on a
// second small list, and the next refill phase — where no lane holds live state — rebuilds the exact position from
// the pixel (generate_ray -> box_entry -> nudge -> advance_exact), decides, and pushes the ray back with a fresh
// model.  The march loop itself therefore contains no call and no FP64.
#ifndef HMRM_K2_RENDER_PACK_CUH
#define HMRM_K2_RENDER_PACK_CUH

#include "k2_render_lin.cuh"

namespace hmrm {

// launch shape: persistent CTAs of HMRM_LIN_THREADS threads, HMRM_PACK_CTAS of them per SM
#ifndef HMRM_PACK_CTAS
#define HMRM_PACK_CTAS 4
#endif

// This kernel keeps the 64-bit form of the integer model (k2_render_lin.cuh, fact 4): a ray's record holds D and
// 2^16 V_0 + 2^15 per axis, and V_j = lin_acc(l, j) >> 16.
struct LinAxis {
	long long d;     // per-step motion in units * 2^16
	long long a0;    // V_0 * 2^16 + 2^15: position of the base sample, pre-shifted, with the rounding half added
};

// 2^16 V_j + (fraction).  One IMAD.WIDE (the 64-bit addend is free) and one IMAD; |a0| < 2^47 + 2^15 and
// j |D| < 2^17 * 2^42, so it cannot wrap.
__device__ __forceinline__ long long lin_acc(const LinAxis &l, unsigned j) {
	return l.a0 + (long long)((unsigned long long)j * (unsigned long long)l.d);
}

#ifndef HMRM_PACK_THRESH
#define HMRM_PACK_THRESH 16
#endif
// Rays of one warp live in three places: its lanes, its stack, its notes.  A tile (<= 32 new rays) is only set up when
// every ray of the warp is on the stack and there are fewer than 32 of them, so the warp never owns more than 63 rays:
// neither the stack nor the list of notes can overflow.
#define HMRM_PACK_QCAP 64          // records per warp
#define HMRM_PACK_WORDS 16         // 32-bit words per record

#define HMRM_PACK_SLOWCAP 64       // notes per warp

enum { kPackContinue = 0, kPackHit = 1, kPackMiss = 2, kPackCutOff = 3, kPackSlow = 4 };
// reasons of a note (bits 8.. of its level word)
enum { kSlowDecide = 0x100, kSlowReanchor = 0x200 };

// One ray in flight.  Everything else the march needs is derived from these (pack_derive).
struct PackRay {
	long long dx, dy, dz;          // LinAxis::d of the three axes
	long long ax, ay, az;          // LinAxis::a0 (valid for the 65536-sample window that contains n)
	unsigned pixel;                // px | py << 16
	unsigned n;                    // sample under examination
	int level;
	uint32_t miss_rgba;            // colour if the ray leaves the grid (needs the exact dir.z: computed at set-up)
};

struct PackDerived {
	float inv_adx, inv_ady, inv_adz;
	int cell_exit;
};

__device__ __forceinline__ PackDerived pack_derive(const RenderParams &P, const PackRay &r) {
	PackDerived d;
	d.inv_adx = fast_rcp(fabsf((float)r.dx) * (1.0f / 65536.0f));
	d.inv_ady = fast_rcp(fabsf((float)r.dy) * (1.0f / 65536.0f));
	const float adz = fabsf((float)r.dz) * (1.0f / 65536.0f);
	d.inv_adz = fast_rcp(adz);
	d.cell_exit = (int)fminf(P.cell_exit_scale * adz + 512.0f, 1.0e9f);
	return d;
}

// The exact state of pixel `pixel` at sample 0: entry point + nudge, per-step addend (main/hmap.cpp:985-998, :1037).
__device__ __forceinline__ void pack_exact_start(const RenderParams &P, const Ray &ray, double ex, double ey, double ez,
                                                 AxisState &ax, AxisState &ay, AxisState &az) {
	ax.p = fadd(ex, fmul(P.nudge, ray.dx));
	ay.p = fadd(ey, fmul(P.nudge, ray.dy));
	az.p = fadd(ez, fmul(P.nudge, ray.dz));
	ax.s = fmul(P.step_dist, ray.dx);
	ay.s = fmul(P.step_dist, ray.dy);
	az.s = fmul(P.step_dist, ray.dz);
	ax.tag = ay.tag = az.tag = INT_MIN;
	ax.S = ay.S = az.S = 0.0;
}

// Slopes of the integer model (k2_render_lin.cuh, fact 4); false if the ray does not fit it.
__device__ __forceinline__ bool pack_slopes(const RenderParams &P, const AxisState &ax, const AxisState &ay, const AxisState &az, PackRay &r) {
	const double zc = P.zq_offset - HMRM_MAGIC;
	const double zs16 = P.zq_scale * 16.0;
	bool model = lin_slope(ax.s * P.fx_scale, r.dx) && lin_slope(-ay.s * P.fx_scale, r.dy) && lin_slope(az.s * zs16, r.dz);
	model = model && fabs(zc) < 1.0e12;
	// no lateral motion and not coming down: such a ray can only end by the reference's hang; the per-step loop cuts it
	return model && (r.dx != 0 || r.dy != 0 || r.dz < 0);
}

// Model offsets for the window that starts at the exact position (ax, ay, az); false if it left the representable range.
__device__ __forceinline__ bool pack_rebase(const RenderParams &P, const AxisState &ax, const AxisState &ay, const AxisState &az, PackRay &r) {
	const double zc = P.zq_offset - HMRM_MAGIC;
	const double zs16 = P.zq_scale * 16.0, zo16 = __fma_rn(16.0, zc, HMRM_MAGIC);
	int vx, vy, vz;
	const bool okx = magic_decode(__fma_rn(ax.p, P.fx_scale, HMRM_MAGIC), vx);
	const bool oky = magic_decode(__fma_rn(ay.p, -P.fx_scale, HMRM_MAGIC), vy);
	const bool okz = magic_decode(__fma_rn(az.p, zs16, zo16), vz);
	r.ax = ((long long)vx << HMRM_LIN_FRAC) + (1LL << (HMRM_LIN_FRAC - 1));
	r.ay = ((long long)vy << HMRM_LIN_FRAC) + (1LL << (HMRM_LIN_FRAC - 1));
	r.az = ((long long)vz << HMRM_LIN_FRAC) + (1LL << (HMRM_LIN_FRAC - 1));
	return okx && oky && okz;
}

// The plain per-step loop (k2_render_brute.cuh) from the exact state (sample `from`) on: rays that do not fit the
// integer model, and rays that left its representable range.  `steps` = samples examined (a hit is sample steps - 1).
template <bool kStats>
__device__ __forceinline__ int pack_fallback(const RenderParams &P, AxisState &ax, AxisState &ay, AxisState &az, unsigned from,
                                             unsigned &hit_cell, unsigned long long &steps, unsigned &fetches) {
	unsigned long long kk = from;
	int verdict = kPackMiss;
	for (;;) {
		const int gx = trunc_cell(fdiv(ax.p, P.gw)), gy = trunc_cell(fdiv(-ay.p, P.gw));
		if (gx < 0 || gy < 0 || gx >= P.map_w || gy >= P.map_h) break;
		const size_t cell = (size_t)gx + (size_t)gy * (size_t)P.map_w;
		kk += 1ULL;
		if (kStats) fetches += 1u;
		if (az.p < __ldg(P.surf + HMRM_CHECKED(P, cell, (size_t)P.map_w * (size_t)P.map_h))) {
			hit_cell = (unsigned)cell;
			verdict = kPackHit;
			break;
		}
		const double nx = fadd(ax.p, ax.s), ny = fadd(ay.p, ay.s), nz = fadd(az.p, az.s);
		if ((nx == ax.p && ny == ay.p && !(nz < az.p)) || kk >= (1ULL << 27)) {
			verdict = kPackCutOff;
			break;
		}
		ax.p = nx; ay.p = ny; az.p = nz;
	}
	steps = kk;
	return verdict;
}

// A sample the integer model could not decide: the reference's own expressions (main/hmap.cpp:1001-1016).  First an
// FP64 linear look from sample 0 (P_n = P_0 + n s up to the roundings of the reference's n adds:
// |P_n - fma(n, s, P_0)| <= (n + 1) 2^-53 max|P|, doubled below), which decides unless the sample is within ~1e-10
// of a cell edge or of the surface; then the exact reconstruction (advance_exact moves the anchor to sample n).
// Returns kPackHit (hit_cell set), kPackMiss (left the grid) or kPackContinue (not below the surface).
template <bool kStats>
__device__ __forceinline__ int pack_decide_exact(const RenderParams &P, AxisState &ax, AxisState &ay, AxisState &az, unsigned &anchor,
                                                 unsigned n, unsigned &hit_cell, unsigned &fetches, unsigned &exact_used) {
	{
		const double mj = (double)n;
		const double rel = fmul(fadd(mj, 2.0), 2.3e-16);
		const double xe = __fma_rn(mj, ax.s, ax.p), ye = __fma_rn(mj, ay.s, ay.p), ze = __fma_rn(mj, az.s, az.p);
		const double bx = fmul(rel, fmax(fabs(ax.p), fabs(xe))), by = fmul(rel, fmax(fabs(ay.p), fabs(ye)));
		const double bz = fmul(rel, fmax(fabs(az.p), fabs(ze)));
		const double qx = fdiv(xe, P.gw), qy = fdiv(-ye, P.gw);
		const double axq = fabs(qx), ayq = fabs(qy);
		const double ex_ = fadd(fmul(bx, P.inv_gw_up), fmul(axq, 4.5e-16)), ey_ = fadd(fmul(by, P.inv_gw_up), fmul(ayq, 4.5e-16));
		const double fxq = fsub(axq, floor(axq)), fyq = fsub(ayq, floor(ayq));
		const double near_x = axq < 1.0 ? fsub(1.0, axq) : fmin(fxq, fsub(1.0, fxq));
		const double near_y = ayq < 1.0 ? fsub(1.0, ayq) : fmin(fyq, fsub(1.0, fyq));
		if (axq < 2.0e9 && ayq < 2.0e9 && near_x > ex_ && near_y > ey_) {
			const int gx = trunc_cell(qx), gy = trunc_cell(qy);
			if (gx < 0 || gy < 0 || gx >= P.map_w || gy >= P.map_h) return kPackMiss;     // :1006-1011
			const size_t cell = (size_t)gx + (size_t)gy * (size_t)P.map_w;
			const double surf = __ldg(P.surf + HMRM_CHECKED(P, cell, (size_t)P.map_w * (size_t)P.map_h));
			if (kStats) fetches += 1u;
			if (fadd(ze, bz) < surf) {
				hit_cell = (unsigned)cell;
				return kPackHit;
			}
			if (fsub(ze, bz) > surf) return kPackContinue;
		}
	}
	exact_used = 1u;
	advance_exact(ax, ay, az, anchor, n);
	const int gx = trunc_cell(fdiv(ax.p, P.gw)), gy = trunc_cell(fdiv(-ay.p, P.gw));
	if (gx < 0 || gy < 0 || gx >= P.map_w || gy >= P.map_h) return kPackMiss;
	const size_t cell = (size_t)gx + (size_t)gy * (size_t)P.map_w;
	if (kStats) fetches += 1u;
	if (az.p < __ldg(P.surf + HMRM_CHECKED(P, cell, (size_t)P.map_w * (size_t)P.map_h))) {
		hit_cell = (unsigned)cell;
		return kPackHit;
	}
	return kPackContinue;
}

// One iteration of the traversal for the ray in `r` (the loop body of march_lin, k2_render_lin.cuh, on the same
// model, with the same margins).  kPackContinue: r advanced to its next sample.  kPackSlow: the sample r.n needs the
// exact arithmetic (r.level carries the reason); the ray leaves the march until the next refill phase.
template <bool kStats, int kLayout>
__device__ __forceinline__ int pack_iterate(const RenderParams &P, PackRay &r, const PackDerived &dv, unsigned &hit_cell,
                                            unsigned &fetches, unsigned *dbg) {
	const int k = P.fx_bits;
	const int cell_mask = (1 << k) - 1;
	// window of the model: V_0 is the exact sample `base`, a multiple of the period (jumps never cross one)
	const unsigned base = r.n & ~(HMRM_LIN_PERIOD - 1u);
	const unsigned j = r.n - base;
	LinAxis lx, ly, lz;
	lx.d = r.dx; lx.a0 = r.ax;
	ly.d = r.dy; ly.a0 = r.ay;
	lz.d = r.dz; lz.a0 = r.az;
	const long long wx = lin_acc(lx, j), wy = lin_acc(ly, j), wz = lin_acc(lz, j);

	auto probe = [&](int lvl, int vx, int vy) -> int {
		const uint2 d = P.lv_desc[lvl];
		const unsigned idx = d.x + pyr_index<kLayout>((unsigned)(vx >> (k + lvl)), (unsigned)(vy >> (k + lvl)), d.y);
		return (int)__ldg(P.lv + HMRM_CHECKED(P, idx, P.lv_total));
	};
	auto above = [&](int vz, int q) -> bool { return vz > (q << 4) + HMRM_LIN_ZMARGIN && q < 65535; };

	bool exact = false;
	const int vx = (int)(wx >> HMRM_LIN_FRAC), vy = (int)(wy >> HMRM_LIN_FRAC);
	const bool inside = ((unsigned)((unsigned long long)wx >> 32) | (unsigned)((unsigned long long)wy >> 32)) < 65536u &&
	                    (unsigned)vx - (unsigned)HMRM_LIN_MARGIN < P.lin_span_x && (unsigned)vy - (unsigned)HMRM_LIN_MARGIN < P.lin_span_y;
	if (!inside) {
		const long long fx = wx >> HMRM_LIN_FRAC, fy = wy >> HMRM_LIN_FRAC;
		const long long low_edge = -(1LL << k) - HMRM_LIN_MARGIN;
		if (fx < low_edge || fy < low_edge || fx >= (long long)P.lin_grid_x + HMRM_LIN_MARGIN ||
		    fy >= (long long)P.lin_grid_y + HMRM_LIN_MARGIN)
			return kPackMiss;
		exact = true;
	}
	const int wz_hi = (int)(wz >> 32);
	int vz = (int)(wz >> HMRM_LIN_FRAC);
	if ((unsigned)(wz_hi + 32768) >= 65536u) vz = wz_hi < 0 ? -1073741824 : 1073741824;

	int level = r.level;
	int q = 0;
	if (!exact) {
		q = probe(level, vx, vy);
		if (kStats) fetches += 1u;
		while (!above(vz, q) && level > 0) {
			level = (level - P.lstride >= P.lmin) ? level - P.lstride : 0;
			q = probe(level, vx, vy);
			if (kStats) { fetches += 1u; dbg[3] += 1u; }
		}
		if (level == 0) {
			const int fx = vx & cell_mask, fy = vy & cell_mask;
			exact = fx < HMRM_LIN_MARGIN || fy < HMRM_LIN_MARGIN || fx > cell_mask - HMRM_LIN_MARGIN || fy > cell_mask - HMRM_LIN_MARGIN;
		}
	}

	unsigned m = 1u;
	if (!exact && above(vz, q)) {
		if (level > 0) {
			float est_xy, est_z;
			for (;;) {
				const unsigned w = 1u << (k + level), mask = w - 1u;
				const unsigned ux = (unsigned)vx, uy = (unsigned)vy;
				const int room_x = (int)(r.dx >= 0 ? min((ux | mask) + 1u + w, P.lin_grid_x) - ux : min((ux & mask) + w, ux));
				const int room_y = (int)(r.dy >= 0 ? min((uy | mask) + 1u + w, P.lin_grid_y) - uy : min((uy & mask) + w, uy));
				est_xy = fminf(__int2float_rz(room_x - (HMRM_LIN_MARGIN + 1)) * dv.inv_adx,
				               __int2float_rz(room_y - (HMRM_LIN_MARGIN + 1)) * dv.inv_ady);
				est_z = r.dz < 0 ? __int2float_rz(vz - (q << 4) - (HMRM_LIN_ZMARGIN + 2)) * dv.inv_adz : 3.0e38f;
				if (!(est_z >= P.climb_ratio * est_xy) || level + P.lstride > P.ltop) break;
				const int q2 = probe(level + P.lstride, vx, vy);
				if (kStats) fetches += 1u;
				if (!above(vz, q2)) break;
				level += P.lstride;
				q = q2;
			}
			// (jumps never cross a window boundary: the next sample examined is at most the first of the next window)
			const float est = fminf(fminf(est_xy, est_z), (float)(HMRM_LIN_PERIOD - j)) * 0.999f;
			m = (est >= 2.0f) ? (unsigned)__float2int_rz(est) : 1u;
			if (kStats) {
				if (m >= 2u) { dbg[0] += 1u; dbg[1] += m; }
				else dbg[2] += 1u;
			}
			if (est_z < est_xy) level = (level - P.lstride >= P.lmin) ? level - P.lstride : 0;
		}
		else {
			if (kStats) dbg[4] += 1u;
			if (vz - (q << 4) > dv.cell_exit) level = P.lmin;
		}
	}
	else if (!exact && vz < (q << 4) - HMRM_LIN_ZMARGIN && q > 0) {
		hit_cell = (unsigned)((size_t)(vx >> k) + (size_t)(vy >> k) * (size_t)P.map_w);
		if (kStats) dbg[5] += 1u;
		return kPackHit;
	}
	else {
		r.level = kSlowDecide;          // undecided: sample r.n goes to the exact arithmetic; the march resumes at level 0
		return kPackSlow;
	}
	r.n += m;
	r.level = level;
	if ((r.n & (HMRM_LIN_PERIOD - 1u)) == 0u) {
		r.level = kSlowReanchor | level;    // the window ran out: a fresh model anchored on the exact sample r.n
		return kPackSlow;
	}
	return kPackContinue;
}

typedef unsigned (*PackQueue)[HMRM_PACK_QCAP];

__device__ __forceinline__ void pack_put(PackQueue Q, int slot, const PackRay &r) {
	Q[0][slot] = (unsigned)r.dx; Q[1][slot] = (unsigned)((unsigned long long)r.dx >> 32);
	Q[2][slot] = (unsigned)r.dy; Q[3][slot] = (unsigned)((unsigned long long)r.dy >> 32);
	Q[4][slot] = (unsigned)r.dz; Q[5][slot] = (unsigned)((unsigned long long)r.dz >> 32);
	Q[6][slot] = (unsigned)r.ax; Q[7][slot] = (unsigned)((unsigned long long)r.ax >> 32);
	Q[8][slot] = (unsigned)r.ay; Q[9][slot] = (unsigned)((unsigned long long)r.ay >> 32);
	Q[10][slot] = (unsigned)r.az; Q[11][slot] = (unsigned)((unsigned long long)r.az >> 32);
	Q[12][slot] = r.pixel;
	Q[13][slot] = r.n;
	Q[14][slot] = (unsigned)r.level;
	Q[15][slot] = r.miss_rgba;
}

__device__ __forceinline__ void pack_get(PackQueue Q, int slot, PackRay &r) {
	r.dx = (long long)((unsigned long long)Q[0][slot] | ((unsigned long long)Q[1][slot] << 32));
	r.dy = (long long)((unsigned long long)Q[2][slot] | ((unsigned long long)Q[3][slot] << 32));
	r.dz = (long long)((unsigned long long)Q[4][slot] | ((unsigned long long)Q[5][slot] << 32));
	r.ax = (long long)((unsigned long long)Q[6][slot] | ((unsigned long long)Q[7][slot] << 32));
	r.ay = (long long)((unsigned long long)Q[8][slot] | ((unsigned long long)Q[9][slot] << 32));
	r.az = (long long)((unsigned long long)Q[10][slot] | ((unsigned long long)Q[11][slot] << 32));
	r.pixel = Q[12][slot];
	r.n = Q[13][slot];
	r.level = (int)Q[14][slot];
	r.miss_rgba = Q[15][slot];
}

// statistics of one finished ray; per-lane atomics: the counting variant is not the timed one
template <bool kStats>
__device__ __forceinline__ void pack_tally(const RenderParams &P, bool surf_hit, unsigned long long steps, bool cut) {
	if (cut) atomicOr(&P.stats->status, 4u);
	if (!kStats) return;
	atomicAdd(&P.stats->box_hits, 1ULL);
	if (surf_hit) atomicAdd(&P.stats->surf_hits, 1ULL);
	atomicAdd(&P.stats->steps, steps);
	atomicMax(&P.stats->max_steps, steps);
}

// (kStats) fetch and event counters of the part of a ray marched so far: flushed whenever the ray changes hands
__device__ __forceinline__ void pack_flush_counters(const RenderParams &P, unsigned &fetches, unsigned *dbg) {
	if (fetches) atomicAdd(&P.stats->fetches, (unsigned long long)fetches);
	fetches = 0u;
	for (int i = 0; i < 8; ++i) {
		if (dbg[i]) atomicAdd(&P.stats->dbg[i], (unsigned long long)dbg[i]);
		dbg[i] = 0u;
	}
}

// one finished pixel (any lane, any time): main/hmap.cpp:139-154
__device__ __forceinline__ void pack_store(const RenderParams &P, unsigned pixel, uint32_t rgba, int first_hit) {
	const size_t at = (size_t)(pixel >> 16) * (size_t)P.W + (size_t)(pixel & 0xFFFFu);
	if (P.pixel_format == 0) store_rgba8(P, HMRM_CHECKED(P, at, (size_t)P.W * (size_t)P.H), rgba);
	else {
		uint8_t *o = (uint8_t *)P.fb + HMRM_CHECKED(P, at * 3, (size_t)P.W * (size_t)P.H * 3);
		o[0] = (uint8_t)rgba;
		o[1] = (uint8_t)(rgba >> 8);
		o[2] = (uint8_t)(rgba >> 16);
	}
	if (P.step_index) P.step_index[at] = first_hit;
}

// REFILL: the warp, with all 32 lanes free and nothing in flight, (1) serves the notes of rays that asked for the
// exact arithmetic — one note per lane — and (2) sets up tiles until its stack holds at least 32 rays or the frame has
// no more tiles.  Pixels that miss the box (or end in the service) are finished here; rays that go on are pushed.
// Not inlined: the FP64-heavy code gets its own register allocation instead of competing with the march loop's.
// io: [0] stack count, [1] cur, [2] end (tile queue batch), [3] tiles_left, [4] notes.
template <bool kStats>
__device__ __noinline__ void pack_refill(const RenderParams &P, PackQueue Q, const unsigned (*S)[HMRM_PACK_SLOWCAP], unsigned io[5]) {
	const int lane = threadIdx.x & 31;
	const unsigned lt_mask = (1u << lane) - 1u;
	const unsigned n_tiles = (unsigned)(P.tiles_x * P.tiles_y);
	int count = (int)io[0];
	unsigned cur = io[1], end = io[2];
	bool tiles_left = io[3] != 0u;
	int notes = (int)io[4];

	// first the notes, 32 at a time (one per lane); then tiles
	for (;;) {
		const bool serving = notes > 0;
		if (!serving && !(count < 32 && tiles_left)) break;
		bool selected = false;
		int px = 0, py = 0;
		unsigned at_n = 0u;          // sample the ray (re)starts at
		int level = P.lstart;
		int reason = 0;
		if (serving) {
			const int take = min(notes, 32);
			if (lane < take) {
				const int at = notes - take + lane;
				const unsigned pixel = S[0][at];
				px = (int)(pixel & 0xFFFFu);
				py = (int)(pixel >> 16);
				at_n = S[1][at];
				reason = (int)S[2][at] & ~0xFF;
				level = (int)S[2][at] & 0xFF;
				selected = true;
			}
			notes -= take;
		}
		else {
			if (cur == end) {
				// (marching tiles are grabbed one at a time, the sky rows at the end of the schedule 8 at a time:
				// k2_render_lin.cuh)
				const unsigned batch = (end != 0u && end >= P.batch_from_tile) ? P.sky_batch : 1u;
				unsigned t = 0u;
				if (lane == 0) t = atomicAdd(P.tile_counter, batch);
				cur = __shfl_sync(0xFFFFFFFFu, t, 0);
				end = min(cur + batch, n_tiles);
				if (cur >= n_tiles) {
					tiles_left = false;
					break;
				}
			}
			const unsigned tile = cur++;
			int ty_seq, tx;
			tile_row_col(P, tile, ty_seq, tx);
			const int ty = P.row_order ? __ldg(P.row_order + HMRM_CHECKED(P, ty_seq, P.tiles_y)) : ty_seq;
			px = tx * 8 + (lane & 7);
			py = P.row_begin + (P.tile_y_first + ty * P.tile_y_step) * 4 + (lane >> 3);
			selected = pixel_selected(P, px, py);
		}
		bool push = false;
		bool resolved = false;       // a pixel of a fresh tile finished at set-up (stored by rows below)
		uint32_t rgba = 0u;
		PackRay nr;
		nr.dx = nr.dy = nr.dz = nr.ax = nr.ay = nr.az = 0;
		nr.pixel = (unsigned)px | ((unsigned)py << 16);
		nr.n = at_n;
		nr.level = level;
		nr.miss_rgba = 0u;
		if (selected) {
			const Ray gr = generate_ray(P, px, py);
			double ex = 0.0, ey = 0.0, ez = 0.0, dist = 0.0;
			// (a note's ray did enter the box: run the slab test itself, not the shortcut that only proves a miss)
			const bool entered = serving ? box_entry_at(P.c0, P.c1, gr, ex, ey, ez, dist) : box_entry(P, gr, ex, ey, ez, dist);
			if (kStats && !serving && P.ray_dump) dump_ray(P, px, py, gr, entered, dist, ex, ey, ez);
			rgba = miss_colour(P, gr.dz);
			if (kStats && !serving) atomicAdd(&P.stats->rays, 1ULL);
			if (!entered) {
				resolved = true;
				if (P.step_index) P.step_index[(size_t)py * (size_t)P.W + (size_t)px] = -1;
			}
			else {
				AxisState ax, ay, az;
				pack_exact_start(P, gr, ex, ey, ez, ax, ay, az);
				unsigned anchor = 0u;          // sample index of (ax.p, ay.p, az.p)
				unsigned hit_cell = 0u, f = 0u, exact_used = 0u;
				int verdict = kPackContinue;   // of this refill: kPackContinue = the ray goes (back) on the stack
				unsigned long long steps = 0ULL;
				bool counted = false;          // `steps` already counts the hit sample
				if (reason == kSlowDecide) {
					verdict = pack_decide_exact<kStats>(P, ax, ay, az, anchor, at_n, hit_cell, f, exact_used);
					steps = at_n;
					if (verdict == kPackContinue) {
						nr.n = at_n + 1u;          // not below the surface: a plain step, cell level next
						nr.level = 0;
						if (kStats) atomicAdd(&P.stats->dbg[4], 1ULL);
					}
					else if (kStats && verdict == kPackHit) atomicAdd(&P.stats->dbg[5], 1ULL);
					if (kStats && exact_used) atomicAdd(&P.stats->dbg[7], 1ULL);
				}
				if (verdict == kPackContinue && nr.n >= 0x7FF00000u && (nr.n & (HMRM_LIN_PERIOD - 1u)) == 0u) {
					verdict = kPackCutOff;         // ~2^31 samples: give up like a hang would, but flagged
					steps = nr.n;
				}
				if (verdict == kPackContinue) {
					// (re)build the integer model for the window that contains nr.n, anchored on its exact first sample
					bool model = pack_slopes(P, ax, ay, az, nr);
					if (model) {
						// an exact decision (advance_exact to sample at_n) may have moved the anchor past the window's first
						// sample, which advance_exact cannot go back to: restart from sample 0
						const unsigned wbase = nr.n & ~(HMRM_LIN_PERIOD - 1u);
						if (anchor > wbase) {
							pack_exact_start(P, gr, ex, ey, ez, ax, ay, az);
							anchor = 0u;
						}
						advance_exact(ax, ay, az, anchor, wbase);
						model = pack_rebase(P, ax, ay, az, nr);
					}
					nr.miss_rgba = rgba;
					push = model;
					if (!model) {
						// does not fit the model (or left its range): the per-step loop from sample nr.n, right here
						advance_exact(ax, ay, az, anchor, nr.n);
						verdict = pack_fallback<kStats>(P, ax, ay, az, nr.n, hit_cell, steps, f);
						counted = true;
					}
				}
				if (kStats && f) atomicAdd(&P.stats->fetches, (unsigned long long)f);
				if (verdict != kPackContinue) {
					int first_hit = -2;
					if (verdict == kPackHit) {
						rgba = hit_colour(P, __ldg(P.color + HMRM_CHECKED(P, hit_cell, (size_t)P.map_w * (size_t)P.map_h)));
						const unsigned long long at = counted ? steps - 1ULL : steps;
						first_hit = (at > 0x7FFFFFFFULL) ? 0x7FFFFFFF : (int)at;
						if (!counted) steps += 1ULL;
					}
					pack_tally<kStats>(P, verdict == kPackHit, steps, verdict == kPackCutOff);
					if (serving) pack_store(P, nr.pixel, rgba, first_hit);
					else {
						if (P.step_index) P.step_index[(size_t)py * (size_t)P.W + (size_t)px] = first_hit;
						resolved = true;
					}
				}
			}
		}
		// finished pixels of a fresh tile: whole rows as words where possible (ray_setup.cuh)
		if (!serving) store_pixel(P, px, py, resolved, rgba);
		const unsigned pm = __ballot_sync(0xFFFFFFFFu, push);
		if (push) pack_put(Q, count + __popc(pm & lt_mask), nr);
		count += __popc(pm);
		__syncwarp();
	}
	io[0] = (unsigned)count;
	io[1] = cur;
	io[2] = end;
	io[3] = tiles_left ? 1u : 0u;
	io[4] = 0u;
}

template <bool kStats, int kLayout>
__global__ void __launch_bounds__(HMRM_LIN_THREADS, HMRM_PACK_CTAS) k2_render_pack(const __grid_constant__ RenderParams P) {
	__shared__ unsigned s_queue[HMRM_LIN_THREADS / 32][HMRM_PACK_WORDS][HMRM_PACK_QCAP];
	__shared__ unsigned s_slow[HMRM_LIN_THREADS / 32][3][HMRM_PACK_SLOWCAP];
	__shared__ unsigned s_tiles[HMRM_LIN_THREADS / 32][2];       // per warp: cur, end of its tile-queue batch
	const int lane = threadIdx.x & 31;
	PackQueue Q = s_queue[threadIdx.x >> 5];
	unsigned(*S)[HMRM_PACK_SLOWCAP] = s_slow[threadIdx.x >> 5];
	unsigned *tq = s_tiles[threadIdx.x >> 5];
	const unsigned lt_mask = (1u << lane) - 1u;
	if (lane == 0) { tq[0] = 0u; tq[1] = 0u; }
	__syncwarp();

	int count = 0;                 // records on this warp's stack (warp-uniform)
	int notes = 0;                 // rays waiting for the exact arithmetic (warp-uniform)
	bool tiles_left = true;

	// Outer loop: refill, then march.  The state of the rays in flight is declared INSIDE the march phase, so that
	// nothing of it is live across the refill call (a value live across a call lives on the stack — for the whole
	// loop).
	for (;;) {
		{
			unsigned io[5] = {(unsigned)count, tq[0], tq[1], tiles_left ? 1u : 0u, (unsigned)notes};
			pack_refill<kStats>(P, Q, S, io);
			count = (int)io[0];
			if (lane == 0) { tq[0] = io[1]; tq[1] = io[2]; }
			tiles_left = io[3] != 0u;
			notes = 0;
			__syncwarp();
		}
		if (count == 0 && !tiles_left) break;

		bool has = false;              // this lane holds a ray
		PackRay ray;
		PackDerived dv;
		unsigned fetches = 0u;         // (kStats) counters of the ray in flight
		unsigned dbg[8] = {0u, 0u, 0u, 0u, 0u, 0u, 0u, 0u};
		ray.dx = ray.dy = ray.dz = ray.ax = ray.ay = ray.az = 0;
		ray.pixel = ray.n = 0u;
		ray.level = 0;
		ray.miss_rgba = 0u;
		dv.inv_adx = dv.inv_ady = dv.inv_adz = 0.f;
		dv.cell_exit = 0;
		for (;;) {
			// ---- idle lanes pop ----
			unsigned active = __ballot_sync(0xFFFFFFFFu, has);
			if (count > 0 && active != 0xFFFFFFFFu) {
				const unsigned idle = ~active;
				const int rank = __popc(idle & lt_mask);
				const int take = min(__popc(idle), count);
				if (!has && rank < take) {
					pack_get(Q, count - 1 - rank, ray);
					dv = pack_derive(P, ray);
					has = true;
				}
				count -= take;
				__syncwarp();
				active = __ballot_sync(0xFFFFFFFFu, has);
			}
			const int n_active = __popc(active);

			// ---- back to the refill phase: when lanes would idle, and with every lane free ----
			const bool want_refill = count == 0 && n_active <= HMRM_PACK_THRESH && (tiles_left || notes > 0);
			if (want_refill || n_active == 0) {
				if (has) {                               // park: records are resumable
					pack_put(Q, count + __popc(active & lt_mask), ray);
					if (kStats) pack_flush_counters(P, fetches, dbg);
				}
				count += n_active;
				__syncwarp();
				break;
			}

			// ---- march: one iteration for every lane that holds a ray ----
			bool slow = false;
			if (has) {
				unsigned hit_cell = 0u;
				const int v = pack_iterate<kStats, kLayout>(P, ray, dv, hit_cell, fetches, dbg);
				if (v == kPackSlow) {
					slow = true;
					has = false;
					if (kStats) pack_flush_counters(P, fetches, dbg);
				}
				else if (v != kPackContinue) {
					uint32_t rgba = ray.miss_rgba;
					int first_hit = -2;
					unsigned long long steps = ray.n;
					if (v == kPackHit) {
						rgba = hit_colour(P, __ldg(P.color + HMRM_CHECKED(P, hit_cell, (size_t)P.map_w * (size_t)P.map_h)));
						first_hit = (steps > 0x7FFFFFFFULL) ? 0x7FFFFFFF : (int)steps;
						steps += 1ULL;
					}
					pack_store(P, ray.pixel, rgba, first_hit);
					pack_tally<kStats>(P, v == kPackHit, steps, v == kPackCutOff);
					if (kStats) pack_flush_counters(P, fetches, dbg);
					has = false;
				}
			}
			// rays that asked for the exact arithmetic leave a note
			const unsigned sm = __ballot_sync(0xFFFFFFFFu, slow);
			if (sm) {
				if (slow) {
					const int at = notes + __popc(sm & lt_mask);
					S[0][at] = ray.pixel;
					S[1][at] = ray.n;
					S[2][at] = (unsigned)ray.level;
				}
				notes += __popc(sm);
				__syncwarp();
			}
			if (kStats && lane == __ffs(active) - 1) {
				// [6]: warp-level march iterations; [8..11]: by busy lanes (1-8, 9-16, 17-24, 25-32)
				atomicAdd(&P.stats->dbg[6], 1ULL);
				atomicAdd(&P.stats->dbg[8 + ((n_active - 1) >> 3)], 1ULL);
			}
		}
	}
}

} // namespace hmrm

#endif
