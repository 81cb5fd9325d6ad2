// K2 (linear-model skip traversal) — production kernel of the exact mode.
//
// Same contract as k2_render_brute.cuh (main/hmap.cpp:978-1058): same framebuffer, same per-pixel first-hit
// sample index, same reference-equivalent step count.  It builds on the three facts of k2_render_skip.cuh
// (closed-form stepping, monotone fixed point, monotone rays + dilated maxima) and adds a fourth that removes
// FP64 — and every divide, refusal and binade check — from the hot loop:
//
// (4) Linear integer model with a proven error bound.  Let P_j be the reference's j-th sample (P_0 exact,
//     P_{j+1} = fl(P_j + s) per axis) and X(x) = x * 2^k / gw its position in fixed-point units (2^-k cells; the
//     height axis uses Zq units).  The kernel tracks   V_j = V_0 + round(j * D / 2^16)   in integers, with
//     V_0 = round(X(P_0)) (one DFMA, |err| <= 0.5 + 2^-22) and D = round(X(s) * 2^16) (|err| <= 0.5 + tiny), so
//       |V_j - X(P_0 + j s)| <= 0.5 + j * 2^-17 + 0.5            (V_0, slope quantisation, final rounding)
//       |X(P_j) - X(P_0 + j s)| <= j * 2^-53 * max|X| <= j * 2^-22   (accumulated FP64 rounding of the adds)
//     and with j < 2^16 between exact re-anchors:   |V_j - X(P_j)| < 1.6 units  (and the reference's rounded
//     quotient fl(x/gw) differs from x/gw by < 2^-22 units).  Everything the march decides is therefore decided
//     from V_j with a margin of HMRM_LIN_MARGIN = 4 units in x and y:
//       * cell index   = V >> k            when V is >= 4 units away from a cell edge,
//       * inside grid / outside grid       when V is >= 4 units away from the grid edge (the low edge is at -1 cell:
//                                          (int) truncates toward zero, so (-1, 0) still is cell 0).
//     The height axis is modelled in 1/16 Zq units (same bound, < 1.6/16 Zq), and Zq16(z) = round(Zr(z)) flips at
//     q +- 1/2, so with HMRM_LIN_ZMARGIN = 8 + 2 sixteenths:
//       * above the (dilated) block max q  when Z_j > 16 q + 10  (q < 65535: clamped values never prove anything),
//       * hit                              when Z_j < 16 q - 10  (q > 0; same monotone Zq16 argument as k2_render_skip.cuh),
//       * a jump of m samples              when m |D| / 2^16 <= (room to the edge of the cleared neighbourhood) - 4 - 1
//                                          per axis and <= (Z_j - 16 q - 10) - 2 in height: the model itself is
//                                          integer-exact (V_{j+m} - V_j is within 1 unit of m D / 2^16, V is monotone
//                                          in j), so the end point needs no test.
//     A sample that is NOT decided with that margin first gets an FP64 linear look (P_n = P_a + (n - a) s up to the
//     accumulated rounding of the reference's adds, a bound of ~(n - a) 2^-53 relative): the reference's own divide /
//     truncate / compare on that estimate decide unless the sample is within ~1e-12 of a cell edge or of the surface.
//     Only then advance_exact() reconstructs the exact FP64 position P_n from the last exact anchor with the
//     binade-aware closed form (fact 1).  On the bench frames that happens 0 times; the model's periodic re-anchoring
//     is its only regular caller.
//
// (Tried and measured in round 2, profiles/r02_kernel_experiments.txt: prefetching the level-0 texels of the next cell
// tests, +1.5..24 % — the kernel is short of issue slots, not of memory parallelism; refilling idle lanes from a
// per-warp stack of rays, k2_render_pack.cuh: 30 of 32 lanes busy instead of 24, but +27..57 % because refilled lanes
// are at unrelated phases of their marches and every warp iteration then runs every path of this loop.)
//
// Rays whose per-step motion or start position does not fit the integer model (steps of thousands of cells, a
// start 2^31 units away, NaNs, no lateral motion at all) take the plain per-step loop of the brute kernel.
#ifndef HMRM_K2_RENDER_LIN_CUH
#define HMRM_K2_RENDER_LIN_CUH

#include "k2_render_skip.cuh"

namespace hmrm {

// Launch shape: persistent CTAs of HMRM_LIN_THREADS threads.  A launch of at least HMRM_LIN_LARGE_TILES tiles runs
// HMRM_LIN_CTAS_LARGE of them per SM (40 registers: more warps to cover the latency of the dependent mip fetches, at
// the price of some spills), a smaller one HMRM_LIN_CTAS (64 registers).  Measured on a B200 at 1000 W
// (profiles/r09_lin32_ab.txt): 6 CTAs are 6-10 % faster than 4 on the 4K and 8K frames, 8-11 % slower on 1280x720.
#ifndef HMRM_LIN_THREADS
#define HMRM_LIN_THREADS 256
#endif
#ifndef HMRM_LIN_CTAS
#define HMRM_LIN_CTAS 4
#endif
#ifndef HMRM_LIN_CTAS_LARGE
#define HMRM_LIN_CTAS_LARGE 6
#endif
#ifndef HMRM_LIN_LARGE_TILES
#define HMRM_LIN_LARGE_TILES 100000     // 3.2 M pixels: a 4K frame is 259200 tiles, one 8-way band of an 8K frame 129600
#endif

#define HMRM_LIN_FRAC 16
#define HMRM_LIN_PERIOD 65536u      // samples between exact re-anchors (keeps the error bound of fact 4)
#define HMRM_LIN_MARGIN 4         // x, y: fixed-point units
#define HMRM_LIN_ZMARGIN 10       // z: 1/16 Zq units = 8 (Zq16 rounds at q +- 1/2) + 2 (model error < 1.6)

// Move the exact anchor (sample index a, position in ax/ay/az.p) forward to sample n.  Exact: closed form inside
// binades (end point checked), plain adds across them.
__device__ __noinline__ void advance_exact(AxisState &ax, AxisState &ay, AxisState &az, unsigned &a, unsigned n) {
	while (a < n) {
		unsigned m = n - a;
		bool jumped = false;
		if (m >= 2u) {
			axis_refresh(ax);
			axis_refresh(ay);
			axis_refresh(az);
			if (ax.tag != INT_MIN && ay.tag != INT_MIN && az.tag != INT_MIN) {
				int lim = (int)min(m, (unsigned)HMRM_JUMP_CAP);
				lim = min(lim, steps_to_binade_edge(ax));
				lim = min(lim, steps_to_binade_edge(ay));
				lim = min(lim, steps_to_binade_edge(az));
				// the edge distances are estimates: verify, and back off a little if the estimate was too long
				for (int tries = 0; lim >= 2 && tries < 3; ++tries) {
					const double md = small_int_to_double(lim);
					const double nx = __fma_rn(md, ax.S, ax.p), ny = __fma_rn(md, ay.S, ay.p), nz = __fma_rn(md, az.S, az.p);
					if (binade_tag(nx) == ax.tag && binade_tag(ny) == ay.tag && binade_tag(nz) == az.tag) {
						ax.p = nx; ay.p = ny; az.p = nz;
						a += (unsigned)lim;
						jumped = true;
						break;
					}
					lim -= 1 + (lim >> 4);
				}
			}
		}
		if (!jumped) {
			ax.p = fadd(ax.p, ax.s);
			ay.p = fadd(ay.p, ay.s);
			az.p = fadd(az.p, az.s);
			a += 1u;
		}
	}
}

// slope of one axis of the integer model; false if it does not fit (|motion| >= 2^26 units per step, NaN)
__device__ __forceinline__ bool lin_slope(double s_units, long long &d) {
	if (!(fabs(s_units) < 67108864.0)) return false;
	d = __double2ll_rn(s_units * 65536.0);
	return true;
}

// One axis of the integer model in 32 bits.  The slope D (units * 2^16, |D| < 2^42) is split once per ray into
// Di = D >> 16 (arithmetic) and Df = D & 0xFFFF, so that D = 2^16 Di + Df and
//     V_j = floor((2^16 V_0 + 2^15 + j D) / 2^16) = V_0 + j Di + floor((j Df + 2^15) / 2^16)
// (j Di 2^16 is a multiple of 2^16 and leaves the floor).  The loop evaluates j < HMRM_LIN_PERIOD = 2^16 only, so
// j Df + 2^15 < 2^16 (2^16 - 1) + 2^15 < 2^32: the last term is exact in unsigned 32 bits, and the sum, taken modulo
// 2^32, is V_j itself whenever V_j fits an int.  Why it does, see march_lin.
struct LinAxis32 {
	int v0;          // V_0: position of the base sample (units)
	int di;          // D >> 16: whole units per step, |di| < 2^26; its sign is the direction of motion
	unsigned df;     // D & 0xFFFF: the fraction of a unit per step, * 2^16
};

__device__ __forceinline__ LinAxis32 lin_split(long long d) {
	return LinAxis32{0, (int)(d >> HMRM_LIN_FRAC), (unsigned)d & 0xFFFFu};
}

__device__ __forceinline__ int lin_at(const LinAxis32 &l, unsigned j) {
	return (int)((unsigned)l.v0 + j * (unsigned)l.di + ((j * l.df + (1u << (HMRM_LIN_FRAC - 1))) >> HMRM_LIN_FRAC));
}

// The first j at which V_j of an axis leaves [-2^31, 2^31), or 0xFFFFFFFF if it does not for any j <= HMRM_LIN_PERIOD.
// V_j is monotone in j, so it stays out from there on.  One 64-bit divide, and only for an axis that could get there
// at all: |V_j - V_0| <= j ((|D| >> 16) + 1) + 1.
__device__ __forceinline__ unsigned lin_exit_j(const LinAxis32 &l) {
	const long long d = ((long long)l.di << HMRM_LIN_FRAC) + (long long)l.df;
	const long long di_abs = (d < 0 ? -d : d) >> HMRM_LIN_FRAC;
	if (d == 0 || llabs((long long)l.v0) + (di_abs + 1) * (long long)HMRM_LIN_PERIOD + 1 <= 2147483647LL) return 0xFFFFFFFFu;
	// a0 = 2^16 V_0 + 2^15 is in (-2^47, 2^47); V_j >= 2^31 iff a0 + j d >= 2^47, V_j < -2^31 iff a0 + j d < -2^47
	const long long a0 = ((long long)l.v0 << HMRM_LIN_FRAC) + (1LL << (HMRM_LIN_FRAC - 1));
	const long long j = d > 0 ? ((1LL << 47) - a0 + d - 1) / d : (a0 + (1LL << 47)) / -d + 1;
	return j > (long long)HMRM_LIN_PERIOD ? 0xFFFFFFFFu : (unsigned)j;
}

template <bool kStats, int kLayout>
__device__ __forceinline__ void march_lin(const RenderParams &P, const Ray &ray, double ex, double ey, double ez,
                                          unsigned &hit_cell, bool &real_hit, int &first_hit, PixelTally &tally) {
	const int k = P.fx_bits;
	// exact state: the anchor sample and the reference's per-step addend
	AxisState ax, ay, az;
	ax.p = fadd(ex, fmul(P.nudge, ray.dx));           // main/hmap.cpp:998
	ay.p = fadd(ey, fmul(P.nudge, ray.dy));
	az.p = fadd(ez, fmul(P.nudge, ray.dz));
	ax.s = fmul(P.step_dist, ray.dx);                  // :1037
	ay.s = fmul(P.step_dist, ray.dy);
	az.s = fmul(P.step_dist, ray.dz);
	ax.tag = ay.tag = az.tag = INT_MIN;
	ax.S = ay.S = az.S = 0.0;
	unsigned anchor = 0u;     // sample index of (ax.p, ay.p, az.p)

	unsigned n = 0u;          // sample under examination
	unsigned fetches = 0u;

	// ---- integer model of this ray ----
	// x, y in fixed-point units (2^-k cells); z in 1/16 Zq units: the extra 4 bits shrink the band in which the model
	// cannot tell `above` from `hit` to ~1.3 Zq units.  Zr(z) = z * zq_scale + c with an integer c, so 16 Zr has the
	// same magic-number form.
	const double zc = P.zq_offset - HMRM_MAGIC;
	const double zs16 = P.zq_scale * 16.0, zo16 = __fma_rn(16.0, zc, HMRM_MAGIC);
	long long dx = 0, dy = 0, dz = 0;
	bool model = lin_slope(ax.s * P.fx_scale, dx) && lin_slope(-ay.s * P.fx_scale, dy) && lin_slope(az.s * zs16, dz);
	model = model && fabs(zc) < 1.0e12;
	// no lateral motion and not coming down: such a ray can only end by the reference's hang; the per-step loop cuts it
	model = model && (dx != 0 || dy != 0 || dz < 0);
	LinAxis32 lx = lin_split(dx), ly = lin_split(dy), lz = lin_split(dz);
	// Every V the loop below evaluates fits an int, so lin_at gives it exactly, in x and y because the loop only moves
	// on from samples that are inside the grid or within the margin of it (otherwise it has decided the ray): a rebase
	// gives |V_0| < 2^31 (magic_decode), a single step adds < 2^26 + 1 units to |V| <= 2^30 + 2^20 + 4 (grid <= 2^30
	// units, k <= 20), and a jump ends inside a cleared neighbourhood clipped to the grid.  Nothing bounds z that way
	// (an ascending ray is never limited by est_z): from the first j at which V_z leaves [-2^31, 2^31), jz_out, the
	// loop uses +-2^30 instead, which is far above or below everything the 16-bit pyramid holds.
	unsigned jz_out = 0xFFFFFFFFu;
	auto rebase = [&]() -> bool {                     // V_0 of the model := the exact anchor
		const bool okx = magic_decode(__fma_rn(ax.p, P.fx_scale, HMRM_MAGIC), lx.v0);
		const bool oky = magic_decode(__fma_rn(ay.p, -P.fx_scale, HMRM_MAGIC), ly.v0);
		const bool okz = magic_decode(__fma_rn(az.p, zs16, zo16), lz.v0);
		jz_out = lin_exit_j(lz);
		return okx && oky && okz;
	};
	unsigned base = 0u;       // sample index of V_0
	model = model && rebase();

	bool finished = false;     // the integer-model loop reached a verdict
	if (model) {
	const float inv_adx = fast_rcp(fabsf((float)dx) * (1.0f / 65536.0f));
	const float inv_ady = fast_rcp(fabsf((float)dy) * (1.0f / 65536.0f));
	const float adz = fabsf((float)dz) * (1.0f / 65536.0f);
	const float inv_adz = fast_rcp(adz);
	const int cell_exit = (int)fminf(P.cell_exit_scale * adz + 512.0f, 1.0e9f);
	const int cell_mask = (1 << k) - 1;
	int level = P.lstart;

	auto probe = [&](int lvl, int vx, int vy) -> int {   // dilated block maximum, in the z units of the model
		const uint2 d = P.lv_desc[lvl];
		const unsigned idx = d.x + pyr_index<kLayout>((unsigned)(vx >> (k + lvl)), (unsigned)(vy >> (k + lvl)), d.y);
		return (int)__ldg(P.lv + HMRM_CHECKED(P, idx, P.lv_total));
	};
	// `above q` / `below q` with the model's error (< 1.6/16 Zq) and Zq16's rounding (ties at q +- 1/2) covered
	auto above = [&](int vz, int q) -> bool { return vz > (q << 4) + HMRM_LIN_ZMARGIN && q < 65535; };

	for (;;) {
		// keep the error bound: re-anchor the model on an exact position every HMRM_LIN_PERIOD samples
		if (n - base >= HMRM_LIN_PERIOD) {
			// (every 65536 samples at most: the place to notice a ray that will never end, ~2^31 samples: give up like a
			// hang would, but flagged)
			if (n >= 0x7FF00000u) {
				tally.cut_off = 1u;
				finished = true;
				break;
			}
			advance_exact(ax, ay, az, anchor, n);
			base = n;
			if (!rebase()) {                 // left the representable range: finish with the per-step loop below
				model = false;
				break;
			}
		}
		const unsigned j = n - base;
		if (kStats) {                        // [6]: warp-level iterations (lane utilisation = lane iterations / 32 / this)
			const unsigned am = __activemask();
			if ((threadIdx.x & 31) == __ffs(am) - 1) {
				tally.dbg[6] += 1u;
				// [8..11]: warp iterations with 1-8, 9-16, 17-24, 25-32 busy lanes
				atomicAdd(&P.stats->dbg[8 + ((__popc(am) - 1) >> 3)], 1ULL);
			}
		}
		// does this sample need the exact treatment?  (within the margin of the grid edge; at level 0 also of a cell edge)
		bool exact = false;
		// (j < HMRM_LIN_PERIOD here, as lin_at requires)
		const int vx = lin_at(lx, j), vy = lin_at(ly, j);
		const bool inside = (unsigned)vx - (unsigned)HMRM_LIN_MARGIN < P.lin_span_x && (unsigned)vy - (unsigned)HMRM_LIN_MARGIN < P.lin_span_y;
		if (!inside) {
			// Certainly outside the grid (main/hmap.cpp:1006-1011)?  The reference truncates toward zero (:1001-1004), so
			// coordinates in (-1, 0) cells still map to cell 0: the low edge of the grid is at -1 cell, not at 0.
			const int low_edge = -(1 << k) - HMRM_LIN_MARGIN;
			if (vx < low_edge || vy < low_edge || vx >= (int)P.lin_grid_x + HMRM_LIN_MARGIN || vy >= (int)P.lin_grid_y + HMRM_LIN_MARGIN) {
				finished = true;
				break;
			}
			exact = true;         // (the whole (-1, 0] strip of the truncation quirk goes the exact way too)
		}
		// height: from jz_out on, far above or far below everything the 16-bit pyramid can hold
		int vz = lin_at(lz, j);
		if (j >= jz_out) vz = lz.di < 0 ? -1073741824 : 1073741824;

		int q = 0;
		if (!exact) {
			// ---- A: find a level whose neighbourhood this sample clears (descend), or reach the cell itself ----
			q = probe(level, vx, vy);
			if (kStats) fetches += 1u;
			while (!above(vz, q) && level > 0) {
				level = (level - P.lstride >= P.lmin) ? level - P.lstride : 0;
				q = probe(level, vx, vy);
				if (kStats) { fetches += 1u; tally.dbg[3] += 1u; }
			}
			if (level == 0) {
				const int fx = vx & cell_mask, fy = vy & cell_mask;
				exact = fx < HMRM_LIN_MARGIN || fy < HMRM_LIN_MARGIN || fx > cell_mask - HMRM_LIN_MARGIN || fy > cell_mask - HMRM_LIN_MARGIN;
			}
		}

		unsigned m = 1u;
		if (!exact && above(vz, q)) {
			// above every surface value of the neighbourhood (or of the cell): this sample cannot hit
			if (level > 0) {
				float est_xy, est_z;
				for (;;) {
					// room (units) along the direction of motion inside the 3x3 neighbourhood of blocks, clipped to the grid
					const unsigned w = 1u << (k + level), mask = w - 1u;
					const unsigned ux = (unsigned)vx, uy = (unsigned)vy;
					const int room_x = (int)(lx.di >= 0 ? min((ux | mask) + 1u + w, P.lin_grid_x) - ux : min((ux & mask) + w, ux));
					const int room_y = (int)(ly.di >= 0 ? min((uy | mask) + 1u + w, P.lin_grid_y) - uy : min((uy & mask) + w, uy));
					est_xy = fminf(__int2float_rz(room_x - (HMRM_LIN_MARGIN + 1)) * inv_adx,
					               __int2float_rz(room_y - (HMRM_LIN_MARGIN + 1)) * inv_ady);
					est_z = lz.di < 0 ? __int2float_rz(vz - (q << 4) - (HMRM_LIN_ZMARGIN + 2)) * inv_adz : 3.0e38f;
					// climb while z leaves room for (much) wider blocks and the wider neighbourhood is cleared too
					if (!(est_z >= P.climb_ratio * est_xy) || level + P.lstride > P.ltop) break;
					const int q2 = probe(level + P.lstride, vx, vy);
					if (kStats) fetches += 1u;
					if (!above(vz, q2)) break;
					level += P.lstride;
					q = q2;
				}
				// Jump length.  The model is integer-exact: V_{j+m} - V_j = round((j+m) D / 2^16) - round(j D / 2^16) lies
				// within 1 unit of m D / 2^16 and V is monotone in j, so any m with m |D| / 2^16 <= room - margin - 1 per
				// axis keeps samples n .. n+m inside the cleared neighbourhood (and above q): no end-point test is needed.
				// The float estimate errs low: conversions round toward zero, and 0.999 covers the ~2^-21 of the reciprocals.
				const float est = fminf(fminf(est_xy, est_z), (float)(HMRM_LIN_PERIOD - j)) * 0.999f;
				m = (est >= 2.0f) ? (unsigned)__float2int_rz(est) : 1u;
				if (kStats) {
					if (m >= 2u) { tally.dbg[0] += 1u; tally.dbg[1] += m; }
					else tally.dbg[2] += 1u;
				}
				// a z-limited jump ends just above q: the next sample will need a finer level
				if (est_z < est_xy) level = (level - P.lstride >= P.lmin) ? level - P.lstride : 0;
			}
			else {
				if (kStats) tally.dbg[4] += 1u;
				if (vz - (q << 4) > cell_exit) level = P.lmin;
			}
		}
		else if (!exact && vz < (q << 4) - HMRM_LIN_ZMARGIN && q > 0) {    // q == 0 may be a clamped value: proves nothing
			// level 0, cell known, clearly below the surface: the reference's test `z < surf` holds (main/hmap.cpp:1016)
			const size_t cell = (size_t)(vx >> k) + (size_t)(vy >> k) * (size_t)P.map_w;
			if (kStats) tally.dbg[5] += 1u;
			hit_cell = (unsigned)cell;      // colour fetched by the caller, once the whole warp is out of the loop
			real_hit = true;
			first_hit = (n > 0x7FFFFFFFu) ? 0x7FFFFFFF : (int)n;
			n += 1u;
			finished = true;
			break;
		}
		else {
			// Undecided in the integer model.  Before paying for an exact reconstruction, take an FP64 look: the reference's
			// sample is P_n = P_a + (n - a) s up to the roundings of its n - a adds, each at most 2^-53 relative and the
			// motion is monotone, so per axis |P_n - fma(n - a, s, P_a)| <= (n - a + 1) * 2^-53 * max(|P_a|, |P_n|).
			// With that bound (doubled below) the reference's own expressions — (int)(x / gw), (int)(-y / gw),
			// z < surf (main/hmap.cpp:1001-1016) — are decided unless the sample is within ~1e-12 of a cell edge or of the
			// surface.  This settles the (-1, 0) truncation strip, cell and grid edges, clamped 16-bit heights and ties.
			{
				const double mj = (double)(n - anchor);
				const double rel = fmul(fadd(mj, 2.0), 2.3e-16);
				const double xe = __fma_rn(mj, ax.s, ax.p), ye = __fma_rn(mj, ay.s, ay.p), ze = __fma_rn(mj, az.s, az.p);
				const double bx = fmul(rel, fmax(fabs(ax.p), fabs(xe))), by = fmul(rel, fmax(fabs(ay.p), fabs(ye)));
				const double bz = fmul(rel, fmax(fabs(az.p), fabs(ze)));
				const double qx = fdiv(xe, P.gw), qy = fdiv(-ye, P.gw);
				// fl(x_true / gw) differs from qx by at most bx / gw + 2^-52 |q|; (int) truncates toward zero, so the only
				// break points are the non-zero integers
				const double axq = fabs(qx), ayq = fabs(qy);
				const double ex_ = fadd(fmul(bx, P.inv_gw_up), fmul(axq, 4.5e-16)), ey_ = fadd(fmul(by, P.inv_gw_up), fmul(ayq, 4.5e-16));
				const double fxq = fsub(axq, floor(axq)), fyq = fsub(ayq, floor(ayq));
				const double near_x = axq < 1.0 ? fsub(1.0, axq) : fmin(fxq, fsub(1.0, fxq));
				const double near_y = ayq < 1.0 ? fsub(1.0, ayq) : fmin(fyq, fsub(1.0, fyq));
				if (axq < 2.0e9 && ayq < 2.0e9 && near_x > ex_ && near_y > ey_) {
					const int gx = trunc_cell(qx), gy = trunc_cell(qy);
					if (gx < 0 || gy < 0 || gx >= P.map_w || gy >= P.map_h) {
						finished = true;                    // the reference's bounds test (:1006-1011): a miss
						break;
					}
					const size_t cell = (size_t)gx + (size_t)gy * (size_t)P.map_w;
					const double surf = __ldg(P.surf + HMRM_CHECKED(P, cell, (size_t)P.map_w * (size_t)P.map_h));
					if (kStats) fetches += 1u;
					if (fadd(ze, bz) < surf) {
						if (kStats) tally.dbg[5] += 1u;
						hit_cell = (unsigned)cell;
						real_hit = true;
						first_hit = (n > 0x7FFFFFFFu) ? 0x7FFFFFFF : (int)n;
						n += 1u;
						finished = true;
						break;
					}
					if (fsub(ze, bz) > surf) {
						if (kStats) tally.dbg[4] += 1u;
						level = 0;
						goto next_sample;                   // certainly not below the surface: plain step, cell level next
					}
				}
			}
			// still undecided: reconstruct the exact sample and let the reference's own expressions decide
			if (kStats) tally.dbg[7] += 1u;
			advance_exact(ax, ay, az, anchor, n);
			const int gx = trunc_cell(fdiv(ax.p, P.gw)), gy = trunc_cell(fdiv(-ay.p, P.gw));
			if (gx < 0 || gy < 0 || gx >= P.map_w || gy >= P.map_h) {
				finished = true;
				break;
			}
			const size_t cell = (size_t)gx + (size_t)gy * (size_t)P.map_w;
			if (kStats) fetches += 1u;
			if (az.p < __ldg(P.surf + HMRM_CHECKED(P, cell, (size_t)P.map_w * (size_t)P.map_h))) {
				hit_cell = (unsigned)cell;      // colour fetched by the caller, once the whole warp is out of the loop
				real_hit = true;
				first_hit = (n > 0x7FFFFFFFu) ? 0x7FFFFFFF : (int)n;
				n += 1u;
				finished = true;
				break;
			}
			level = 0;
		}
next_sample:
		n += m;
	}
	}   // if (model)

	if (!finished) {
		// The plain per-step loop (k2_render_brute.cuh) from the exact anchor on, with a cap instead of a hang: rays
		// that do not fit the integer model, and rays that left its representable range.
		advance_exact(ax, ay, az, anchor, n);
		unsigned long long kk = n;
		for (;;) {
			const int gx = trunc_cell(fdiv(ax.p, P.gw)), gy = trunc_cell(fdiv(-ay.p, P.gw));
			if (gx < 0 || gy < 0 || gx >= P.map_w || gy >= P.map_h) break;
			const size_t cell = (size_t)gx + (size_t)gy * (size_t)P.map_w;
			kk += 1ULL;
			if (kStats) fetches += 1u;
			if (az.p < __ldg(P.surf + HMRM_CHECKED(P, cell, (size_t)P.map_w * (size_t)P.map_h))) {
				hit_cell = (unsigned)cell;      // colour fetched by the caller, once the whole warp is out of the loop
				real_hit = true;
				first_hit = (kk - 1ULL > 0x7FFFFFFFULL) ? 0x7FFFFFFF : (int)(kk - 1ULL);
				break;
			}
			const double nx = fadd(ax.p, ax.s), ny = fadd(ay.p, ay.s), nz = fadd(az.p, az.s);
			if ((nx == ax.p && ny == ay.p && !(nz < az.p)) || kk >= (1ULL << 27)) {
				tally.cut_off = 1u;
				break;
			}
			ax.p = nx; ay.p = ny; az.p = nz;
		}
		tally.steps = kk;
		tally.fetches = fetches;
		return;
	}
	tally.steps = n;
	tally.fetches = fetches;
}

template <bool kStats, int kLayout, int kCtas>
__global__ void __launch_bounds__(HMRM_LIN_THREADS, kCtas) k2_render_lin(const __grid_constant__ RenderParams P) {
	const int lane = threadIdx.x & 31;
	const unsigned n_tiles = (unsigned)(P.tiles_x * P.tiles_y);

	// Tile queue: one atomic per grab.  Marching tiles are grabbed one at a time (their costs are heavy-tailed and a
	// wide grab that swallows several heavy tiles doubles the frame time), but the tile rows the host has placed at
	// the end of the schedule because they look above the horizon are grabbed 8 tiles at a time: a sky tile costs
	// ~25 ns of SM time and a frame's worth of them is otherwise bound by the single-address atomic.
	// (Issuing the next grab before the current tile is processed hides the atomic's round trip but makes every warp
	// sit on a reserved tile: measured 0.53 -> 0.56 ms on the bench frame, dropped.  A CTA-level pool in shared memory
	// refilled with one global atomic per 4/8/16 tiles changed nothing, 0.526 vs 0.528 ms: the wait on the atomic shows
	// in the stall samples but other warps fill the issue slots.)
	unsigned cur = 0u, end = 0u;
	for (;;) {
		if (cur == end) {
			const unsigned batch = (end != 0u && end >= P.batch_from_tile) ? P.sky_batch : 1u;
			unsigned t = 0u;
			if (lane == 0) t = atomicAdd(P.tile_counter, batch);
			cur = __shfl_sync(0xFFFFFFFFu, t, 0);
			end = min(cur + batch, n_tiles);
			if (cur >= n_tiles) break;
		}
		const unsigned tile = cur++;
		int ty_seq, tx;
		tile_row_col(P, tile, ty_seq, tx);
		// longest-processing-time-first: a few grazing tiles take ~50x the mean, so they must start early
		const int ty = P.row_order ? __ldg(P.row_order + HMRM_CHECKED(P, ty_seq, P.tiles_y)) : ty_seq;
		const int px = tx * 8 + (lane & 7);
		const int py = P.row_begin + (P.tile_y_first + ty * P.tile_y_step) * 4 + (lane >> 3);
		const bool active = pixel_selected(P, px, py);

		PixelTally tally = {0ULL, 0ULL, 0u, 0u, 0u, {0u, 0u, 0u, 0u, 0u, 0u, 0u, 0u}};
		uint32_t rgba = 0u;
		if (active) {
			bool real_hit = false;
			int first_hit = -1;
			unsigned hit_cell = 0u;
			const Ray ray = generate_ray(P, px, py);
			double ex, ey, ez, lo = 0.0;
			const bool entered = box_entry(P, ray, ex, ey, ez, lo);
			if (kStats && P.ray_dump) dump_ray(P, px, py, ray, entered, lo, ex, ey, ez);
			if (entered) {
				tally.box_hit = 1u;
				first_hit = -2;
				march_lin<kStats, kLayout>(P, ray, ex, ey, ez, hit_cell, real_hit, first_hit, tally);
			}
			if (!real_hit) rgba = miss_colour(P, ray.dz);
			else {
				rgba = hit_colour(P, __ldg(P.color + HMRM_CHECKED(P, hit_cell, (size_t)P.map_w * (size_t)P.map_h)));
				tally.surf_hit = 1u;
			}
			if (P.step_index) P.step_index[(size_t)py * (size_t)P.W + (size_t)px] = first_hit;
		}
		store_pixel(P, px, py, active, rgba);       // main/hmap.cpp:139-154 (RGBA8), or packed RGB8
		commit_tally<kStats>(P, active, tally);
	}
}

} // namespace hmrm

#endif
