// rg_grid.cuh — Scene::trace with EXACT spatial culling (SURVEY.md section 8f row 1).
//
// Scene::trace is a pure minimum over bodies (scene.rs:34-39), so any body that provably
// returns None — or a distance no smaller than one already found — may be skipped without
// changing the result.  Spheres are binned into a uniform grid; a ray walks the cells it
// pierces (3-D DDA in FP32 grid coordinates) and runs, per listed sphere, the FP32
// conservative cull and then the reference's exact FP64 test.  The result is the same
// lexicographic (distance, body index) minimum as the brute-force scan.
//
// Why no hit can be missed (derivation: DESIGN.md section 4.2):
//   * a sphere is listed in every cell its bounding box, inflated by 2 * kGridInflate = 4e-3 cell,
//     overlaps (binning is done in FP64);
//   * the FP32 walk follows the true ray to within 8.1e-4 cell in every axis (u = 2^-24, grid
//     coordinates <= 1024 in magnitude, <= 256 cells per axis: origin and direction rounding
//     u * 8197, boundary parameters u * 5380), so every point of the true ray lies within that distance
//     of a cell the walk visits, and a sphere hit there is listed in that cell;
//   * the walk stops only at the entry of a cell whose entry parameter lies beyond the best exact
//     distance (with slack): everything nearer lies in — or within the same 8.1e-4 cell of — a cell
//     visited before;
//   * rays the argument does not cover (direction not unit within 1e-9 — reflections off
//     un-normalised plane normals — non-finite origins, origins farther than 1e9 cells) skip the
//     grid and scan every sphere exactly; origins farther than 1024 cells are first moved along
//     the ray, in FP64, to one cell before the grid box;
//   * spheres too large for the grid ("loose") and the non-sphere bodies the grid does not hold are tested per ray;
//   * boxes and disks with sound geometry are binned as enclosing spheres ("proxies", rg_scene.cuh): a line that
//     misses the ball misses the body, and every point the body's test returns lies in the ball, except in one
//     case of the box test (an origin exactly on a face plane of an axis whose 1.0 / d_k is infinite), which the
//     ray set-up finds through the sorted face planes and tests exactly.
//
// Execution model.  Ray lengths differ wildly (a lit shadow ray crosses the whole grid, an
// occluded one stops after a few cells) and the exact FP64 test is ~10x a cull test, so a
// one-thread-per-ray loop leaves most lanes of a warp idle (measured: 6 of 32 active).  The
// kernel therefore runs PERSISTENT warps, and every phase is written so that the lanes that take
// part run ONE instruction stream (a path that is rare per lane is frequent per warp: the SIMT tax):
//   * lanes whose ray is finished retire it and fetch new rays from a global counter (warp ballot +
//     one atomic per refill) instead of waiting for the slowest lane;
//   * scanning lanes fetch one 48-byte record per step — a new cell's first record or the next
//     chained record of a crowded cell, the same code either way — and cull its two items;
//   * a lane that finds a cull survivor parks it ("pending"); the warp evaluates pending
//     candidates together, so the expensive exact test runs with many lanes active instead of one.
#pragma once
#include "rg_trace.cuh"

namespace rg {

#ifndef RG_GRID_THREADS
#define RG_GRID_THREADS 32    // warps of a CTA share nothing: the size only sets how finely finished CTAs make room for the
                              // next kernel's (measured 256 / 128 / 64 / 32 threads: C4 18.94 / 18.02 / 17.98 / 17.82 ms)
#endif
constexpr int kGridTraceThreads = RG_GRID_THREADS;
constexpr float kGridInflate = 2e-3f;       // in cells; see above
constexpr float kGridMaxCoord = 2048.0f;    // |grid coordinate| limit for FP32 traversal
constexpr double kGridUnitTol = 1e-9;
constexpr int kGridRefill = 12;             // refill when at least this many lanes are idle
constexpr int kGridExactQuorum = 6;         // evaluate pending candidates when this many lanes wait
constexpr int kGridScanBurst = 4;           // scan steps between quorum checks
#ifndef RG_GRID_MINB
#define RG_GRID_MINB (7 * 128 / RG_GRID_THREADS)   // CTAs per SM the register budget is set for: 28 warps per SM = 72 registers (measured 16..32 warps)
#endif
constexpr uint32_t kNoSphere = 0xFFFFFFFFu;
constexpr float kFltBig = 3.4e38f;
#define kFltInf __int_as_float(0x7f800000)

// Chained cell records (rg_grid.cu): the record that holds item list positions pos, pos + 1 of a cell whose
// first two items sit in the cell's own record.  Positions of different cells never share a pair, so
// ncells + pos / 2 is collision-free and needs no allocation pass.
__host__ __device__ inline uint32_t grid_chain_record(uint32_t ncells, uint32_t pos) { return ncells + (pos >> 1); }
__host__ __device__ inline size_t grid_record_count(size_t ncells, size_t total_items) { return ncells + total_items / 2 + 1; }

#ifdef RG_GRID_DEBUG
static __device__ unsigned long long rg_grid_dbg[2][16];
#endif

template <bool ANY>
struct GridHit {
    Nearest best;
    bool occluded;
    double tmax;
    __device__ __forceinline__ void offer(double t, uint32_t body) {
        if (ANY) occluded = occluded || (t <= tmax);
        else best.offer(t, body);
    }
    // upper bound on distances still worth looking at (FP32, rounded up generously)
    __device__ __forceinline__ float bound() const {
        if (ANY) return tmax < 3.0e38 ? (float)tmax * 1.000001f + 1e-30f : kFltBig;
        return best.found() ? (float)best.t * 1.000001f + 1e-30f : kFltBig;
    }
};

// One item of the sphere list: a sphere, or (PROXY, index >= n_spheres) a box / disk binned through its enclosing
// sphere, which runs the body's own test.
template <bool ANY, bool PROXY>
__device__ __forceinline__ void exact_sphere(const DScene &s, const Ray &ray, uint32_t sph, GridHit<ANY> &h,
                                             unsigned &n_exact, unsigned &nan_count) {
    const double4 sp = s.sph[sph];
    double t;
    ++n_exact;
    if (PROXY && sph >= s.n_spheres) {
        const uint32_t b = s.sph_body[sph];
        if (misc_intersect(s, b, ray, t)) {
            if (t != t) { ++nan_count; return; }
            h.offer(t, b);
        }
        return;
    }
    if (sphere_intersect(sp.x, sp.y, sp.z, sp.w, ray, t)) {
        if (t != t) { ++nan_count; return; }
        h.offer(t, s.sph_body[sph]);
    }
}

// STATS = true: the instrumented build of the same kernel (RG_OPT_TRACE_STATS) that counts cells visited,
// records fetched, cull tests, refills and lane use into DCounters::grid_*; results are unchanged.
// PROXY = true: the grid also holds boxes and disks (`gp`, rg_scene.cuh); false: spheres only, `gp` is not read.
template <bool ANY, bool STATS = false, bool PROXY = false>
__global__ void __launch_bounds__(kGridTraceThreads, RG_GRID_MINB) k_trace_grid(const DScene s, const TraceArgs a,
                                                                                const GridProxies gp) {
    const GridDev &g = s.grid;
    const uint32_t lane = threadIdx.x & 31u;
    const uint32_t lanemask_lt = (1u << lane) - 1u;
    const uint32_t n_rays = ray_count(a);
    const uint32_t seg_len = segment_length(a);
    unsigned n_exact = 0, nan_count = 0;
    unsigned long long st_cells = 0, st_fetch = 0, st_culls = 0, st_refills = 0, st_lane_steps = 0, st_lane_slots = 0;
#ifdef RG_GRID_DEBUG
    unsigned long long dbg[16] = {0};
    uint32_t last_sph = kNoSphere, last_sph2 = kNoSphere;
    long long tmark = clock64();
#define DBG_PHASE(k) if (STATS) { long long now_ = clock64(); dbg[k] += (unsigned long long)(now_ - tmark); tmark = now_; }
#else
#define DBG_PHASE(k)
#endif

    // ---- per-lane ray state
    bool active = false;        // this lane owns an unfinished ray
    bool walking = false;       // ... and it is inside the grid walk (else it only waits to be written out)
    uint32_t pi = 0;            // physical queue index of the ray
    CullRay cr;
    GridHit<ANY> h;
    // 3-D DDA, per axis: the ray parameter at the next cell boundary is  tn = tex + k * dt  (ONE fmaf, never
    // accumulated), where tex = parameter at the grid's exit plane of that axis, dt = |1 / direction| and
    // -k = boundaries still ahead of the exit plane (a float counter: k > 0 after a step = left the grid)
    float tnx = 0, tny = 0, tnz = 0;
    float kx = 0, ky = 0, kz = 0;
    float dtx = 0, dty = 0, dtz = 0;
    float tex = 0, tey = 0, tez = 0;
    float tcur = 0;                                            // parameter at which the walk enters `cell` (+inf: it has left the grid)
    float boundf = 0;                                          // distances worth looking at, in walk parameter units (FP32, rounded up)
    float t0f = 0;                                             // the walk is parameterised from o + t0*d (far origins)
    int cell = 0, scx = 0, scy = 0, scz = 0;                   // linear index of the next cell to examine, per-axis stride (signed)
    uint32_t pend0 = kNoSphere, pend1 = kNoSphere;             // cull survivors waiting for their exact test
    uint32_t chain = 0;                                        // next record of the cell being examined (0: none, enter the next cell)
    uint32_t skip = kNoSphere;                                 // a sphere whose exact result for this ray is already known: the origin hint
                                                               // (rg_trace.cuh), then the sphere tested last (it is listed in the next cells too)
    bool exhausted = false;                                    // warp-uniform: the queue has no more rays
    h.best.init();
    h.occluded = false;
    h.tmax = 0.0;
    {
        Ray none;
        none.o = d3(0, 0, 0);
        none.d = d3(0, 0, 0);
        cr = make_cull_ray(s, none, false);
    }


    for (;;) {
        // ================= (A) retire finished rays, refill idle lanes from the global ray counter ==========
        if (active && !walking && pend0 == kNoSphere && pend1 == kNoSphere) {
            if (ANY) a.out_lit[pi] = h.occluded ? 0 : 1;
            else { a.out_t[pi] = h.best.t; a.out_body[pi] = h.best.body; }
            active = false;
        }
        const uint32_t idle = __ballot_sync(0xffffffffu, !active);
        if (idle == 0xffffffffu && exhausted) break;
        if (!exhausted && (__popc(idle) >= a.g_refill)) {
            uint32_t base = 0;
            if (lane == 0) base = atomicAdd(a.fetch, (unsigned)__popc(idle));
            base = __shfl_sync(0xffffffffu, base, 0);
            exhausted = base + (uint32_t)__popc(idle) >= n_rays;
            if (STATS && lane == 0) ++st_refills;
#ifdef RG_GRID_DEBUG
            if (STATS && lane == 0) dbg[12] += __popc(idle);
            last_sph = last_sph2 = (!active) ? kNoSphere : last_sph;
#endif
            const uint32_t ri = base + __popc(idle & lanemask_lt);
            if (!active && ri < n_rays) {
                // ---- set a new ray up: non-sphere bodies, loose spheres, clip to the grid
                active = true;
                walking = false;
                pend0 = pend1 = kNoSphere;
                chain = 0;
                pi = phys_index(seg_len, a.seg_stride, ri);
                const Ray ray = load_ray(a.q, pi);
                skip = a.q.hint[pi];
                h.best.init();
                h.occluded = false;
                h.tmax = ANY ? a.tmax[pi] : 0.0;
                if (!PROXY) {   // (verbatim as before proxies: the sphere-only kernels compile to the same SASS)
                for (uint32_t m = 0; m < s.n_misc; ++m) {          // planes, disks, boxes: exact, per ray
                    const uint32_t b = s.misc_body[m];
                    double t;
                    if (misc_intersect(s, b, ray, t)) {
                        if (t != t) { ++nan_count; continue; }
                        h.offer(t, b);
                    }
                }
                n_exact += s.n_misc;
                } else {
                    for (uint32_t m = 0; m < gp.n_misc; ++m) {     // non-sphere bodies kept out of the grid: exact, per ray
                        const uint32_t b = gp.misc_body[m];
                        double t;
                        if (misc_intersect(s, b, ray, t)) {
                            if (t != t) { ++nan_count; continue; }
                            h.offer(t, b);
                        }
                    }
                    n_exact += gp.n_misc;
                    // The one case where the reference's box test can return a point outside the box: 1.0 / d_k is
                    // infinite and o_k lies exactly on a face plane of axis k (0 * inf = NaN drops a slab check).
                    // Such boxes are found through the sorted face planes and tested here, whatever else happens.
                    const double od[3] = {ray.o.x, ray.o.y, ray.o.z}, dd[3] = {ray.d.x, ray.d.y, ray.d.z};
#pragma unroll 1
                    for (int k = 0; k < 3; ++k) {
                        if (!isinf(1.0 / dd[k])) continue;
                        const FaceRef *f = gp.faces + (size_t)k * gp.n_faces;
                        uint32_t lo = 0, hi = gp.n_faces;
                        while (lo < hi) {
                            const uint32_t mid = (lo + hi) >> 1;
                            if (f[mid].c < od[k]) lo = mid + 1; else hi = mid;
                        }
                        for (; lo < gp.n_faces && f[lo].c == od[k]; ++lo) {
                            const uint32_t b = f[lo].body;
                            double t;
                            ++n_exact;
                            if (aabb_intersect(s.geom + 8 * (size_t)b, ray, t)) {
                                if (t != t) { ++nan_count; continue; }
                                h.offer(t, b);
                            }
                        }
                    }
                }
                if (ANY && skip == kHintOccluded) h.occluded = true;   // the sphere the ray starts on is in the way
                if (!(ANY && h.occluded)) {
                cr = make_cull_ray(s, ray, true);
                D3 op = ray.o - d3(s.cull_ref[0], s.cull_ref[1], s.cull_ref[2]);
                const double D2 = dot(ray.d, ray.d);
                // Far-away origins (e.g. hits on an infinite plane near the horizon) would lose FP32
                // position accuracy inside the grid.  Clip such rays against the grid box in FP64 and
                // start the FP32 walk from o + t0*d, a point on the same ray just before the box.
                bool misses_box = false;
                t0f = 0.0f;
                {
                    const double gx = (op.x - (double)g.lo[0]) * (double)g.inv_cell[0];
                    const double gy = (op.y - (double)g.lo[1]) * (double)g.inv_cell[1];
                    const double gz = (op.z - (double)g.lo[2]) * (double)g.inv_cell[2];
                    const double lim = 0.5 * (double)kGridMaxCoord;
                    const bool near_box = fabs(gx) <= lim && fabs(gy) <= lim && fabs(gz) <= lim;   // false on NaN
                    // (beyond 1e9 cells the FP64 move along the ray would itself cost more than 1e-6 cell: such rays scan every sphere)
                    const bool finite = fabs(gx) < 1e9 && fabs(gy) < 1e9 && fabs(gz) < 1e9;
                    if (!near_box && finite) {
                        const double ddx = ray.d.x * (double)g.inv_cell[0], ddy = ray.d.y * (double)g.inv_cell[1],
                                     ddz = ray.d.z * (double)g.inv_cell[2];
                        double tmin = 0.0, tmax = 1e300;
                        const double gs[3] = {gx, gy, gz}, ds[3] = {ddx, ddy, ddz};
#pragma unroll
                        for (int k = 0; k < 3; ++k) {
                            const double dimk = (double)g.dim[k];
                            if (ds[k] == 0.0) {
                                if (gs[k] < -1.0 || gs[k] > dimk + 1.0) misses_box = true;
                            } else {
                                const double ta = (-1.0 - gs[k]) / ds[k], tb = (dimk + 1.0 - gs[k]) / ds[k];   // box padded by a cell
                                tmin = fmax(tmin, fmin(ta, tb));
                                tmax = fmin(tmax, fmax(ta, tb));
                            }
                        }
                        if (!(tmin <= tmax)) misses_box = true;   // also on NaN
                        if (!misses_box) {
                            op = op + ray.d * tmin;                // still on the ray, one cell before the box
                            t0f = __double2float_rd(tmin);         // rounded down: bounds stay conservative
                        }
                    }
                }
                const float ogx = ((float)op.x - g.lo[0]) * g.inv_cell[0];
                const float ogy = ((float)op.y - g.lo[1]) * g.inv_cell[1];
                const float ogz = ((float)op.z - g.lo[2]) * g.inv_cell[2];
                const float dgx = (float)ray.d.x * g.inv_cell[0], dgy = (float)ray.d.y * g.inv_cell[1],
                            dgz = (float)ray.d.z * g.inv_cell[2];
                const bool walkable = fabs(D2 - 1.0) <= kGridUnitTol && (misses_box || (fabsf(ogx) <= kGridMaxCoord &&
                                      fabsf(ogy) <= kGridMaxCoord && fabsf(ogz) <= kGridMaxCoord));   // false on NaN
                {
                    if (!walkable) {
                        // outside the conservativeness argument: scan every sphere (cull + exact) and every proxy's
                        // body (exact: the cull's bound on a proxy assumes |d| = 1 within the walk's 1e-9, DESIGN 4.2)
                        for (uint32_t q = 0; q < s.n_spheres; ++q)
                            if (q != skip && !cull_reject(cr, s.cull4[q])) exact_sphere<ANY, PROXY>(s, ray, q, h, n_exact, nan_count);
                        if (PROXY)
                            for (uint32_t q = s.n_spheres; q < s.n_spheres + gp.n_proxies; ++q)
                                exact_sphere<ANY, PROXY>(s, ray, q, h, n_exact, nan_count);
                    } else {
                        for (uint32_t q = 0; q < g.n_loose; ++q) {
                            const uint32_t sp = g.loose[q];
                            if (sp != skip && !cull_reject(cr, s.cull4[sp])) exact_sphere<ANY, PROXY>(s, ray, sp, h, n_exact, nan_count);
                        }
                        // clip the ray to the grid box [0, dim]
                        const float ix = 1.0f / dgx, iy = 1.0f / dgy, iz = 1.0f / dgz;
                        const float dimx = (float)g.dim[0], dimy = (float)g.dim[1], dimz = (float)g.dim[2];
                        float t0x = (0.0f - ogx) * ix, t1x = (dimx - ogx) * ix;
                        float t0y = (0.0f - ogy) * iy, t1y = (dimy - ogy) * iy;
                        float t0z = (0.0f - ogz) * iz, t1z = (dimz - ogz) * iz;
                        // a ray parallel to a slab (d = 0): inside -> (-inf, +inf), outside -> empty
                        if (dgx == 0.0f) { bool in = ogx >= 0.0f && ogx <= dimx; t0x = in ? -kFltBig : kFltBig; t1x = in ? kFltBig : -kFltBig; }
                        if (dgy == 0.0f) { bool in = ogy >= 0.0f && ogy <= dimy; t0y = in ? -kFltBig : kFltBig; t1y = in ? kFltBig : -kFltBig; }
                        if (dgz == 0.0f) { bool in = ogz >= 0.0f && ogz <= dimz; t0z = in ? -kFltBig : kFltBig; t1z = in ? kFltBig : -kFltBig; }
                        const float tenter = fmaxf(fmaxf(fminf(t0x, t1x), fminf(t0y, t1y)), fmaxf(fminf(t0z, t1z), 0.0f));
                        const float texit = fminf(fminf(fmaxf(t0x, t1x), fmaxf(t0y, t1y)), fmaxf(t0z, t1z));
                        // slack: the box walls are padded away from every sphere, so grazing rays may go either way
                        boundf = h.bound() - t0f;
                        if (!misses_box && tenter <= texit * 1.000001f + 1e-6f && tenter <= boundf) {
                            const int cx = min(max((int)floorf(ogx + tenter * dgx), 0), g.dim[0] - 1);
                            const int cy = min(max((int)floorf(ogy + tenter * dgy), 0), g.dim[1] - 1);
                            const int cz = min(max((int)floorf(ogz + tenter * dgz), 0), g.dim[2] - 1);
                            // per axis: exit plane of the grid (dim when stepping up, 0 when stepping down), the
                            // parameter there, the parameter step per cell, and minus the boundaries before it.
                            // An axis the ray does not move along never steps: tn = +big.
                            tex = dgx > 0.0f ? (dimx - ogx) * ix : (dgx < 0.0f ? (0.0f - ogx) * ix : kFltBig);
                            tey = dgy > 0.0f ? (dimy - ogy) * iy : (dgy < 0.0f ? (0.0f - ogy) * iy : kFltBig);
                            tez = dgz > 0.0f ? (dimz - ogz) * iz : (dgz < 0.0f ? (0.0f - ogz) * iz : kFltBig);
                            dtx = dgx != 0.0f ? fabsf(ix) : 0.0f;
                            dty = dgy != 0.0f ? fabsf(iy) : 0.0f;
                            dtz = dgz != 0.0f ? fabsf(iz) : 0.0f;
                            kx = dgx > 0.0f ? (float)(cx + 1 - g.dim[0]) : (float)(-cx);
                            ky = dgy > 0.0f ? (float)(cy + 1 - g.dim[1]) : (float)(-cy);
                            kz = dgz > 0.0f ? (float)(cz + 1 - g.dim[2]) : (float)(-cz);
                            tnx = fmaf(kx, dtx, tex);
                            tny = fmaf(ky, dty, tey);
                            tnz = fmaf(kz, dtz, tez);
                            cell = (cz * g.dim[1] + cy) * g.dim[0] + cx;
                            scx = dgx > 0.0f ? 1 : -1;
                            scy = dgy > 0.0f ? g.dim[0] : -g.dim[0];
                            scz = dgz > 0.0f ? g.dim[0] * g.dim[1] : -(g.dim[0] * g.dim[1]);
                            tcur = tenter;
                            walking = true;
                        }
                    }
                }
                }   // not occluded by a body tested above / by the origin hint
            }
        }

        DBG_PHASE(0)
        // ================= (B) scan: one 48-byte record per step ======================================
        // A scanning lane fetches ONE record per step and culls its two items: either the first record of
        // the next cell of its walk — the DDA then advances to the cell after it WHILE the fetch is in flight
        // (the step does not depend on what the cell holds) — or the next chained record of the cell it is
        // in (cells with more than two items).  Both cases run the same instruction stream (the step is
        // predicated), so a warp never serialises a rare per-lane path.  Records live only inside one
        // iteration: nothing of them stays in registers across the refill and exact-test phases.
#pragma unroll 1
        for (int burst = 0; burst < a.g_burst; ++burst) {
            bool go = active && walking && pend0 == kNoSphere && pend1 == kNoSphere;
            const bool enter = chain == 0u;   // the next record is a new cell's first
            if (go && enter && ((ANY && h.occluded) || boundf < fmaf(tcur, 0.99999f, -1e-5f))) {
                walking = false;   // nothing nearer can lie in or beyond this cell (or the walk has left the grid)
                go = false;
            }
            if (STATS) {
                st_lane_steps += go ? 1u : 0u;
                if (lane == 0) st_lane_slots += 32u;
            }
            if (go) {
                const float4 *rec = g.cell_rec + 3 * (size_t)(enter ? (uint32_t)cell : chain);
                const float4 c0 = rec[0], c1 = rec[1];
                const uint4 cm = *reinterpret_cast<const uint4 *>(rec + 2);
                if (enter) {
                    // step: the axis whose boundary comes first; tn = tex + k * dt recomputed, never accumulated
                    const float tnext = fminf(tnx, fminf(tny, tnz));
                    const bool ax = tnx <= tny && tnx <= tnz;
                    const bool ay = !ax && tny <= tnz;
                    const bool az = !ax && !ay;
                    kx += ax ? 1.0f : 0.0f;
                    ky += ay ? 1.0f : 0.0f;
                    kz += az ? 1.0f : 0.0f;
                    tnx = fmaf(kx, dtx, tex);
                    tny = fmaf(ky, dty, tey);
                    tnz = fmaf(kz, dtz, tez);
                    cell += ax ? scx : (ay ? scy : scz);
                    // k > 0: that boundary was the grid's exit plane (+inf beats every bound).  (A prefetch.global.L1 of the
                    // next cell's record at this point — it is known before this cell's culls run — was measured: 19.8 -> 25.0 ms.)
                    tcur = fmaxf(kx, fmaxf(ky, kz)) > 0.0f ? kFltInf : tnext;
                }
                if (STATS) { st_cells += enter ? 1u : 0u; st_fetch += (cm.x != kNoSphere) ? 1u : 0u; st_culls += (cm.x != kNoSphere) + (cm.y != kNoSphere); }
                // (an empty slot holds kNoSphere: "parking" it parks nothing, so it needs no test of its own)
                if (cm.x != skip && !cull_reject(cr, c0)) pend0 = cm.x;
                if (cm.y != skip && !cull_reject(cr, c1)) pend1 = cm.y;
                chain = cm.z;
            }
        }

        DBG_PHASE(1)
        // ================= (C) exact tests of the parked candidates, many lanes at a time ==========
        const bool has_pending = pend0 != kNoSphere || pend1 != kNoSphere;
        const uint32_t waiting = __ballot_sync(0xffffffffu, has_pending);
        const uint32_t scanning = __ballot_sync(0xffffffffu, active && walking && !has_pending);
        if (waiting && (__popc(waiting) >= a.g_quorum || scanning == 0u ||
                        (exhausted && __popc(waiting) * 2 >= __popc(waiting | scanning)))) {
#ifdef RG_GRID_DEBUG
            if (STATS) {
                if (lane == 0) { dbg[3] += 1; dbg[4] += __popc(waiting); }
                if (RG_GRID_DEBUG >= 2 && has_pending) {
                    const Ray ray = load_ray(a.q, pi);
                    for (int w = 0; w < 2; ++w) {
                        const uint32_t sp_i = w ? pend1 : pend0;
                        if (sp_i == kNoSphere) continue;
                        dbg[5] += 1;
                        if (sp_i == last_sph || sp_i == last_sph2) dbg[10] += 1;
                        last_sph2 = last_sph; last_sph = sp_i;
                        const double4 sp = s.sph[sp_i];
                        D3 hyp = d3(sp.x, sp.y, sp.z) - ray.o;
                        double adj = dot(hyp, ray.d);
                        double opp2 = dot(hyp, hyp) - (adj * adj);
                        double r2 = sp.w * sp.w;
                        double t;
                        if (opp2 > r2) dbg[6] += 1;
                        else if (!sphere_intersect(sp.x, sp.y, sp.z, sp.w, ray, t)) { dbg[7] += 1; if (fabs(dot(hyp, hyp) - r2) < 1e-6 * r2) dbg[11] += 1; }
                        else if (ANY ? !(t <= h.tmax) : !(t < h.best.t || !h.best.found())) dbg[8] += 1;
                        else dbg[9] += 1;
                    }
                }
            }
#endif
            if (has_pending) {
                // every waiting lane runs the first test together; a second survivor of the same record is rare
                const Ray ray = load_ray(a.q, pi);
                const uint32_t first = pend0 != kNoSphere ? pend0 : pend1;
                const uint32_t second = pend0 != kNoSphere ? pend1 : kNoSphere;
                exact_sphere<ANY, PROXY>(s, ray, first, h, n_exact, nan_count);
                if (second != kNoSphere) exact_sphere<ANY, PROXY>(s, ray, second, h, n_exact, nan_count);
                skip = second != kNoSphere ? second : first;   // re-listed in the cells that follow: same ray, same answer
                pend0 = pend1 = kNoSphere;
                boundf = h.bound() - t0f;
            }
        }
        DBG_PHASE(2)
#ifdef RG_GRID_DEBUG
        if (STATS && lane == 0) dbg[13] += 1;
#endif
    }
#ifdef RG_GRID_DEBUG
    if (STATS) {
        for (int k = 0; k < 16; ++k) {
            unsigned long long v = dbg[k];
            const bool lane0_only = k <= 4 || k == 13 || k == 12;
            if (!lane0_only) for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
            if (lane == 0 && v) atomicAdd(&rg_grid_dbg[ANY ? 1 : 0][k], v);
        }
    }
#endif

    unsigned long long ne = n_exact;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        ne += __shfl_xor_sync(0xffffffffu, ne, o);
        nan_count += __shfl_xor_sync(0xffffffffu, nan_count, o);
    }
    if (lane == 0) {
        if (ne) atomicAdd(&a.ctr->exact_tests, ne);
        if (nan_count) atomicAdd(&a.ctr->err_nan, (unsigned long long)nan_count);
    }
    if (STATS) {
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            st_cells += __shfl_xor_sync(0xffffffffu, st_cells, o);
            st_fetch += __shfl_xor_sync(0xffffffffu, st_fetch, o);
            st_culls += __shfl_xor_sync(0xffffffffu, st_culls, o);
            st_lane_steps += __shfl_xor_sync(0xffffffffu, st_lane_steps, o);
        }
        if (lane == 0) {
            atomicAdd(&a.ctr->grid_cells, st_cells);
            atomicAdd(&a.ctr->grid_fetches, st_fetch);
            atomicAdd(&a.ctr->grid_culls, st_culls);
            atomicAdd(&a.ctr->grid_refills, st_refills);
            atomicAdd(&a.ctr->grid_lane_steps, st_lane_steps);
            atomicAdd(&a.ctr->grid_lane_slots, st_lane_slots);
        }
    }
}

}  // namespace rg
