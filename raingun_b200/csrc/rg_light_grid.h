// rg_light_grid.h — per-light 2-D grids for shadow rays (DESIGN.md section 4.2, "Light grids"), shared by the
// device build and tracer (rg_grid.cu, rg_grid.cuh) and the host unit test (tests/test_light_grid_cpu.py).
//
// Every shadow ray of one light lies on a line the light fixes up to a 2-D key: a directional light's rays all run
// along d = l.v, so the key is where the origin projects onto a plane perpendicular to d; a spherical light's rays
// all run through its position L, so the key is the direction o - L, looked up in a cube map around L.  A sphere
// (or a box / disk proxy) is listed in every cell of the key space its ball, inflated by kLgInflate * scale,
// can reach; one that would cover more than kLgMaxCells cells, or that is not finite, goes on the light's
// "always" list, which every ray of the light tests.  Each list is sorted from the light outward by the item's
// light-space depth, so a ray can stop at the first record that lies beyond its own origin.
//
// Cells of all lights share one index space: cell 0 is an empty placeholder (so that record 0 is never a cell's
// first record and chain = 0 keeps meaning "no more records"), then per light its key cells and its always list.
#pragma once
#include <stdint.h>

#include <algorithm>
#include <cmath>
#include <cstring>

#ifdef __CUDACC__
#define RG_LG_HD __host__ __device__
#else
#define RG_LG_HD
#endif

namespace rg {

constexpr uint32_t kLightGrids = 8;        // lights [0, kLightGrids) of a scene get a grid
constexpr double kLgInflate = 1e-5;        // x scale: added to every radius (covers the FP64 exact test and |o + tmax d - L|)
constexpr double kLgOriginMax = 16.0;      // x scale: rays from farther origins keep the 3-D walk
constexpr double kLgUnitTol = 1e-14;       // | |d|^2 - 1 | above this: the 3-D walk
constexpr double kLgEndTol = 1e-9;         // x scale: spherical lights, |o + tmax d - L| per axis above this: the 3-D walk
constexpr double kLgPad = 1e-3;            // cells: every binned range is widened by this much on both sides
constexpr uint32_t kLgMaxCells = 1024;     // an item that would cover more cells of one light goes on its always list
constexpr int kLgMaxDim = 1024;            // cells per axis (directional) or per cube face edge (spherical)

struct LightGridInfo {
    double v[3];          // directional: the rays' direction l.v; spherical: the light's position L
    double U[3], W[3];    // directional: orthonormal basis of the key plane (perpendicular to v)
    double lo[2], inv[2]; // directional: key-plane origin and inverse cell size per axis
    double scale;         // 1 + the largest |coordinate| of the scene's items and of the light
    int32_t dim[2];       // directional: cells per axis; spherical: cells per cube face edge (both)
    uint32_t kind;        // RG_LIGHT_DIRECTIONAL (0) | RG_LIGHT_SPHERICAL (1)
    uint32_t base;        // index of the light's first key cell
    uint32_t always;      // index of the light's always list (= base + key cells)
    uint32_t pad;
};

RG_LG_HD inline uint32_t lg_key_cells(const LightGridInfo &g) {
    return g.kind == 0 ? (uint32_t)g.dim[0] * (uint32_t)g.dim[1] : 6u * (uint32_t)g.dim[0] * (uint32_t)g.dim[0];
}

RG_LG_HD inline int lg_floor_clamp(double x, int n) {
    const double f = std::floor(x);
    return f < 0.0 ? 0 : (f > (double)(n - 1) ? n - 1 : (int)f);
}

// Where an item lies in one light's key space.  Returns the number of key cells it covers (ranges: per face, or
// face 0 for a directional light, cells [r[f][0], r[f][1]] x [r[f][2], r[f][3]], empty when r[f][0] > r[f][1]),
// or -1: the item goes on the always list.  Binning runs in FP64 on the device and in the host test alike.
RG_LG_HD inline int lg_item_ranges(const LightGridInfo &g, const double c[3], double r, int rng[6][4]) {
    r = std::fabs(r);
    const bool ok = std::isfinite(c[0]) && std::isfinite(c[1]) && std::isfinite(c[2]) && std::isfinite(r) &&
                    std::fabs(c[0]) < 1e6 && std::fabs(c[1]) < 1e6 && std::fabs(c[2]) < 1e6 && r < 1e6;
    if (!ok) return -1;
    const double R = r + kLgInflate * g.scale;
    for (int f = 0; f < 6; ++f) { rng[f][0] = 1; rng[f][1] = 0; rng[f][2] = 1; rng[f][3] = 0; }
    long long cells = 0;
    if (g.kind == 0) {
        const double cu = (c[0] * g.U[0] + c[1] * g.U[1]) + c[2] * g.U[2];
        const double cw = (c[0] * g.W[0] + c[1] * g.W[1]) + c[2] * g.W[2];
        rng[0][0] = lg_floor_clamp((cu - R - g.lo[0]) * g.inv[0] - kLgPad, g.dim[0]);
        rng[0][1] = lg_floor_clamp((cu + R - g.lo[0]) * g.inv[0] + kLgPad, g.dim[0]);
        rng[0][2] = lg_floor_clamp((cw - R - g.lo[1]) * g.inv[1] - kLgPad, g.dim[1]);
        rng[0][3] = lg_floor_clamp((cw + R - g.lo[1]) * g.inv[1] + kLgPad, g.dim[1]);
        cells = (long long)(rng[0][1] - rng[0][0] + 1) * (rng[0][3] - rng[0][2] + 1);
    } else {
        // The ball's bounding box relative to L; on face (m, s) a direction v has coordinates (v_a, v_b) / (s v_m)
        // with s v_m > 0.  Over the box, with w = s v_m in (max(w0, 0), w1], a / w is bounded as below.
        const int N = g.dim[0];
        const double rel[3] = {c[0] - g.v[0], c[1] - g.v[1], c[2] - g.v[2]};
        for (int f = 0; f < 6; ++f) {
            const int m = f >> 1, a = m == 0 ? 1 : 0, b = m == 2 ? 1 : 2;
            const double s = (f & 1) ? -1.0 : 1.0;
            const double w0 = s * rel[m] - R, w1 = s * rel[m] + R;
            if (!(w1 > 0.0)) continue;
            double lim[2][2];
            const int ax[2] = {a, b};
            for (int k = 0; k < 2; ++k) {
                const double A0 = rel[ax[k]] - R, A1 = rel[ax[k]] + R;
                lim[k][0] = A0 >= 0.0 ? A0 / w1 : (w0 > 0.0 ? A0 / w0 : -2.0);
                lim[k][1] = A1 <= 0.0 ? A1 / w1 : (w0 > 0.0 ? A1 / w0 : 2.0);
            }
            if (lim[0][0] > 1.0 + 1e-9 || lim[0][1] < -1.0 - 1e-9 || lim[1][0] > 1.0 + 1e-9 || lim[1][1] < -1.0 - 1e-9) continue;
            for (int k = 0; k < 2; ++k) {
                const double u0 = lim[k][0] < -1.0 ? -1.0 : lim[k][0], u1 = lim[k][1] > 1.0 ? 1.0 : lim[k][1];
                rng[f][2 * k] = lg_floor_clamp((u0 + 1.0) * 0.5 * N - kLgPad, N);
                rng[f][2 * k + 1] = lg_floor_clamp((u1 + 1.0) * 0.5 * N + kLgPad, N);
            }
            cells += (long long)(rng[f][1] - rng[f][0] + 1) * (rng[f][3] - rng[f][2] + 1);
        }
    }
    return cells > (long long)kLgMaxCells ? -1 : (int)cells;
}

// Cell index (relative to g.base) of key-cell (x, y) on face f.
RG_LG_HD inline uint32_t lg_cell_index(const LightGridInfo &g, int f, int x, int y) {
    return ((uint32_t)f * (uint32_t)g.dim[1] + (uint32_t)y) * (uint32_t)g.dim[0] + (uint32_t)x;
}

// Light-space depth of an item, smallest where the item is nearest the light (directional: -(v.c + R); spherical:
// |c - L| - R).  Lists are sorted by it, rounded down to FP32.
RG_LG_HD inline double lg_item_depth(const LightGridInfo &g, const double c[3], double r) {
    const double R = std::fabs(r) + kLgInflate * g.scale;
    if (g.kind == 0) return -(((c[0] * g.v[0] + c[1] * g.v[1]) + c[2] * g.v[2]) + R);
    const double x = c[0] - g.v[0], y = c[1] - g.v[1], z = c[2] - g.v[2];
    return std::sqrt((x * x + y * y) + z * z) - R;
}

// Key of a shadow ray of this light: its key cell (relative to g.base), or -1 when its key lies outside the
// directional grid (no listed item can then be hit: only the always list is left), or -2 when the ray lies outside
// the argument of DESIGN.md 4.2 and keeps the 3-D walk.  `depth` receives the ray's own light-space depth.
RG_LG_HD inline long long lg_ray_key(const LightGridInfo &g, const double o[3], const double d[3], double tmax, double &depth) {
    const double lim = kLgOriginMax * g.scale;
    if (!(std::fabs(o[0]) <= lim && std::fabs(o[1]) <= lim && std::fabs(o[2]) <= lim)) return -2;   // also NaN
    const double D2 = (d[0] * d[0] + d[1] * d[1]) + d[2] * d[2];
    if (!(std::fabs(D2 - 1.0) <= kLgUnitTol)) return -2;
    if (g.kind == 0) {
        if (!(d[0] == g.v[0] && d[1] == g.v[1] && d[2] == g.v[2])) return -2;
        depth = -((o[0] * g.v[0] + o[1] * g.v[1]) + o[2] * g.v[2]);
        const double x = (((o[0] * g.U[0] + o[1] * g.U[1]) + o[2] * g.U[2]) - g.lo[0]) * g.inv[0];
        const double y = (((o[0] * g.W[0] + o[1] * g.W[1]) + o[2] * g.W[2]) - g.lo[1]) * g.inv[1];
        if (!(x >= 0.0 && x < (double)g.dim[0] && y >= 0.0 && y < (double)g.dim[1])) return -1;
        return (long long)lg_cell_index(g, 0, lg_floor_clamp(x, g.dim[0]), lg_floor_clamp(y, g.dim[1]));
    }
    const double tol = kLgEndTol * g.scale;
    const double v[3] = {o[0] - g.v[0], o[1] - g.v[1], o[2] - g.v[2]};
    for (int k = 0; k < 3; ++k)
        if (!(std::fabs((o[k] + tmax * d[k]) - g.v[k]) <= tol)) return -2;   // the ray does not end at L (also NaN tmax)
    const double ax = std::fabs(v[0]), ay = std::fabs(v[1]), az = std::fabs(v[2]);
    const int m = (ax >= ay && ax >= az) ? 0 : (ay >= az ? 1 : 2);
    const double vm = v[m];
    if (vm == 0.0) return -2;
    const int a = m == 0 ? 1 : 0, b = m == 2 ? 1 : 2;
    const int f = 2 * m + (vm < 0.0 ? 1 : 0);
    const double am = std::fabs(vm);
    const int N = g.dim[0];
    depth = std::sqrt((v[0] * v[0] + v[1] * v[1]) + v[2] * v[2]);
    return (long long)lg_cell_index(g, f, lg_floor_clamp((v[a] / am + 1.0) * 0.5 * N, N), lg_floor_clamp((v[b] / am + 1.0) * 0.5 * N, N));
}

// Sort key of a list entry: FP32 depth rounded down, mapped to an unsigned order, then the item index.
RG_LG_HD inline uint32_t lg_float_order(float f) {
    uint32_t u;
    std::memcpy(&u, &f, 4);
    return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}
RG_LG_HD inline float lg_order_float(uint32_t u) {
    u = (u & 0x80000000u) ? (u & 0x7FFFFFFFu) : ~u;
    float f;
    std::memcpy(&f, &u, 4);
    return f;
}
RG_LG_HD inline float lg_float_down(double x) {
#ifdef __CUDA_ARCH__
    return __double2float_rd(x);
#else
    float f = (float)x;
    if ((double)f > x) f = std::nextafter(f, -INFINITY);
    return f;
#endif
}

// Ascending in-place sort of a list's keys: insertion sort for short lists, heap sort beyond (cf. gb_sort_u32).
RG_LG_HD inline void lg_sort_u64(uint64_t *v, uint32_t n) {
    if (n <= 32u) {
        for (uint32_t i = 1; i < n; ++i) {
            const uint64_t x = v[i];
            uint32_t j = i;
            while (j > 0 && v[j - 1] > x) { v[j] = v[j - 1]; --j; }
            v[j] = x;
        }
        return;
    }
    for (uint32_t i = n / 2u; i-- > 0;) {
        uint32_t root = i;
        const uint64_t x = v[root];
        for (;;) {
            uint32_t child = 2u * root + 1u;
            if (child >= n) break;
            if (child + 1u < n && v[child + 1u] > v[child]) ++child;
            if (v[child] <= x) break;
            v[root] = v[child];
            root = child;
        }
        v[root] = x;
    }
    for (uint32_t end = n - 1u; end > 0; --end) {
        const uint64_t t = v[0];
        v[0] = v[end];
        v[end] = t;
        uint32_t root = 0;
        const uint64_t x = v[0];
        for (;;) {
            uint32_t child = 2u * root + 1u;
            if (child >= end) break;
            if (child + 1u < end && v[child + 1u] > v[child]) ++child;
            if (v[child] <= x) break;
            v[root] = v[child];
            root = child;
        }
        v[root] = x;
    }
}

// Host: the geometry of one light's grid from the item list (n x 4: centre, radius) and the scene's scale;
// `cells_per_item` sets the resolution.  Returns false when the light gets no grid.
inline bool lg_setup(LightGridInfo &g, uint32_t kind, const double v[3], const double *items, uint32_t n, double scale,
                     double cells_per_item) {
    g = LightGridInfo{};
    g.kind = kind;
    g.scale = scale;
    for (int k = 0; k < 3; ++k) g.v[k] = v[k];
    if (!(std::isfinite(v[0]) && std::isfinite(v[1]) && std::isfinite(v[2])) || n == 0) return false;
    const double cells = std::max(1.0, cells_per_item * (double)n);
    if (kind != 0) {
        const int N = (int)std::min((double)kLgMaxDim, std::max(1.0, std::ceil(std::sqrt(cells / 6.0))));
        g.dim[0] = g.dim[1] = N;
        return true;
    }
    const double D2 = (v[0] * v[0] + v[1] * v[1]) + v[2] * v[2];
    if (!(std::fabs(D2 - 1.0) <= kLgUnitTol)) return false;
    // U: v x (the axis least aligned with v), normalised; W = v x U
    const int k = (std::fabs(v[0]) <= std::fabs(v[1]) && std::fabs(v[0]) <= std::fabs(v[2])) ? 0 : (std::fabs(v[1]) <= std::fabs(v[2]) ? 1 : 2);
    const double e[3] = {k == 0 ? 1.0 : 0.0, k == 1 ? 1.0 : 0.0, k == 2 ? 1.0 : 0.0};
    double U[3] = {v[1] * e[2] - v[2] * e[1], v[2] * e[0] - v[0] * e[2], v[0] * e[1] - v[1] * e[0]};
    const double un = std::sqrt((U[0] * U[0] + U[1] * U[1]) + U[2] * U[2]);
    for (int j = 0; j < 3; ++j) U[j] /= un;
    double W[3] = {v[1] * U[2] - v[2] * U[1], v[2] * U[0] - v[0] * U[2], v[0] * U[1] - v[1] * U[0]};
    const double wn = std::sqrt((W[0] * W[0] + W[1] * W[1]) + W[2] * W[2]);
    for (int j = 0; j < 3; ++j) { W[j] /= wn; g.U[j] = U[j]; g.W[j] = W[j]; }
    double lo[2] = {0, 0}, hi[2] = {0, 0};
    bool have = false;
    for (uint32_t i = 0; i < n; ++i) {
        const double *c = items + 4 * (size_t)i;
        const double r = std::fabs(c[3]);
        if (!(std::isfinite(c[0]) && std::isfinite(c[1]) && std::isfinite(c[2]) && std::isfinite(r) && std::fabs(c[0]) < 1e6 &&
              std::fabs(c[1]) < 1e6 && std::fabs(c[2]) < 1e6 && r < 1e6))
            continue;
        const double R = r + kLgInflate * scale;
        const double p[2] = {(c[0] * U[0] + c[1] * U[1]) + c[2] * U[2], (c[0] * W[0] + c[1] * W[1]) + c[2] * W[2]};
        for (int j = 0; j < 2; ++j) {
            if (!have || p[j] - R < lo[j]) lo[j] = p[j] - R;
            if (!have || p[j] + R > hi[j]) hi[j] = p[j] + R;
        }
        have = true;
    }
    if (!have) return false;
    const double ext[2] = {std::max(hi[0] - lo[0], 1e-9), std::max(hi[1] - lo[1], 1e-9)};
    const double cell = std::sqrt(ext[0] * ext[1] / cells);
    for (int j = 0; j < 2; ++j) {
        g.dim[j] = (int)std::min((double)kLgMaxDim, std::max(1.0, std::ceil(ext[j] / cell)));
        const double pad = 0.01 * ext[j] / g.dim[j];   // no item ends within kLgPad cells of an edge
        g.lo[j] = lo[j] - pad;
        g.inv[j] = g.dim[j] / (ext[j] + 2.0 * pad);
    }
    return true;
}

}  // namespace rg
