// rg_grid.cu — host-side construction of the exact-culling grid (rg_grid.cuh) at scene upload.
#include <algorithm>
#include <cmath>
#include <cstdlib>
#include <cstring>
#include <limits>

#include "rg_cull.h"
#include "rg_grid.cuh"
#include "rg_host.h"

namespace rg {

// cells per sphere (RG_GRID_DENSITY overrides, for tuning runs).  Measured on the B200, C4 / C5 ms per frame.  Round 1's
// kernel: 2 -> 26.20 / 266.9, 3 -> 25.71 / 263.9, 4 -> 25.96 / 268.3, 6 -> 26.67 / 282.0.  Round 2's (chained records: a
// crowded cell costs one more record, exactly what a cell visit costs, so fewer, fuller cells win): 0.5 -> 19.76 / 200.2,
// 0.75 -> 19.02 / 187.9, 1 -> 18.90 / 183.5, 1.25 -> 18.77 / 184.1, 1.5 -> 18.86 / 185.6, 2 -> 19.21 / 189.7, 3 -> 19.84 / 200.4,
// 4 -> 20.58 / 209.7, 6 -> 21.71 / 227.6.
static double grid_density() {
    static const double d = [] { const char *e = getenv("RG_GRID_DENSITY"); double v = e ? atof(e) : 0.0; return v > 0.0 ? v : 1.25; }();
    return d;
}

template <typename T>
static int upload_vec(rg_scene *sc, const std::vector<T> &v, const T **out) {
    *out = nullptr;
    if (v.empty()) return RG_OK;
    void *p = sc->arena.alloc(v.size() * sizeof(T));
    if (!p) return RG_E_NOMEM;
    RG_CUDA(cudaMemcpy(p, v.data(), v.size() * sizeof(T), cudaMemcpyHostToDevice));
    *out = reinterpret_cast<const T *>(p);
    return RG_OK;
}

// the FP32 cull record of one sphere as k_cull_records (rg_api.cu) computes it on the device
static float4 host_cull_record(const double *sp, const double *P) {
    const double cx = sp[0] - P[0], cy = sp[1] - P[1], cz = sp[2] - P[2], r = sp[3];
    const double C2 = cx * cx + cy * cy + cz * cz, r2 = r * r;
    if (C2 < kCullHuge && r2 < kCullHuge) {
        const double K = (C2 - r2) - kCullU * (kCullSphereC2 * C2 + kCullSphereR2 * r2);
        return make_float4((float)cx, (float)cy, (float)cz, (float)K);
    }
    return make_float4(0.f, 0.f, 0.f, -std::numeric_limits<float>::infinity());
}

static int grid_build_host(rg_scene *sc, const double *sph, uint32_t n) {
    GridDev &g = sc->ds.grid;
    g = GridDev{};
    if (n < 8) return RG_OK;   // brute force is the right tool for a handful of bodies
    std::vector<float4> cull(n);
    for (uint32_t i = 0; i < n; ++i) cull[i] = host_cull_record(sph + 4 * (size_t)i, sc->ds.cull_ref);

    // bounds of the finite spheres, relative to the cull reference point P
    const double *P = sc->ds.cull_ref;
    std::vector<uint32_t> loose, binned;
    double lo[3] = {0, 0, 0}, hi[3] = {0, 0, 0};
    bool have = false;
    std::vector<double> rel((size_t)n * 4);
    for (uint32_t i = 0; i < n; ++i) {
        double c[3] = {sph[4 * (size_t)i] - P[0], sph[4 * (size_t)i + 1] - P[1], sph[4 * (size_t)i + 2] - P[2]};
        double r = std::fabs(sph[4 * (size_t)i + 3]);
        bool ok = std::isfinite(c[0]) && std::isfinite(c[1]) && std::isfinite(c[2]) && std::isfinite(r) &&
                  std::fabs(c[0]) < 1e6 && std::fabs(c[1]) < 1e6 && std::fabs(c[2]) < 1e6 && r < 1e6;
        rel[4 * (size_t)i] = c[0]; rel[4 * (size_t)i + 1] = c[1]; rel[4 * (size_t)i + 2] = c[2]; rel[4 * (size_t)i + 3] = r;
        if (!ok) { loose.push_back(i); continue; }
        binned.push_back(i);
        for (int k = 0; k < 3; ++k) {
            if (!have) { lo[k] = c[k] - r; hi[k] = c[k] + r; }
            else { lo[k] = std::fmin(lo[k], c[k] - r); hi[k] = std::fmax(hi[k], c[k] + r); }
        }
        have = true;
    }
    if (binned.size() < 8) return RG_OK;

    // resolution: ~kDensity cells per sphere, cubic cells, at most 256 per axis
    const double kDensity = grid_density();
    double ext[3], vol = 1.0;
    for (int k = 0; k < 3; ++k) { ext[k] = std::fmax(hi[k] - lo[k], 1e-9); vol *= ext[k]; }
    double cell = std::cbrt(vol / (kDensity * (double)binned.size()));
    if (!(cell > 0.0) || !std::isfinite(cell)) return RG_OK;
    int dim[3];
    for (int k = 0; k < 3; ++k) dim[k] = (int)std::min(256.0, std::max(1.0, std::ceil(ext[k] / cell)));
    // pad the box so that no sphere comes within the inflation distance of a wall
    double csz[3];
    for (int k = 0; k < 3; ++k) {
        double c0 = ext[k] / dim[k];
        lo[k] -= 0.02 * c0;
        hi[k] += 0.02 * c0;
        csz[k] = (hi[k] - lo[k]) / dim[k];
    }
    const size_t ncells = (size_t)dim[0] * dim[1] * dim[2];

    // a sphere is listed in every cell its bounding box inflated by kGridInflate cells overlaps
    auto cell_range = [&](uint32_t i, int k, int &a, int &b) {
        double c = rel[4 * (size_t)i + k], r = rel[4 * (size_t)i + 3];
        double fa = (c - r - lo[k]) / csz[k] - 2.0 * kGridInflate;
        double fb = (c + r - lo[k]) / csz[k] + 2.0 * kGridInflate;
        a = std::max(0, std::min(dim[k] - 1, (int)std::floor(fa)));
        b = std::max(0, std::min(dim[k] - 1, (int)std::floor(fb)));
    };
    const uint64_t kMaxCellsPerSphere = 512;
    std::vector<uint32_t> count(ncells + 1, 0);
    std::vector<uint32_t> kept;
    for (uint32_t i : binned) {
        int a[3], b[3];
        for (int k = 0; k < 3; ++k) cell_range(i, k, a[k], b[k]);
        uint64_t span = (uint64_t)(b[0] - a[0] + 1) * (b[1] - a[1] + 1) * (b[2] - a[2] + 1);
        if (span > kMaxCellsPerSphere) { loose.push_back(i); continue; }
        kept.push_back(i);
        for (int z = a[2]; z <= b[2]; ++z)
            for (int y = a[1]; y <= b[1]; ++y)
                for (int x = a[0]; x <= b[0]; ++x) count[((size_t)z * dim[1] + y) * dim[0] + x + 1]++;
    }
    if (loose.size() > 256 || kept.size() < 8) return RG_OK;   // not a scene a uniform grid suits
    for (size_t c = 0; c < ncells; ++c) count[c + 1] += count[c];
    std::vector<uint32_t> start(count.begin(), count.end());
    std::vector<uint32_t> items(start[ncells]);
    std::vector<float4> items_cull(start[ncells]);
    std::vector<uint32_t> fill(start.begin(), start.end() - 1);
    for (uint32_t i : kept) {   // ascending sphere index, so every cell list is sorted
        int a[3], b[3];
        for (int k = 0; k < 3; ++k) cell_range(i, k, a[k], b[k]);
        for (int z = a[2]; z <= b[2]; ++z)
            for (int y = a[1]; y <= b[1]; ++y)
                for (int x = a[0]; x <= b[0]; ++x) {
                    uint32_t pos = fill[((size_t)z * dim[1] + y) * dim[0] + x]++;
                    items[pos] = i;
                    items_cull[pos] = cull[i];
                }
    }
    std::sort(loose.begin(), loose.end());

    // Cell records: the items of a cell live IN 48-byte records (two cull records + their sphere indices +
    // the index of the cell's next record), so a visit is one fixed-size fetch and two culls for every
    // lane.  Record c is cell c's first; a cell with more than two items (a few per cent at the default
    // density) continues in chained records behind the cells' own (grid_chain_record), which the tracer reads
    // exactly like a first record: one instruction stream for every scanning lane, no separate overflow
    // path.  Empty slots hold a record that every cullable ray rejects.  (Three items per 64-byte record — fewer
    // chained records, one more cull per visit — was measured: C4 18.8 -> 19.5 ms, C5 186 -> 198 ms at its own best density.)
    const float kInf = std::numeric_limits<float>::infinity();
    const size_t nrecs = grid_record_count(ncells, start[ncells]);
    std::vector<float4> recs(nrecs * 3, make_float4(0.f, 0.f, 0.f, kInf));
    for (size_t c = 0; c < ncells; ++c) {
        const uint32_t b0 = start[c], b1 = start[c + 1];
        for (uint32_t pos = b0, r = (uint32_t)c; pos < b1 || pos == b0; pos += 2) {   // every cell has its first record, even when empty
            const uint32_t n = b1 - pos > 2 ? 2 : b1 - pos;
            const uint32_t next = pos + 2 < b1 ? grid_chain_record((uint32_t)ncells, pos + 2) : 0u;
            recs[3 * (size_t)r] = n > 0 ? items_cull[pos] : make_float4(0.f, 0.f, 0.f, kInf);
            recs[3 * (size_t)r + 1] = n > 1 ? items_cull[pos + 1] : make_float4(0.f, 0.f, 0.f, kInf);
            const uint4 meta = make_uint4(n > 0 ? items[pos] : 0xFFFFFFFFu, n > 1 ? items[pos + 1] : 0xFFFFFFFFu, next, 0u);
            std::memcpy(&recs[3 * (size_t)r + 2], &meta, sizeof(meta));
            r = next;
            if (!next) break;
        }
    }

    int rc;
    if ((rc = upload_vec(sc, recs, &g.cell_rec))) return rc;
    if ((rc = upload_vec(sc, start, &g.cell_start))) return rc;
    if ((rc = upload_vec(sc, items, &g.cell_items))) return rc;
    if ((rc = upload_vec(sc, items_cull, &g.cell_cull4))) return rc;
    if ((rc = upload_vec(sc, loose, &g.loose))) return rc;
    g.n_loose = (uint32_t)loose.size();
    for (int k = 0; k < 3; ++k) {
        g.lo[k] = (float)lo[k];
        g.cell[k] = (float)csz[k];
        g.inv_cell[k] = (float)(1.0 / csz[k]);
        g.dim[k] = dim[k];
    }
    g.enabled = 1;
    return RG_OK;
}

// ---- the same structure built ON THE DEVICE ---------------------------------------------------
// The host loops above cost 1.4 ms for 10,000 spheres and 20 ms for 100,000 (measured on the B200
// box), i.e. most of a scene upload; the sphere list and the cull records are already in HBM at
// this point, so binning is four small kernels.  Only the bounding box (one pass over the
// centres), the resolution and two counters stay on the host.  All binning arithmetic is the host
// builder's, in FP64 without contraction, and every cell list is sorted by sphere index, so both
// builders produce the same records bit for bit (RG_GRID_BUILD=host selects the host one; the
// parity tests compare images and exact-test counts of the two).
struct GridBuildParams {
    double lo[3], csz[3], P[3];
    int dim[3];
    uint32_t n;
};
enum : uint32_t { GB_LOOSE = 0, GB_KEPT = 1, GB_TOTAL = 2 };
constexpr uint32_t kGbLooseTmp = 1024;
constexpr uint64_t kGbMaxCellsPerSphere = 512;

// 0 = not binned (non-finite / huge), 1 = loose (spans too many cells), 2 = kept; cell range in a, b
__device__ __forceinline__ int gb_classify(const GridBuildParams &p, const double4 sp, int a[3], int b[3]) {
    const double c[3] = {sp.x - p.P[0], sp.y - p.P[1], sp.z - p.P[2]};
    const double r = fabs(sp.w);
    const bool ok = isfinite(c[0]) && isfinite(c[1]) && isfinite(c[2]) && isfinite(r) && fabs(c[0]) < 1e6 &&
                    fabs(c[1]) < 1e6 && fabs(c[2]) < 1e6 && r < 1e6;
    if (!ok) return 0;
    uint64_t span = 1;
#pragma unroll
    for (int k = 0; k < 3; ++k) {
        const double fa = (c[k] - r - p.lo[k]) / p.csz[k] - 2.0 * kGridInflate;
        const double fb = (c[k] + r - p.lo[k]) / p.csz[k] + 2.0 * kGridInflate;
        a[k] = max(0, min(p.dim[k] - 1, (int)floor(fa)));
        b[k] = max(0, min(p.dim[k] - 1, (int)floor(fb)));
        span *= (uint64_t)(b[k] - a[k] + 1);
    }
    return span > kGbMaxCellsPerSphere ? 1 : 2;
}

__global__ void __launch_bounds__(256) k_gb_count(const GridBuildParams p, const double4 *__restrict__ sph, uint32_t *count,
                                                  uint32_t *ctr, uint32_t *loose_tmp) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= p.n) return;
    int a[3], b[3];
    const int kind = gb_classify(p, sph[i], a, b);
    if (kind != 2) {   // loose: tested per ray (non-finite spheres are never culled by their records)
        const uint32_t pos = atomicAdd(&ctr[GB_LOOSE], 1u);
        if (pos < kGbLooseTmp) loose_tmp[pos] = i;
        return;
    }
    atomicAdd(&ctr[GB_KEPT], 1u);
    for (int z = a[2]; z <= b[2]; ++z)
        for (int y = a[1]; y <= b[1]; ++y)
            for (int x = a[0]; x <= b[0]; ++x) atomicAdd(&count[((size_t)z * p.dim[1] + y) * p.dim[0] + x], 1u);
}

// exclusive prefix sum of count[0, n) in place, count[n] = total; one 1024-thread block walking the array in
// tiles of 4096 (one coalesced 128-bit load per thread, warp shuffles, 32 warp sums through shared memory)
__global__ void __launch_bounds__(1024) k_gb_scan(uint32_t *count, uint32_t n, uint32_t *ctr) {
    __shared__ uint32_t warp_sum[32];
    __shared__ uint32_t carry;
    const uint32_t t = threadIdx.x, lane = t & 31u, warp = t >> 5;
    if (t == 0) carry = 0;
    __syncthreads();
    for (uint32_t base = 0; base < n; base += 4096u) {
        const uint32_t i = base + 4u * t;
        uint4 v = make_uint4(0u, 0u, 0u, 0u);
        if (i + 3u < n) v = *reinterpret_cast<const uint4 *>(count + i);
        else {
            if (i < n) v.x = count[i];
            if (i + 1u < n) v.y = count[i + 1];
            if (i + 2u < n) v.z = count[i + 2];
        }
        const uint32_t mine = v.x + v.y + v.z + v.w;
        uint32_t incl = mine;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const uint32_t up = __shfl_up_sync(0xffffffffu, incl, o);
            if ((int)lane >= o) incl += up;
        }
        if (lane == 31u) warp_sum[warp] = incl;
        __syncthreads();
        if (warp == 0) {
            uint32_t w = warp_sum[lane];
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const uint32_t up = __shfl_up_sync(0xffffffffu, w, o);
                if ((int)lane >= o) w += up;
            }
            warp_sum[lane] = w;   // inclusive over warps
        }
        __syncthreads();
        const uint32_t before = carry + (warp ? warp_sum[warp - 1] : 0u) + (incl - mine);
        const uint4 o4 = make_uint4(before, before + v.x, before + v.x + v.y, before + v.x + v.y + v.z);
        if (i + 3u < n) *reinterpret_cast<uint4 *>(count + i) = o4;
        else {
            if (i < n) count[i] = o4.x;
            if (i + 1u < n) count[i + 1] = o4.y;
            if (i + 2u < n) count[i + 2] = o4.z;
        }
        __syncthreads();
        if (t == 1023u) carry += warp_sum[31];
        __syncthreads();
    }
    if (t == 0) {
        count[n] = carry;
        ctr[GB_TOTAL] = carry;
    }
}

// (the lists are written only if they fit the capacity the host allocated before it knew their size:
// k_gb_* run back to back with no read-back in between; the host checks the total afterwards)
__global__ void __launch_bounds__(256) k_gb_fill(const GridBuildParams p, const double4 *__restrict__ sph,
                                                 const uint32_t *__restrict__ start, uint32_t *cursor, uint32_t *items,
                                                 const uint32_t *__restrict__ ctr, uint32_t items_cap) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= p.n || ctr[GB_TOTAL] > items_cap) return;
    int a[3], b[3];
    if (gb_classify(p, sph[i], a, b) != 2) return;
    for (int z = a[2]; z <= b[2]; ++z)
        for (int y = a[1]; y <= b[1]; ++y)
            for (int x = a[0]; x <= b[0]; ++x) {
                const size_t c = ((size_t)z * p.dim[1] + y) * p.dim[0] + x;
                items[start[c] + atomicAdd(&cursor[c], 1u)] = i;
            }
}

// Ascending in-place sort of a cell's list: insertion sort for the usual handful of items, heap sort
// beyond that, so that a degenerate scene (tens of thousands of spheres in one cell) costs
// O(n log n) in its one thread instead of O(n^2).  Host-callable for the unit test in rg_sort_test.
__host__ __device__ inline void gb_sort_u32(uint32_t *v, uint32_t n) {
    if (n <= 32u) {
        for (uint32_t i = 1; i < n; ++i) {
            const uint32_t x = v[i];
            uint32_t j = i;
            while (j > 0 && v[j - 1] > x) { v[j] = v[j - 1]; --j; }
            v[j] = x;
        }
        return;
    }
    auto sift = [&](uint32_t root, uint32_t end) {   // max-heap sift-down over v[0, end)
        const uint32_t x = v[root];
        for (;;) {
            uint32_t child = 2u * root + 1u;
            if (child >= end) break;
            if (child + 1u < end && v[child + 1u] > v[child]) ++child;
            if (v[child] <= x) break;
            v[root] = v[child];
            root = child;
        }
        v[root] = x;
    };
    for (uint32_t i = n / 2u; i-- > 0;) sift(i, n);
    for (uint32_t end = n - 1u; end > 0; --end) {
        const uint32_t t = v[0];
        v[0] = v[end];
        v[end] = t;
        sift(0u, end);
    }
}

// per cell: sort its list by sphere index (the atomics above fill it in arbitrary order), copy the
// cull records next to it and write the inline 48-byte record (see grid_build_host)
__global__ void __launch_bounds__(256) k_gb_finish(uint32_t ncells, const uint32_t *__restrict__ start, uint32_t *items,
                                                   const float4 *__restrict__ cull4, float4 *items_cull, float4 *recs,
                                                   const uint32_t *__restrict__ ctr, uint32_t items_cap) {
    const uint32_t c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= ncells || ctr[GB_TOTAL] > items_cap) return;
    const uint32_t b0 = start[c], b1 = start[c + 1], n = b1 - b0;
    gb_sort_u32(items + b0, n);   // lists are short (mean < 1, rarely > 8)
    for (uint32_t i = b0; i < b1; ++i) items_cull[i] = cull4[items[i]];
    const float kInf = __int_as_float(0x7f800000);
    for (uint32_t pos = b0, r = c;; pos += 2) {   // the cell's chain of records (see grid_build_host)
        const uint32_t m = b1 - pos > 2 ? 2 : b1 - pos;
        const uint32_t next = pos + 2 < b1 ? grid_chain_record(ncells, pos + 2) : 0u;
        recs[3 * (size_t)r] = m > 0 ? items_cull[pos] : make_float4(0.f, 0.f, 0.f, kInf);
        recs[3 * (size_t)r + 1] = m > 1 ? items_cull[pos + 1] : make_float4(0.f, 0.f, 0.f, kInf);
        *reinterpret_cast<uint4 *>(&recs[3 * (size_t)r + 2]) =
            make_uint4(m > 0 ? items[pos] : 0xFFFFFFFFu, m > 1 ? items[pos + 1] : 0xFFFFFFFFu, next, 0u);
        if (!next) break;
        r = next;
    }
}

__global__ void k_gb_sort_loose(const uint32_t *tmp, const uint32_t *__restrict__ ctr, uint32_t *out) {   // <= 256 entries: one thread
    if (blockIdx.x || threadIdx.x) return;
    const uint32_t n = ctr[GB_LOOSE] <= 256u ? ctr[GB_LOOSE] : 0u;
    for (uint32_t i = 0; i < n; ++i) {
        const uint32_t v = tmp[i];
        uint32_t j = i;
        while (j > 0 && out[j - 1] > v) { out[j] = out[j - 1]; --j; }
        out[j] = v;
    }
}

static int grid_build_device(rg_scene *sc, const double *sph, uint32_t n) {
    GridDev &g = sc->ds.grid;
    g = GridDev{};
    if (n < 8) return RG_OK;
    // host: bounding box of the binnable spheres and the resolution (same arithmetic as grid_build_host)
    const double *P = sc->ds.cull_ref;
    double lo[3] = {0, 0, 0}, hi[3] = {0, 0, 0};
    bool have = false;
    size_t binned = 0;
    for (uint32_t i = 0; i < n; ++i) {
        const double c[3] = {sph[4 * (size_t)i] - P[0], sph[4 * (size_t)i + 1] - P[1], sph[4 * (size_t)i + 2] - P[2]};
        const double r = std::fabs(sph[4 * (size_t)i + 3]);
        const bool ok = std::isfinite(c[0]) && std::isfinite(c[1]) && std::isfinite(c[2]) && std::isfinite(r) &&
                        std::fabs(c[0]) < 1e6 && std::fabs(c[1]) < 1e6 && std::fabs(c[2]) < 1e6 && r < 1e6;
        if (!ok) continue;
        ++binned;
        for (int k = 0; k < 3; ++k) {   // (finite operands: plain comparisons give what fmin / fmax give)
            const double a = c[k] - r, b = c[k] + r;
            if (!have || a < lo[k]) lo[k] = a;
            if (!have || b > hi[k]) hi[k] = b;
        }
        have = true;
    }
    if (binned < 8) return RG_OK;
    const double kDensity = grid_density();
    double ext[3], vol = 1.0;
    for (int k = 0; k < 3; ++k) { ext[k] = std::fmax(hi[k] - lo[k], 1e-9); vol *= ext[k]; }
    const double cell = std::cbrt(vol / (kDensity * (double)binned));
    if (!(cell > 0.0) || !std::isfinite(cell)) return RG_OK;
    GridBuildParams p{};
    p.n = n;
    for (int k = 0; k < 3; ++k) {
        p.dim[k] = (int)std::min(256.0, std::max(1.0, std::ceil(ext[k] / cell)));
        const double c0 = ext[k] / p.dim[k];
        lo[k] -= 0.02 * c0;
        hi[k] += 0.02 * c0;
        p.lo[k] = lo[k];
        p.csz[k] = (hi[k] - lo[k]) / p.dim[k];
        p.P[k] = P[k];
    }
    const size_t ncells = (size_t)p.dim[0] * p.dim[1] * p.dim[2];

    // Capacity of the cell lists before their size is known: a sphere lands in ~2.7 cells at the default density;
    // 8 per sphere (and never less than 4096) is generous, and a scene that needs more takes a second, exact pass.
    uint32_t items_cap = (uint32_t)std::min<uint64_t>(std::max<uint64_t>(8ull * n, 4096), 0x7FFFFFFFull);
    cudaStream_t st = sc->stream;
    uint32_t h_ctr[4] = {0, 0, 0, 0};
    uint32_t *start = nullptr, *cursor = nullptr, *ctr = nullptr, *loose_tmp = nullptr, *items = nullptr, *loose = nullptr;
    float4 *items_cull = nullptr, *recs = nullptr;
    for (int pass = 0; pass < 2; ++pass) {
        start = static_cast<uint32_t *>(sc->arena.alloc((ncells + 1) * sizeof(uint32_t)));
        cursor = static_cast<uint32_t *>(sc->arena.alloc(ncells * sizeof(uint32_t)));
        ctr = static_cast<uint32_t *>(sc->arena.alloc(4 * sizeof(uint32_t)));
        loose_tmp = static_cast<uint32_t *>(sc->arena.alloc(kGbLooseTmp * sizeof(uint32_t)));
        items = static_cast<uint32_t *>(sc->arena.alloc((size_t)items_cap * sizeof(uint32_t)));
        items_cull = static_cast<float4 *>(sc->arena.alloc((size_t)items_cap * sizeof(float4)));
        loose = static_cast<uint32_t *>(sc->arena.alloc(256 * sizeof(uint32_t)));
        recs = static_cast<float4 *>(sc->arena.alloc(grid_record_count(ncells, items_cap) * 3 * sizeof(float4)));
        if (!start || !cursor || !ctr || !loose_tmp || !items || !items_cull || !loose || !recs) return RG_E_NOMEM;
        RG_CUDA(cudaMemsetAsync(start, 0, (ncells + 1) * sizeof(uint32_t), st));
        RG_CUDA(cudaMemsetAsync(cursor, 0, ncells * sizeof(uint32_t), st));
        RG_CUDA(cudaMemsetAsync(ctr, 0, 4 * sizeof(uint32_t), st));
        const unsigned sblocks = (n + 255) / 256;
        k_gb_count<<<sblocks, 256, 0, st>>>(p, sc->ds.sph, start, ctr, loose_tmp);
        k_gb_scan<<<1, 1024, 0, st>>>(start, (uint32_t)ncells, ctr);
        k_gb_fill<<<sblocks, 256, 0, st>>>(p, sc->ds.sph, start, cursor, items, ctr, items_cap);
        k_gb_finish<<<(unsigned)((ncells + 255) / 256), 256, 0, st>>>((uint32_t)ncells, start, items, sc->ds.cull4, items_cull, recs, ctr, items_cap);
        k_gb_sort_loose<<<1, 32, 0, st>>>(loose_tmp, ctr, loose);
        RG_CUDA(cudaGetLastError());
        RG_CUDA(cudaMemcpyAsync(h_ctr, ctr, sizeof h_ctr, cudaMemcpyDeviceToHost, st));
        RG_CUDA(cudaStreamSynchronize(st));   // the one synchronisation of the build (and of the scene upload before it)
        if (h_ctr[GB_TOTAL] <= items_cap) break;
        items_cap = h_ctr[GB_TOTAL];          // rare: lists longer than the generous guess — once more, exactly sized
    }
    const uint32_t n_loose = h_ctr[GB_LOOSE], n_kept = h_ctr[GB_KEPT];
    if (n_loose > 256 || n_kept < 8) return RG_OK;   // not a scene a uniform grid suits

    g.cell_rec = recs;
    g.cell_start = start;
    g.cell_items = items;
    g.cell_cull4 = items_cull;
    g.loose = loose;
    g.n_loose = n_loose;
    for (int k = 0; k < 3; ++k) {
        g.lo[k] = (float)p.lo[k];
        g.cell[k] = (float)p.csz[k];
        g.inv_cell[k] = (float)(1.0 / p.csz[k]);
        g.dim[k] = p.dim[k];
    }
    g.enabled = 1;
    return RG_OK;
}

int grid_build(rg_scene *sc, const double *sph, uint32_t n) {
    static const bool on_host = [] { const char *e = getenv("RG_GRID_BUILD"); return e && std::strcmp(e, "host") == 0; }();
    return on_host ? grid_build_host(sc, sph, n) : grid_build_device(sc, sph, n);
}

// ---- light grids (rg_light_grid.h) -------------------------------------------------------------
// Built like the 3-D grid on the device: count -> scan -> fill -> per-cell sort -> records, over the items of
// every light at once (one thread per (light, item)).  Lists are sorted by (FP32 depth rounded down, item index),
// so the build is deterministic; a record's 4th word holds the depth of its first item.
static double light_grid_density() {   // key cells per item (RG_LIGHT_GRID_DENSITY overrides, for tuning runs)
    static const double d = [] { const char *e = getenv("RG_LIGHT_GRID_DENSITY"); double v = e ? atof(e) : 0.0; return v > 0.0 ? v : 2.0; }();
    return d;
}

__device__ __forceinline__ uint64_t lg_sort_key(const LightGridInfo &g, const double4 sp, uint32_t i) {
    const double c[3] = {sp.x, sp.y, sp.z};
    return ((uint64_t)lg_float_order(lg_float_down(lg_item_depth(g, c, sp.w))) << 32) | i;
}

// FILL = false: count the entries of every cell; true: write them (sort keys) at start[c] + cursor[c]
template <bool FILL>
__global__ void __launch_bounds__(256) k_lg_bin(const LightGridInfo *__restrict__ info, uint32_t n_lights, const double4 *__restrict__ sph,
                                                uint32_t n, uint32_t *count, const uint32_t *__restrict__ start, uint64_t *keys,
                                                const uint32_t *__restrict__ ctr, uint32_t items_cap) {
    const uint64_t t = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= (uint64_t)n * n_lights) return;
    if (FILL && ctr[GB_TOTAL] > items_cap) return;
    const uint32_t l = (uint32_t)(t / n), i = (uint32_t)(t % n);
    const LightGridInfo g = info[l];
    const double4 sp = sph[i];
    const double c[3] = {sp.x, sp.y, sp.z};
    int rng[6][4];
    const int k = lg_item_ranges(g, c, sp.w, rng);
    const uint64_t key = FILL ? lg_sort_key(g, sp, i) : 0ull;
    auto put = [&](uint32_t cell) {
        if (FILL) keys[start[cell] + atomicAdd(&count[cell], 1u)] = key;
        else atomicAdd(&count[cell], 1u);
    };
    if (k < 0) { put(g.always); return; }
    for (int f = 0; f < 6; ++f)
        for (int y = rng[f][2]; y <= rng[f][3]; ++y)
            for (int x = rng[f][0]; x <= rng[f][1]; ++x) put(g.base + lg_cell_index(g, f, x, y));
}

// per cell: sort the keys, then the item list and the chain of 48-byte records (as k_gb_finish)
__global__ void __launch_bounds__(256) k_lg_finish(uint32_t ncells, const uint32_t *__restrict__ start, uint64_t *keys, uint32_t *items,
                                                   const float4 *__restrict__ cull4, float4 *recs, const uint32_t *__restrict__ ctr,
                                                   uint32_t items_cap) {
    const uint32_t c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= ncells || ctr[GB_TOTAL] > items_cap) return;
    const uint32_t b0 = start[c], b1 = start[c + 1];
    lg_sort_u64(keys + b0, b1 - b0);
    for (uint32_t i = b0; i < b1; ++i) items[i] = (uint32_t)keys[i];
    const float kInf = __int_as_float(0x7f800000);
    for (uint32_t pos = b0, r = c;; pos += 2) {
        const uint32_t m = b1 - pos > 2 ? 2 : b1 - pos;
        const uint32_t next = pos + 2 < b1 ? grid_chain_record(ncells, pos + 2) : 0u;
        recs[3 * (size_t)r] = m > 0 ? cull4[items[pos]] : make_float4(0.f, 0.f, 0.f, kInf);
        recs[3 * (size_t)r + 1] = m > 1 ? cull4[items[pos + 1]] : make_float4(0.f, 0.f, 0.f, kInf);
        const float depth = m > 0 ? lg_order_float((uint32_t)(keys[pos] >> 32)) : kInf;
        *reinterpret_cast<uint4 *>(&recs[3 * (size_t)r + 2]) =
            make_uint4(m > 0 ? items[pos] : 0xFFFFFFFFu, m > 1 ? items[pos + 1] : 0xFFFFFFFFu, next, __float_as_uint(depth));
        if (!next) break;
        r = next;
    }
}

int light_grid_build(rg_scene *sc, const double *sph, uint32_t n) {
    sc->lg = LightGrids{};
    const uint32_t nl = std::min<uint32_t>((uint32_t)sc->lights.size(), kLightGrids);
    if (!sc->ds.grid.enabled || nl == 0 || n == 0) return RG_OK;   // only the grid tracer reads light grids
    double scale = 1.0;
    for (uint32_t i = 0; i < n; ++i) {
        const double *c = sph + 4 * (size_t)i;
        const double m = std::max(std::max(std::fabs(c[0]), std::fabs(c[1])), std::fabs(c[2])) + std::fabs(c[3]);
        if (m < 1e6) scale = std::max(scale, 1.0 + m);   // (false on NaN: such items go on the always lists)
    }
    std::vector<LightGridInfo> info;
    uint32_t ncells = 1;   // cell 0: the empty placeholder (rg_light_grid.h)
    for (uint32_t l = 0; l < nl; ++l) {
        const DLight &L = sc->lights[l];
        double sl = scale;
        if (L.kind != RG_LIGHT_DIRECTIONAL) {
            const double m = std::max(std::max(std::fabs(L.v[0]), std::fabs(L.v[1])), std::fabs(L.v[2]));
            if (!(m < 1e6)) break;
            sl = std::max(sl, 1.0 + m);
        }
        LightGridInfo g;
        if (!lg_setup(g, L.kind == RG_LIGHT_DIRECTIONAL ? 0u : 1u, L.v, sph, n, sl, light_grid_density())) break;   // lights [0, l) keep theirs
        g.base = ncells;
        g.always = ncells + lg_key_cells(g);
        ncells = g.always + 1;
        info.push_back(g);
    }
    if (info.empty()) return RG_OK;
    const uint32_t nlg = (uint32_t)info.size();
    const LightGridInfo *d_info = nullptr;
    int rc;
    if ((rc = upload_vec(sc, info, &d_info))) return rc;
    uint32_t items_cap = (uint32_t)std::min<uint64_t>(std::max<uint64_t>(4ull * n * nlg, 4096), 0x7FFFFFFFull);
    cudaStream_t st = sc->stream;
    uint32_t h_ctr[4] = {0, 0, 0, 0};
    uint32_t *start = nullptr, *cursor = nullptr, *ctr = nullptr, *items = nullptr;
    uint64_t *keys = nullptr;
    float4 *recs = nullptr;
    const unsigned bblocks = (unsigned)(((uint64_t)n * nlg + 255) / 256);
    for (int pass = 0; pass < 2; ++pass) {
        start = static_cast<uint32_t *>(sc->arena.alloc(((size_t)ncells + 1) * sizeof(uint32_t)));
        cursor = static_cast<uint32_t *>(sc->arena.alloc((size_t)ncells * sizeof(uint32_t)));
        ctr = static_cast<uint32_t *>(sc->arena.alloc(4 * sizeof(uint32_t)));
        keys = static_cast<uint64_t *>(sc->arena.alloc((size_t)items_cap * sizeof(uint64_t)));
        items = static_cast<uint32_t *>(sc->arena.alloc((size_t)items_cap * sizeof(uint32_t)));
        recs = static_cast<float4 *>(sc->arena.alloc(grid_record_count(ncells, items_cap) * 3 * sizeof(float4)));
        if (!start || !cursor || !ctr || !keys || !items || !recs) return RG_E_NOMEM;
        RG_CUDA(cudaMemsetAsync(start, 0, ((size_t)ncells + 1) * sizeof(uint32_t), st));
        RG_CUDA(cudaMemsetAsync(cursor, 0, (size_t)ncells * sizeof(uint32_t), st));
        RG_CUDA(cudaMemsetAsync(ctr, 0, 4 * sizeof(uint32_t), st));
        k_lg_bin<false><<<bblocks, 256, 0, st>>>(d_info, nlg, sc->ds.sph, n, start, nullptr, nullptr, ctr, items_cap);
        k_gb_scan<<<1, 1024, 0, st>>>(start, ncells, ctr);
        k_lg_bin<true><<<bblocks, 256, 0, st>>>(d_info, nlg, sc->ds.sph, n, cursor, start, keys, ctr, items_cap);
        k_lg_finish<<<(ncells + 255) / 256, 256, 0, st>>>(ncells, start, keys, items, sc->ds.cull4, recs, ctr, items_cap);
        RG_CUDA(cudaGetLastError());
        RG_CUDA(cudaMemcpyAsync(h_ctr, ctr, sizeof h_ctr, cudaMemcpyDeviceToHost, st));
        RG_CUDA(cudaStreamSynchronize(st));
        if (h_ctr[GB_TOTAL] <= items_cap) break;
        items_cap = h_ctr[GB_TOTAL];   // lists longer than the guess: once more, exactly sized
    }
    LightGrids &lg = sc->lg;
    lg.n_lights = nlg;
    lg.info = d_info;
    lg.cell_rec = recs;
    lg.cell_start = start;
    lg.cell_items = items;
    return RG_OK;
}

}  // namespace rg
