// rg_scene.cuh — the scene as it lives in HBM (the "scene-upload layer").
//
// Layout (all read-only during a render):
//   * bodies in ORIGINAL order: kind[n], geom[n][8] (f64), mat[n] — used by shading, which
//     touches one body per hit;
//   * intersection lists: spheres as double4 (cx,cy,cz,r) + their original body index, and
//     the "misc" list (planes, disks, boxes: few, tested one by one in f64).  The original
//     index travels with every candidate because Scene::trace keeps the FIRST of equal
//     minima (scene.rs:34-39);
//   * cull4[n_spheres]: the FP32 conservative-cull record of each sphere (rg_trace.cuh), followed by those of
//     the grid's box / disk proxies (GridProxies below);
//   * the exact-culling grid (rg_grid.cuh);
//   * lights by value inside the struct (<= RG_MAX_LIGHTS), textures as CUDA texture objects.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/raingun_b200.h"

namespace rg {

struct BodyMat {            // material.rs:7-12 flattened; 48 bytes
    float color[3];         // Coloration::Color
    float albedo;
    float p0, p1;           // Reflecting{reflectivity} | Refractive{index, transparency}
    float tex_off[2];       // Texture{x_offset, y_offset}
    int32_t tex;            // texture index or -1
    uint8_t coloration;     // RG_COLORATION_*
    uint8_t surface;        // RG_SURFACE_*
    uint8_t pad[2];
    uint32_t pad2[2];
};
static_assert(sizeof(BodyMat) == 48, "BodyMat layout");

struct DLight {             // lights.rs:8-26
    double v[3];            // Spherical: position.  Directional: normalize(-direction), hoisted
                            // (lights.rs:48 — a pure function of the light)
    float color[3];
    float intensity;
    uint32_t kind;
    uint32_t pad;
};

struct DTex {
    cudaTextureObject_t obj;  // uchar4 texels, point sampling, unnormalised coordinates
    uint32_t w, h;
};

struct GridDev {            // see rg_grid.cuh
    float lo[3];            // grid origin, relative to cull_ref
    float inv_cell[3];
    float cell[3];
    int32_t dim[3];
    const uint32_t *cell_start;   // [ncells + 1]
    const uint32_t *cell_items;   // sphere indices (into the sphere list), cell by cell
    const float4 *cell_cull4;     // the same spheres' FP32 cull records, in the same order
    const float4 *cell_rec;       // [nrecords][3]: cull record of item 0, of item 1, (idx0, idx1, next record of the cell | 0, -);
                                  // records [0, ncells) are the cells' first, chained ones follow (rg_grid.cuh)
    uint32_t n_loose;             // spheres kept out of the grid (too large): brute-forced
    const uint32_t *loose;        // their sphere-list indices
    uint32_t enabled;
};

struct DScene {
    uint32_t n_bodies;
    uint32_t n_spheres;
    uint32_t n_misc;
    uint32_t n_lights;
    const uint8_t *kind;
    const double *geom;           // [n_bodies][8]
    const BodyMat *mat;
    const double4 *sph;           // [n_spheres] cx, cy, cz, r (+ the grid's proxies behind them, GridProxies)
    const uint32_t *sph_body;     // [n_spheres] original body index (+ the proxies')
    const uint32_t *body_sph;     // [n_bodies] the body's index in the sphere list (0xFFFFFFFF: not a sphere)
    const float4 *cull4;          // [n_spheres] c - P (f32), K - m_s       (rg_trace.cuh)
    const float4 *cull2;          // the same records pair-interleaved for FFMA2: (x0,x1,y0,y1)(z0,z1,-K0,-K1)
    const uint32_t *misc_body;    // [n_misc] original body index
    const DTex *tex;
    double fov_adj;               // tan(fov.to_radians() / 2), ray.rs:46 (host libm, once)
    double cull_ref[3];           // P: reference point of the FP32 cull coordinates
    float default_color[3];
    uint32_t max_depth;
    GridDev grid;
    DLight lights[RG_MAX_LIGHTS];
};

// Boxes and disks in the grid (rg_grid.cuh, DESIGN.md section 4.2).  A binnable box or disk enters the grid as
// a sphere that encloses it (its "proxy"): DScene::sph[n_spheres, n_spheres + n_proxies), with its body index in
// sph_body[] and its FP32 cull record in cull4[].  Only k_trace_grid reads this struct; it travels as a kernel
// argument of its own, so that DScene — and every kernel that takes it — is what it is in a sphere-only scene.
struct FaceRef {                  // one face plane of a binned box: the bound's coordinate and the box's body index
    double c;
    uint32_t body;
    uint32_t pad;
};
struct GridProxies {
    uint32_t n_proxies;
    uint32_t n_misc;              // non-sphere bodies kept out of the grid (planes, inverted boxes, ...): tested per ray
    const uint32_t *misc_body;    // [n_misc] original body index
    uint32_t n_faces;             // = 2 x binned boxes
    const FaceRef *faces;         // [3][n_faces]: per axis k, (lo_k, box) and (hi_k, box) of every binned box, sorted by c
};

// Per recursion level, for the host-free wavefront loop (rg_wavefront.cu): every launch of a
// level reads its size from here instead of from the host.  Zeroed at the start of a batch.
struct DLevelCtr {
    unsigned int n;                    // path rays of this level (written by k_generate / the level above's k_shade)
    unsigned int n_lit;                // hits of this level that need shadow rays
    unsigned int fetch;                // persistent nearest-hit trace of this level: next unclaimed ray
    unsigned int fetch_shadow;         // ... of this level's shadow trace
};

// Device-side counters of one render call (zeroed by the host before the call).
struct DCounters {
    unsigned long long rays[4];        // primary, shadow, reflection, transmission (megakernel only)
    unsigned long long exact_tests;
    unsigned long long cull_unsound;
    unsigned long long err_nan, err_trans, err_aabb;
    unsigned int q_next;               // wavefront: children emitted into the next level
    unsigned int q_lit;                // wavefront: hits that need shadow rays
    unsigned int fetch;                // persistent trace kernels: next unclaimed ray of the queue
    unsigned int fetch_shadow;         // ... of the shadow queue (the two kinds of trace run concurrently)
    // ---- host-free loop
    unsigned int overflow;             // a level outgrew its queue capacity: the frame is void, the host re-renders
    unsigned int max_level;            // deepest level that held a ray
    unsigned int deeper;               // the last enqueued level emitted children (depth hint too small): frame void
    unsigned int pad_;
    unsigned long long grid_cells;     // RG_OPT_TRACE_STATS: cells visited / records fetched / cull tests / refills
    unsigned long long grid_fetches;
    unsigned long long grid_culls;
    unsigned long long grid_refills;
    unsigned long long grid_lane_steps;   // active lanes summed over scan iterations, and the iterations x 32
    unsigned long long grid_lane_slots;
    DLevelCtr lvl[RG_MAX_DEPTH + 2];
};

}  // namespace rg
