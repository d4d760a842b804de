// rg_host.h — host-side state behind the opaque `rg_scene` handle.
#pragma once
#include <cuda_runtime.h>

#include <atomic>
#include <cstdarg>
#include <cstdio>
#include <string>
#include <vector>

#include "rg_scene.cuh"

namespace rg {

void set_error(const char *fmt, ...);
int cuda_fail(cudaError_t e, const char *what, const char *file, int line);

#define RG_CUDA(call)                                                      \
    do {                                                                   \
        cudaError_t _e = (call);                                           \
        if (_e != cudaSuccess) return rg::cuda_fail(_e, #call, __FILE__, __LINE__); \
    } while (0)

// A device allocation that only ever grows; kept across frames so that a steady-state
// render performs no cudaMalloc.
struct DeviceBuffer {
    void *ptr = nullptr;
    size_t cap = 0;
    int reserve(size_t bytes);
    void release();
    template <typename T> T *as() const { return reinterpret_cast<T *>(ptr); }
};

// Scene arrays are carved out of a few large blocks instead of one cudaMalloc each, and the
// blocks survive the scene (see DeviceContext): re-uploading a scene every frame then costs
// H2D copies only.
struct SceneArena {
    std::vector<DeviceBuffer> blocks;
    size_t cur = 0, off = 0;
    void *alloc(size_t bytes);   // nullptr on failure (error already set)
    void reset() { cur = 0; off = 0; }
    void release();
};

// Scratch of the wavefront pipeline (rg_wavefront.cu).
struct WavefrontScratch {
    DeviceBuffer ray[2];        // ping-pong path-ray queues: 3 x double2 per ray
    DeviceBuffer hit_t, hit_body;
    // Shadow-side buffers exist twice (level parity): the shadow trace + diffuse of level d run on
    // the auxiliary stream WHILE the main stream traces and shades level d+1.
    DeviceBuffer sray[2];       // shadow-ray queue: 3 x double2 per ray
    DeviceBuffer s_tmax[2];     // light.distance(hit_point) per shadow ray
    DeviceBuffer s_ab[2];       // (max(n.L,0), intensity) per shadow ray
    DeviceBuffer s_lit[2];      // in_light byte per shadow ray
    DeviceBuffer lit_bc[2];     // float4 (body colour, albedo) per lit hit
    DeviceBuffer lit_node[2];   // node index per lit hit
    // Scenes with more than RG_MAX_LIGHTS lights only (light chunks after the first, rg_wavefront.cu):
    DeviceBuffer lit_geo[2];    // per lit hit: hit point and normal (f64, a RayQueue with o = point, d = normal) + body
    DeviceBuffer lit_acc[2];    // per lit hit: float4 RGB sum of the chunks so far
    std::vector<DeviceBuffer> nodes;   // per level: NodeA float4 + NodeB uint4
    std::vector<cudaEvent_t> events;   // timing events of the trace launches, reused across frames
    cudaStream_t aux = nullptr;        // shadow-side stream (created on first use)
    std::vector<cudaEvent_t> sync_events;   // cross-stream dependencies (no timing), reused across frames
    void release();
};

// Captured wavefront frames (rg_wavefront.cu): the launch sequence of a batch depends only on its
// key (batch geometry, output pointers, options, scratch addresses), so it is captured once into a
// CUDA graph and replayed; a key must be seen twice before it is worth an instantiation.
struct GraphEntry {
    std::vector<uint64_t> key;
    cudaGraphExec_t exec = nullptr;
    uint32_t launches = 0;
    uint64_t last_use = 0;
};
struct GraphCache {
    std::vector<GraphEntry> entries;
    std::vector<std::vector<uint64_t>> seen;
    uint64_t tick = 0;
    void release();
};

// The device-side state of a scene that does not depend on the scene's content.  Destroying a scene
// parks it (rg_api.cu) and the next scene created on the same device adopts it, so a host that
// re-uploads the scene every frame does not pay cudaMalloc / cudaFree for its (possibly multi-GB)
// scratch each time.
struct DeviceContext {
    WavefrontScratch wf;
    DeviceBuffer frame;                // staging of host-buffer renders
    DeviceBuffer rowlist;              // device copy of a caller's row list
    DeviceBuffer samples;              // megakernel with RG_OPT_SUPERSAMPLE > 1: f32 RGB of a band of samples
    // RG_OPT_SUPERSAMPLE_EDGES (rg_api.cu adaptive_render)
    DeviceBuffer edge_ref;             // the reference frame of the requested rows and their neighbours: f32 RGB
    DeviceBuffer edge_rows;            // requested rows, their neighbours' rows in edge_ref, and those rows' image rows
    DeviceBuffer edge_flag;            // per requested pixel: refined; then per emit block: refined count / offset
    DeviceBuffer edge_list;            // the refined pixels (EdgeList)
    SceneArena arena;                  // scene arrays
    DCounters *d_counters = nullptr;
    DCounters *h_counters = nullptr;   // pinned
    cudaStream_t stream = nullptr;     // library-owned stream for host-buffer renders
    cudaEvent_t ev[4] = {nullptr, nullptr, nullptr, nullptr};
    uint8_t *h_stage = nullptr;        // pinned staging of the scene upload (one H2D copy per scene)
    size_t h_stage_cap = 0;
    // every handle exists: a create() that failed half-way must not hand its holes to the next scene
    bool complete() const { return stream && d_counters && h_counters && ev[0] && ev[1] && ev[2] && ev[3]; }
    void release();                    // frees everything; the context's device must be current
};

// RG_OPT_SUPERSAMPLE_EDGES: the refined pixels of an adaptive frame (rg_api.cu adaptive_render), in device memory.
// Entry (k, x) is column x of the call's k-th requested row, which is image row req_rows[k].
struct EdgeList {
    const uint2 *entries;
    uint32_t count;
    const uint32_t *req_rows;
};

// What a render call delivers: RGBA8 rows in order, RGBA8 rows stored at their place in a full frame
// (rg_render_rowlist_scatter), unquantised f32 RGB rows in order (rg_render_rows_f32), or f32 RGB rows stored at
// their place in a full frame (rg_render_rowlist_f32_scatter).
enum class OutKind { Rgba8, Rgba8Scatter, F32, F32Scatter };
constexpr size_t bytes_per_pixel(OutKind k) { return k == OutKind::F32 || k == OutKind::F32Scatter ? 12 : 4; }
// the output pointer is a full frame (address of image row 0), not the batch's first row
constexpr bool is_scatter(OutKind k) { return k == OutKind::Rgba8Scatter || k == OutKind::F32Scatter; }

}  // namespace rg

namespace rg { struct MultiState; }

// Parking moves the DeviceContext base out (its DeviceBuffers are plain pointer pairs, so they are
// copied) and deletes the scene without releasing anything: rg_scene must not free in a destructor.
struct rg_scene : rg::DeviceContext {
    int device = 0;
    rg::MultiState *multi = nullptr;       // set: this handle spans several GPUs (rg_multi.cu) and owns no device state itself
    std::atomic<bool> busy{false};         // a render call is running on this handle (second callers get RG_E_BUSY)
    rg::DScene ds{};                    // device pointers inside
    rg::GridProxies gp{};               // boxes and disks binned into the grid (rg_scene.cuh)
    rg::LightGrids lg{};                // per-light grids of the shadow rays (rg_light_grid.h)
    std::vector<rg::DLight> lights;        // every light, as uploaded (light_all): the host builds each light chunk's
                                           // DScene from these without reading the device
    std::vector<cudaTextureObject_t> tex_objs;
    uint8_t *h_frame = nullptr;            // pinned staging of the streaming renders (not parked; a multi-GPU handle has one too)
    size_t h_frame_cap = 0;
    rg::GraphCache graphs;                 // dies with the scene (kernel parameters hold scene pointers by value)
    // options
    int pipeline = RG_PIPELINE_AUTO;
    int accel = RG_ACCEL_AUTO;
    uint32_t scene_max_depth = 0;          // as given in the desc
    uint64_t batch_pixels = 0;
    int verify_cull = 0;
    int overlap = 0;                       // RG_OPT_OVERLAP: 0 auto (on with the grid tracer), 1 off, 2 on
    int graph = 0;                         // RG_OPT_GRAPH: 0 auto, 1 off, 2 on
    int trace_stats = 0;                   // RG_OPT_TRACE_STATS: 0 off, 1 every grid trace launch, 2 any-hit only, 3 nearest-hit only
    bool origin_hints = true;              // RG_OPT_ORIGIN_HINTS
    bool light_grids = true;               // RG_OPT_LIGHT_GRIDS
    uint32_t supersample = 1;              // RG_OPT_SUPERSAMPLE: n x n samples per pixel (a multi-GPU handle keeps a copy
                                           // for its size checks)
    int supersample_edges = -1;            // RG_OPT_SUPERSAMPLE_EDGES: -1 off, else the mask's threshold T (0 ... 255)
    uint32_t depth_hint = 0;               // levels the ray tree of this scene has been seen to use (0 = unknown)
    uint32_t level_growth = 2;             // wavefront queue of level d holds min(2^d, level_growth) x the batch's pixels;
                                           // doubled when a level outgrows its queue (the frame is then repeated)
    // derived
    uint32_t n_bodies = 0;
    int sm_count = 0;
};

namespace rg {
// rg_wavefront.cu
// rows [y0, y1) of the image, or — when d_rows is given — entries [y0, y1) of that row list, at n x n samples per
// pixel (n > 1: d_rows is the expanded list of sample rows, n per listed row, render_rowlist_device).  With `list`, the
// refined pixels of an adaptive frame instead (y0, y1 and d_rows unused), each stored at its place (EdgeList).
int wavefront_render(rg_scene *sc, uint32_t width, uint32_t height, uint32_t y0, uint32_t y1,
                     const uint32_t *d_rows, OutKind kind, uchar4 *d_out, cudaStream_t stream, rg_stats *st, uint32_t n,
                     const EdgeList *list = nullptr);
// RG_OPT_SUPERSAMPLE = n > 1: writes `out_rows` output rows of `width` pixels, each the average of its n x n samples,
// which are f32 RGB at src + stride * i, i in the order of the level-0 queue with strips of `strip` rows over the
// batch's n out_rows sample rows (strip 1: row-major).  Scatter: output row r goes to image row d_rows[row0 + r n] / n.
int launch_resolve(OutKind kind, const float *src, uint32_t stride, uint32_t strip, uint32_t n, uint32_t width, uint32_t out_rows,
                   const uint32_t *d_rows, uint32_t row0, void *out, cudaStream_t stream);
// RG_OPT_SUPERSAMPLE_EDGES: stores the average of each listed pixel's n x n samples (f32 RGB at src + stride * i, pixel-
// major, sub-row-major) at the pixel's place: row k of `out`, or image row req_rows[k] of a full frame (scatter kinds)
int launch_resolve_list(OutKind kind, const float *src, uint32_t stride, uint32_t n, uint32_t width, const uint2 *list, uint32_t count,
                        const uint32_t *req_rows, void *out, cudaStream_t stream);
// RG_OPT_SUPERSAMPLE_EDGES: mask, emit and compact over the npix = K width requested pixels (k_edge_emit): the unrefined
// pixels get their reference value in `out`, the refined ones go to `list`, their count to block_count[(npix + 255) / 256]
int launch_edge_mask(OutKind kind, const float *ref, const int32_t *nb, uint32_t width, uint32_t npix, uint32_t t,
                     const uint32_t *req_rows, void *out, uint8_t *flag, uint32_t *block_count, uint2 *list, cudaStream_t stream);
// rg_api.cu
// rg_render_rowlist_device / rg_render_rowlist_f32_device (kind Rgba8 / F32) and rg_render_rowlist_scatter /
// rg_render_rowlist_f32_scatter (Rgba8Scatter / F32Scatter) without the one-render-at-a-time guard (for callers that hold it)
int render_rowlist_device(rg_scene *sc, uint32_t w, uint32_t h, const uint32_t *rows, uint32_t n_rows, OutKind kind, void *d_out,
                          cudaStream_t stream, rg_stats *stats);
// adds the stats of one part of a call to `total`; device times add up for parts that ran one after another and
// overlap for `concurrent` ones (the slowest counts)
void merge_stats(rg_stats &total, const rg_stats &part, bool concurrent);
// rg_multi.cu
// kind Rgba8 or F32: row rows[k] goes to frame + rows[k] * w * bytes_per_pixel(kind)
int render_rowlist_to_host(rg_scene *sc, uint32_t w, uint32_t h, const uint32_t *rows, uint32_t n_rows, OutKind kind, uint8_t *frame,
                           rg_stats *st);
int multi_create(const rg_scene_desc *desc, const int32_t *devices, uint32_t n_devices, rg_scene **out);
void multi_destroy(rg_scene *sc);
int multi_set_option(rg_scene *sc, int32_t key, int64_t value);
uint32_t multi_device_count(const rg_scene *sc);
int multi_render_rows(rg_scene *sc, uint32_t w, uint32_t h, uint32_t y0, uint32_t y1, uint8_t *rgba_out, rg_stats *stats);
// rg_grid.cu
int grid_build(rg_scene *sc, const double *sph /* n x 4, host */, uint32_t n);
// after grid_build: the light grids of the scene's first kLightGrids lights (none without the 3-D grid)
int light_grid_build(rg_scene *sc, const double *sph /* n x 4, host */, uint32_t n);
}  // namespace rg
