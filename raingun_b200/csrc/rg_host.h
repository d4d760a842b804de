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
// blocks survive the scene (see ParkedContext in rg_api.cu): re-uploading a scene every frame
// then costs H2D copies only.
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
    std::vector<DeviceBuffer> nodes;   // per level: NodeA float4 + NodeB uint4
    std::vector<cudaEvent_t> events;   // timing events of the trace launches, reused across frames
    cudaStream_t aux = nullptr;        // shadow-side stream (created on first use)
    cudaStream_t rb = nullptr;         // counter read-back stream (lets the main stream run ahead of the host)
    std::vector<cudaEvent_t> sync_events;   // cross-stream dependencies (no timing), reused across frames
    void release();
};

// Captured host-free frames (rg_wavefront.cu): the launch sequence of a batch depends only on its
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

}  // namespace rg

namespace rg { struct MultiState; }

struct rg_scene {
    int device = 0;
    rg::MultiState *multi = nullptr;       // set: this handle spans several GPUs (rg_multi.cu) and owns no device state itself
    std::atomic<bool> busy{false};         // a render call is running on this handle (second callers get RG_E_BUSY)
    rg::DScene ds{};                    // device pointers inside
    rg::GridProxies gp{};               // boxes and disks binned into the grid (rg_scene.cuh)
    rg::SceneArena arena;               // scene arrays
    std::vector<cudaTextureObject_t> tex_objs;
    rg::DCounters *d_counters = nullptr;
    rg::DCounters *h_counters = nullptr;   // pinned
    cudaStream_t stream = nullptr;         // library-owned stream for host-buffer renders
    cudaEvent_t ev[4] = {nullptr, nullptr, nullptr, nullptr};
    rg::DeviceBuffer frame;                // RGBA8 staging for host-buffer renders
    rg::DeviceBuffer rowlist;              // device copy of a caller's row list
    uint8_t *h_stage = nullptr;            // pinned staging of the scene upload (one H2D copy per scene)
    size_t h_stage_cap = 0;
    uint8_t *h_frame = nullptr;            // pinned staging
    size_t h_frame_cap = 0;
    rg::WavefrontScratch wf;
    rg::GraphCache graphs;                 // dies with the scene (kernel parameters hold scene pointers by value)
    // options
    int pipeline = RG_PIPELINE_AUTO;
    int accel = RG_ACCEL_AUTO;
    uint32_t scene_max_depth = 0;          // as given in the desc
    uint64_t batch_pixels = 0;
    int verify_cull = 0;
    int overlap = 0;                       // RG_OPT_OVERLAP: 0 auto (on with the grid tracer), 1 off, 2 on
    int host_free = 0;                     // RG_OPT_HOST_FREE: 0 auto (on), 1 off (host-sized loop), 2 on
    int graph = 0;                         // RG_OPT_GRAPH: 0 auto, 1 off, 2 on
    bool trace_stats = false;              // RG_OPT_TRACE_STATS
    bool origin_hints = true;              // RG_OPT_ORIGIN_HINTS
    uint32_t depth_hint = 0;               // levels the ray tree of this scene has been seen to use (0 = unknown)
    bool host_free_overflowed = false;     // a level once outgrew the default queue capacity: stay with the host-sized loop
    bool out_f32 = false;                  // this call delivers unquantised f32 colours, 3 per pixel (rg_render_rows_f32)
    bool scatter_out = false;              // this call stores rows at their place in a full frame (rg_render_rowlist_scatter)
    // derived
    uint32_t n_bodies = 0;
    int sm_count = 0;
};

namespace rg {
// rg_wavefront.cu
// rows [y0, y1) of the image, or — when d_rows is given — entries [y0, y1) of that row list
int wavefront_render(rg_scene *sc, uint32_t width, uint32_t height, uint32_t y0, uint32_t y1,
                     const uint32_t *d_rows, uchar4 *d_out, cudaStream_t stream, rg_stats *st);
// rg_api.cu: rg_render_rowlist_device without the one-render-at-a-time guard (for callers that hold it)
int rowlist_device_unguarded(rg_scene *sc, uint32_t w, uint32_t h, const uint32_t *rows, uint32_t n_rows, void *d_rgba_out,
                             void *cuda_stream, rg_stats *stats);
// rg_multi.cu
int render_rowlist_to_host(rg_scene *sc, uint32_t w, uint32_t h, const uint32_t *rows, uint32_t n_rows, uint8_t *frame, rg_stats *st);
int multi_create(const rg_scene_desc *desc, const int32_t *devices, uint32_t n_devices, rg_scene **out);
void multi_destroy(rg_scene *sc);
int multi_set_option(rg_scene *sc, int32_t key, int64_t value);
uint32_t multi_device_count(const rg_scene *sc);
int multi_render_rows(rg_scene *sc, uint32_t w, uint32_t h, uint32_t y0, uint32_t y1, uint8_t *rgba_out, rg_stats *stats);
// rg_grid.cu
int grid_build(rg_scene *sc, const double *sph /* n x 4, host */, uint32_t n);
}  // namespace rg
