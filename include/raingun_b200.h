/*
 * raingun_b200.h — C ABI of the B200-native render hot path.
 *
 * This is the drop-in boundary for raingun-lib's per-pixel render path. The
 * reference has no FFI today; the path sits behind two inherent methods of a
 * plain Rust struct:
 *
 *     pub struct Scene { fov, default_color, max_recursion_depth, bodies, lights }
 *                                                   raingun-lib/src/scene.rs:11-19
 *     Scene::render_image(&self, w, h) -> ImageBuffer<Rgba<u8>>      scene.rs:41-43
 *     Scene::streaming_render(&self, w, h, Sender<RenderedPixel>)    scene.rs:45-51
 *
 * A host (the Rust `-sys` shim shown in INTEGRATION.md, the C++ host in
 * raingun_b200/host, or the Python ctypes mirror in raingun_b200/) parses the
 * YAML scene and decodes textures exactly as the reference does, flattens the
 * `Vec<Body>` / `Vec<Light>` into the body-indexed arrays of `rg_scene_desc`,
 * and calls the entry points below.  Plain pointers and sizes only; the library
 * copies everything it is given (host buffers stay caller-owned).
 *
 * There is no CPU fallback: every entry point that renders fails with
 * RG_E_CUDA when no sm_100 device is usable.
 */
#ifndef RAINGUN_B200_H
#define RAINGUN_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define RG_ABI_VERSION 2u

/* Largest scene.max_recursion_depth the device path accepts (the reference's
 * default is 10, scene.rs:26; `--draft` lowers it to 4, src/main.rs:74-75). */
#define RG_MAX_DEPTH 64u
/* Obsolete: scenes may have any number of lights.  Kept so that existing hosts compile.  It is
 * still the size of one light chunk: the device shades a scene's lights RG_MAX_LIGHTS at a time,
 * so a scene with at most this many lights takes exactly the path it always took. */
#define RG_MAX_LIGHTS 32u

/* ---- error codes (0 = ok, negative = failure; never unwinds across the ABI) */
enum {
    RG_OK = 0,
    RG_E_INVALID = -1,    /* null pointer, bad enum value, bad index            */
    RG_E_PORTRAIT = -2,   /* width < height: `assert!(width >= height)` ray.rs:42 */
    RG_E_TOO_LARGE = -3,  /* width*height does not fit u32 (rendering.rs:27)    */
    RG_E_DEPTH = -4,      /* max_recursion_depth > RG_MAX_DEPTH                 */
    RG_E_CUDA = -5,       /* CUDA runtime failure / no usable device            */
    RG_E_NOMEM = -6,      /* device or host allocation failed                   */
    RG_E_CANCELLED = -7,  /* streaming callback asked to stop (rendering.rs:53-54,67) */
    RG_E_LIGHTS = -8,     /* obsolete: no longer returned (any light count is accepted) */
    RG_E_BUSY = -9        /* the handle is already rendering on another thread (the reference's &Scene
                             is Sync; a device scene owns its scratch: one render at a time per handle) */
};

/* `device` value for rg_scene_create: upload to EVERY visible GPU; renders are then split into row
 * tiles across them inside the library (rayon's par_iter, rendering.rs:27-35). */
#define RG_DEVICE_ALL (-1)

/* ---- enums mirroring the reference's serde enums --------------------------- */
enum { RG_BODY_SPHERE = 0, RG_BODY_PLANE = 1, RG_BODY_DISK = 2, RG_BODY_AABB = 3 }; /* bodies.rs:41-47 */
enum { RG_COLORATION_COLOR = 0, RG_COLORATION_TEXTURE = 1 };                        /* material.rs:20-24 */
enum { RG_SURFACE_DIFFUSE = 0, RG_SURFACE_REFLECTING = 1, RG_SURFACE_REFRACTIVE = 2 }; /* material.rs:49-54 */
enum { RG_LIGHT_DIRECTIONAL = 0, RG_LIGHT_SPHERICAL = 1 };                          /* lights.rs:22-26 */

/* One decoded texture (`DynamicImage`, material.rs:26-32).  `channels` is 3
 * (RGB8) or 4 (RGBA8); rows are tightly packed, row-major, top row first —
 * `get_pixel(x, y)` order (material.rs:67). */
typedef struct rg_texture_desc {
    uint32_t width;
    uint32_t height;
    uint32_t channels;
    uint32_t reserved;
    const uint8_t *pixels;
} rg_texture_desc;

/* The flattened `Scene` (scene.rs:11-19).  All per-body arrays are indexed by
 * the body's position in `Scene::bodies`, which is what the first-minimum
 * tie-break of `Scene::trace` (scene.rs:34-39) depends on.
 *
 * body_geom[i][8] (f64), by kind:
 *   SPHERE  center.x,y,z, radius                              bodies.rs:13-18
 *   PLANE   origin.x,y,z, normal.x,y,z   (normal NOT normalised) bodies.rs:20-25
 *   DISK    origin.x,y,z, normal.x,y,z, radius                bodies.rs:27-33
 *   AABB    bounds[0].x,y,z, bounds[1].x,y,z                  bodies.rs:35-39
 * f32 material fields are the YAML numbers parsed as f64 and then narrowed,
 * as serde does (material.rs:10,30-31,52-53; lights.rs:12,19).
 */
typedef struct rg_scene_desc {
    uint32_t abi_version;          /* RG_ABI_VERSION */
    uint32_t max_recursion_depth;  /* scene.rs:16, default 10 */
    double fov;                    /* degrees, scene.rs:14, default 90 */
    float default_color[3];        /* scene.rs:15 */
    uint32_t n_bodies;

    const uint8_t *body_kind;       /* [n_bodies] RG_BODY_*            */
    const double *body_geom;        /* [n_bodies][8]                   */
    const uint8_t *coloration_kind; /* [n_bodies] RG_COLORATION_*      */
    const float *color;             /* [n_bodies][3] (Color variant)   */
    const int32_t *texture_id;      /* [n_bodies] index into textures, or -1 */
    const float *texture_offset;    /* [n_bodies][2] x_offset, y_offset */
    const float *albedo;            /* [n_bodies]                      */
    const uint8_t *surface_kind;    /* [n_bodies] RG_SURFACE_*         */
    const float *surface_param;     /* [n_bodies][2]: Reflecting{reflectivity,-};
                                       Refractive{index, transparency} */

    uint32_t n_lights;
    uint32_t n_textures;
    const uint8_t *light_kind;      /* [n_lights] RG_LIGHT_*           */
    const double *light_vec;        /* [n_lights][3] direction | position */
    const float *light_color;       /* [n_lights][3]                   */
    const float *light_intensity;   /* [n_lights]                      */

    const rg_texture_desc *textures; /* [n_textures] */
} rg_scene_desc;

/* Which device pipeline renders (all are bit-identical in their output). */
enum {
    RG_PIPELINE_WAVEFRONT = 0, /* per-bounce ray queues                            */
    RG_PIPELINE_MEGAKERNEL = 1,/* one thread per pixel, explicit stack, every body tested in FP64 */
    RG_PIPELINE_AUTO = 2       /* default: the megakernel for scenes of a handful of bodies (the shipped
                                  examples: no queue traffic at all, 2-3x faster there), else the wavefront */
};
/* How `Scene::trace` is evaluated (results identical; see DESIGN.md). */
enum {
    RG_ACCEL_AUTO = 0,  /* grid when it pays (64 or more spheres, boxes and disks it can bin), brute force otherwise */
    RG_ACCEL_BRUTE = 1, /* the reference algorithm: every ray x every body */
    RG_ACCEL_GRID = 2   /* exact culling through a uniform grid + brute-force rest: spheres, and boxes (lo <= hi) and
                           disks (radius > 0) of finite geometry through enclosing spheres; planes and other
                           bodies are tested per ray */
};
/* Option keys for rg_scene_set_option. */
enum {
    RG_OPT_PIPELINE = 1,
    RG_OPT_ACCEL = 2,
    RG_OPT_MAX_DEPTH = 3,    /* like main.rs:119-123: lowers max_recursion_depth  */
    RG_OPT_BATCH_PIXELS = 4, /* pixels per wavefront batch (0 = automatic); with RG_OPT_SUPERSAMPLE > 1, samples per
                                batch, and per band of the megakernel's sample scratch */
    RG_OPT_VERIFY_CULL = 5,  /* debug: count FP32-culled pairs the FP64 test hits  */
    RG_OPT_OVERLAP = 6,      /* shadow side of a level concurrent with the next level's path side:
                                0 = automatic (on with the grid tracer), 1 = off, 2 = on */
    RG_OPT_HOST_FREE = 7,    /* obsolete: every wavefront frame runs the host-free level loop (device-sized
                                launches, one synchronisation per frame; render_image is one call,
                                rendering.rs:24-38).  Values 0-2 are accepted and ignored */
    RG_OPT_GRAPH = 8,        /* replay the host-free frame as one CUDA graph: 0 = automatic, 1 = off, 2 = on */
    RG_OPT_TRACE_STATS = 9,  /* 1 = the grid tracer counts cells / fetches / cull tests / lane use
                                (rg_stats.grid_*); an instrumented kernel, slower; results unchanged.
                                2 = count the any-hit (shadow) launches only, 3 = the nearest-hit ones only */
    RG_OPT_SCHEDULE = 11,    /* multi-GPU scenes: 0 = automatic, 1 = static (tile t on device t mod N),
                                2 = static share + a stealable tail handed out by an atomic tile counter */
    RG_OPT_TILE_ROWS = 12,   /* multi-GPU scenes: rows per tile (default 8) */
    RG_OPT_ORIGIN_HINTS = 13, /* 1 (default) = every secondary ray carries the outcome of the reference's test against the
                                sphere it starts on, and the grid tracer skips that test; 0 = off.  Results unchanged
                                (Scene::trace is a minimum: a body proven to return None may be left out, scene.rs:34-39) */
    RG_OPT_SUPERSAMPLE = 14, /* n x n primary rays per pixel, box-filtered on the device; 1 (default) ... 8, anything else
                                is RG_E_INVALID.  A (w x h) frame is the reference's render at (n*w x n*h) reduced n x n:
                                sample (X, Y) is the f32 Color of create_prime(X, Y, n*w, n*h) (ray.rs:37-54), and per
                                channel, in f32, s = 0; for j in 0..n, for i in 0..n: s = s + sample(n*x + i, n*y + j);
                                avg = s / (n*n), rounded to nearest.  The RGBA8 entry points store Color::rgba(avg)
                                (color.rs:32-37), the f32 ones avg.  Output buffers keep their sizes; the ray and error
                                counters count every sample's rays.  (n*w)*(n*h) must fit in u32, else RG_E_TOO_LARGE. */
    RG_OPT_LIGHT_GRIDS = 15, /* 1 (default) = the grid tracer traces the shadow rays of a scene's first 8 lights through
                                per-light 2-D grids (one short list per ray instead of a 3-D walk); 0 = the 3-D walk for
                                every ray.  Results unchanged (DESIGN.md section 4.2) */
    RG_OPT_SUPERSAMPLE_EDGES = 16 /* edge-adaptive RG_OPT_SUPERSAMPLE: -1 (default) = off, every pixel gets n x n samples;
                                T = 0 ... 255 = only pixels on an edge of the reference frame do; anything else is
                                RG_E_INVALID.  No effect with n = 1.  With n > 1 and T >= 0, for a (w x h) image:
                                R is the reference's own RGBA8 frame of the WHOLE image (Color::rgba of
                                create_prime(x, y, w, h), the n = 1 frame).  Pixel (x, y) is refined iff some
                                8-neighbour (x + dx, y + dy) inside the image has |R(x,y)_c - R(x+dx,y+dy)_c| > T, in
                                integer bytes, for some c in r, g, b (alpha is ignored; a NaN colour is 0 in R).  A
                                refined pixel is what RG_OPT_SUPERSAMPLE = n delivers for it; any other pixel is the
                                n = 1 pixel (R's bytes, or its f32 colour).  The mask is a function of the whole frame:
                                every entry point (row ranges, row lists in any order with duplicates, scatter, host,
                                device, f32, streaming, multi-GPU at any tile height) gives the pixels of a full-frame
                                render.  Counters count every ray traced: with R' = the requested rows and their
                                in-image neighbours y +- 1, once each, rays_primary = |R'| w + n*n (refined requested
                                pixels), the other counters those rays' trees.  Output sizes, refusals and size checks
                                are those of RG_OPT_SUPERSAMPLE (DESIGN.md section 4.6) */
};

/* Counters and timings of one render call.  A "ray" is one `Scene::trace`
 * invocation (rendering.rs:73 primary, :126 reflection/transmission, :150 shadow). */
typedef struct rg_stats {
    uint64_t rays_primary;
    uint64_t rays_shadow;
    uint64_t rays_reflection;
    uint64_t rays_transmission;
    uint64_t body_tests;           /* sum over rays of n_bodies (brute-force charge) */
    uint64_t exact_tests;          /* FP64 intersect evaluations actually executed (the grid tracer
                                      counts a box or disk it tests twice for one ray twice) */
    uint64_t cull_unsound;         /* RG_OPT_VERIFY_CULL: must be 0                   */
    /* conditions on which the reference would have panicked */
    uint64_t err_nan_distance;     /* scene.rs:38 partial_cmp().unwrap()             */
    uint64_t err_transmission_none;/* rendering.rs:106 .unwrap() on None             */
    uint64_t err_aabb_normal;      /* bodies.rs:324 assert!(false)                   */
    double ms_device;              /* CUDA-event time of all device work             */
    double ms_trace;               /* ... of the nearest-hit + shadow kernels        */
    double ms_wall;                /* host wall clock of the call                    */
    uint32_t gpu_launches;         /* kernels launched by this call                  */
    uint32_t batches;              /* wavefront batches                              */
    uint32_t max_level;            /* deepest level that traced a ray                */
    uint32_t accel_used;           /* RG_ACCEL_BRUTE | RG_ACCEL_GRID                 */
    uint32_t host_free;            /* 1 = the frame ran without host synchronisation (every wavefront frame;
                                      0 for the megakernel) */
    uint32_t graph_replays;        /* batches replayed from a captured CUDA graph    */
    /* RG_OPT_TRACE_STATS (grid tracer only; zero otherwise) */
    uint64_t grid_cells;           /* grid cells visited by all rays                 */
    uint64_t grid_fetches;         /* cell records fetched (occupied cells)          */
    uint64_t grid_culls;           /* FP32 cull tests                                */
    uint64_t grid_refills;         /* warp refills from the ray counter              */
    uint64_t grid_lane_steps;      /* lanes doing scan work, summed over scan iterations */
    uint64_t grid_lane_slots;      /* 32 x scan iterations (the denominator)         */
    uint32_t pipeline_used;        /* RG_PIPELINE_WAVEFRONT | RG_PIPELINE_MEGAKERNEL */
    uint32_t devices_used;         /* GPUs that rendered rows of this call (multi-GPU scenes) */
} rg_stats;

typedef struct rg_scene rg_scene;

/* Streaming callback: one finished band of rows (the analogue of the
 * `RenderedPixel` messages, rendering.rs:18-22,59-65).  `rgba` holds
 * `rows * width * 4` bytes and is only valid during the call.  Return 0 to
 * continue, non-zero to cancel (a closed channel, rendering.rs:53-54,67). */
typedef int (*rg_rows_cb)(uint32_t y0, uint32_t rows, uint32_t width,
                          const uint8_t *rgba, void *user);

/* Copies the flattened scene, uploads it to CUDA device `device`, builds the
 * exact-culling grid.  Replaces the serde construction of `Scene`
 * (scene.rs:11-31) + `load_texture` (material.rs:34-47) as the upload layer. */
int rg_scene_create(const rg_scene_desc *desc, int32_t device, rg_scene **out);
/* The same on an explicit list of devices (n_devices >= 1; a device listed twice gets two lanes).  With more than one device the
 * handle spans them: rg_render / rg_render_rows / rg_render_stream cut the image into row tiles, one
 * library thread per GPU renders the tiles it owns or claims from the shared tile counter and copies its
 * rows over its own PCIe link into the caller's buffer.  The *_device entry points need a single-device
 * handle. */
int rg_scene_create_multi(const rg_scene_desc *desc, const int32_t *devices, uint32_t n_devices, rg_scene **out);
/* GPUs a handle spans (1 for rg_scene_create on one device). */
int rg_scene_device_count(const rg_scene *scene);
void rg_scene_destroy(rg_scene *scene);
int rg_scene_set_option(rg_scene *scene, int32_t key, int64_t value);

/* Scene::render_image (scene.rs:41-43 -> rendering.rs:24-38).  Blocking; writes
 * width*height*4 bytes of row-major RGBA8 (alpha 255, color.rs:32-37) into
 * caller-owned HOST memory. `stats` may be NULL. */
int rg_render(rg_scene *scene, uint32_t width, uint32_t height,
              uint8_t *rgba_out, rg_stats *stats);

/* The same, restricted to image rows [y0, y1): the unit multi-GPU sharding
 * works in.  Writes (y1-y0)*width*4 bytes. */
int rg_render_rows(rg_scene *scene, uint32_t width, uint32_t height,
                   uint32_t y0, uint32_t y1, uint8_t *rgba_out, rg_stats *stats);

/* As rg_render_rows but the result stays in DEVICE memory (`d_rgba_out`, on the
 * scene's device, (y1-y0)*width*4 bytes) and the work is enqueued on
 * `cuda_stream` (a cudaStream_t, NULL = the legacy default stream).  The call
 * returns after the device work has finished (per-level queue sizes are read
 * back on the host). */
int rg_render_rows_device(rg_scene *scene, uint32_t width, uint32_t height,
                          uint32_t y0, uint32_t y1, void *d_rgba_out,
                          void *cuda_stream, rg_stats *stats);

/* Row-tile sharding: renders the image rows listed in `rows` (n_rows entries, any order, HOST
 * array) and writes them compacted, in list order, to DEVICE memory (n_rows*width*4 bytes).
 * This is the unit a multi-GPU host uses: each GPU renders the row tiles it claimed from a
 * work-stealing counter, then the tiles are gathered (raingun_b200/dist.py). */
int rg_render_rowlist_device(rg_scene *scene, uint32_t width, uint32_t height,
                             const uint32_t *rows, uint32_t n_rows, void *d_rgba_out,
                             void *cuda_stream, rg_stats *stats);

/* The same with the gather FUSED into the last kernel: row `rows[k]` is stored at its own place,
 * `d_frame + rows[k]*width*4`, of a full width*height*4 frame.  `d_frame` may be another GPU's
 * memory mapped with rg_shared_frame_open: every GPU of a box then quantises its rows straight
 * into the one frame on GPU 0 over NVLink / NVSwitch, and `collect` (rendering.rs:34-35) needs no
 * separate exchange — only a barrier.  Wavefront pipeline only. */
int rg_render_rowlist_scatter(rg_scene *scene, uint32_t width, uint32_t height,
                              const uint32_t *rows, uint32_t n_rows, void *d_frame,
                              void *cuda_stream, rg_stats *stats);

/* Row-tile sharding with the frame in HOST memory: renders the listed image rows on the scene's device and
 * copies row rows[k] to `frame + rows[k]*width*4` (`frame` = address of image row 0 of a full
 * width*height*4 frame; runs of adjacent rows travel as one copy, an interleaved share as one strided
 * copy).  With one process (or thread) per GPU and `frame` a pinned buffer all of them see — the caller's
 * own, or a shared-memory file registered with rg_host_register in every process — every GPU delivers its
 * rows over its own PCIe link and nothing is gathered on a GPU first. */
int rg_render_rowlist_host(rg_scene *scene, uint32_t width, uint32_t height,
                           const uint32_t *rows, uint32_t n_rows, uint8_t *frame, rg_stats *stats);
/* Pins caller-owned host memory (cudaHostRegister, portable) so that device-to-host copies into it run at
 * full PCIe speed; undo with rg_host_unregister before freeing it. */
int rg_host_register(void *ptr, size_t bytes);
int rg_host_unregister(void *ptr);

/* One process driving several GPUs: lets kernels running on `device` store into memory that lives on `peer`
 * (cudaDeviceEnablePeerAccess; NVLink / NVSwitch on a B200 box), so that rg_render_rowlist_scatter on one GPU
 * can write its rows into a frame on another.  Harmless if already enabled. */
int rg_device_enable_peer(int32_t device, int32_t peer);

/* A barrier for the processes of one box (one per GPU) in POSIX shared memory: the creator (create = 1) makes
 * it for `parties` processes and hands `name` ("/something") to the others by any channel; every process then
 * calls rg_shm_barrier_wait at the end of a sharded frame.  Each rank has synchronised its own stream by then
 * (the render calls block), so a sense-reversing counter does in microseconds what a GPU collective does in
 * 60-100 us.  Close in every process; the creator also unlinks the name. */
int rg_shm_barrier_open(const char *name, uint32_t parties, int32_t create, void **handle);
int rg_shm_barrier_wait(void *handle);
int rg_shm_barrier_close(void *handle);

/* A device frame that other PROCESSES (one per GPU) can map: create on the owning rank, pass the
 * opaque handle bytes to the others (any channel), open there.  Close with is_owner = 1 on the
 * creating rank (frees the memory), 0 elsewhere (unmaps). */
#define RG_IPC_HANDLE_BYTES 64u
int rg_shared_frame_create(int32_t device, size_t bytes, void **d_ptr, uint8_t *handle /* [RG_IPC_HANDLE_BYTES] */);
int rg_shared_frame_open(int32_t device, const uint8_t *handle, void **d_ptr);
int rg_shared_frame_close(int32_t device, void *d_ptr, int32_t is_owner);

/* Scene::streaming_render (scene.rs:45-51 -> rendering.rs:40-69): renders in
 * bands of `band_rows` rows (0 = automatic) and hands each finished band to
 * `cb` from the calling thread.  Returns RG_E_CANCELLED if `cb` returned
 * non-zero. */
int rg_render_stream(rg_scene *scene, uint32_t width, uint32_t height,
                     uint32_t band_rows, rg_rows_cb cb, void *user, rg_stats *stats);

/* Destroying a scene parks its device-side context (scratch queues of possibly several GB, frame, arena,
 * stream, pinned buffers) for the next scene created on the same device, so that a host that re-uploads
 * the scene every frame never pays cudaMalloc again.  rg_trim releases everything parked (on all devices)
 * and returns the number of contexts freed; the library also does so itself before reporting RG_E_NOMEM. */
int rg_trim(void);

/* Unquantised output.  `RenderedPixel.color` is an f32 `Color` (rendering.rs:18-22,59-65): streaming_render's
 * consumers receive the colour BEFORE `Color::rgba` (color.rs:32-37) narrows it to bytes.  These two entry
 * points deliver exactly that — 3 floats (r, g, b) per pixel, row-major, bit-identical to the reference's
 * f32 values — for hosts whose consumer is not the CLI's RGBA8 collector.  Single-device scenes. */
typedef int (*rg_rows_f32_cb)(uint32_t y0, uint32_t rows, uint32_t width,
                              const float *rgb, void *user);
int rg_render_rows_f32(rg_scene *scene, uint32_t width, uint32_t height,
                       uint32_t y0, uint32_t y1, float *rgb_out, rg_stats *stats);
int rg_render_stream_f32(rg_scene *scene, uint32_t width, uint32_t height,
                         uint32_t band_rows, rg_rows_f32_cb cb, void *user, rg_stats *stats);

/* The f32 twins of rg_render_rows_device, rg_render_rowlist_device, rg_render_rowlist_scatter and
 * rg_render_rowlist_host: the same rows, destinations, streams, checks, refusals and stats, with 3 floats
 * (12 bytes) per pixel holding the bits rg_render_rows_f32 delivers for the same pixels.  The scatter and
 * host forms store row rows[k] at `d_frame` / `frame` + rows[k]*width*3 floats of a full width*height*3
 * frame; the scatter form needs the wavefront pipeline and writes 128-bit stores when width % 4 == 0 and
 * the frame is 16-byte aligned.  Single-device scenes. */
int rg_render_rows_f32_device(rg_scene *scene, uint32_t width, uint32_t height, uint32_t y0, uint32_t y1,
                              float *d_rgb_out, void *cuda_stream, rg_stats *stats);
int rg_render_rowlist_f32_device(rg_scene *scene, uint32_t width, uint32_t height, const uint32_t *rows,
                                 uint32_t n_rows, float *d_rgb_out, void *cuda_stream, rg_stats *stats);
int rg_render_rowlist_f32_scatter(rg_scene *scene, uint32_t width, uint32_t height, const uint32_t *rows,
                                  uint32_t n_rows, float *d_frame, void *cuda_stream, rg_stats *stats);
int rg_render_rowlist_f32_host(rg_scene *scene, uint32_t width, uint32_t height, const uint32_t *rows,
                               uint32_t n_rows, float *frame, rg_stats *stats);

/* Thread-local description of the last failure in this thread. */
const char *rg_last_error(void);

/* Roofline denominators measured on the scene-independent device: a register-
 * resident FFMA / DFMA loop over the whole chip.  Results in TFLOP/s
 * (2 flops per FMA).  Used by bench.py; not part of the render path. */
int rg_measure_peaks(int32_t device, double *fp32_tflops, double *fp64_tflops,
                     double *sm_clock_mhz);

/* Number of usable CUDA devices (0 if none / no driver). */
int rg_device_count(void);

#ifdef __cplusplus
}
#endif
#endif /* RAINGUN_B200_H */
