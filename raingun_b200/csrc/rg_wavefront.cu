// rg_wavefront.cu — the wavefront pipeline: render_image's pixel loop (rendering.rs:24-38)
// turned inside out.
//
// The reference recurses per pixel (get_color <-> cast_ray, rendering.rs:80-130).  Here all
// rays of one recursion depth form a queue ("level"); per level:
//     k_trace_*  nearest hit of every path ray           Scene::trace            scene.rs:34-39
//     k_shade    hit point, normal, material; emits the level's shadow rays and the next
//                level's reflection / transmission rays, compacted with warp ballot + popc
//                                                         get_color, fresnel, Ray::create_*
//     k_trace_*  (ANY) the shadow rays                    shade_diffuse           rendering.rs:150-155
//     k_diffuse  the per-light sum, in light order        shade_diffuse           rendering.rs:157-171
// (a scene with more than RG_MAX_LIGHTS lights runs the last two per chunk of RG_MAX_LIGHTS lights,
// k_shadow_rays setting up every chunk after the first: see enqueue_batch_dev)
// and after the deepest level, bottom-up:
//     k_combine  parent colour from its children's        get_color               rendering.rs:88-116
//     k_quantise Color::rgba                                                      color.rs:32-37
// Every hit keeps a 32-byte node (colour + child links), so colours are combined in exactly
// the reference's order and the image is bit-identical to the recursive evaluation —
// no throughput-weight reformulation, no atomics on pixels.
#include <algorithm>
#include <cstdlib>

#include "rg_grid.cuh"
#include "rg_host.h"
#include "rg_trace.cuh"

#ifdef RG_GRID_DEBUG
extern "C" int rg_debug_grid_counters(unsigned long long *out, int reset) {
    if (out && cudaMemcpyFromSymbol(out, rg::rg_grid_dbg, sizeof(unsigned long long) * 32) != cudaSuccess) return -1;
    if (reset) { unsigned long long z[32] = {0}; if (cudaMemcpyToSymbol(rg::rg_grid_dbg, z, sizeof z) != cudaSuccess) return -1; }
    return 0;
}
#endif

namespace rg {

constexpr uint32_t kChildDefault = 0xFFFFFFFFu;   // child colour is scene.default_color (no node)
enum : uint32_t { NODE_MISS = 0, NODE_DIFFUSE = 1, NODE_REFLECTING = 2, NODE_REFRACTIVE = 3 };

struct LevelBuffers {
    RayQueue cur, next, shadow;
    const double *hit_t;
    const uint32_t *hit_body;
    float4 *node_a;        // rgb (final colour after k_combine) + p0 (reflectivity | kr)
    uint4 *node_b;         // child_reflection, child_transmission, kind, transparency bits
    double *s_tmax;
    float2 *s_ab;
    float4 *lit_bc;
    uint32_t *lit_node;
    uint32_t cap;          // capacity of this level's queue
    uint32_t shadow_sl, shadow_sj;   // shadow ray of (lit hit j, light l) lives at l * shadow_sl + j * shadow_sj
    uint32_t can_spawn;    // depth + 1 < max_recursion_depth
    // sizes live on the device
    const unsigned int *n_dev;       // the level's ray count
    unsigned int *q_next, *q_lit;    // counters k_shade appends to: children (= next level's n_dev), lit hits
    uint32_t cap_next;               // capacity of the next level's queue
    unsigned int *void_flag;         // set when a queue overflows; once set, every later launch does nothing
    uint32_t level;                  // recursion depth of this level
    uint32_t last_enqueued;          // no launch follows for this level's children (depth hint): flag them
    uint32_t hints;                  // the tracer reads origin hints (rg_trace.cuh): 1 = compute them, 2 = write kHintNone
                                     // (RG_OPT_ORIGIN_HINTS = 0), 0 = the tracer ignores them (brute force): write nothing
    uint32_t n_lights;               // lights of the scene: shadow rays per lit hit, all chunks together
    RayQueue lit_geo;                // light chunks after the first follow (k_shadow_rays): per lit hit, hit point (o),
                                     // normal (d) and body (hint); a == nullptr: not kept
};

// Lights are shaded in chunks of this many (a scene with at most this many lights has exactly one).  It bounds the
// shadow queues at cap x kLightChunk rays per level parity whatever the scene's light count.
constexpr uint32_t kLightChunk = RG_MAX_LIGHTS;

// Size of a level as its kernels see it: read from the device and clamped to the capacity (0 once the frame is void).
__device__ __forceinline__ uint32_t level_size(uint32_t cap, const unsigned int *n_dev, const unsigned int *void_flag) {
    if (*void_flag) return 0u;
    const uint32_t v = *n_dev;
    return v < cap ? v : cap;
}

// Order of the level-0 queue.  Rows of a batch are taken in strips of `strip` rows and a strip is
// walked column by column, so 32 consecutive rays (a warp of every later kernel) cover a compact
// (32 / strip) x strip tile of the image instead of a 32 x 1 run: neighbouring lanes hit the same
// body, their shadow rays and children stay together, and the whole ray tree below inherits the
// locality (queues are compacted in parent order).  Pure index permutation: results are unchanged.
struct PixelOrder {
    uint32_t width, rows, strip;   // batch geometry
    // queue index -> (x, batch row)
    __device__ __forceinline__ void pixel(uint32_t i, uint32_t &x, uint32_t &r) const {
        const uint32_t per = strip * width, sidx = i / per, j = i - sidx * per;
        const uint32_t hs = min(strip, rows - sidx * strip);
        x = j / hs;
        r = sidx * strip + (j - x * hs);
    }
    // (x, batch row) -> queue index
    __device__ __forceinline__ uint32_t index(uint32_t x, uint32_t r) const {
        const uint32_t sidx = r / strip, hs = min(strip, rows - sidx * strip);
        return sidx * strip * width + x * hs + (r - sidx * strip);
    }
};

// rendering.rs:71-72 + ray.rs:37-54: the level-0 queue, one ray per pixel of rows [y0, y1)
// `rows` (optional) maps the k-th row of the batch to an image row, for row-tile sharding.
__global__ void __launch_bounds__(256) k_generate(const DScene s, RayQueue q, uint32_t width, uint32_t height,
                                                  uint32_t y0, uint32_t npix, const uint32_t *__restrict__ rows,
                                                  unsigned int *n_level0, const PixelOrder po) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i == 0 && n_level0) *n_level0 = npix;
    if (i >= npix) return;
    uint32_t x, r;
    po.pixel(i, x, r);
    const uint32_t k = y0 + r;
    const uint32_t y = rows ? rows[k] : k;
    store_ray(q, i, create_prime(s, x, y, width, height));
    q.hint[i] = kHintNone;   // camera rays start on no body
}

// Origin hints of the rays k_shade makes (rg_trace.cuh): `og` = geom of the sphere the ray starts on (nullptr: none,
// or hints are off), `own` = its sphere-list index.
__device__ __forceinline__ uint32_t path_origin_hint(const double *og, uint32_t own, const Ray &r) {
    if (!og) return kHintNone;
    double t;
    return sphere_intersect(og[0], og[1], og[2], og[3], r, t) ? kHintNone : own;   // a hit: the tracer finds it itself
}
__device__ __forceinline__ uint32_t shadow_origin_hint(const double *og, uint32_t own, const Ray &r, double tmax) {
    if (!og) return kHintNone;
    double t;
    if (!sphere_intersect(og[0], og[1], og[2], og[3], r, t)) return own;
    if (t <= tmax) return kHintOccluded;   // rendering.rs:150-155: nearest.distance <= light distance for some body
    return t == t ? own : kHintNone;       // beyond the light: contributes nothing; NaN: the tracer counts it (scene.rs:38)
}

// shade_diffuse's per-(hit, light) setup (rendering.rs:141-149,163): the shadow ray from hit_point + n * SHADOW_BIAS
// towards the light, stored at slot k with the light's distance (the trace's tmax), the ray's origin hint and the
// light-dependent scalars (max(n.L, 0), intensity) that k_diffuse needs.  k_shade runs it for the first light chunk,
// k_shadow_rays for the later ones: the arithmetic exists once.
__device__ __forceinline__ void shadow_ray_setup(const LevelBuffers &lb, uint32_t k, const DLight &L, D3 hp, D3 n,
                                                 const double *og, uint32_t own) {
    Ray sh;
    sh.o = hp + n * kShadowBias;
    sh.d = light_direction_from(L, hp);
    store_ray(lb.shadow, k, sh);
    const double tmax = light_distance(L, hp);
    lb.s_tmax[k] = tmax;
    if (lb.hints) lb.shadow.hint[k] = shadow_origin_hint(og, own, sh, tmax);
    lb.s_ab[k] = make_float2(fmaxf((float)dot(n, sh.d), 0.0f), light_intensity(L, hp));
}

#ifndef RG_SHADE_MINB
#define RG_SHADE_MINB 4   // 64 registers: the kernel waits on gathers (long scoreboard), occupancy pays (measured 3 / 4 / 5 CTAs per SM)
#endif
__global__ void __launch_bounds__(256, RG_SHADE_MINB) k_shade(const DScene s, const LevelBuffers lb, DCounters *ctr) {
    const uint32_t lane = threadIdx.x & 31u, lt = (1u << lane) - 1u;
    const uint32_t n_level = level_size(lb.cap, lb.n_dev, lb.void_flag);
    if (blockIdx.x == 0 && threadIdx.x == 0 && n_level) atomicMax(&ctr->max_level, lb.level);
    __shared__ uint32_t sh_cnt[3];     // lit, reflection, transmission entries of this block
    __shared__ uint32_t sh_base[2];    // block base in the lit / next-level queues
    __shared__ uint32_t sh_drop;       // the next level's queue is full: this block's children are dropped (frame void)
    // grid-stride over the level: the launch is sized by the queue's capacity
    for (uint32_t base = blockIdx.x * blockDim.x; base < n_level; base += gridDim.x * blockDim.x) {
    const uint32_t i = base + threadIdx.x;
    const bool active = i < n_level;
    bool want_lit = false, want_refl = false, want_trans = false;
    Ray ray, refl, trans;
    D3 hp = d3(0, 0, 0), n = d3(0, 0, 0);
    uint32_t body = kNoBody, kind = NODE_MISS;
    float4 na = make_float4(s.default_color[0], s.default_color[1], s.default_color[2], 0.0f);
    float transparency = 0.0f;
    C3 bc = c3(0, 0, 0);
    if (active) {
        body = lb.hit_body[i];
        if (body != kNoBody) {
            ray = load_ray(lb.cur, i);
            hp = ray.o + ray.d * lb.hit_t[i];                       // rendering.rs:81
            n = surface_normal(s, body, hp, ctr);                  // :83
            const BodyMat &m = s.mat[body];
            bc = body_color_at(s, body, hp);
            if (m.surface == RG_SURFACE_REFRACTIVE) {              // :95-117
                kind = NODE_REFRACTIVE;
                float kr = (float)fresnel(ray.d, n, m.p0);
                na = make_float4(bc.r, bc.g, bc.b, kr);
                transparency = m.p1;
                if (kr < 1.0f) {
                    if (create_transmission(n, ray.d, hp, kShadowBias, m.p0, trans)) want_trans = lb.can_spawn != 0;
                    else atomicAdd(&ctr->err_trans, 1ull);         // :106 unwrap() on None
                }
                refl = create_reflection(n, ray.d, hp);
                want_refl = lb.can_spawn != 0;
            } else {
                want_lit = true;                                   // :87 / :89 shade_diffuse
                if (m.surface == RG_SURFACE_REFLECTING) {
                    kind = NODE_REFLECTING;
                    na.w = m.p0;
                    refl = create_reflection(n, ray.d, hp);
                    want_refl = lb.can_spawn != 0;
                } else {
                    kind = NODE_DIFFUSE;
                }
            }
        }
    }
    // ---- queue compaction: slots by warp ballot + popc, warps ranked inside the block through
    // shared-memory counters, ONE global atomic per block per queue (the per-warp version spent
    // half of this kernel serialised on three L2 addresses).
    if (threadIdx.x < 3) sh_cnt[threadIdx.x] = 0;
    __syncthreads();
    const uint32_t m_lit = __ballot_sync(0xffffffffu, want_lit);
    const uint32_t m_refl = __ballot_sync(0xffffffffu, want_refl);
    const uint32_t m_trans = __ballot_sync(0xffffffffu, want_trans);
    uint32_t w_lit = 0, w_next = 0;
    if (lane == 0) {
        if (m_lit) w_lit = atomicAdd(&sh_cnt[0], (unsigned)__popc(m_lit));
        // a warp's children are laid out [reflections..., transmissions...]; the block interleaves warps
        if (m_refl | m_trans) w_next = atomicAdd(&sh_cnt[1], (unsigned)(__popc(m_refl) + __popc(m_trans)));
        if (m_trans) atomicAdd(&sh_cnt[2], (unsigned)__popc(m_trans));
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        const uint32_t n_lit_b = sh_cnt[0], n_next_b = sh_cnt[1], n_trans_b = sh_cnt[2];
        sh_base[0] = n_lit_b ? atomicAdd(lb.q_lit, n_lit_b) : 0u;
        sh_drop = 0u;
        if (lb.last_enqueued) {   // depth hint: nobody will trace this level's children — they must not exist
            sh_base[1] = 0u;
            sh_drop = 1u;
            if (n_next_b) ctr->deeper = 1u;   // the host repeats the frame with every level
        } else {
            sh_base[1] = n_next_b ? atomicAdd(lb.q_next, n_next_b) : 0u;
            if (n_next_b && (uint64_t)sh_base[1] + n_next_b > lb.cap_next) {   // the host repeats the frame with larger queues
                sh_drop = 1u;
                atomicExch(lb.void_flag, 1u);
            }
        }
        if (n_next_b - n_trans_b) atomicAdd(&ctr->rays[2], (unsigned long long)(n_next_b - n_trans_b));
        if (n_trans_b) atomicAdd(&ctr->rays[3], (unsigned long long)n_trans_b);
        if (n_lit_b) atomicAdd(&ctr->rays[1], (unsigned long long)n_lit_b * lb.n_lights);
    }
    __syncthreads();
    if (sh_drop) { want_refl = false; want_trans = false; }
    const uint32_t base_lit = sh_base[0] + __shfl_sync(0xffffffffu, w_lit, 0);
    const uint32_t base_next = sh_base[1] + __shfl_sync(0xffffffffu, w_next, 0);
    uint32_t child_refl = kChildDefault, child_trans = kChildDefault;
    // origin hints (rg_trace.cuh): every ray made here starts on `body`; if that is a sphere, run the reference's
    // test of this very ray against it now (geom[body] holds the same four doubles as the sphere list)
    const double *og = nullptr;
    uint32_t own = kHintNone;
    if (lb.hints == 1u && body != kNoBody && s.kind[body] == RG_BODY_SPHERE) {
        own = s.body_sph[body];
        og = s.geom + 8 * (size_t)body;
    }
    if (want_refl) {
        child_refl = base_next + __popc(m_refl & lt);
        store_ray(lb.next, child_refl, refl);
        if (lb.hints) lb.next.hint[child_refl] = path_origin_hint(og, own, refl);
    }
    if (want_trans) {
        child_trans = base_next + __popc(m_refl) + __popc(m_trans & lt);
        store_ray(lb.next, child_trans, trans);
        if (lb.hints) lb.next.hint[child_trans] = path_origin_hint(og, own, trans);
    }
    if (want_lit) {
        // shade_diffuse's per-light setup of the lights in `s` (all of them, or the first chunk).  (Doing this warp-cooperatively — one (hit, light) pair per lane instead of a
        // per-light loop in the ~third of the lanes that are lit — was measured: no gain once the kernel
        // runs at 64 registers; it waits on gathers, not on issue slots.  Likewise partitioning a block's rays
        // into misses / refractive hits / lit hits so that every warp runs one path: 18.83 vs 18.93 ms.)
        const uint32_t j = base_lit + __popc(m_lit & lt);
        lb.lit_node[j] = i;
        lb.lit_bc[j] = make_float4(bc.r, bc.g, bc.b, s.mat[body].albedo);
        if (lb.lit_geo.a) {   // more light chunks follow: keep what k_shadow_rays needs (the path side reuses hit_t / hit_body)
            Ray g;
            g.o = hp;
            g.d = n;
            store_ray(lb.lit_geo, j, g);
            lb.lit_geo.hint[j] = body;
        }
        for (uint32_t l = 0; l < s.n_lights; ++l) shadow_ray_setup(lb, l * lb.shadow_sl + j * lb.shadow_sj, s.lights[l], hp, n, og, own);
    }
    if (active) {
        lb.node_a[i] = na;
        lb.node_b[i] = make_uint4(child_refl, child_trans, kind, __float_as_uint(transparency));
    }
    }   // grid-stride loop
}

// Shadow rays of a light chunk after the first (scenes with more than kLightChunk lights), from the lit-hit geometry
// k_shade kept: one thread per (light of the chunk, lit hit), light-major like the queue, so that neighbouring threads
// store neighbouring slots of one light's segment.  `s` holds the chunk's lights.  Block 0 rearms the level's
// shadow-trace counter for this chunk's trace: the previous chunk's trace, earlier on the same stream, used it up.
__global__ void __launch_bounds__(256) k_shadow_rays(const DScene s, const LevelBuffers lb, unsigned int *fetch_shadow) {
    if (blockIdx.x == 0 && threadIdx.x == 0) *fetch_shadow = 0u;
    const uint32_t n_lit = level_size(lb.cap, lb.q_lit, lb.void_flag);
    const uint32_t n = n_lit * s.n_lights;   // <= cap x kLightChunk < 2^31 (plan_batch_dev)
    for (uint32_t t = blockIdx.x * blockDim.x + threadIdx.x; t < n; t += gridDim.x * blockDim.x) {
        const uint32_t l = t / n_lit, j = t - l * n_lit;
        const Ray g = load_ray(lb.lit_geo, j);   // o = hit point, d = normal
        const uint32_t body = lb.lit_geo.hint[j];
        const double *og = nullptr;
        uint32_t own = kHintNone;
        if (lb.hints == 1u && s.kind[body] == RG_BODY_SPHERE) {   // as in k_shade
            own = s.body_sph[body];
            og = s.geom + 8 * (size_t)body;
        }
        shadow_ray_setup(lb, l * lb.shadow_sl + j * lb.shadow_sj, s.lights[l], g.o, g.d, og, own);
    }
}

// rendering.rs:140,157-171: final_color accumulates light by light, in scene order, then clamps.  With several light
// chunks (`s` holds one), `acc_in` (nullptr: the first chunk, start from 0) is the sum of the chunks before, and
// `acc_out` (nullptr: the last chunk, clamp and write the node) receives the sum so far.  An f32 stored and loaded
// keeps its bits and the chunks run in light order, so the sum is ((0 + t0) + t1) + ..., the reference's.
__global__ void __launch_bounds__(256) k_diffuse(const DScene s, const float4 *__restrict__ lit_bc,
                                                 const uint32_t *__restrict__ lit_node, const float2 *__restrict__ s_ab,
                                                 const uint8_t *__restrict__ s_lit, float4 *node_a, uint32_t cap,
                                                 uint32_t shadow_sl, uint32_t shadow_sj, const unsigned int *n_lit_dev,
                                                 const unsigned int *void_flag, const float4 *acc_in, float4 *acc_out) {
    const uint32_t n_lit = level_size(cap, n_lit_dev, void_flag);
    for (uint32_t j = blockIdx.x * blockDim.x + threadIdx.x; j < n_lit; j += gridDim.x * blockDim.x) {
    const float4 b = lit_bc[j];
    const C3 bc = c3(b.x, b.y, b.z);
    C3 fin = c3(0.0f, 0.0f, 0.0f);
    if (acc_in) { const float4 c = acc_in[j]; fin = c3(c.x, c.y, c.z); }
    for (uint32_t l = 0; l < s.n_lights; ++l) {
        const uint32_t k = l * shadow_sl + j * shadow_sj;
        const float2 ab = s_ab[k];
        fin = fin + light_term(bc, s.lights[l], b.w, ab.x, ab.y, s_lit[k] != 0);
    }
    if (acc_out) { acc_out[j] = make_float4(fin.r, fin.g, fin.b, 0.0f); continue; }
    fin = clamp01(fin);
    const uint32_t node = lit_node[j];
    float4 a = node_a[node];
    a.x = fin.r; a.y = fin.g; a.z = fin.b;
    node_a[node] = a;
    }
}

// get_color's combination of child colours (rendering.rs:88-93, 112-116), one level at a time,
// deepest level first.  `child_a` is the (already final) level below.
__global__ void __launch_bounds__(256) k_combine(const DScene s, float4 *node_a, const uint4 *__restrict__ node_b,
                                                 const float4 *__restrict__ child_a, uint32_t cap,
                                                 const unsigned int *n_dev, const unsigned int *void_flag) {
    const uint32_t n = level_size(cap, n_dev, void_flag);
    const C3 dflt = c3(s.default_color[0], s.default_color[1], s.default_color[2]);
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
    const uint4 b = node_b[i];
    if (b.z != NODE_REFLECTING && b.z != NODE_REFRACTIVE) continue;
    float4 a = node_a[i];
    C3 refl = dflt, refr = dflt;
    if (b.x != kChildDefault) { float4 c = child_a[b.x]; refl = c3(c.x, c.y, c.z); }
    if (b.y != kChildDefault) { float4 c = child_a[b.y]; refr = c3(c.x, c.y, c.z); }
    C3 out;
    if (b.z == NODE_REFLECTING) {
        out = (c3(a.x, a.y, a.z) * (1.0f - a.w)) + (refl * a.w);
    } else {
        C3 col = (refl * a.w) + (refr * (1.0f - a.w));
        out = (col * __uint_as_float(b.w)) * c3(a.x, a.y, a.z);
    }
    a.x = out.r; a.y = out.g; a.z = out.b;
    node_a[i] = a;
    }
}

__device__ __forceinline__ uint32_t pack_rgba(uchar4 c) {
    return (uint32_t)c.x | ((uint32_t)c.y << 8) | ((uint32_t)c.z << 16) | ((uint32_t)c.w << 24);
}

// Color::rgba (color.rs:32-37): 4 pixels of a row per thread, one 128-bit store; the level-0 nodes are
// gathered through the queue order (PixelOrder).
__global__ void __launch_bounds__(256) k_quantise(const float4 *__restrict__ node_a, uchar4 *out, uint32_t npix, const PixelOrder po) {
    const uint32_t p4 = (blockIdx.x * blockDim.x + threadIdx.x) * 4u;   // first of 4 pixels, row-major in the batch
    if (p4 >= npix) return;
    const uint32_t r = p4 / po.width, x = p4 - r * po.width;
    if (x + 4u <= po.width && (reinterpret_cast<uintptr_t>(out + p4) & 15u) == 0) {
        uint32_t p[4];   // one packed RGBA8 word per pixel, stored as one 128-bit word
#pragma unroll
        for (uint32_t k = 0; k < 4; ++k) { float4 a = node_a[po.index(x + k, r)]; p[k] = pack_rgba(quantise(c3(a.x, a.y, a.z))); }
        *reinterpret_cast<uint4 *>(out + p4) = make_uint4(p[0], p[1], p[2], p[3]);
    } else {
        for (uint32_t k = p4; k < npix && k < p4 + 4u; ++k) {
            const uint32_t rk = k / po.width;
            float4 a = node_a[po.index(k - rk * po.width, rk)];
            out[k] = quantise(c3(a.x, a.y, a.z));
        }
    }
}

// RenderedPixel.color (rendering.rs:18-22,59-65): the UNQUANTISED f32 colour of every pixel, 3 floats per pixel
// row-major in the batch — what Scene::streaming_render sends down its channel.
__global__ void __launch_bounds__(256) k_export_f32(const float4 *__restrict__ node_a, float *out, uint32_t npix, const PixelOrder po) {
    const uint32_t p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= npix) return;
    const uint32_t r = p / po.width, x = p - r * po.width;
    const float4 a = node_a[po.index(x, r)];
    out[3 * (size_t)p] = a.x;
    out[3 * (size_t)p + 1] = a.y;
    out[3 * (size_t)p + 2] = a.z;
}

// The same, fused with the gather of a sharded frame: batch row r belongs to image row
// rows[row0 + r] and is stored at its place in a FULL frame that may live in another
// GPU's memory (a CUDA-IPC mapping written over NVLink) or in pinned host memory: the "collective"
// of this path is these stores, and nothing is left to exchange when the kernel retires.
__global__ void __launch_bounds__(256) k_quantise_scatter(const float4 *__restrict__ node_a, uchar4 *frame, uint32_t npix,
                                                          const uint32_t *__restrict__ rows, uint32_t row0, const PixelOrder po) {
    const uint32_t p4 = (blockIdx.x * blockDim.x + threadIdx.x) * 4u;
    if (p4 >= npix) return;
    const uint32_t width = po.width;
    const uint32_t r = p4 / width, x = p4 - r * width;
    if (x + 4u <= width) {
        uchar4 *dst = frame + (size_t)rows[row0 + r] * width + x;
        uint32_t p[4];
#pragma unroll
        for (uint32_t k = 0; k < 4; ++k) { float4 a = node_a[po.index(x + k, r)]; p[k] = pack_rgba(quantise(c3(a.x, a.y, a.z))); }
        if ((reinterpret_cast<uintptr_t>(dst) & 15u) == 0) *reinterpret_cast<uint4 *>(dst) = make_uint4(p[0], p[1], p[2], p[3]);
        else { uint32_t *d32 = reinterpret_cast<uint32_t *>(dst); d32[0] = p[0]; d32[1] = p[1]; d32[2] = p[2]; d32[3] = p[3]; }
    } else {
        for (uint32_t k = p4; k < npix && k < p4 + 4u; ++k) {
            const uint32_t rk = k / width, xk = k - rk * width;
            float4 a = node_a[po.index(xk, rk)];
            frame[(size_t)rows[row0 + rk] * width + xk] = quantise(c3(a.x, a.y, a.z));
        }
    }
}

// RG_OPT_SUPERSAMPLE = n > 1: the last kernel of a batch, in place of k_quantise / k_quantise_scatter / k_export_f32.
// One thread per output pixel averages its n x n samples as include/raingun_b200.h specifies: per channel s = 0, then
// s + sample in sub-row, sub-column order, then s / (n n) rounded to nearest (a sum without products: nothing for
// FMA contraction to fuse).  `po` spans the batch's sample rows; sample (X, Y) is f32 RGB at src + stride * po.index(X, Y)
// (the level-0 nodes: stride 4, queue order; the megakernel's f32 output: stride 3, row-major = strip 1).  Scatter:
// output row r of the batch is image row rows[row0 + r n] / n (the row list holds n sample rows per listed row).
template <OutKind K>
__global__ void __launch_bounds__(256) k_resolve_ss(const float *__restrict__ src, uint32_t stride, const PixelOrder po, uint32_t n,
                                                    uint32_t npix, const uint32_t *__restrict__ rows, uint32_t row0, void *out) {
    const uint32_t p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= npix) return;
    const uint32_t w = po.width / n, r = p / w, x = p - r * w;
    float s[3] = {0.0f, 0.0f, 0.0f};
    for (uint32_t j = 0; j < n; ++j)
        for (uint32_t i = 0; i < n; ++i) {
            const float *c = src + (size_t)stride * po.index(n * x + i, n * r + j);
            float v[3];
            if (stride == 4) { const float4 a = *reinterpret_cast<const float4 *>(c); v[0] = a.x; v[1] = a.y; v[2] = a.z; }
            else { v[0] = c[0]; v[1] = c[1]; v[2] = c[2]; }
#pragma unroll
            for (int k = 0; k < 3; ++k) s[k] = __fadd_rn(s[k], v[k]);
        }
    const float nn = (float)(n * n);
    const C3 avg = c3(__fdiv_rn(s[0], nn), __fdiv_rn(s[1], nn), __fdiv_rn(s[2], nn));
    if constexpr (K == OutKind::F32) {
        float *o = static_cast<float *>(out) + 3 * (size_t)p;
        o[0] = avg.r; o[1] = avg.g; o[2] = avg.b;
    } else if constexpr (K == OutKind::Rgba8Scatter) {
        static_cast<uchar4 *>(out)[(size_t)(rows[row0 + r * n] / n) * w + x] = quantise(avg);
    } else {
        static_cast<uchar4 *>(out)[p] = quantise(avg);
    }
}

int launch_resolve(OutKind kind, const float *src, uint32_t stride, uint32_t strip, uint32_t n, uint32_t width, uint32_t out_rows,
                   const uint32_t *d_rows, uint32_t row0, void *out, cudaStream_t stream) {
    const uint32_t npix = out_rows * width;
    if (npix == 0) return RG_OK;
    PixelOrder po;
    po.width = n * width;
    po.rows = n * out_rows;
    po.strip = strip;
    const unsigned blocks = (npix + 255) / 256;
    if (kind == OutKind::F32) k_resolve_ss<OutKind::F32><<<blocks, 256, 0, stream>>>(src, stride, po, n, npix, d_rows, row0, out);
    else if (kind == OutKind::Rgba8Scatter) k_resolve_ss<OutKind::Rgba8Scatter><<<blocks, 256, 0, stream>>>(src, stride, po, n, npix, d_rows, row0, out);
    else k_resolve_ss<OutKind::Rgba8><<<blocks, 256, 0, stream>>>(src, stride, po, n, npix, d_rows, row0, out);
    RG_CUDA(cudaGetLastError());
    return RG_OK;
}

// RG_OPT_VERIFY_CULL >= 2: re-trace every ray of a queue with the verbatim reference scan and
// count results that differ from what the production trace kernel wrote (must be 0).
template <bool ANY>
__global__ void __launch_bounds__(128) k_verify_trace(const DScene s, const TraceArgs a, int level) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= ray_count(a)) return;
    const uint32_t pi = phys_index(segment_length(a), a.seg_stride, i);
    const Ray ray = load_ray(a.q, pi);
    const Nearest h = trace_exact_all(s, ray, a.ctr);
    bool bad;
    if (ANY) {
        const bool lit = !h.found() || h.t > a.tmax[pi];
        bad = (a.out_lit[pi] != 0) != lit;
    } else {
        bad = a.out_body[pi] != h.body || (h.found() && a.out_t[pi] != h.t);
    }
    if (bad) {
        unsigned long long k = atomicAdd(&a.ctr->cull_unsound, 1ull);
        if (k < 8)
            printf("verify: level %d %s ray %u o=(%.17g,%.17g,%.17g) d=(%.17g,%.17g,%.17g) exact=(%.17g,%u) got=(%.17g,%u)\n", level,
                   ANY ? "shadow" : "path", i, ray.o.x, ray.o.y, ray.o.z, ray.d.x, ray.d.y, ray.d.z, h.t, h.body,
                   ANY ? (double)a.out_lit[pi] : a.out_t[pi], ANY ? 0u : a.out_body[pi]);
    }
}

// shadow-queue order: light-major (one segment per light: neighbouring lanes trace neighbouring hits towards
// the same light; default) or hit-major (the L rays of a hit adjacent; RG_SHADOW_LIGHT_MAJOR=0, for comparison)
static bool shadow_light_major() {
    static const bool v = [] { const char *e = getenv("RG_SHADOW_LIGHT_MAJOR"); return !e || atoi(e) != 0; }();
    return v;
}

// strip height of the level-0 queue order (RG_STRIP_ROWS for tuning; 1 = plain row-major)
static PixelOrder pixel_order(uint32_t width, uint32_t rows) {
    static const uint32_t strip = [] { const char *e = getenv("RG_STRIP_ROWS"); const int v = e ? atoi(e) : 4; return (uint32_t)(v >= 1 && v <= 32 ? v : 4); }();
    PixelOrder po;
    po.width = width;
    po.rows = rows;
    po.strip = strip;
    return po;
}

static RayQueue make_queue(DeviceBuffer &b, size_t cap) {
    RayQueue q;
    q.a = b.as<double2>();
    q.b = q.a + cap;
    q.c = q.b + cap;
    q.hint = reinterpret_cast<uint32_t *>(q.c + cap);
    return q;
}

struct EventPool {
    std::vector<cudaEvent_t> &ev;   // owned by the scratch (kept across frames)
    size_t used = 0;
    unsigned flags;
    explicit EventPool(std::vector<cudaEvent_t> &store, unsigned f = cudaEventDefault) : ev(store), flags(f) {}
    cudaEvent_t get() {
        if (used == ev.size()) {
            cudaEvent_t e;
            if (cudaEventCreateWithFlags(&e, flags) != cudaSuccess) return nullptr;
            ev.push_back(e);
        }
        return ev[used++];
    }
};

constexpr int kResidentSmemMax = 232448 - 1024;   // opt-in shared memory of one CTA on sm_100 (227 KB), minus the static part

// Can k_trace_brute_resident hold this scene's cull records (plus its per-warp scratch) in the
// shared memory one CTA may use?  (RG_BRUTE_RESIDENT=0 forces the streaming kernel.)
static bool brute_resident_fits(const rg_scene *sc) {
    static const bool enabled = [] { const char *e = getenv("RG_BRUTE_RESIDENT"); return !e || atoi(e) != 0; }();
    if (!enabled || sc->ds.n_spheres == 0) return false;
    const uint32_t n_records = (uint32_t)(((size_t)sc->ds.n_spheres + 3) / 4 * 4);
    return resident_smem_bytes(n_records, 4, 20) <= (size_t)kResidentSmemMax;
}

template <bool ANY>
static int launch_trace(rg_scene *sc, const TraceArgs &ta, bool use_grid, cudaStream_t stream) {
    if (ta.n == 0) return RG_OK;
    if (use_grid) {
        // persistent warps: enough blocks to fill the chip, each pulling rays from ta.fetch
        const unsigned want = (ta.n + kGridTraceThreads - 1) / kGridTraceThreads;
        static const int bps = [] { const char *e = getenv("RG_GRID_BPS"); return e ? atoi(e) : RG_GRID_MINB; }();
        static const int t_refill = [] { const char *e = getenv("RG_GRID_REFILL"); return e ? atoi(e) : kGridRefill; }();
        static const int t_quorum = [] { const char *e = getenv("RG_GRID_QUORUM"); return e ? atoi(e) : kGridExactQuorum; }();
        static const int t_burst = [] { const char *e = getenv("RG_GRID_BURST"); return e ? atoi(e) : kGridScanBurst; }();
        const unsigned blocks = std::min<unsigned>(want, (unsigned)(sc->sm_count * bps));
        TraceArgs tuned = ta;
        tuned.g_refill = t_refill; tuned.g_quorum = t_quorum; tuned.g_burst = t_burst;
        if (sc->gp.n_proxies) {   // boxes / disks in the grid
            if (sc->trace_stats) k_trace_grid<ANY, true, true><<<blocks, kGridTraceThreads, 0, stream>>>(sc->ds, tuned, sc->gp);
            else k_trace_grid<ANY, false, true><<<blocks, kGridTraceThreads, 0, stream>>>(sc->ds, tuned, sc->gp);
        } else {
            if (sc->trace_stats) k_trace_grid<ANY, true><<<blocks, kGridTraceThreads, 0, stream>>>(sc->ds, tuned, sc->gp);
            else k_trace_grid<ANY, false><<<blocks, kGridTraceThreads, 0, stream>>>(sc->ds, tuned, sc->gp);
        }
    } else if (brute_resident_fits(sc) && ta.n >= (uint32_t)sc->sm_count * 64u * 32u) {
        // the whole cull array fits in one SM's shared memory: one persistent CTA per SM, warps
        // pull ray tiles from a counter and never meet at a barrier again (rg_trace.cuh)
        static const int variant = [] { const char *e = getenv("RG_RESIDENT_VARIANT"); return e ? atoi(e) : 0; }();
        const uint32_t n_records = (uint32_t)(((size_t)sc->ds.n_spheres + 3) / 4 * 4);
#define RG_LAUNCH_RESIDENT(R_, U_, T_, PF_)                                                                                   \
    do {                                                                                                                      \
        static std::atomic<uint64_t> attr_set{0}; /* per device: the attribute belongs to the device's copy of the function */ \
        const uint64_t dev_bit = 1ull << (sc->device & 63);                                                                   \
        if (!(attr_set.load() & dev_bit)) {                                                                                   \
            RG_CUDA(cudaFuncSetAttribute(k_trace_brute_resident<ANY, R_, U_, T_, PF_>, cudaFuncAttributeMaxDynamicSharedMemorySize, \
                                         kResidentSmemMax));                                                                  \
            attr_set.fetch_or(dev_bit);                                                                                       \
        }                                                                                                                     \
        const uint64_t tiles = ((uint64_t)ta.n + 32 * R_ - 1) / (32 * R_);                                                     \
        const unsigned blocks = (unsigned)std::min<uint64_t>((uint64_t)sc->sm_count, (tiles + (T_ / 32) - 1) / (T_ / 32));      \
        k_trace_brute_resident<ANY, R_, U_, T_, PF_><<<blocks, T_, resident_smem_bytes(n_records, R_, T_ / 32), stream>>>(sc->ds, ta, n_records); \
    } while (0)
        // Measured on C4 / C3 (ms per 4K brute-force frame) with the software-pipelined loop of round 2 (rg_trace.cuh):
        // R=4,U=2,512 thr 310.0 / 14.3;  R=3,U=2: 512 thr 313.4 / 17.6, 576 thr 322.1 / 9.1, 608 thr 322.1 / 10.1,
        // 640 thr 326.7 / 9.8;  R=2,U=4,512 thr 353.5.  (The loop before it, R=3,U=2,640 thr: 373.5 / 9.3; the streaming
        // kernel 394.7.)  More rays per lane amortise the record loads and the vote over more
        // FFMA2s and win on long scans; short scans (C3: 500 groups per tile) want more warps to hide the tile prologue.
        switch (variant ? variant : (sc->ds.n_spheres >= 4096u ? 1 : 4)) {
            case 1: RG_LAUNCH_RESIDENT(4, 2, 512, true); break;
            case 2: RG_LAUNCH_RESIDENT(2, 4, 512, true); break;
            case 3: RG_LAUNCH_RESIDENT(3, 2, 608, true); break;
            case 4: RG_LAUNCH_RESIDENT(3, 2, 576, true); break;
            case 5: RG_LAUNCH_RESIDENT(3, 2, 512, true); break;
            default: RG_LAUNCH_RESIDENT(3, 2, 640, true); break;
        }
#undef RG_LAUNCH_RESIDENT
    } else {
        // register tiling R: 4 rays per thread when there is enough work to fill the chip
        const uint64_t full = (uint64_t)sc->sm_count * 2 * kTraceThreads;
        static const int variant = [] { const char *e = getenv("RG_BRUTE_VARIANT"); return e ? atoi(e) : 0; }();
#define RG_LAUNCH_BRUTE(R_, U_, M_) \
    k_trace_brute<ANY, R_, U_, M_><<<(ta.n + R_ * kTraceThreads - 1) / (R_ * kTraceThreads), kTraceThreads, 0, stream>>>(sc->ds, ta)
        if (ta.n >= full * 4 * 2) {
            switch (variant) {
                case 1: RG_LAUNCH_BRUTE(4, 4, 2); break;
                case 2: RG_LAUNCH_BRUTE(2, 2, 3); break;
                case 3: RG_LAUNCH_BRUTE(2, 4, 3); break;
                case 4: RG_LAUNCH_BRUTE(2, 4, 4); break;
                case 5: RG_LAUNCH_BRUTE(2, 2, 4); break;
                case 6: RG_LAUNCH_BRUTE(4, 2, 3); break;
                case 7: RG_LAUNCH_BRUTE(4, 4, 3); break;
                case 8: RG_LAUNCH_BRUTE(4, 2, 2); break;
                case 9: RG_LAUNCH_BRUTE(2, 4, 4); break;
                default: RG_LAUNCH_BRUTE(4, 2, 2); break;   // with round 2's loop (C4, streaming kernel only): 366 ms; (2,4,3) 375, (2,4,4) 386, (4,4,2) 405
            }
        } else if (ta.n >= full * 2 * 2) {
            RG_LAUNCH_BRUTE(2, 4, 4);
        } else {
            RG_LAUNCH_BRUTE(1, 2, 3);
        }
#undef RG_LAUNCH_BRUTE
    }
    RG_CUDA(cudaGetLastError());
    return RG_OK;
}

// ---- the host-free level loop ------------------------------------------------------------------
// render_image is one call with no per-depth host involvement (rendering.rs:24-38).  Here the
// whole batch — every level's trace, shade, shadow trace, diffuse, then combine and quantise —
// is ENQUEUED without a single host synchronisation: each launch reads its level's size from
// DCounters::lvl[] (written by the level above) and is sized for the queue's CAPACITY; persistent
// / grid-stride kernels make surplus blocks free.  Queue capacities are fixed up front:
//     cap[0] = pixels,   cap[d] = min(2 cap[d-1], rg_scene::level_growth * pixels)
// (a hit spawns <= 2 rays, so 2 cap[d-1] is exact; real scenes stay far below the initial growth of 2x).
// A level that would outgrow its queue sets DCounters::overflow, every later launch of the frame then
// does nothing, and the host doubles the scene's level_growth and repeats the render (sticky per scene).
// Once level_growth >= 2^(levels-1) the clamp is inactive and no level can overflow, so a scene repeats
// at most levels - 2 frames over its lifetime.
// The launch sequence depends only on (pixels, depth, lights, capacities, buffers), so it can be
// captured once into a CUDA graph and replayed per frame (RG_OPT_GRAPH).
struct DevPlan {
    uint32_t levels = 0;                    // levels 0 .. levels-1 are enqueued
    uint32_t cap[RG_MAX_DEPTH + 2] = {0};
};

static int plan_batch_dev(rg_scene *sc, uint32_t npix, DevPlan &plan, bool use_grid) {
    const DScene &ds = sc->ds;
    const uint32_t L = ds.n_lights;
    WavefrontScratch &wf = sc->wf;
    // Levels to enqueue: all the recursion depth allows, or — once a frame of this scene has shown how deep
    // its ray tree really goes — just those (a shallow scene with the default depth of 10 would otherwise pay
    // for dozens of empty launches).  The frame is checked afterwards: the last enqueued level must not have
    // emitted children (wavefront_render), else it is repeated with every level.
    plan.levels = std::max<uint32_t>(ds.max_depth, 1u);
    if (sc->depth_hint && sc->depth_hint < plan.levels) plan.levels = sc->depth_hint;
    const uint32_t C = std::min(L, kLightChunk);   // lights per chunk: the shadow queues hold one chunk at a time
    uint64_t cap_max[2] = {0, 0}, cap_all = 0;
    for (uint32_t d = 0; d < plan.levels; ++d) {
        const uint64_t c = d == 0 ? npix : std::min<uint64_t>(2ull * plan.cap[d - 1], (uint64_t)sc->level_growth * npix);
        if (c > 0x7FFFFFFFull || c * std::max<uint32_t>(C, 1u) > 0x7FFFFFFFull) {
            set_error("level %u could hold more than 2^31 rays; use a smaller batch", d);
            return RG_E_NOMEM;
        }
        plan.cap[d] = (uint32_t)c;
        cap_max[d & 1] = std::max(cap_max[d & 1], c);
        cap_all = std::max(cap_all, c);
    }
    int rc;
    if (wf.nodes.size() < plan.levels) wf.nodes.resize(plan.levels);
    for (uint32_t d = 0; d < plan.levels; ++d)
        if ((rc = wf.nodes[d].reserve((size_t)plan.cap[d] * 32))) return rc;
    if ((rc = wf.hit_t.reserve((size_t)cap_all * 8))) return rc;
    if ((rc = wf.hit_body.reserve((size_t)cap_all * 4))) return rc;
    for (int p = 0; p < 2; ++p) {
        const uint64_t c = std::max<uint64_t>(cap_max[p], 1), sc_ = std::max<uint64_t>(c * C, 1);
        if ((rc = wf.ray[p].reserve((size_t)c * kRayBytes))) return rc;
        if ((rc = wf.sray[p].reserve((size_t)sc_ * kRayBytes))) return rc;
        if ((rc = wf.s_tmax[p].reserve((size_t)sc_ * 8))) return rc;
        if ((rc = wf.s_ab[p].reserve((size_t)sc_ * 8))) return rc;
        if ((rc = wf.s_lit[p].reserve((size_t)sc_))) return rc;
        if ((rc = wf.lit_bc[p].reserve((size_t)c * 16))) return rc;
        if ((rc = wf.lit_node[p].reserve((size_t)c * 4))) return rc;
        if (L > kLightChunk) {   // the lit hits' geometry and partial sums outlive k_shade by the later chunks
            if ((rc = wf.lit_geo[p].reserve((size_t)c * kRayBytes))) return rc;
            if ((rc = wf.lit_acc[p].reserve((size_t)c * 16))) return rc;
        }
    }
    return RG_OK;
}

// The DScene of light chunk c: lights [c * kLightChunk, ...) inline, the rest of the struct as the scene's.
static DScene chunk_scene(const rg_scene *sc, uint32_t c) {
    DScene cs = sc->ds;
    const uint32_t first = c * kLightChunk;
    cs.n_lights = std::min<uint32_t>(kLightChunk, (uint32_t)sc->lights.size() - first);
    std::copy(sc->lights.begin() + first, sc->lights.begin() + first + cs.n_lights, cs.lights);
    return cs;
}

// Enqueues one batch.  No allocation, no synchronisation, no host read: legal inside a stream capture.
// `timed` = record CUDA events around the trace launches (not possible while capturing).
static int enqueue_batch_dev(rg_scene *sc, const DevPlan &plan, uint32_t width, uint32_t height, uint32_t y0, uint32_t npix,
                             const uint32_t *d_rows, OutKind kind, uchar4 *d_out, cudaStream_t stream, rg_stats *st, bool use_grid,
                             EventPool *events, EventPool &sync_events,
                             std::vector<std::pair<cudaEvent_t, cudaEvent_t>> *trace_spans) {
    const DScene &ds = sc->ds;
    const uint32_t L = ds.n_lights;
    WavefrontScratch &wf = sc->wf;
    DCounters *dc = sc->d_counters;
    int rc;
    // enough blocks to fill the chip several times over; grid-stride loops do the rest
    const unsigned max_blocks = (unsigned)sc->sm_count * 16u;
    auto blocks = [&](uint64_t n) { return (unsigned)std::max<uint64_t>(1, std::min<uint64_t>((n + 255) / 256, max_blocks)); };
    // Two-stream schedule.  The shadow side of level d (any-hit trace + k_diffuse) depends only on
    // k_shade(d); the path side of level d+1 (nearest trace + k_shade) depends only on k_shade(d)
    // too.  With the grid tracer both are latency-bound persistent kernels with long tails, so the
    // shadow side runs on an auxiliary stream, concurrently with the next level's path side; its
    // buffers exist twice (level parity) and k_shade(d+2) waits for the shadow side of level d.
    // The brute-force tracer fills the chip on its own and keeps the single-stream order (its
    // per-kernel times are also what the roofline figure is computed from).  (A second auxiliary stream
    // for the odd levels, so that two shadow sides overlap as well, was measured: no gain at any batch size.)
    const bool overlap = L > 0 && (sc->overlap == 2 || (sc->overlap == 0 && use_grid));
    cudaStream_t aux = overlap ? wf.aux : stream;
    cudaEvent_t shadow_done[2] = {nullptr, nullptr};
    // Light chunks.  A scene with more than kLightChunk lights shades them kLightChunk at a time: k_shade sets up the
    // first chunk's shadow rays and keeps each lit hit's geometry; every later chunk gets its rays from k_shadow_rays.
    // Each chunk is traced and summed by k_diffuse into a per-hit f32 accumulator; the last chunk clamps.  Each chunk's
    // launches take a DScene holding that chunk's lights, so the kernels read them from the constant bank as always.
    const bool chunked = L > kLightChunk;
    const uint32_t n_chunks = chunked ? (L + kLightChunk - 1) / kLightChunk : 1u;
    const uint32_t C = std::min(L, kLightChunk);
    std::vector<DScene> chunks;
    if (chunked)
        for (uint32_t c = 0; c < n_chunks; ++c) chunks.push_back(chunk_scene(sc, c));

    RG_CUDA(cudaMemsetAsync(dc->lvl, 0, sizeof(dc->lvl), stream));
    RayQueue cur = make_queue(wf.ray[0], plan.cap[0]);
    const PixelOrder po = pixel_order(width, npix / width);
    k_generate<<<(npix + 255) / 256, 256, 0, stream>>>(ds, cur, width, height, y0, npix, d_rows, &dc->lvl[0].n, po);
    RG_CUDA(cudaGetLastError());
    st->gpu_launches++;
    st->rays_primary += npix;

    for (uint32_t d = 0; d < plan.levels; ++d) {
        const bool can_spawn = d + 1 < ds.max_depth;
        const uint32_t cap = plan.cap[d], cap_next = can_spawn ? plan.cap[d + 1] : 0u;
        const int p = overlap ? (int)(d & 1u) : 0;
        TraceArgs ta{};
        ta.q = cur;
        ta.n = cap;
        ta.n_dev = &dc->lvl[d].n;
        ta.n_mul = 1;
        ta.void_flag = &dc->overflow;
        ta.fetch = &dc->lvl[d].fetch;
        ta.out_t = wf.hit_t.as<double>();
        ta.out_body = wf.hit_body.as<uint32_t>();
        ta.ctr = dc;
        ta.verify = sc->verify_cull == 1;
        cudaEvent_t e0 = nullptr, e1 = nullptr;
        if (events) { e0 = events->get(); e1 = events->get(); RG_CUDA(cudaEventRecord(e0, stream)); }
        if ((rc = launch_trace<false>(sc, ta, use_grid, stream))) return rc;
        if (events) { RG_CUDA(cudaEventRecord(e1, stream)); trace_spans->emplace_back(e0, e1); }
        st->gpu_launches++;
        if (sc->verify_cull >= 2) k_verify_trace<false><<<(cap + 127) / 128, 128, 0, stream>>>(ds, ta, (int)d);

        LevelBuffers lb{};
        lb.cur = cur;
        lb.next = make_queue(wf.ray[(d + 1) & 1], std::max<uint32_t>(cap_next, 1u));
        lb.shadow = make_queue(wf.sray[p], (size_t)std::max<uint64_t>((uint64_t)cap * C, 1));
        lb.hit_t = wf.hit_t.as<double>();
        lb.hit_body = wf.hit_body.as<uint32_t>();
        lb.node_a = wf.nodes[d].as<float4>();
        lb.node_b = reinterpret_cast<uint4 *>(wf.nodes[d].as<float4>() + cap);
        lb.s_tmax = wf.s_tmax[p].as<double>();
        lb.s_ab = wf.s_ab[p].as<float2>();
        lb.lit_bc = wf.lit_bc[p].as<float4>();
        lb.lit_node = wf.lit_node[p].as<uint32_t>();
        lb.cap = cap;
        lb.n_dev = &dc->lvl[d].n;
        const bool light_major = shadow_light_major();
        lb.shadow_sl = light_major ? cap : 1u;   // one segment of `cap` slots per light, or the L rays of a hit adjacent
        lb.shadow_sj = light_major ? 1u : C;
        lb.can_spawn = can_spawn ? 1u : 0u;
        lb.q_next = &dc->lvl[d + 1].n;
        lb.q_lit = &dc->lvl[d].n_lit;
        lb.cap_next = cap_next;
        lb.void_flag = &dc->overflow;
        lb.level = d;
        lb.hints = use_grid ? (sc->origin_hints ? 1u : 2u) : 0u;
        lb.last_enqueued = (d + 1 == plan.levels && can_spawn) ? 1u : 0u;
        lb.n_lights = L;
        if (chunked) lb.lit_geo = make_queue(wf.lit_geo[p], cap);
        if (shadow_done[p]) RG_CUDA(cudaStreamWaitEvent(stream, shadow_done[p], 0));   // level d-2 still reads these buffers
        k_shade<<<blocks(cap), 256, 0, stream>>>(chunked ? chunks[0] : ds, lb, dc);
        RG_CUDA(cudaGetLastError());
        st->gpu_launches++;

        if (L && overlap) {   // shadow side, concurrent with the next level's path side
            cudaEvent_t shaded = sync_events.get();
            RG_CUDA(cudaEventRecord(shaded, stream));
            RG_CUDA(cudaStreamWaitEvent(aux, shaded, 0));
        }
        float4 *acc = chunked ? wf.lit_acc[p].as<float4>() : nullptr;
        for (uint32_t c = 0; c < n_chunks; ++c) {   // (one pass, c = 0, unless the scene has more than kLightChunk lights)
            const DScene &cs = chunked ? chunks[c] : ds;
            const uint32_t Lc = cs.n_lights;
            LevelBuffers lc = lb;
            lc.shadow_sj = light_major ? 1u : Lc;
            if (c > 0) {
                k_shadow_rays<<<blocks((uint64_t)cap * Lc), 256, 0, aux>>>(cs, lc, &dc->lvl[d].fetch_shadow);
                RG_CUDA(cudaGetLastError());
                st->gpu_launches++;
            }
            if (Lc) {
                TraceArgs sa{};
                sa.q = lc.shadow;
                sa.tmax = lc.s_tmax;
                sa.n = cap * Lc;
                sa.n_dev = &dc->lvl[d].n_lit;
                sa.n_mul = Lc;
                sa.seg_len_dev = light_major ? &dc->lvl[d].n_lit : nullptr;
                sa.seg_stride = cap;
                sa.void_flag = &dc->overflow;
                sa.fetch = &dc->lvl[d].fetch_shadow;
                sa.out_lit = wf.s_lit[p].as<uint8_t>();
                sa.ctr = dc;
                sa.verify = sc->verify_cull == 1;
                if (events) { e0 = events->get(); e1 = events->get(); RG_CUDA(cudaEventRecord(e0, aux)); }
                if ((rc = launch_trace<true>(sc, sa, use_grid, aux))) return rc;
                if (events) { RG_CUDA(cudaEventRecord(e1, aux)); trace_spans->emplace_back(e0, e1); }
                st->gpu_launches++;
                if (sc->verify_cull >= 2) k_verify_trace<true><<<(sa.n + 127) / 128, 128, 0, aux>>>(cs, sa, (int)d);
            }
            k_diffuse<<<blocks(cap), 256, 0, aux>>>(cs, lc.lit_bc, lc.lit_node, lc.s_ab, wf.s_lit[p].as<uint8_t>(), lc.node_a, cap,
                                                    lc.shadow_sl, lc.shadow_sj, &dc->lvl[d].n_lit, &dc->overflow,
                                                    c > 0 ? acc : nullptr, c + 1 < n_chunks ? acc : nullptr);
            RG_CUDA(cudaGetLastError());
            st->gpu_launches++;
        }
        if (overlap) {
            shadow_done[p] = sync_events.get();
            RG_CUDA(cudaEventRecord(shadow_done[p], aux));
        }
        cur = lb.next;
    }
    for (int q = 0; q < 2; ++q)
        if (shadow_done[q]) RG_CUDA(cudaStreamWaitEvent(stream, shadow_done[q], 0));
    for (int lvl = (int)plan.levels - 1; lvl >= 0; --lvl) {
        float4 *a = wf.nodes[lvl].as<float4>();
        const uint4 *b = reinterpret_cast<const uint4 *>(a + plan.cap[lvl]);
        const float4 *child = (uint32_t)lvl + 1 < plan.levels ? wf.nodes[lvl + 1].as<float4>() : nullptr;
        k_combine<<<blocks(plan.cap[lvl]), 256, 0, stream>>>(ds, a, b, child, plan.cap[lvl], &dc->lvl[lvl].n, &dc->overflow);
        RG_CUDA(cudaGetLastError());
        st->gpu_launches++;
    }
    if (sc->supersample > 1) {   // width, height, y0 and npix are in sample space: npix / (n n) output pixels
        const uint32_t n = sc->supersample;
        if ((rc = launch_resolve(kind, reinterpret_cast<const float *>(wf.nodes[0].as<float4>()), 4, po.strip, n, width / n,
                                 po.rows / n, d_rows, y0, d_out, stream)))
            return rc;
    } else if (kind == OutKind::F32)
        k_export_f32<<<(npix + 255) / 256, 256, 0, stream>>>(wf.nodes[0].as<float4>(), reinterpret_cast<float *>(d_out), npix, po);
    else if (kind == OutKind::Rgba8Scatter)
        k_quantise_scatter<<<(unsigned)((((uint64_t)npix + 3) / 4 + 255) / 256), 256, 0, stream>>>(wf.nodes[0].as<float4>(), d_out, npix, d_rows, y0, po);
    else
        k_quantise<<<(unsigned)((((uint64_t)npix + 3) / 4 + 255) / 256), 256, 0, stream>>>(wf.nodes[0].as<float4>(), d_out, npix, po);
    RG_CUDA(cudaGetLastError());
    st->gpu_launches++;
    st->batches++;
    return RG_OK;
}

// ---- one CUDA graph per batch shape --------------------------------------------------------------
static std::vector<uint64_t> graph_key(const rg_scene *sc, const DevPlan &plan, uint32_t width, uint32_t height, uint32_t y0,
                                       uint32_t npix, const uint32_t *d_rows, OutKind kind, const uchar4 *d_out, bool use_grid) {
    const WavefrontScratch &wf = sc->wf;
    std::vector<uint64_t> k = {width, height, y0, npix, (uint64_t)(uintptr_t)d_rows, (uint64_t)(uintptr_t)d_out,
                               (uint64_t)use_grid, (uint64_t)kind, (uint64_t)sc->ds.max_depth, (uint64_t)sc->overlap,
                               (uint64_t)sc->verify_cull, (uint64_t)sc->trace_stats | ((uint64_t)sc->origin_hints << 1), (uint64_t)plan.levels,
                               (uint64_t)sc->level_growth,    // the capacities are baked into the captured launches
                               (uint64_t)sc->supersample};    // the last launch: (n, w, h) and (1, n w, n h) share a sample space
    auto add = [&](const DeviceBuffer &b) { k.push_back((uint64_t)(uintptr_t)b.ptr); };
    add(wf.ray[0]); add(wf.ray[1]); add(wf.hit_t); add(wf.hit_body);
    for (int p = 0; p < 2; ++p) { add(wf.sray[p]); add(wf.s_tmax[p]); add(wf.s_ab[p]); add(wf.s_lit[p]); add(wf.lit_bc[p]); add(wf.lit_node[p]); }
    for (uint32_t d = 0; d < plan.levels; ++d) add(wf.nodes[d]);
    // The light-chunk count needs no entry: it is fixed by the handle's scene, and a graph dies with its scene.
    if (sc->ds.n_lights > kLightChunk)
        for (int p = 0; p < 2; ++p) { add(wf.lit_geo[p]); add(wf.lit_acc[p]); }
    return k;
}

// Replays the batch from a captured graph; captures it when its key is seen for the second time.
// Returns RG_OK with *done = false when the batch should be enqueued the ordinary way.
static int graph_batch(rg_scene *sc, const DevPlan &plan, uint32_t width, uint32_t height, uint32_t y0, uint32_t npix,
                       const uint32_t *d_rows, OutKind kind, uchar4 *d_out, cudaStream_t stream, rg_stats *st, bool use_grid,
                       EventPool &sync_events, bool *done) {
    *done = false;
    GraphCache &gc = sc->graphs;
    const std::vector<uint64_t> key = graph_key(sc, plan, width, height, y0, npix, d_rows, kind, d_out, use_grid);
    GraphEntry *hit = nullptr;
    for (auto &e : gc.entries)
        if (e.key == key) { hit = &e; break; }
    if (!hit) {
        bool seen = false;
        for (auto &k : gc.seen) seen = seen || k == key;
        if (getenv("RG_DEBUG_GRAPH")) fprintf(stderr, "[graph] dev %d key npix %u y0 %u rows %p out %p levels %u: %s\n", sc->device, npix, y0, (const void *)d_rows, (void *)d_out, plan.levels, seen ? "capture" : "first sight");
        if (!seen) {   // first time: run it eagerly (also warms every lazily initialised launch path)
            if (gc.seen.size() >= 32) gc.seen.erase(gc.seen.begin());
            gc.seen.push_back(key);
            return RG_OK;
        }
        // capture on the library's own stream (the caller's may be the legacy stream, which cannot capture)
        cudaStream_t cs = sc->stream;
        rg_stats tmp{};
        const size_t sync_used = sync_events.used;
        RG_CUDA(cudaStreamBeginCapture(cs, cudaStreamCaptureModeThreadLocal));
        const int rc = enqueue_batch_dev(sc, plan, width, height, y0, npix, d_rows, kind, d_out, cs, &tmp, use_grid, nullptr, sync_events, nullptr);
        cudaGraph_t graph = nullptr;
        const cudaError_t ce = cudaStreamEndCapture(cs, &graph);
        sync_events.used = sync_used;
        if (rc != RG_OK || ce != cudaSuccess || !graph) {
            if (getenv("RG_DEBUG_GRAPH")) fprintf(stderr, "[graph] capture failed: rc %d, cuda %d (%s)\n", rc, (int)ce, cudaGetErrorString(ce));
            if (graph) cudaGraphDestroy(graph);
            cudaGetLastError();
            sc->graph = 1;   // capture is not possible here: stay with eager launches
            return rc != RG_OK ? rc : RG_OK;
        }
        cudaGraphExec_t exec = nullptr;
        const cudaError_t ie = cudaGraphInstantiate(&exec, graph, 0);
        cudaGraphDestroy(graph);
        if (ie != cudaSuccess) { cudaGetLastError(); sc->graph = 1; return RG_OK; }
        if (gc.entries.size() >= 8) {   // evict the least recently used
            size_t lru = 0;
            for (size_t i = 1; i < gc.entries.size(); ++i)
                if (gc.entries[i].last_use < gc.entries[lru].last_use) lru = i;
            cudaGraphExecDestroy(gc.entries[lru].exec);
            gc.entries.erase(gc.entries.begin() + (long)lru);
        }
        GraphEntry e;
        e.key = key;
        e.exec = exec;
        e.launches = tmp.gpu_launches;
        gc.entries.push_back(std::move(e));
        hit = &gc.entries.back();
    }
    hit->last_use = ++gc.tick;
    RG_CUDA(cudaGraphLaunch(hit->exec, stream));
    st->gpu_launches += hit->launches;
    st->rays_primary += npix;
    st->batches++;
    st->graph_replays++;
    *done = true;
    return RG_OK;
}

int wavefront_render(rg_scene *sc, uint32_t width, uint32_t height, uint32_t y0, uint32_t y1,
                     const uint32_t *d_rows, OutKind kind, uchar4 *d_out, cudaStream_t stream, rg_stats *st) {
    const DScene &ds = sc->ds;
    bool use_grid = false;
    if (sc->accel == RG_ACCEL_GRID) use_grid = ds.grid.enabled != 0;
    else if (sc->accel == RG_ACCEL_AUTO) use_grid = ds.grid.enabled != 0 && ds.n_spheres + sc->gp.n_proxies >= 64;
    st->accel_used = use_grid ? RG_ACCEL_GRID : RG_ACCEL_BRUTE;

    EventPool events(sc->wf.events);
    EventPool sync_events(sc->wf.sync_events, cudaEventDisableTiming);
    std::vector<std::pair<cudaEvent_t, cudaEvent_t>> trace_spans;
    // RG_OPT_SUPERSAMPLE: the batches trace the (n width x n height) sample image, output row y being sample rows
    // [n y, n y + n) (or, with a row list, entries [n k, n k + n) of the expanded list); batches are cut in whole output rows.
    const uint32_t n = sc->supersample, sw = n * width, sh = n * height;
    const uint32_t rows = y1 - y0;
    const uint64_t batch_pixels = sc->batch_pixels ? sc->batch_pixels : (16ull << 20);
    uint32_t batch_rows = (uint32_t)std::max<uint64_t>(1, std::min<uint64_t>(rows ? rows : 1, batch_pixels / ((uint64_t)n * sw)));
    const rg_stats st0 = *st;
    for (;;) {   // a ray tree larger than device memory restarts the render with half the rows per batch
        *st = st0;
        events.used = 0;
        sync_events.used = 0;
        trace_spans.clear();
        RG_CUDA(cudaMemsetAsync(sc->d_counters, 0, sizeof(DCounters), stream));
        RG_CUDA(cudaEventRecord(sc->ev[0], stream));
        int rc = RG_OK;
        if (sc->ds.n_lights > 0 && (sc->overlap == 2 || (sc->overlap == 0 && use_grid))) {
            if (!sc->wf.aux) RG_CUDA(cudaStreamCreateWithFlags(&sc->wf.aux, cudaStreamNonBlocking));
        }
        for (uint32_t y = y0; y < y1 && rc == RG_OK;) {
            const uint32_t ye = (uint32_t)std::min<uint64_t>((uint64_t)y + batch_rows, y1);
            uchar4 *out = kind == OutKind::Rgba8Scatter ? d_out
                        : reinterpret_cast<uchar4 *>(reinterpret_cast<unsigned char *>(d_out) + (size_t)(y - y0) * width * bytes_per_pixel(kind));
            DevPlan plan;
            const uint64_t npix64 = (uint64_t)(ye - y) * n * sw;
            if (npix64 > 0x7FFFFFFFull) { set_error("batch of %llu pixels is too large", (unsigned long long)npix64); rc = RG_E_NOMEM; }
            else if (npix64 && (rc = plan_batch_dev(sc, (uint32_t)npix64, plan, use_grid)) == RG_OK) {
                bool done = false;
                if (sc->graph != 1 && sc->verify_cull == 0)
                    rc = graph_batch(sc, plan, sw, sh, n * y, (uint32_t)npix64, d_rows, kind, out, stream, st, use_grid, sync_events, &done);
                if (rc == RG_OK && !done)
                    rc = enqueue_batch_dev(sc, plan, sw, sh, n * y, (uint32_t)npix64, d_rows, kind, out, stream, st, use_grid, &events,
                                           sync_events, &trace_spans);
            }
            y = ye;
        }
        if (rc == RG_E_NOMEM && batch_rows > 1) {
            cudaStreamSynchronize(stream);
            if (sc->wf.aux) cudaStreamSynchronize(sc->wf.aux);
            sc->wf.release();
            batch_rows = (batch_rows + 1) / 2;
            continue;
        }
        if (rc) return rc;
        RG_CUDA(cudaEventRecord(sc->ev[1], stream));
        RG_CUDA(cudaMemcpyAsync(sc->h_counters, sc->d_counters, sizeof(DCounters), cudaMemcpyDeviceToHost, stream));
        RG_CUDA(cudaStreamSynchronize(stream));
        if (sc->h_counters->overflow) {   // a level outgrew its queue: repeat with twice the growth per level
            sc->level_growth *= 2;
            continue;
        }
        if (sc->depth_hint && sc->depth_hint < std::max<uint32_t>(sc->ds.max_depth, 1u) &&
            sc->h_counters->deeper) {   // the ray tree went deeper than the hint: repeat with every level
            sc->depth_hint = 0;
            continue;
        }
        break;
    }
    // what the next frame of this scene may assume about the depth of the ray tree
    {
        const uint32_t used = std::max(st->max_level, sc->h_counters->max_level) + 1u;
        sc->depth_hint = std::max(sc->depth_hint, used);
    }
    st->host_free = 1;
    float ms = 0.f;
    RG_CUDA(cudaEventElapsedTime(&ms, sc->ev[0], sc->ev[1]));
    st->ms_device = ms;
    double tr = 0.0;
    for (auto &p : trace_spans) {
        float t = 0.f;
        if (cudaEventElapsedTime(&t, p.first, p.second) == cudaSuccess) tr += t;
    }
    st->ms_trace = tr;
    const DCounters &c = *sc->h_counters;
    st->rays_shadow += c.rays[1];                        // counted on the device
    if (c.max_level > st->max_level) st->max_level = c.max_level;
    st->grid_cells = c.grid_cells;
    st->grid_fetches = c.grid_fetches;
    st->grid_culls = c.grid_culls;
    st->grid_refills = c.grid_refills;
    st->grid_lane_steps = c.grid_lane_steps;
    st->grid_lane_slots = c.grid_lane_slots;
    st->rays_reflection = c.rays[2];
    st->rays_transmission = c.rays[3];
    st->exact_tests = c.exact_tests;
    st->cull_unsound = c.cull_unsound;
    st->err_nan_distance = c.err_nan;
    st->err_transmission_none = c.err_trans;
    st->err_aabb_normal = c.err_aabb;
    st->body_tests = (st->rays_primary + st->rays_shadow + st->rays_reflection + st->rays_transmission) * (uint64_t)sc->n_bodies;
    return RG_OK;
}

}  // namespace rg
