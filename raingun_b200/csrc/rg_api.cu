// rg_api.cu — the C ABI (include/raingun_b200.h): scene upload, render entry points,
// error reporting.  Host-side hoists are limited to values that are pure functions of the
// scene and are computed with the reference's own operation order (this file is compiled
// with -ffp-contract=off on the host side).
#include <algorithm>
#include <chrono>
#include <cstdlib>
#include <cmath>
#include <cstring>
#include <limits>
#include <map>
#include <mutex>

#include "rg_cull.h"
#include "rg_host.h"
#include "rg_mega.cuh"

namespace rg {

constexpr uint32_t kMegaAutoBodies = 24;   // measured crossover (C4-style scenes, 1080p and 4K): megakernel ahead up to 24 spheres, level at 32
static thread_local std::string g_last_error;
static double g_last_ffma2_tflops = 0.0, g_last_ffma_tflops = 0.0;   // rg_measure_peaks detail

void set_error(const char *fmt, ...) {
    char buf[1024];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof(buf), fmt, ap);
    va_end(ap);
    g_last_error = buf;
}

int cuda_fail(cudaError_t e, const char *what, const char *file, int line) {
    set_error("CUDA error %d (%s) at %s:%d: %s", (int)e, cudaGetErrorString(e), file, line, what);
    if (e == cudaErrorMemoryAllocation) {
        cudaGetLastError();
        return RG_E_NOMEM;
    }
    return RG_E_CUDA;
}

static size_t trim_parked(int device);

int DeviceBuffer::reserve(size_t bytes) {
    if (bytes <= cap) return RG_OK;
    if (ptr) { cudaFree(ptr); ptr = nullptr; cap = 0; }
    size_t want = bytes + bytes / 8 + 256;   // headroom: neighbouring frames differ slightly
    cudaError_t e = cudaMalloc(&ptr, want);
    if (e != cudaSuccess) {
        cudaGetLastError();
        e = cudaMalloc(&ptr, bytes);
        want = bytes;
    }
    if (e != cudaSuccess) {   // scratch parked by earlier scenes of this device may be what is in the way
        cudaGetLastError();
        int dev = 0;
        if (cudaGetDevice(&dev) == cudaSuccess && trim_parked(dev) > 0) e = cudaMalloc(&ptr, bytes);
    }
    if (e != cudaSuccess) { ptr = nullptr; return cuda_fail(e, "cudaMalloc(scratch)", __FILE__, __LINE__); }
    cap = want;
    return RG_OK;
}
void DeviceBuffer::release() {
    if (ptr) cudaFree(ptr);
    ptr = nullptr;
    cap = 0;
}
void WavefrontScratch::release() {
    ray[0].release(); ray[1].release(); hit_t.release(); hit_body.release();
    for (int p = 0; p < 2; ++p) {
        sray[p].release(); s_tmax[p].release(); s_ab[p].release(); s_lit[p].release(); lit_bc[p].release(); lit_node[p].release();
    }
    for (auto &b : nodes) b.release();
    nodes.clear();
    for (auto e : events) cudaEventDestroy(e);
    events.clear();
    for (auto e : sync_events) cudaEventDestroy(e);
    sync_events.clear();
    if (aux) cudaStreamDestroy(aux);
    aux = nullptr;
    if (rb) cudaStreamDestroy(rb);
    rb = nullptr;
}

void GraphCache::release() {
    for (auto &e : entries)
        if (e.exec) cudaGraphExecDestroy(e.exec);
    entries.clear();
    seen.clear();
}

// Scratch arenas outlive a scene: destroying a scene parks its (possibly multi-GB) wavefront
// buffers here and the next scene created on the same device adopts them, so a host that
// re-uploads the scene every frame does not pay cudaMalloc/cudaFree for them each time.
struct ParkedContext {
    bool used = false;
    WavefrontScratch wf;
    DeviceBuffer frame, rowlist;
    SceneArena arena;
    DCounters *d_counters = nullptr, *h_counters = nullptr;
    cudaStream_t stream = nullptr;
    cudaEvent_t ev[4] = {nullptr, nullptr, nullptr, nullptr};
    uint8_t *h_stage = nullptr;   // pinned staging of the scene upload
    size_t h_stage_cap = 0;
};
static void free_parked(ParkedContext &p) {   // device of the context must be current
    p.wf.release();
    p.frame.release();
    p.rowlist.release();
    p.arena.release();
    if (p.d_counters) cudaFree(p.d_counters);
    if (p.h_counters) cudaFreeHost(p.h_counters);
    if (p.h_stage) cudaFreeHost(p.h_stage);
    for (auto &e : p.ev) if (e) cudaEventDestroy(e);
    if (p.stream) cudaStreamDestroy(p.stream);
}
static std::mutex g_park_mutex;
// a few per device: a multi-GPU host keeps several batches (scene handles) in flight per GPU
static std::map<int, std::vector<ParkedContext>> g_parked;
constexpr size_t kMaxParkedPerDevice = 4;

// frees every context parked on `device` (-1: on all devices); returns how many were freed
static size_t trim_parked(int device) {
    std::vector<std::pair<int, ParkedContext>> victims;
    {
        std::lock_guard<std::mutex> lock(g_park_mutex);
        for (auto &kv : g_parked) {
            if (device >= 0 && kv.first != device) continue;
            for (auto &p : kv.second) victims.emplace_back(kv.first, std::move(p));
            kv.second.clear();
        }
    }
    int cur = 0;
    cudaGetDevice(&cur);
    for (auto &v : victims) {
        cudaSetDevice(v.first);
        free_parked(v.second);
    }
    cudaSetDevice(cur);
    return victims.size();
}

void *SceneArena::alloc(size_t bytes) {
    bytes = (bytes + 255) & ~(size_t)255;
    if (bytes == 0) bytes = 256;
    for (;;) {
        if (cur < blocks.size() && off + bytes <= blocks[cur].cap) {
            void *p = static_cast<char *>(blocks[cur].ptr) + off;
            off += bytes;
            return p;
        }
        if (cur + 1 < blocks.size()) { ++cur; off = 0; continue; }
        DeviceBuffer b;
        if (b.reserve(std::max<size_t>(bytes, (size_t)16 << 20)) != RG_OK) return nullptr;
        blocks.push_back(b);
        cur = blocks.size() - 1;
        off = 0;
    }
}
void SceneArena::release() {
    for (auto &b : blocks) b.release();
    blocks.clear();
    reset();
}

template <typename T>
static int upload(rg_scene *sc, const T *host, size_t count, const T **out) {
    *out = nullptr;
    if (count == 0) return RG_OK;
    void *p = sc->arena.alloc(count * sizeof(T));
    if (!p) return RG_E_NOMEM;
    RG_CUDA(cudaMemcpy(p, host, count * sizeof(T), cudaMemcpyHostToDevice));
    *out = reinterpret_cast<const T *>(p);
    return RG_OK;
}

static int validate(const rg_scene_desc *d) {
    if (!d) { set_error("scene desc is NULL"); return RG_E_INVALID; }
    if (d->abi_version != RG_ABI_VERSION) { set_error("abi_version %u != %u", d->abi_version, RG_ABI_VERSION); return RG_E_INVALID; }
    if (d->max_recursion_depth > RG_MAX_DEPTH) { set_error("max_recursion_depth %u > %u", d->max_recursion_depth, RG_MAX_DEPTH); return RG_E_DEPTH; }
    if (d->n_lights > RG_MAX_LIGHTS) { set_error("%u lights > %u", d->n_lights, RG_MAX_LIGHTS); return RG_E_LIGHTS; }
    if (d->n_bodies && (!d->body_kind || !d->body_geom || !d->coloration_kind || !d->color || !d->texture_id ||
                        !d->texture_offset || !d->albedo || !d->surface_kind || !d->surface_param)) {
        set_error("a per-body array is NULL");
        return RG_E_INVALID;
    }
    if (d->n_lights && (!d->light_kind || !d->light_vec || !d->light_color || !d->light_intensity)) {
        set_error("a per-light array is NULL");
        return RG_E_INVALID;
    }
    if (d->n_textures && !d->textures) { set_error("textures is NULL"); return RG_E_INVALID; }
    for (uint32_t i = 0; i < d->n_bodies; ++i) {
        if (d->body_kind[i] > RG_BODY_AABB) { set_error("bodies[%u]: bad kind %u", i, d->body_kind[i]); return RG_E_INVALID; }
        if (d->surface_kind[i] > RG_SURFACE_REFRACTIVE) { set_error("bodies[%u]: bad surface %u", i, d->surface_kind[i]); return RG_E_INVALID; }
        if (d->coloration_kind[i] > RG_COLORATION_TEXTURE) { set_error("bodies[%u]: bad coloration", i); return RG_E_INVALID; }
        if (d->coloration_kind[i] == RG_COLORATION_TEXTURE &&
            (d->texture_id[i] < 0 || (uint32_t)d->texture_id[i] >= d->n_textures)) {
            set_error("bodies[%u]: texture_id %d out of range", i, d->texture_id[i]);
            return RG_E_INVALID;
        }
    }
    for (uint32_t i = 0; i < d->n_lights; ++i)
        if (d->light_kind[i] > RG_LIGHT_SPHERICAL) { set_error("lights[%u]: bad kind", i); return RG_E_INVALID; }
    for (uint32_t i = 0; i < d->n_textures; ++i) {
        const rg_texture_desc &t = d->textures[i];
        if (!t.pixels || t.width == 0 || t.height == 0 || (t.channels != 3 && t.channels != 4) ||
            t.width > 0x7FFFFFFFu || t.height > 0x7FFFFFFFu) {
            set_error("textures[%u]: bad descriptor", i);
            return RG_E_INVALID;
        }
    }
    return RG_OK;
}

// ray.rs:46: (fov.to_radians() / 2.0).tan(); f64::to_radians is `self * (PI / 180.0)`.
static double fov_adjustment(double fov_degrees) {
    const double pi = 3.14159265358979323846264338327950288;
    return std::tan((fov_degrees * (pi / 180.0)) / 2.0);
}

// RGB8 / RGBA8 texels as uploaded -> the uchar4 rows of a pitch-linear texture.
// DynamicImage::get_pixel yields Rgba<u8> (material.rs:67); RGB sources get alpha 255.
__global__ void __launch_bounds__(256) k_tex_expand(const uint8_t *__restrict__ src, uint32_t channels, uint32_t w, uint32_t h,
                                                    uint8_t *dst, size_t pitch) {
    const uint32_t x = blockIdx.x * blockDim.x + threadIdx.x, y = blockIdx.y;
    if (x >= w || y >= h) return;
    const uint8_t *p = src + ((size_t)y * w + x) * channels;
    *reinterpret_cast<uchar4 *>(dst + (size_t)y * pitch + (size_t)x * 4) = make_uchar4(p[0], p[1], p[2], channels == 4 ? p[3] : 255);
}

// Textures are CUDA texture objects (point sampling, unnormalised coordinates: the integer texel is
// computed exactly as Texture::wrap does, material.rs:70-79) over PITCH-LINEAR memory carved from the
// scene arena: cudaMallocArray / cudaFreeArray cost 8-100 ms per scene on this driver (measured),
// the arena costs nothing once it exists, and the RGB -> RGBA expansion runs on the device.
static int create_textures(rg_scene *sc, const rg_scene_desc *d) {
    std::vector<DTex> host(d->n_textures);
    for (uint32_t i = 0; i < d->n_textures; ++i) {
        const rg_texture_desc &t = d->textures[i];
        const size_t raw_bytes = (size_t)t.width * t.height * t.channels;
        const size_t pitch = ((size_t)t.width * 4 + 511) & ~(size_t)511;
        uint8_t *raw = static_cast<uint8_t *>(sc->arena.alloc(raw_bytes));
        uint8_t *lin = static_cast<uint8_t *>(sc->arena.alloc(pitch * t.height + 512));
        if (!raw || !lin) return RG_E_NOMEM;
        lin = reinterpret_cast<uint8_t *>((reinterpret_cast<uintptr_t>(lin) + 511) & ~(uintptr_t)511);   // textureAlignment
        RG_CUDA(cudaMemcpyAsync(raw, t.pixels, raw_bytes, cudaMemcpyHostToDevice, sc->stream));
        k_tex_expand<<<dim3((t.width + 255) / 256, t.height), 256, 0, sc->stream>>>(raw, t.channels, t.width, t.height, lin, pitch);
        RG_CUDA(cudaGetLastError());
        cudaResourceDesc res{};
        res.resType = cudaResourceTypePitch2D;
        res.res.pitch2D.devPtr = lin;
        res.res.pitch2D.desc = cudaCreateChannelDesc<uchar4>();
        res.res.pitch2D.width = t.width;
        res.res.pitch2D.height = t.height;
        res.res.pitch2D.pitchInBytes = pitch;
        cudaTextureDesc td{};
        td.addressMode[0] = cudaAddressModeClamp;
        td.addressMode[1] = cudaAddressModeClamp;
        td.filterMode = cudaFilterModePoint;        // nearest texel: material.rs:63-68 does no filtering
        td.readMode = cudaReadModeElementType;
        td.normalizedCoords = 0;
        cudaTextureObject_t obj = 0;
        RG_CUDA(cudaCreateTextureObject(&obj, &res, &td, nullptr));
        sc->tex_objs.push_back(obj);
        host[i].obj = obj;
        host[i].w = t.width;
        host[i].h = t.height;
    }
    if (d->n_textures) RG_CUDA(cudaStreamSynchronize(sc->stream));   // the caller's pixel buffers may go away
    return upload(sc, host.data(), host.size(), &sc->ds.tex);
}

// FP32 cull records (rg_cull.h) of every sphere, computed where the sphere list already is.  The arithmetic is
// the host builder's of round 1 operation for operation (FP64, no contraction: this file is compiled with
// -fmad=false), so the records are the same bits; cull2 is the pair-interleaved copy for the packed FFMA2 kernel.
__global__ void __launch_bounds__(256) k_cull_records(const double4 *__restrict__ sph, uint32_t n, uint32_t n_padded, double px, double py,
                                                      double pz, float4 *cull4, float4 *cull2) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;   // (no early return: the pair exchange below needs whole warps)
    const float kInf = __int_as_float(0x7f800000);
    float4 rec = make_float4(0.f, 0.f, 0.f, kInf);   // padding: rejects everything
    if (i < n) {
        const double4 sp = sph[i];
        const double cx = sp.x - px, cy = sp.y - py, cz = sp.z - pz, r = sp.w;
        const double C2 = cx * cx + cy * cy + cz * cz, r2 = r * r;
        if (C2 < kCullHuge && r2 < kCullHuge) {   // also false for NaN
            const double K = (C2 - r2) - kCullU * (kCullSphereC2 * C2 + kCullSphereR2 * r2);
            rec = make_float4((float)cx, (float)cy, (float)cz, (float)K);
        } else {
            rec = make_float4(0.f, 0.f, 0.f, -kInf);   // never rejected
        }
    }
    // pair (2k, 2k+1) -> cull2[2k] = (x0, x1, y0, y1), cull2[2k+1] = (z0, z1, -K0, -K1)
    const float ox = __shfl_xor_sync(0xffffffffu, rec.x, 1), oy = __shfl_xor_sync(0xffffffffu, rec.y, 1),
                oz = __shfl_xor_sync(0xffffffffu, rec.z, 1), ow = __shfl_xor_sync(0xffffffffu, rec.w, 1);
    if (i >= n_padded) return;
    cull4[i] = rec;
    if (!cull2) return;   // grid proxies (rg_scene.cuh): records for the grid only
    if ((i & 1u) == 0) cull2[i] = make_float4(rec.x, ox, rec.y, oy);
    else cull2[i] = make_float4(oz, rec.z, -ow, -rec.w);
}

// A box or disk the grid may bin through an enclosing sphere (DESIGN.md section 4.2): finite geometry, a disk of
// positive radius, a box with lo <= hi on every axis.  Everything else (planes, inverted boxes, ...) is tested per ray.
// The proxy is the box's centre and half-diagonal, the disk's origin and radius, with the radius inflated by
// 1e-9 (|c|_inf + r): far more than the rounding of the centre and of the radius, and than the distance by which
// the reference's FP64 tests can place a hit outside the body for origins within 1e6 (|c|_inf + r) of it.
static bool grid_proxy(uint8_t kind, const double *g, double out[4]) {
    double c[3], r;
    if (kind == RG_BODY_DISK) {
        for (int k = 0; k < 7; ++k)
            if (!std::isfinite(g[k])) return false;
        if (!(g[6] > 0.0)) return false;
        c[0] = g[0]; c[1] = g[1]; c[2] = g[2];
        r = g[6];
    } else if (kind == RG_BODY_AABB) {
        double h2 = 0.0;
        for (int k = 0; k < 3; ++k) {
            if (!std::isfinite(g[k]) || !std::isfinite(g[k + 3]) || !(g[k] <= g[k + 3])) return false;
            c[k] = 0.5 * g[k] + 0.5 * g[k + 3];
            const double e = 0.5 * g[k + 3] - 0.5 * g[k];
            h2 += e * e;
        }
        r = std::sqrt(h2);
    } else {
        return false;
    }
    const double cmax = std::max(std::fabs(c[0]), std::max(std::fabs(c[1]), std::fabs(c[2])));
    r = r + 1e-9 * (cmax + r);
    if (!std::isfinite(r)) return false;
    out[0] = c[0]; out[1] = c[1]; out[2] = c[2]; out[3] = r;
    return true;
}

static int build_scene(rg_scene *sc, const rg_scene_desc *d) {
    DScene &ds = sc->ds;
    const uint32_t n = d->n_bodies;
    ds.n_bodies = n;
    ds.n_lights = d->n_lights;
    ds.max_depth = d->max_recursion_depth;
    sc->scene_max_depth = d->max_recursion_depth;
    sc->n_bodies = n;
    ds.fov_adj = fov_adjustment(d->fov);
    for (int k = 0; k < 3; ++k) ds.default_color[k] = d->default_color[k];

    static const bool dbg_timing = getenv("RG_DEBUG_TIMING") != nullptr;
    auto T0 = std::chrono::steady_clock::now();
    auto lap = [&](const char *what) {
        if (!dbg_timing) return;
        auto t = std::chrono::steady_clock::now();
        fprintf(stderr, "[build_scene] %-14s %.3f ms\n", what, std::chrono::duration<double, std::milli>(t - T0).count());
        T0 = t;
    };
    // ---- everything the device needs from the host, laid out in ONE pinned staging buffer -> one async copy
    // (the sphere / non-sphere lists are laid out for the worst case, so that one pass over the bodies fills everything)
    auto align = [](size_t x) { return (x + 255) & ~(size_t)255; };
    size_t n_boxes = 0;
    for (uint32_t i = 0; i < n; ++i) n_boxes += d->body_kind[i] == RG_BODY_AABB;
    const size_t off_kind = 0, off_geom = align(off_kind + n), off_mat = align(off_geom + (size_t)n * 64),
                 off_sph = align(off_mat + (size_t)n * sizeof(BodyMat)), off_sphb = align(off_sph + (size_t)n * 32),
                 off_misc = align(off_sphb + (size_t)n * 4), off_bsph = align(off_misc + (size_t)n * 4),
                 off_gmisc = align(off_bsph + (size_t)n * 4), off_face = align(off_gmisc + (size_t)n * 4),
                 total = align(off_face + n_boxes * 6 * sizeof(FaceRef));
    if (sc->h_stage_cap < total) {
        if (sc->h_stage) cudaFreeHost(sc->h_stage);
        sc->h_stage = nullptr;
        sc->h_stage_cap = 0;
        const size_t want = total + total / 4 + 4096;
        RG_CUDA(cudaMallocHost(&sc->h_stage, want));
        sc->h_stage_cap = want;
    }
    uint8_t *hs = sc->h_stage;
    if (n) {
        std::memcpy(hs + off_kind, d->body_kind, n);
        std::memcpy(hs + off_geom, d->body_geom, (size_t)n * 64);
    }
    BodyMat *mats = reinterpret_cast<BodyMat *>(hs + off_mat);
    double *sph = reinterpret_cast<double *>(hs + off_sph);
    uint32_t *sph_body = reinterpret_cast<uint32_t *>(hs + off_sphb), *misc_body = reinterpret_cast<uint32_t *>(hs + off_misc);
    uint32_t *body_sph = reinterpret_cast<uint32_t *>(hs + off_bsph), *gmisc_body = reinterpret_cast<uint32_t *>(hs + off_gmisc);
    double lo[3] = {0, 0, 0}, hi[3] = {0, 0, 0};   // bounding box of the finite sphere and proxy centres
    bool have = false;
    auto extend = [&](const double *c) {
        if (!(std::isfinite(c[0]) && std::isfinite(c[1]) && std::isfinite(c[2]))) return;
        if (!have) {
            for (int k = 0; k < 3; ++k) lo[k] = hi[k] = c[k];
            have = true;
        } else {   // plain comparisons: the operands are finite (fmin / fmax are library calls here)
            for (int k = 0; k < 3; ++k) {
                if (c[k] < lo[k]) lo[k] = c[k];
                if (c[k] > hi[k]) hi[k] = c[k];
            }
        }
    };
    std::vector<double> prox;            // proxies (grid_proxy), appended to the sphere list below
    std::vector<uint32_t> prox_body;
    std::vector<FaceRef> faces[3];       // face planes of the binned boxes, per axis
    uint32_t ns = 0, nm = 0, ngm = 0;
    for (uint32_t i = 0; i < n; ++i) {
        BodyMat m;
        m.color[0] = d->color[3 * (size_t)i]; m.color[1] = d->color[3 * (size_t)i + 1]; m.color[2] = d->color[3 * (size_t)i + 2];
        m.albedo = d->albedo[i];
        m.p0 = d->surface_param[2 * (size_t)i];
        m.p1 = d->surface_param[2 * (size_t)i + 1];
        m.tex_off[0] = d->texture_offset[2 * (size_t)i];
        m.tex_off[1] = d->texture_offset[2 * (size_t)i + 1];
        m.tex = d->coloration_kind[i] == RG_COLORATION_TEXTURE ? d->texture_id[i] : -1;
        m.coloration = d->coloration_kind[i];
        m.surface = d->surface_kind[i];
        m.pad[0] = m.pad[1] = 0;
        m.pad2[0] = m.pad2[1] = 0;
        mats[i] = m;
        const double *g = d->body_geom + 8 * (size_t)i;
        if (d->body_kind[i] == RG_BODY_SPHERE) {
            std::memcpy(sph + 4 * (size_t)ns, g, 32);
            body_sph[i] = ns;
            sph_body[ns++] = i;
            extend(g);
        } else {
            body_sph[i] = 0xFFFFFFFFu;
            misc_body[nm++] = i;
            double p[4];
            if (grid_proxy(d->body_kind[i], g, p)) {
                prox.insert(prox.end(), p, p + 4);
                prox_body.push_back(i);
                extend(p);
                if (d->body_kind[i] == RG_BODY_AABB)
                    for (int k = 0; k < 3; ++k) {
                        faces[k].push_back(FaceRef{g[k], i, 0u});
                        faces[k].push_back(FaceRef{g[k + 3], i, 0u});
                    }
            } else {
                gmisc_body[ngm++] = i;
            }
        }
    }
    const uint32_t np = (uint32_t)prox_body.size(), nsp = ns + np;
    if (np) {   // the combined list: spheres, then proxies
        std::memcpy(sph + 4 * (size_t)ns, prox.data(), prox.size() * sizeof(double));
        std::memcpy(sph_body + ns, prox_body.data(), np * sizeof(uint32_t));
    }
    FaceRef *face = reinterpret_cast<FaceRef *>(hs + off_face);
    const size_t n_faces = faces[0].size();
    for (int k = 0; k < 3; ++k) {
        std::sort(faces[k].begin(), faces[k].end(),
                  [](const FaceRef &a, const FaceRef &b) { return a.c < b.c || (a.c == b.c && a.body < b.body); });
        if (n_faces) std::memcpy(face + k * n_faces, faces[k].data(), n_faces * sizeof(FaceRef));
    }
    ds.n_spheres = ns;
    ds.n_misc = nm;
    const size_t cull_padded = ((size_t)ns + 3) / 4 * 4;
    // P = centre of the bounding box of the sphere and proxy centres: reference point of the FP32 cull coordinates
    for (int k = 0; k < 3; ++k) ds.cull_ref[k] = have ? 0.5 * (lo[k] + hi[k]) : 0.0;

    for (uint32_t l = 0; l < d->n_lights; ++l) {
        DLight &L = ds.lights[l];
        L.kind = d->light_kind[l];
        const double *v = d->light_vec + 3 * (size_t)l;
        if (L.kind == RG_LIGHT_DIRECTIONAL) {
            // lights.rs:48: (-directional.direction).normalize(), cgmath order
            double nx = -v[0], ny = -v[1], nz = -v[2];
            double inv = 1.0 / std::sqrt((nx * nx + ny * ny) + nz * nz);
            L.v[0] = nx * inv; L.v[1] = ny * inv; L.v[2] = nz * inv;
        } else {
            L.v[0] = v[0]; L.v[1] = v[1]; L.v[2] = v[2];
        }
        for (int k = 0; k < 3; ++k) L.color[k] = d->light_color[3 * (size_t)l + k];
        L.intensity = d->light_intensity[l];
    }

    lap("host flatten");
    uint8_t *dev = static_cast<uint8_t *>(sc->arena.alloc(total));
    float4 *cull4 = static_cast<float4 *>(sc->arena.alloc(std::max<size_t>(std::max<size_t>(cull_padded, nsp), 1) * sizeof(float4)));
    float4 *cull2 = static_cast<float4 *>(sc->arena.alloc(std::max<size_t>(cull_padded, 1) * sizeof(float4)));
    if (!dev || !cull4 || !cull2) return RG_E_NOMEM;
    RG_CUDA(cudaMemcpyAsync(dev, hs, total, cudaMemcpyHostToDevice, sc->stream));
    ds.kind = n ? dev + off_kind : nullptr;
    ds.geom = n ? reinterpret_cast<const double *>(dev + off_geom) : nullptr;
    ds.mat = n ? reinterpret_cast<const BodyMat *>(dev + off_mat) : nullptr;
    ds.sph = nsp ? reinterpret_cast<const double4 *>(dev + off_sph) : nullptr;
    ds.sph_body = nsp ? reinterpret_cast<const uint32_t *>(dev + off_sphb) : nullptr;
    ds.misc_body = nm ? reinterpret_cast<const uint32_t *>(dev + off_misc) : nullptr;
    ds.body_sph = n ? reinterpret_cast<const uint32_t *>(dev + off_bsph) : nullptr;
    ds.cull4 = nsp ? cull4 : nullptr;
    ds.cull2 = ns ? cull2 : nullptr;
    if (cull_padded) {
        k_cull_records<<<(unsigned)((cull_padded + 255) / 256), 256, 0, sc->stream>>>(ds.sph, ns, (uint32_t)cull_padded, ds.cull_ref[0],
                                                                                      ds.cull_ref[1], ds.cull_ref[2], cull4, cull2);
        RG_CUDA(cudaGetLastError());
    }
    if (np) {   // (after the spheres' launch, whose padding records it overwrites)
        k_cull_records<<<(np + 255) / 256, 256, 0, sc->stream>>>(ds.sph + ns, np, np, ds.cull_ref[0], ds.cull_ref[1], ds.cull_ref[2],
                                                                 cull4 + ns, nullptr);
        RG_CUDA(cudaGetLastError());
    }
    GridProxies &gp = sc->gp;
    gp = GridProxies{};
    gp.n_proxies = np;
    gp.n_misc = ngm;
    gp.misc_body = ngm ? reinterpret_cast<const uint32_t *>(dev + off_gmisc) : nullptr;
    gp.n_faces = (uint32_t)n_faces;
    gp.faces = n_faces ? reinterpret_cast<const FaceRef *>(dev + off_face) : nullptr;
    lap("enqueue upload");
    if (dbg_timing) { cudaStreamSynchronize(sc->stream); lap("(upload done)"); }
    int rc;
    if ((rc = create_textures(sc, d))) return rc;
    lap("textures");
    if ((rc = grid_build(sc, sph, nsp))) return rc;   // (synchronises the stream: the staging buffer is free again)
    lap("grid");
    RG_CUDA(cudaStreamSynchronize(sc->stream));
    return RG_OK;
}

// ---- roofline denominators: register-resident FMA loops ---------------------------------
__global__ void __launch_bounds__(256) k_ffma2_peak(float2 *out, int iters, float2 a, float2 b) {
    float2 x0 = make_float2(threadIdx.x, 1.f), x1 = make_float2(2.f, 3.f), x2 = make_float2(4.f, 5.f), x3 = make_float2(6.f, 7.f);
    float2 x4 = x0, x5 = x1, x6 = x2, x7 = x3;
    for (int i = 0; i < iters; ++i) {
        x0 = __ffma2_rn(x0, a, b); x1 = __ffma2_rn(x1, a, b); x2 = __ffma2_rn(x2, a, b); x3 = __ffma2_rn(x3, a, b);
        x4 = __ffma2_rn(x4, a, b); x5 = __ffma2_rn(x5, a, b); x6 = __ffma2_rn(x6, a, b); x7 = __ffma2_rn(x7, a, b);
    }
    float sx = ((x0.x + x1.x) + (x2.x + x3.x)) + ((x4.y + x5.y) + (x6.y + x7.y));
    if (sx == 123456789.f) out[0] = make_float2(sx, sx);
}

template <typename T>
__global__ void __launch_bounds__(256) k_fma_peak(T *out, int iters, T a, T b, long long *cycles) {
    T x0 = (T)threadIdx.x, x1 = x0 + 1, x2 = x0 + 2, x3 = x0 + 3, x4 = x0 + 4, x5 = x0 + 5, x6 = x0 + 6, x7 = x0 + 7;
    long long c0 = clock64();
    for (int i = 0; i < iters; ++i) {
        if constexpr (sizeof(T) == 4) {
            x0 = fmaf(x0, a, b); x1 = fmaf(x1, a, b); x2 = fmaf(x2, a, b); x3 = fmaf(x3, a, b);
            x4 = fmaf(x4, a, b); x5 = fmaf(x5, a, b); x6 = fmaf(x6, a, b); x7 = fmaf(x7, a, b);
        } else {
            x0 = fma(x0, a, b); x1 = fma(x1, a, b); x2 = fma(x2, a, b); x3 = fma(x3, a, b);
            x4 = fma(x4, a, b); x5 = fma(x5, a, b); x6 = fma(x6, a, b); x7 = fma(x7, a, b);
        }
    }
    long long c1 = clock64();
    T s = ((x0 + x1) + (x2 + x3)) + ((x4 + x5) + (x6 + x7));
    if (s == (T)123456789) out[0] = s;   // keeps the loop alive, never true in practice
    if (blockIdx.x == 0 && threadIdx.x == 0 && cycles) *cycles = c1 - c0;
}

}  // namespace rg

using namespace rg;

extern "C" {
static int rg_render_rowlist_device_impl(rg_scene *sc, uint32_t w, uint32_t h, const uint32_t *rows, uint32_t n_rows, void *d_rgba_out,
                                         void *cuda_stream, rg_stats *stats);
}
namespace rg {
int rowlist_device_unguarded(rg_scene *sc, uint32_t w, uint32_t h, const uint32_t *rows, uint32_t n_rows, void *d_rgba_out,
                             void *cuda_stream, rg_stats *stats) {
    return rg_render_rowlist_device_impl(sc, w, h, rows, n_rows, d_rgba_out, cuda_stream, stats);
}
}  // namespace rg

extern "C" {

const char *rg_last_error(void) { return g_last_error.c_str(); }

int rg_device_count(void) {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) { cudaGetLastError(); return 0; }
    return n;
}

void rg_scene_destroy(rg_scene *sc) {
    if (!sc) return;
    if (sc->multi) { multi_destroy(sc); return; }
    cudaSetDevice(sc->device);
    sc->graphs.release();
    for (auto o : sc->tex_objs) cudaDestroyTextureObject(o);
    {
        std::lock_guard<std::mutex> lock(g_park_mutex);
        std::vector<ParkedContext> &parked = g_parked[sc->device];
        // park the device-side context for the next scene on this device — only a COMPLETE one (a create() that
        // failed half-way must not hand its holes to the next scene)
        const bool complete = sc->stream && sc->d_counters && sc->h_counters && sc->ev[0] && sc->ev[1] && sc->ev[2] && sc->ev[3];
        if (parked.size() < kMaxParkedPerDevice && complete) {
            if (sc->h_frame) cudaFreeHost(sc->h_frame);
            parked.emplace_back();
            ParkedContext &slot = parked.back();
            slot.used = true;
            slot.wf = std::move(sc->wf);
            slot.frame = sc->frame;
            slot.rowlist = sc->rowlist;
            slot.arena = std::move(sc->arena);
            slot.d_counters = sc->d_counters;
            slot.h_counters = sc->h_counters;
            slot.stream = sc->stream;
            slot.h_stage = sc->h_stage;
            slot.h_stage_cap = sc->h_stage_cap;
            for (int k = 0; k < 4; ++k) slot.ev[k] = sc->ev[k];
            delete sc;
            return;
        }
    }
    sc->arena.release();
    sc->wf.release();
    sc->frame.release();
    sc->rowlist.release();
    if (sc->h_frame) cudaFreeHost(sc->h_frame);
    if (sc->h_stage) cudaFreeHost(sc->h_stage);
    if (sc->d_counters) cudaFree(sc->d_counters);
    if (sc->h_counters) cudaFreeHost(sc->h_counters);
    for (auto &e : sc->ev) if (e) cudaEventDestroy(e);
    if (sc->stream) cudaStreamDestroy(sc->stream);
    delete sc;
}

int rg_scene_create(const rg_scene_desc *desc, int32_t device, rg_scene **out) {
    if (!out) { set_error("out is NULL"); return RG_E_INVALID; }
    *out = nullptr;
    static const bool dbg_timing = getenv("RG_DEBUG_TIMING") != nullptr;
    auto T0 = std::chrono::steady_clock::now();
    auto lap = [&](const char *what) {
        if (!dbg_timing) return;
        auto t = std::chrono::steady_clock::now();
        fprintf(stderr, "[rg_scene_create] %-12s %.3f ms\n", what, std::chrono::duration<double, std::milli>(t - T0).count());
        T0 = t;
    };
    int rc = validate(desc);
    lap("validate");
    if (rc) return rc;
    int ndev = 0;
    cudaError_t e = cudaGetDeviceCount(&ndev);
    if (e != cudaSuccess || ndev == 0) {
        cudaGetLastError();
        set_error("no CUDA device available (%s); this library has no CPU path", cudaGetErrorString(e));
        return RG_E_CUDA;
    }
    if (device == RG_DEVICE_ALL) {   // every visible GPU (RG_DEVICES=n: the first n)
        const char *e = getenv("RG_DEVICES");
        int n = e ? atoi(e) : ndev;
        if (n < 1 || n > ndev) n = ndev;
        std::vector<int32_t> all((size_t)n);
        for (int k = 0; k < n; ++k) all[(size_t)k] = k;
        if (n == 1) return rg_scene_create(desc, 0, out);
        return multi_create(desc, all.data(), (uint32_t)n, out);
    }
    if (device < 0 || device >= ndev) { set_error("device %d out of range (%d devices)", device, ndev); return RG_E_INVALID; }
    RG_CUDA(cudaSetDevice(device));
    // cudaGetDeviceProperties costs ~2.6 ms per call on this driver (measured); three attribute
    // queries, cached per device, cost nothing on the re-upload-per-frame path
    struct DevInfo { int major = 0, minor = 0, sms = 0; };
    static std::mutex dev_mutex;
    static std::map<int, DevInfo> dev_cache;
    DevInfo info;
    {
        std::lock_guard<std::mutex> lock(dev_mutex);
        auto it = dev_cache.find(device);
        if (it == dev_cache.end()) {
            RG_CUDA(cudaDeviceGetAttribute(&info.major, cudaDevAttrComputeCapabilityMajor, device));
            RG_CUDA(cudaDeviceGetAttribute(&info.minor, cudaDevAttrComputeCapabilityMinor, device));
            RG_CUDA(cudaDeviceGetAttribute(&info.sms, cudaDevAttrMultiProcessorCount, device));
            dev_cache[device] = info;
        } else {
            info = it->second;
        }
    }
    if (info.major < 10) {
        set_error("device %d is sm_%d%d; this library is built for sm_100a only", device, info.major, info.minor);
        return RG_E_CUDA;
    }
    lap("device props");
    rg_scene *sc = new rg_scene();
    sc->device = device;
    sc->sm_count = info.sms;
    auto fail = [&](int code) { rg_scene_destroy(sc); return code; };
    {
        std::lock_guard<std::mutex> lock(g_park_mutex);
        auto it = g_parked.find(device);
        if (it != g_parked.end() && !it->second.empty()) {   // adopt a context an earlier scene left behind
            ParkedContext slot = std::move(it->second.back());
            it->second.pop_back();
            sc->wf = std::move(slot.wf);
            sc->frame = slot.frame;
            sc->rowlist = slot.rowlist;
            sc->arena = std::move(slot.arena);
            sc->arena.reset();
            sc->d_counters = slot.d_counters;
            sc->h_counters = slot.h_counters;
            sc->stream = slot.stream;
            sc->h_stage = slot.h_stage;
            sc->h_stage_cap = slot.h_stage_cap;
            for (int k = 0; k < 4; ++k) sc->ev[k] = slot.ev[k];
        }
    }
    if (!sc->stream) {
        if (cudaStreamCreateWithFlags(&sc->stream, cudaStreamNonBlocking) != cudaSuccess) return fail(cuda_fail(cudaGetLastError(), "stream", __FILE__, __LINE__));
        for (auto &ev : sc->ev)
            if (cudaEventCreate(&ev) != cudaSuccess) return fail(cuda_fail(cudaGetLastError(), "event", __FILE__, __LINE__));
        if (cudaMalloc(&sc->d_counters, sizeof(DCounters)) != cudaSuccess) return fail(cuda_fail(cudaGetLastError(), "counters", __FILE__, __LINE__));
        if (cudaMallocHost(&sc->h_counters, sizeof(DCounters)) != cudaSuccess) return fail(cuda_fail(cudaGetLastError(), "counters", __FILE__, __LINE__));
    }
    lap("context");
    rc = build_scene(sc, desc);
    if (rc) return fail(rc);
    lap("build_scene");
    *out = sc;
    return RG_OK;
}

int rg_scene_set_option(rg_scene *sc, int32_t key, int64_t value) {
    if (!sc) { set_error("scene is NULL"); return RG_E_INVALID; }
    if (sc->multi) return multi_set_option(sc, key, value);
    switch (key) {
        case RG_OPT_SCHEDULE:    // multi-GPU scenes only; accepted and ignored on one device
        case RG_OPT_TILE_ROWS:
            return RG_OK;
        case RG_OPT_PIPELINE:
            if (value != RG_PIPELINE_WAVEFRONT && value != RG_PIPELINE_MEGAKERNEL && value != RG_PIPELINE_AUTO) break;
            sc->pipeline = (int)value;
            return RG_OK;
        case RG_OPT_ACCEL:
            if (value < RG_ACCEL_AUTO || value > RG_ACCEL_GRID) break;
            sc->accel = (int)value;
            return RG_OK;
        case RG_OPT_MAX_DEPTH:   // main.rs:119-123: a limit only lowers the scene's own depth
            if (value < 0) break;
            sc->ds.max_depth = (uint64_t)value < sc->scene_max_depth ? (uint32_t)value : sc->scene_max_depth;
            return RG_OK;
        case RG_OPT_BATCH_PIXELS:
            if (value < 0) break;
            sc->batch_pixels = (uint64_t)value;
            return RG_OK;
        case RG_OPT_VERIFY_CULL:
            sc->verify_cull = (int)value;
            return RG_OK;
        case RG_OPT_OVERLAP:
            if (value < 0 || value > 2) break;
            sc->overlap = (int)value;
            return RG_OK;
        case RG_OPT_HOST_FREE:
            if (value < 0 || value > 2) break;
            sc->host_free = (int)value;
            return RG_OK;
        case RG_OPT_GRAPH:
            if (value < 0 || value > 2) break;
            sc->graph = (int)value;
            return RG_OK;
        case RG_OPT_TRACE_STATS:
            sc->trace_stats = value != 0;
            return RG_OK;
        case RG_OPT_ORIGIN_HINTS:
            sc->origin_hints = value != 0;
            return RG_OK;
        default: break;
    }
    set_error("bad option key %d / value %lld", key, (long long)value);
    return RG_E_INVALID;
}

static int check_dims(rg_scene *sc, uint32_t w, uint32_t h, uint32_t y0, uint32_t y1) {
    if (!sc) { set_error("scene is NULL"); return RG_E_INVALID; }
    if (w == 0 || h == 0) { set_error("empty image %ux%u", w, h); return RG_E_INVALID; }
    if (w < h) { set_error("width %u < height %u: portrait images are not supported (ray.rs:42)", w, h); return RG_E_PORTRAIT; }
    if ((uint64_t)w * h > 0xFFFFFFFFull) { set_error("width*height overflows u32 (rendering.rs:27)"); return RG_E_TOO_LARGE; }
    if (y0 > y1 || y1 > h) { set_error("bad row range [%u, %u) of %u", y0, y1, h); return RG_E_INVALID; }
    return RG_OK;
}

static int mega_render(rg_scene *sc, uint32_t w, uint32_t h, uint32_t y0, uint32_t y1, const uint32_t *d_rows,
                       uchar4 *d_out, cudaStream_t stream, rg_stats *st) {
    const uint64_t npix = (uint64_t)(y1 - y0) * w;
    RG_CUDA(cudaMemsetAsync(sc->d_counters, 0, sizeof(DCounters), stream));
    RG_CUDA(cudaEventRecord(sc->ev[0], stream));
    if (npix) {
        const unsigned blocks = (unsigned)((npix + 127) / 128);
        float *f32 = sc->out_f32 ? reinterpret_cast<float *>(d_out) : nullptr;
        if (sc->ds.max_depth <= 12) k_render_mega<12><<<blocks, 128, 0, stream>>>(sc->ds, w, h, y0, y1, d_rows, d_out, f32, sc->d_counters);
        else k_render_mega<RG_MAX_DEPTH><<<blocks, 128, 0, stream>>>(sc->ds, w, h, y0, y1, d_rows, d_out, f32, sc->d_counters);
        RG_CUDA(cudaGetLastError());
    }
    RG_CUDA(cudaEventRecord(sc->ev[1], stream));
    RG_CUDA(cudaMemcpyAsync(sc->h_counters, sc->d_counters, sizeof(DCounters), cudaMemcpyDeviceToHost, stream));
    RG_CUDA(cudaStreamSynchronize(stream));
    float ms = 0.f;
    RG_CUDA(cudaEventElapsedTime(&ms, sc->ev[0], sc->ev[1]));
    const DCounters &c = *sc->h_counters;
    st->rays_primary = c.rays[0];
    st->rays_shadow = c.rays[1];
    st->rays_reflection = c.rays[2];
    st->rays_transmission = c.rays[3];
    st->err_nan_distance = c.err_nan;
    st->err_transmission_none = c.err_trans;
    st->err_aabb_normal = c.err_aabb;
    st->ms_device = ms;
    st->ms_trace = ms;
    st->gpu_launches = npix ? 1 : 0;
    st->batches = 1;
    st->accel_used = RG_ACCEL_BRUTE;
    uint64_t rays = c.rays[0] + c.rays[1] + c.rays[2] + c.rays[3];
    st->body_tests = rays * sc->n_bodies;
    st->exact_tests = st->body_tests;
    return RG_OK;
}

// Common tail of the device-output entry points: rows [y0, y1), or entries [0, n) of a row list.
static int render_device(rg_scene *sc, uint32_t w, uint32_t h, uint32_t y0, uint32_t y1, const uint32_t *d_rows,
                         void *d_rgba_out, cudaStream_t stream, rg_stats *stats) {
    auto t0 = std::chrono::steady_clock::now();
    rg_stats local;
    std::memset(&local, 0, sizeof(local));
    int rc;
    // RG_PIPELINE_AUTO: with a handful of bodies the per-pixel recursion (every body tested in FP64, no queues)
    // beats the wavefront at every image size (measured on the shipped examples, 800x600 .. 4K: 2-3x);
    // the crossover lies near kMegaAutoBodies bodies (RG_MEGA_AUTO_BODIES for tuning runs)
    static const uint32_t mega_auto_bodies = [] { const char *e = getenv("RG_MEGA_AUTO_BODIES"); return e ? (uint32_t)atoi(e) : kMegaAutoBodies; }();
    const bool mega = sc->pipeline == RG_PIPELINE_MEGAKERNEL ||
                      (sc->pipeline == RG_PIPELINE_AUTO && !sc->scatter_out && sc->n_bodies <= mega_auto_bodies && sc->verify_cull == 0);
    if (mega) rc = mega_render(sc, w, h, y0, y1, d_rows, (uchar4 *)d_rgba_out, stream, &local);
    else rc = wavefront_render(sc, w, h, y0, y1, d_rows, (uchar4 *)d_rgba_out, stream, &local);
    local.pipeline_used = mega ? RG_PIPELINE_MEGAKERNEL : RG_PIPELINE_WAVEFRONT;
    local.devices_used = 1;
    local.ms_wall = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count();
    if (stats) *stats = local;
    return rc;
}

static int single_device_only(const rg_scene *sc, const char *what) {
    if (sc && sc->multi) { set_error("%s needs a single-device scene (this one spans %u GPUs)", what, multi_device_count(sc)); return RG_E_INVALID; }
    return RG_OK;
}

static int rg_render_rows_device_impl(rg_scene *sc, uint32_t w, uint32_t h, uint32_t y0, uint32_t y1, void *d_rgba_out,
                          void *cuda_stream, rg_stats *stats) {
    int rc = check_dims(sc, w, h, y0, y1);
    if (rc) return rc;
    if ((rc = single_device_only(sc, "rg_render_rows_device"))) return rc;
    if (!d_rgba_out && y1 > y0) { set_error("output pointer is NULL"); return RG_E_INVALID; }
    RG_CUDA(cudaSetDevice(sc->device));
    return render_device(sc, w, h, y0, y1, nullptr, d_rgba_out, reinterpret_cast<cudaStream_t>(cuda_stream), stats);
}

static int rg_render_rowlist_device_impl(rg_scene *sc, uint32_t w, uint32_t h, const uint32_t *rows, uint32_t n_rows,
                             void *d_rgba_out, void *cuda_stream, rg_stats *stats) {
    int rc = check_dims(sc, w, h, 0, h);
    if (rc) return rc;
    if ((rc = single_device_only(sc, "rg_render_rowlist_device"))) return rc;
    if (n_rows && (!rows || !d_rgba_out)) { set_error("rows / output pointer is NULL"); return RG_E_INVALID; }
    for (uint32_t k = 0; k < n_rows; ++k)
        if (rows[k] >= h) { set_error("rows[%u] = %u is outside the image (height %u)", k, rows[k], h); return RG_E_INVALID; }
    RG_CUDA(cudaSetDevice(sc->device));
    cudaStream_t stream = reinterpret_cast<cudaStream_t>(cuda_stream);
    if (n_rows) {
        if ((rc = sc->rowlist.reserve((size_t)n_rows * sizeof(uint32_t)))) return rc;
        RG_CUDA(cudaMemcpyAsync(sc->rowlist.ptr, rows, (size_t)n_rows * sizeof(uint32_t), cudaMemcpyHostToDevice, stream));
        RG_CUDA(cudaStreamSynchronize(stream));   // `rows` may be pageable and reused by the caller
    }
    return render_device(sc, w, h, 0, n_rows, sc->rowlist.as<uint32_t>(), d_rgba_out, stream, stats);
}

static int rg_render_rowlist_scatter_impl(rg_scene *sc, uint32_t w, uint32_t h, const uint32_t *rows, uint32_t n_rows,
                              void *d_frame, void *cuda_stream, rg_stats *stats) {
    if (sc && sc->pipeline == RG_PIPELINE_MEGAKERNEL) { set_error("rg_render_rowlist_scatter needs the wavefront pipeline"); return RG_E_INVALID; }
    if (!sc) { set_error("scene is NULL"); return RG_E_INVALID; }
    sc->scatter_out = true;
    const int rc = rg_render_rowlist_device_impl(sc, w, h, rows, n_rows, d_frame, cuda_stream, stats);
    sc->scatter_out = false;
    return rc;
}

// ---- frames another process' GPU can write into (CUDA IPC; peer stores travel over NVLink) ----
static_assert(sizeof(cudaIpcMemHandle_t) == RG_IPC_HANDLE_BYTES, "RG_IPC_HANDLE_BYTES");

int rg_shared_frame_create(int32_t device, size_t bytes, void **d_ptr, uint8_t *handle) {
    if (!d_ptr || !handle || bytes == 0) { set_error("rg_shared_frame_create: bad argument"); return RG_E_INVALID; }
    RG_CUDA(cudaSetDevice(device));
    void *p = nullptr;
    if (cudaMalloc(&p, bytes) != cudaSuccess) return cuda_fail(cudaGetLastError(), "cudaMalloc(shared frame)", __FILE__, __LINE__);
    cudaIpcMemHandle_t hnd;
    cudaError_t e = cudaIpcGetMemHandle(&hnd, p);
    if (e != cudaSuccess) { cudaFree(p); return cuda_fail(e, "cudaIpcGetMemHandle", __FILE__, __LINE__); }
    std::memcpy(handle, &hnd, sizeof hnd);
    *d_ptr = p;
    return RG_OK;
}

int rg_shared_frame_open(int32_t device, const uint8_t *handle, void **d_ptr) {
    if (!d_ptr || !handle) { set_error("rg_shared_frame_open: bad argument"); return RG_E_INVALID; }
    RG_CUDA(cudaSetDevice(device));
    cudaIpcMemHandle_t hnd;
    std::memcpy(&hnd, handle, sizeof hnd);
    void *p = nullptr;
    RG_CUDA(cudaIpcOpenMemHandle(&p, hnd, cudaIpcMemLazyEnablePeerAccess));
    *d_ptr = p;
    return RG_OK;
}

int rg_shared_frame_close(int32_t device, void *d_ptr, int32_t is_owner) {
    if (!d_ptr) return RG_OK;
    RG_CUDA(cudaSetDevice(device));
    if (is_owner) RG_CUDA(cudaFree(d_ptr));
    else RG_CUDA(cudaIpcCloseMemHandle(d_ptr));
    return RG_OK;
}

static int rg_render_rows_impl(rg_scene *sc, uint32_t w, uint32_t h, uint32_t y0, uint32_t y1, uint8_t *rgba_out, rg_stats *stats) {
    int rc = check_dims(sc, w, h, y0, y1);
    if (rc) return rc;
    if (!rgba_out && y1 > y0) { set_error("output pointer is NULL"); return RG_E_INVALID; }
    if (sc->multi) return multi_render_rows(sc, w, h, y0, y1, rgba_out, stats);   // every GPU of the scene takes its row tiles
    auto t0 = std::chrono::steady_clock::now();
    RG_CUDA(cudaSetDevice(sc->device));
    const size_t bytes = (size_t)(y1 - y0) * w * 4;
    if ((rc = sc->frame.reserve(bytes ? bytes : 4))) return rc;
    rg_stats local;
    std::memset(&local, 0, sizeof(local));
    rc = rg_render_rows_device_impl(sc, w, h, y0, y1, sc->frame.ptr, sc->stream, &local);
    if (rc) return rc;
    if (bytes) {
        RG_CUDA(cudaMemcpyAsync(rgba_out, sc->frame.ptr, bytes, cudaMemcpyDeviceToHost, sc->stream));
        RG_CUDA(cudaStreamSynchronize(sc->stream));
    }
    local.ms_wall = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count();
    if (stats) *stats = local;
    return RG_OK;
}

static int rg_render_impl(rg_scene *sc, uint32_t w, uint32_t h, uint8_t *rgba_out, rg_stats *stats) {
    return rg_render_rows_impl(sc, w, h, 0, h, rgba_out, stats);
}

static void accumulate(rg_stats *total, const rg_stats &s) {
    total->rays_primary += s.rays_primary;
    total->rays_shadow += s.rays_shadow;
    total->rays_reflection += s.rays_reflection;
    total->rays_transmission += s.rays_transmission;
    total->body_tests += s.body_tests;
    total->exact_tests += s.exact_tests;
    total->cull_unsound += s.cull_unsound;
    total->err_nan_distance += s.err_nan_distance;
    total->err_transmission_none += s.err_transmission_none;
    total->err_aabb_normal += s.err_aabb_normal;
    total->ms_device += s.ms_device;
    total->ms_trace += s.ms_trace;
    total->gpu_launches += s.gpu_launches;
    total->batches += s.batches;
    total->graph_replays += s.graph_replays;
    total->host_free = s.host_free;
    total->pipeline_used = s.pipeline_used;
    total->grid_cells += s.grid_cells;
    total->grid_fetches += s.grid_fetches;
    total->grid_culls += s.grid_culls;
    total->grid_refills += s.grid_refills;
    total->grid_lane_steps += s.grid_lane_steps;
    total->grid_lane_slots += s.grid_lane_slots;
    if (s.max_level > total->max_level) total->max_level = s.max_level;
    total->accel_used = s.accel_used;
}

static int rg_render_stream_impl(rg_scene *sc, uint32_t w, uint32_t h, uint32_t band_rows, rg_rows_cb cb, void *user, rg_stats *stats) {
    int rc = check_dims(sc, w, h, 0, h);
    if (rc) return rc;
    if (!cb) { set_error("callback is NULL"); return RG_E_INVALID; }
    auto t0 = std::chrono::steady_clock::now();
    RG_CUDA(cudaSetDevice(sc->device));
    if (band_rows == 0) {
        uint64_t rows = (1ull << 20) / w;   // ~1 Mpixel per band
        band_rows = (uint32_t)(rows < 1 ? 1 : rows);
    }
    if (band_rows > h) band_rows = h;
    const size_t band_bytes = (size_t)band_rows * w * 4;
    if (sc->h_frame_cap < band_bytes) {
        if (sc->h_frame) cudaFreeHost(sc->h_frame);
        sc->h_frame = nullptr;
        sc->h_frame_cap = 0;
        RG_CUDA(cudaMallocHost(&sc->h_frame, band_bytes));
        sc->h_frame_cap = band_bytes;
    }
    rg_stats total;
    std::memset(&total, 0, sizeof(total));
    for (uint32_t y0 = 0; y0 < h; y0 += band_rows) {
        uint32_t y1 = y0 + band_rows < h ? y0 + band_rows : h;
        rg_stats s;
        rc = rg_render_rows_impl(sc, w, h, y0, y1, sc->h_frame, &s);
        if (rc) return rc;
        accumulate(&total, s);
        if (cb(y0, y1 - y0, w, sc->h_frame, user) != 0) {   // closed channel: rendering.rs:53-54,67
            set_error("render cancelled by the row callback at row %u", y0);
            total.ms_wall = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count();
            if (stats) *stats = total;
            return RG_E_CANCELLED;
        }
    }
    total.ms_wall = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count();
    if (stats) *stats = total;
    return RG_OK;
}

// ---- public render entry points: one call at a time per handle ---------------------------------------
// The reference's &Scene is Sync; a device-side scene is not (its scratch queues belong to the handle), so a
// second render on a handle that is already rendering is refused with RG_E_BUSY instead of corrupting both.
struct BusyGuard {
    rg_scene *sc;
    bool ok;
    explicit BusyGuard(rg_scene *s) : sc(s), ok(true) {
        if (sc && sc->busy.exchange(true, std::memory_order_acquire)) {
            ok = false;
            set_error("this scene handle is already rendering on another thread (one render at a time per handle; create one handle per thread)");
        }
    }
    ~BusyGuard() { if (sc && ok) sc->busy.store(false, std::memory_order_release); }
};
#define RG_ENTER(sc) BusyGuard _guard(sc); if (!_guard.ok) return RG_E_BUSY

int rg_render_rows_device(rg_scene *sc, uint32_t w, uint32_t h, uint32_t y0, uint32_t y1, void *d_rgba_out, void *cuda_stream, rg_stats *stats) {
    RG_ENTER(sc);
    return rg_render_rows_device_impl(sc, w, h, y0, y1, d_rgba_out, cuda_stream, stats);
}
int rg_render_rowlist_device(rg_scene *sc, uint32_t w, uint32_t h, const uint32_t *rows, uint32_t n_rows, void *d_rgba_out, void *cuda_stream, rg_stats *stats) {
    RG_ENTER(sc);
    return rg_render_rowlist_device_impl(sc, w, h, rows, n_rows, d_rgba_out, cuda_stream, stats);
}
int rg_render_rowlist_scatter(rg_scene *sc, uint32_t w, uint32_t h, const uint32_t *rows, uint32_t n_rows, void *d_frame, void *cuda_stream, rg_stats *stats) {
    RG_ENTER(sc);
    return rg_render_rowlist_scatter_impl(sc, w, h, rows, n_rows, d_frame, cuda_stream, stats);
}
int rg_render_rows(rg_scene *sc, uint32_t w, uint32_t h, uint32_t y0, uint32_t y1, uint8_t *rgba_out, rg_stats *stats) {
    RG_ENTER(sc);
    return rg_render_rows_impl(sc, w, h, y0, y1, rgba_out, stats);
}
int rg_render(rg_scene *sc, uint32_t w, uint32_t h, uint8_t *rgba_out, rg_stats *stats) {
    RG_ENTER(sc);
    return rg_render_impl(sc, w, h, rgba_out, stats);
}
int rg_render_stream(rg_scene *sc, uint32_t w, uint32_t h, uint32_t band_rows, rg_rows_cb cb, void *user, rg_stats *stats) {
    RG_ENTER(sc);
    return rg_render_stream_impl(sc, w, h, band_rows, cb, user, stats);
}

// ---- unquantised colours: RenderedPixel.color is an f32 Color (rendering.rs:18-22), quantised only by the consumer
static int render_rows_f32_impl(rg_scene *sc, uint32_t w, uint32_t h, uint32_t y0, uint32_t y1, float *rgb_out, rg_stats *stats) {
    int rc = check_dims(sc, w, h, y0, y1);
    if (rc) return rc;
    if ((rc = single_device_only(sc, "rg_render_rows_f32"))) return rc;
    if (!rgb_out && y1 > y0) { set_error("output pointer is NULL"); return RG_E_INVALID; }
    RG_CUDA(cudaSetDevice(sc->device));
    const size_t bytes = (size_t)(y1 - y0) * w * 12;
    if ((rc = sc->frame.reserve(bytes ? bytes : 4))) return rc;
    sc->out_f32 = true;
    rc = render_device(sc, w, h, y0, y1, nullptr, sc->frame.ptr, sc->stream, stats);
    sc->out_f32 = false;
    if (rc) return rc;
    if (bytes) {
        RG_CUDA(cudaMemcpyAsync(rgb_out, sc->frame.ptr, bytes, cudaMemcpyDeviceToHost, sc->stream));
        RG_CUDA(cudaStreamSynchronize(sc->stream));
    }
    return RG_OK;
}

int rg_render_rows_f32(rg_scene *sc, uint32_t w, uint32_t h, uint32_t y0, uint32_t y1, float *rgb_out, rg_stats *stats) {
    RG_ENTER(sc);
    return render_rows_f32_impl(sc, w, h, y0, y1, rgb_out, stats);
}

int rg_render_stream_f32(rg_scene *sc, uint32_t w, uint32_t h, uint32_t band_rows, rg_rows_f32_cb cb, void *user, rg_stats *stats) {
    RG_ENTER(sc);
    int rc = check_dims(sc, w, h, 0, h);
    if (rc) return rc;
    if (!cb) { set_error("callback is NULL"); return RG_E_INVALID; }
    if ((rc = single_device_only(sc, "rg_render_stream_f32"))) return rc;
    RG_CUDA(cudaSetDevice(sc->device));
    if (band_rows == 0) band_rows = (uint32_t)std::max<uint64_t>(1, (1ull << 20) / w);
    if (band_rows > h) band_rows = h;
    const size_t band_bytes = (size_t)band_rows * w * 12;
    if (sc->h_frame_cap < band_bytes) {
        if (sc->h_frame) cudaFreeHost(sc->h_frame);
        sc->h_frame = nullptr;
        sc->h_frame_cap = 0;
        RG_CUDA(cudaMallocHost(&sc->h_frame, band_bytes));
        sc->h_frame_cap = band_bytes;
    }
    rg_stats total;
    std::memset(&total, 0, sizeof(total));
    for (uint32_t y0 = 0; y0 < h; y0 += band_rows) {
        const uint32_t y1 = y0 + band_rows < h ? y0 + band_rows : h;
        rg_stats s;
        std::memset(&s, 0, sizeof s);
        rc = render_rows_f32_impl(sc, w, h, y0, y1, reinterpret_cast<float *>(sc->h_frame), &s);
        if (rc) return rc;
        accumulate(&total, s);
        if (cb(y0, y1 - y0, w, reinterpret_cast<const float *>(sc->h_frame), user) != 0) {   // closed channel: rendering.rs:53-54,67
            set_error("render cancelled by the row callback at row %u", y0);
            if (stats) *stats = total;
            return RG_E_CANCELLED;
        }
    }
    if (stats) *stats = total;
    return RG_OK;
}

int rg_render_rowlist_host(rg_scene *sc, uint32_t w, uint32_t h, const uint32_t *rows, uint32_t n_rows, uint8_t *frame, rg_stats *stats) {
    RG_ENTER(sc);
    int rc = check_dims(sc, w, h, 0, h);
    if (rc) return rc;
    if ((rc = single_device_only(sc, "rg_render_rowlist_host"))) return rc;
    if (n_rows && (!rows || !frame)) { set_error("rows / frame pointer is NULL"); return RG_E_INVALID; }
    RG_CUDA(cudaSetDevice(sc->device));
    return render_rowlist_to_host(sc, w, h, rows, n_rows, frame, stats);
}

int rg_trim(void) { return (int)trim_parked(-1); }

int rg_device_enable_peer(int32_t device, int32_t peer) {
    int ndev = rg_device_count();
    if (device < 0 || device >= ndev || peer < 0 || peer >= ndev) { set_error("device %d / peer %d out of range (%d devices)", device, peer, ndev); return RG_E_INVALID; }
    if (device == peer) return RG_OK;
    int can = 0;
    RG_CUDA(cudaDeviceCanAccessPeer(&can, device, peer));
    if (!can) { set_error("GPU %d cannot address GPU %d's memory", device, peer); return RG_E_CUDA; }
    RG_CUDA(cudaSetDevice(device));
    const cudaError_t e = cudaDeviceEnablePeerAccess(peer, 0);
    if (e == cudaErrorPeerAccessAlreadyEnabled) { cudaGetLastError(); return RG_OK; }
    RG_CUDA(e);
    return RG_OK;
}

int rg_host_register(void *ptr, size_t bytes) {
    if (!ptr || !bytes) { set_error("rg_host_register: bad argument"); return RG_E_INVALID; }
    RG_CUDA(cudaHostRegister(ptr, bytes, cudaHostRegisterPortable));
    return RG_OK;
}

int rg_host_unregister(void *ptr) {
    if (!ptr) return RG_OK;
    RG_CUDA(cudaHostUnregister(ptr));
    return RG_OK;
}

int rg_scene_create_multi(const rg_scene_desc *desc, const int32_t *devices, uint32_t n_devices, rg_scene **out) {
    if (!out) { set_error("out is NULL"); return RG_E_INVALID; }
    *out = nullptr;
    if (!devices || n_devices == 0) { set_error("no devices given"); return RG_E_INVALID; }
    if (n_devices == 1) return rg_scene_create(desc, devices[0], out);
    int rc = validate(desc);   // (a device listed twice simply gets two lanes: its own scene copy, stream and thread each)
    if (rc) return rc;
    return multi_create(desc, devices, n_devices, out);
}

int rg_scene_device_count(const rg_scene *sc) {
    if (!sc) return 0;
    return sc->multi ? (int)multi_device_count(sc) : 1;
}

int rg_measure_peaks(int32_t device, double *fp32_tflops, double *fp64_tflops, double *sm_clock_mhz) {
    int ndev = rg_device_count();
    if (device < 0 || device >= ndev) { set_error("device %d out of range (%d devices)", device, ndev); return ndev ? RG_E_INVALID : RG_E_CUDA; }
    RG_CUDA(cudaSetDevice(device));
    cudaDeviceProp prop{};
    RG_CUDA(cudaGetDeviceProperties(&prop, device));
    const int blocks = prop.multiProcessorCount * 8, threads = 256;
    void *out = nullptr;
    long long *cyc = nullptr;
    RG_CUDA(cudaMalloc(&out, 64));
    RG_CUDA(cudaMalloc(&cyc, sizeof(long long)));
    cudaEvent_t e0, e1;
    RG_CUDA(cudaEventCreate(&e0));
    RG_CUDA(cudaEventCreate(&e1));
    double best32 = 0, best64 = 0, best32x2 = 0, mhz = 0;
    for (int rep = 0; rep < 4; ++rep) {
        const int it32 = 1 << 16, it64 = 1 << 14;
        float ms = 0;
        RG_CUDA(cudaEventRecord(e0));
        k_fma_peak<float><<<blocks, threads>>>((float *)out, it32, 1.0000001f, 1e-9f, cyc);
        RG_CUDA(cudaEventRecord(e1));
        RG_CUDA(cudaEventSynchronize(e1));
        RG_CUDA(cudaEventElapsedTime(&ms, e0, e1));
        double tf = (double)blocks * threads * it32 * 8.0 * 2.0 / (ms * 1e-3) / 1e12;
        if (rep && tf > best32) {
            best32 = tf;
            long long c = 0;
            RG_CUDA(cudaMemcpy(&c, cyc, sizeof(c), cudaMemcpyDeviceToHost));
            // the sampled block runs for the kernel's whole life only approximately; a clock estimate
            mhz = (double)c / (ms * 1e-3) / 1e6;
        }
        RG_CUDA(cudaEventRecord(e0));
        k_fma_peak<double><<<blocks, threads>>>((double *)out, it64, 1.0000001, 1e-9, nullptr);
        RG_CUDA(cudaEventRecord(e1));
        RG_CUDA(cudaEventSynchronize(e1));
        RG_CUDA(cudaEventElapsedTime(&ms, e0, e1));
        tf = (double)blocks * threads * it64 * 8.0 * 2.0 / (ms * 1e-3) / 1e12;
        if (rep && tf > best64) best64 = tf;
        // packed FFMA2 (fma.rn.f32x2): the same FP32 pipe, half the issue slots per flop
        RG_CUDA(cudaEventRecord(e0));
        k_ffma2_peak<<<blocks, threads>>>((float2 *)out, it32, make_float2(1.0000001f, 0.9999999f), make_float2(1e-9f, 1e-9f));
        RG_CUDA(cudaEventRecord(e1));
        RG_CUDA(cudaEventSynchronize(e1));
        RG_CUDA(cudaEventElapsedTime(&ms, e0, e1));
        tf = (double)blocks * threads * it32 * 8.0 * 4.0 / (ms * 1e-3) / 1e12;
        if (rep && tf > best32x2) best32x2 = tf;
    }
    cudaEventDestroy(e0);
    cudaEventDestroy(e1);
    cudaFree(out);
    cudaFree(cyc);
    if (fp32_tflops) *fp32_tflops = best32 > best32x2 ? best32 : best32x2;
    g_last_ffma2_tflops = best32x2;
    g_last_ffma_tflops = best32;
    if (getenv("RG_DEBUG_PEAKS")) fprintf(stderr, "peaks: FFMA %.2f TFLOP/s, FFMA2 %.2f TFLOP/s, DFMA %.2f TFLOP/s\n", best32, best32x2, best64);
    if (fp64_tflops) *fp64_tflops = best64;
    if (sm_clock_mhz) *sm_clock_mhz = mhz;
    return RG_OK;
}

}  // extern "C"
