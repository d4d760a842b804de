// rg_mega.cuh — validation pipeline: one thread per pixel, the reference's recursion
// (rendering.rs:71-130) unrolled into an explicit stack, brute-force FP64 Scene::trace.
// It is the device restatement the wavefront pipeline is cross-checked against on the GPU
// (both must produce identical bytes); it is not the performance path.
#pragma once
#include "rg_exact.cuh"

namespace rg {

struct MegaFrame {
    Ray pending;      // Refractive: the reflection ray, cast after the refraction returns
    C3 a;             // Reflecting: diffuse colour.  Refractive: surface colour
    C3 b;             // Refractive: refraction colour once known
    float p0, p1;     // reflectivity | kr, transparency
    uint8_t kind;     // RG_SURFACE_REFLECTING | RG_SURFACE_REFRACTIVE
    uint8_t stage;    // Refractive: 0 = refraction in flight, 1 = reflection in flight
};

// rendering.rs:132-172 with a full nearest-hit trace per light, exactly as written there.  MANY_LIGHTS (a scene with
// more than RG_MAX_LIGHTS lights): the lights come from the arena copy (DScene::light_all) instead of the constant
// bank.  (One kernel for both costs the common case 14 registers: lights read from global memory stay in registers
// across the trace, where constant-bank ones are read again.)
template <bool MANY_LIGHTS>
__device__ __forceinline__ C3 mega_shade_diffuse(const DScene &s, uint32_t body, D3 hp, D3 n,
                                                 DCounters *ctr, unsigned long long &n_shadow) {
    C3 bc = body_color_at(s, body, hp);
    float albedo = s.mat[body].albedo;
    C3 fin = c3(0.0f, 0.0f, 0.0f);
    for (uint32_t l = 0; l < s.n_lights; ++l) {
        const DLight &L = MANY_LIGHTS ? s.light_all[l] : s.lights[l];
        D3 dir = light_direction_from(L, hp);
        Ray shadow;
        shadow.o = hp + n * kShadowBias;
        shadow.d = dir;
        ++n_shadow;
        Nearest h = trace_exact_all(s, shadow, ctr);
        bool in_light = !h.found() || h.t > light_distance(L, hp);
        float a = fmaxf((float)dot(n, dir), 0.0f);
        fin = fin + light_term(bc, L, albedo, a, light_intensity(L, hp), in_light);
    }
    return clamp01(fin);
}

template <int STACK, bool MANY_LIGHTS>
__global__ void __launch_bounds__(128)
k_render_mega(DScene s, uint32_t width, uint32_t height, uint32_t y0, uint32_t y1, const uint32_t *__restrict__ rows,
              uchar4 *__restrict__ out, float *__restrict__ out_f32, DCounters *ctr) {
    const uint64_t npix = (uint64_t)(y1 - y0) * width;
    const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    unsigned long long cnt[4] = {0, 0, 0, 0};   // primary, shadow, reflection, transmission
    if (i < npix) {
        const uint32_t k = y0 + (uint32_t)(i / width);
        const uint32_t x = (uint32_t)(i - (uint64_t)(k - y0) * width);
        const uint32_t y = rows ? rows[k] : k;
        const C3 dflt = c3(s.default_color[0], s.default_color[1], s.default_color[2]);
        MegaFrame stack[STACK];
        int sp = 0;
        Ray ray = create_prime(s, x, y, width, height);
        int ray_kind = 0;
        C3 ret = dflt;
        bool calling = true;
        for (;;) {
            if (calling) {
                // cast_ray (rendering.rs:122-130); the primary ray is always traced (:71-78)
                if (sp > 0 && (uint32_t)sp >= s.max_depth) { ret = dflt; calling = false; continue; }
                ++cnt[ray_kind];
                Nearest h = trace_exact_all(s, ray, ctr);
                if (!h.found()) { ret = dflt; calling = false; continue; }
                // get_color (rendering.rs:80-120)
                D3 hp = ray.o + ray.d * h.t;
                D3 n = surface_normal(s, h.body, hp, ctr);
                const BodyMat &m = s.mat[h.body];
                if (m.surface == RG_SURFACE_DIFFUSE) {
                    ret = mega_shade_diffuse<MANY_LIGHTS>(s, h.body, hp, n, ctr, cnt[1]);
                    calling = false;
                } else if (m.surface == RG_SURFACE_REFLECTING) {
                    MegaFrame &f = stack[sp++];
                    f.kind = RG_SURFACE_REFLECTING;
                    f.p0 = m.p0;
                    f.a = mega_shade_diffuse<MANY_LIGHTS>(s, h.body, hp, n, ctr, cnt[1]);
                    ray = create_reflection(n, ray.d, hp);
                    ray_kind = 2;
                } else {
                    MegaFrame &f = stack[sp++];
                    f.kind = RG_SURFACE_REFRACTIVE;
                    float kr = (float)fresnel(ray.d, n, m.p0);
                    f.p0 = kr;
                    f.p1 = m.p1;
                    f.a = body_color_at(s, h.body, hp);
                    f.pending = create_reflection(n, ray.d, hp);
                    f.b = dflt;
                    f.stage = 1;
                    Ray tr;
                    bool go_refract = false;
                    if (kr < 1.0f) {
                        if (create_transmission(n, ray.d, hp, kShadowBias, m.p0, tr)) go_refract = true;
                        else atomicAdd(&ctr->err_trans, 1ull);   // rendering.rs:106 unwrap() on None
                    }
                    if (go_refract) { f.stage = 0; ray = tr; ray_kind = 3; }
                    else { ray = f.pending; ray_kind = 2; }
                }
            } else {
                if (sp == 0) break;
                MegaFrame &f = stack[sp - 1];
                if (f.kind == RG_SURFACE_REFLECTING) {
                    ret = (f.a * (1.0f - f.p0)) + (ret * f.p0);          // rendering.rs:92-93
                    --sp;
                } else if (f.stage == 0) {
                    f.b = ret;
                    f.stage = 1;
                    ray = f.pending;
                    ray_kind = 2;
                    calling = true;
                } else {
                    C3 col = (ret * f.p0) + (f.b * (1.0f - f.p0));        // rendering.rs:115
                    ret = (col * f.p1) * f.a;                             // rendering.rs:116
                    --sp;
                }
            }
        }
        if (out_f32) { out_f32[3 * i] = ret.r; out_f32[3 * i + 1] = ret.g; out_f32[3 * i + 2] = ret.b; }   // RenderedPixel.color
        else out[i] = quantise(ret);
    }
    // ray counters: warp-reduce, one atomic per warp per type
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        unsigned long long v = cnt[k];
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
        if ((threadIdx.x & 31) == 0 && v) atomicAdd(&ctr->rays[k], v);
    }
}

}  // namespace rg
