// rg_trace.cuh — Scene::trace (scene.rs:34-39) for a queue of rays: the hot loop.
//
// k_trace_brute is the reference algorithm — every ray against every body — arranged for
// the B200:
//   * the sphere list is streamed through shared memory in chunks by 1-D bulk async copies
//     (cp.async.bulk + mbarrier, double-buffered), one 16-byte FP32 cull record per sphere;
//   * each thread owns R rays (register-tiled), so one broadcast LDS.128 feeds 32*R tests;
//   * a test is a CONSERVATIVE reject in FP32 (rg_cull.h); two spheres are tested per
//     instruction with Blackwell's packed FFMA2 (fma.rn.f32x2): 7 FFMA2 + one FMNMX.NAN + one FSETP per
//     ray and sphere pair; the loop is software-pipelined by hand (see k_trace_brute_resident);
//   * the rare survivors are not evaluated in the divergent inner loop: they are appended
//     to a per-warp candidate queue with __ballot_sync/__popc and evaluated 32 at a time,
//     one candidate per lane, with the reference's exact FP64 test (rg_exact.cuh);
//   * the per-ray result is the lexicographic min of (distance, original body index), the
//     order-independent form of min_by's first-minimum rule.
// ANY = true is the shadow-ray variant: shade_diffuse only asks whether the nearest hit is
// farther than the light (rendering.rs:150-155), which is false exactly when SOME body is
// hit at t <= light.distance; so any such hit decides and no minimum is needed.
#pragma once
#include <cstdio>
#include "rg_cull.h"
#include "rg_exact.cuh"

namespace rg {

constexpr int kTraceThreads = 256;
constexpr int kTraceWarps = kTraceThreads / 32;
constexpr int kChunkSpheres = 1024;                 // 16 KB per stage
constexpr int kCullPad = 4;                         // cull4[] is padded to a multiple of this
constexpr int kSlotBits = 10;                       // local ray slot: r * 256 + tid  (R <= 4)

struct RayQueue {            // 3 x double2 per ray: (ox,oy) (oz,dx) (dy,dz) — 128-bit coalesced traffic
    double2 *a, *b, *c;
    uint32_t *hint;          // per ray, from the kernel that made it (k_shade): see kHintOccluded / origin_hint
};
constexpr size_t kRayBytes = 48 + 4;     // bytes of queue storage per ray

// Origin hints.  A secondary ray starts on the body it leaves, 1e-13 outside (or inside) its surface: far too
// close for the FP32 cull to tell, so the grid tracer used to spend one exact FP64 test per ray on that sphere
// just to learn "behind the origin" (a third of all its exact tests, measured).  k_shade knows the body, runs the
// reference's test (sphere_intersect, the same function on the same FP64 ray the tracer would load) once, at
// full lane occupancy, and leaves the outcome with the ray:
//   a sphere-list index   that sphere returns None (or, for a shadow ray, a hit beyond the light) for this ray:
//                         the tracer may skip it — Scene::trace is a minimum, a None contributes nothing;
//   kHintOccluded         (shadow rays) the ray's own sphere is hit before the light: shade_diffuse's answer is
//                         "not in light" whatever else the ray meets (rendering.rs:150-155);
//   0xFFFFFFFF            nothing known.
// Trace kernels are free to ignore hints (the brute-force ones do): the result is the same.
constexpr uint32_t kHintNone = 0xFFFFFFFFu;
constexpr uint32_t kHintOccluded = 0xFFFFFFFEu;

struct TraceArgs {
    RayQueue q;
    const double *tmax;      // ANY: light.distance(hit_point) per ray
    uint32_t n;              // capacity of the queue: an upper bound of the ray count
    uint32_t seg_stride;     // light-major shadow queues: ray i lives at (i / seg_len) * seg_stride + i % seg_len
    const unsigned int *seg_len_dev;   // ... with seg_len (= lit hits of the level) read from device memory; nullptr: dense
    double *out_t;           // nearest: distance (undefined when body == kNoBody)
    uint32_t *out_body;      // nearest: original body index or kNoBody
    uint8_t *out_lit;        // ANY: 1 = in light
    DCounters *ctr;
    unsigned int *fetch;     // persistent kernels: the ray counter of THIS launch (one per level and kind, zeroed per batch)
    const unsigned int *n_dev;   // the ray count is *n_dev * n_mul, read from device memory (a launch issued
                                 // before the host knows it)
    uint32_t n_mul;              // path queues: 1; shadow queues: lights per lit hit
    const unsigned int *void_flag;   // if set and non-zero, the frame is void (a queue overflowed): trace nothing
    int verify;              // RG_OPT_VERIFY_CULL
    int g_refill, g_quorum, g_burst;   // persistent grid kernel tuning (rg_grid.cuh)
};

// Number of rays this launch has to trace (see TraceArgs::n_dev).
__device__ __forceinline__ uint32_t ray_count(const TraceArgs &a) {
    if (a.void_flag && *a.void_flag) return 0u;
    const unsigned long long v = (unsigned long long)*a.n_dev * a.n_mul;
    return v < a.n ? (uint32_t)v : a.n;
}

// Path queues are dense (seg_len = 0, no seg_len_dev).  Shadow queues hold one segment per light so that
// neighbouring lanes trace neighbouring hits towards the SAME light (coherent origins AND directions:
// measured -23 % on the all-diffuse C3 frame, -4 % on C4 against hit-major order).
__device__ __forceinline__ uint32_t segment_length(const TraceArgs &a) {
    if (!a.seg_len_dev) return 0u;
    const uint32_t v = *a.seg_len_dev;
    return v < a.seg_stride ? v : a.seg_stride;
}
__device__ __forceinline__ uint32_t phys_index(uint32_t seg_len, uint32_t seg_stride, uint32_t i) {
    return seg_len ? (i / seg_len) * seg_stride + (i % seg_len) : i;
}
__device__ __forceinline__ Ray load_ray(const RayQueue &q, uint32_t i) {
    double2 a = q.a[i], b = q.b[i], c = q.c[i];
    Ray r;
    r.o = d3(a.x, a.y, b.x);
    r.d = d3(b.y, c.x, c.y);
    return r;
}
__device__ __forceinline__ void store_ray(const RayQueue &q, uint32_t i, const Ray &r) {
    q.a[i] = make_double2(r.o.x, r.o.y);
    q.b[i] = make_double2(r.o.z, r.d.x);
    q.c[i] = make_double2(r.d.y, r.d.z);
}

// ---- mbarrier / bulk-copy primitives (sm_90+ PTX; SASS: SYNCS.*, UBLKCP) ------------------
__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t *bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t *bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t *bar, uint32_t parity) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "WAIT_%=:\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
        "@p bra DONE_%=;\n\t"
        "bra WAIT_%=;\n\t"
        "DONE_%=:\n\t}" ::"r"(smem_u32(bar)), "r"(parity) : "memory");
}
__device__ __forceinline__ void bulk_g2s(void *dst_smem, const void *src_gmem, uint32_t bytes, uint64_t *bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                     smem_u32(dst_smem)),
                 "l"(src_gmem), "r"(bytes), "r"(smem_u32(bar))
                 : "memory");
}

// max that returns NaN when either operand is NaN (SASS FMNMX.NAN); fmaxf would drop the NaN
__device__ __forceinline__ float max_nan(float a, float b) {
    float d;
    asm("max.NaN.f32 %0, %1, %2;" : "=f"(d) : "f"(a), "f"(b));
    return d;
}
__device__ __forceinline__ float4 lds128(uint32_t shared_addr) {
    float4 v;
    asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(shared_addr));
    return v;
}

// Per-ray constants of the FP32 cull (rg_cull.h), derived once from the FP64 ray.
struct CullRay {
    float dx, dy, dz, nod;      // d, -(o'.d)
    float o2x, o2y, o2z, thr;   // -2 o', -|o'|^2 + m_r   (thr = +inf: never reject)
};
__device__ __forceinline__ CullRay make_cull_ray(const DScene &s, const Ray &ray, bool active) {
    CullRay c;
    D3 op = ray.o - d3(s.cull_ref[0], s.cull_ref[1], s.cull_ref[2]);
    double O2 = dot(op, op), D2 = dot(ray.d, ray.d), od = dot(op, ray.d);
    bool cullable = fabs(D2 - 1.0) <= kCullUnitTol && O2 < kCullHuge;    // false on NaN
    c.dx = (float)ray.d.x; c.dy = (float)ray.d.y; c.dz = (float)ray.d.z;
    c.nod = (float)(-od);
    c.o2x = (float)(-2.0 * op.x); c.o2y = (float)(-2.0 * op.y); c.o2z = (float)(-2.0 * op.z);
    c.thr = cullable ? (float)(-O2 + kCullU * kCullRayO2 * O2) : __int_as_float(0x7f800000);
    if (!active) {   // a lane without a ray rejects everything it can
        c.dx = c.dy = c.dz = c.nod = c.o2x = c.o2y = c.o2z = 0.0f;
        c.thr = __int_as_float(0xff800000);
    }
    return c;
}
// true = the sphere is certainly missed (the reference's `opp2 > r2` holds); false = must be
// tested exactly.  NaN anywhere compares false, i.e. "test exactly".
__device__ __forceinline__ bool cull_reject(const CullRay &c, float4 sp) {
    float s = fmaf(sp.x, c.dx, fmaf(sp.y, c.dy, fmaf(sp.z, c.dz, c.nod)));
    float q = fmaf(sp.x, c.o2x, fmaf(sp.y, c.o2y, fmaf(sp.z, c.o2z, sp.w)));
    float g = fmaf(-s, s, q);
    return g > c.thr;
}

// ---- packed form: two spheres per instruction (sm_100 FFMA2) --------------------------------
// The brute-force kernel reads the records pair-interleaved: for spheres (2k, 2k+1)
//     A = (x0, x1, y0, y1)      B = (z0, z1, -K0, -K1)
// and evaluates h = s*s - q = -g with every per-ray constant of the q-chain negated, which is
// bit-for-bit the negation of the scalar form (round-to-nearest is symmetric), so
// "g > thr"  <=>  "h < -thr": the decisions, and the soundness argument, are unchanged.
struct CullRay2 {
    float2 dx, dy, dz, nod;     // (d, d), (-(o'.d), -(o'.d))
    float2 px, py, pz;          // +2 o' duplicated  (= -o2)
    float nthr;                 // -thr   (-inf: never reject;  +inf: lane without a ray)
};
__device__ __forceinline__ CullRay2 make_cull_ray2(const CullRay &c) {
    CullRay2 p;
    p.dx = make_float2(c.dx, c.dx); p.dy = make_float2(c.dy, c.dy); p.dz = make_float2(c.dz, c.dz);
    p.nod = make_float2(c.nod, c.nod);
    p.px = make_float2(-c.o2x, -c.o2x); p.py = make_float2(-c.o2y, -c.o2y); p.pz = make_float2(-c.o2z, -c.o2z);
    p.nthr = -c.thr;
    return p;
}
// h for the two spheres of a pair: (h.x < nthr) = sphere 2k rejected, (h.y < nthr) = sphere 2k+1.
__device__ __forceinline__ float2 cull_h2(const CullRay2 &c, float4 A, float4 B) {
    const float2 X = make_float2(A.x, A.y), Y = make_float2(A.z, A.w), Z = make_float2(B.x, B.y), NK = make_float2(B.z, B.w);
    const float2 s = __ffma2_rn(X, c.dx, __ffma2_rn(Y, c.dy, __ffma2_rn(Z, c.dz, c.nod)));
    const float2 nq = __ffma2_rn(X, c.px, __ffma2_rn(Y, c.py, __ffma2_rn(Z, c.pz, NK)));
    return __ffma2_rn(s, s, nq);
}
// the scalar decision for one sphere of a pair, from the packed constants (rare path)
__device__ __forceinline__ bool cull_reject_half(const CullRay2 &c, float4 A, float4 B, int half) {
    const float x = half ? A.y : A.x, y = half ? A.w : A.z, z = half ? B.y : B.x, nk = half ? B.w : B.z;
    const float s = fmaf(x, c.dx.x, fmaf(y, c.dy.x, fmaf(z, c.dz.x, c.nod.x)));
    const float nq = fmaf(x, c.px.x, fmaf(y, c.py.x, fmaf(z, c.pz.x, nk)));
    return fmaf(s, s, nq) < c.nthr;
}

template <bool ANY, int R, int U, int MINB>
__global__ void __launch_bounds__(kTraceThreads, MINB)
k_trace_brute(const DScene s, const TraceArgs a) {
    static_assert(R * kTraceThreads <= (1 << kSlotBits), "slot bits");
    static_assert(U == 2 || U == 4, "U spheres = U/2 pairs per iteration");
    static_assert(kCullPad % U == 0 && U <= kCullPad, "records are padded to kCullPad");
    __shared__ __align__(128) float4 stage[2][kChunkSpheres + 3 * kCullPad];   // + slack for the prefetch (two groups ahead)
    __shared__ uint64_t mbar[2];
    __shared__ uint32_t cq[kTraceWarps][64];
    __shared__ double best_t[R * kTraceThreads];
    __shared__ uint32_t best_b[R * kTraceThreads];   // nearest: body; ANY: 1 = occluded
    __shared__ uint8_t tag[R * kTraceThreads];

    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const uint32_t block_base = blockIdx.x * (uint32_t)(R * kTraceThreads);
    const uint32_t n_rays = ray_count(a);
    if (block_base >= n_rays) return;   // device-sized launches cover the queue's capacity: surplus blocks leave at once
    const uint32_t seg_len = segment_length(a);
    const uint32_t lanemask_lt = (1u << lane) - 1u;
    const uint32_t nsph = s.n_spheres;
    const uint32_t nchunks = (nsph + kChunkSpheres - 1) / kChunkSpheres;
    unsigned long long n_exact = 0;
    unsigned nan_count = 0, unsound = 0;

    auto chunk_records = [&](uint32_t c) -> uint32_t {
        uint32_t cnt = nsph - c * kChunkSpheres;
        if (cnt > (uint32_t)kChunkSpheres) cnt = kChunkSpheres;
        return (cnt + kCullPad - 1) / kCullPad * kCullPad;
    };
    if (tid == 0) {
        mbar_init(&mbar[0], 1);
        mbar_init(&mbar[1], 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();
    if (tid == 0 && nchunks > 0) {
        uint32_t bytes = chunk_records(0) * 16u;
        mbar_expect_tx(&mbar[0], bytes);
        bulk_g2s(&stage[0][0], s.cull2, bytes, &mbar[0]);
    }

    // ---- prologue: my R rays; the few non-sphere bodies are tested exactly right here
    CullRay2 cr[R];
#pragma unroll
    for (int r = 0; r < R; ++r) {
        const uint32_t slot = r * kTraceThreads + tid;
        const uint32_t i = block_base + slot;
        const bool active = i < n_rays;
        Ray ray;
        ray.o = d3(0, 0, 0);
        ray.d = d3(0, 0, 0);
        const uint32_t pi = active ? phys_index(seg_len, a.seg_stride, i) : 0u;
        if (active) ray = load_ray(a.q, pi);
        cr[r] = make_cull_ray2(make_cull_ray(s, ray, active));
        Nearest best;
        best.init();
        bool occluded = false;
        if (active) {
            const double tmax = ANY ? a.tmax[pi] : 0.0;
            for (uint32_t m = 0; m < s.n_misc; ++m) {
                uint32_t b = s.misc_body[m];
                double t;
                if (misc_intersect(s, b, ray, t)) {
                    if (t != t) { ++nan_count; continue; }
                    if (ANY) occluded = occluded || (t <= tmax);
                    else best.offer(t, b);
                }
            }
            n_exact += s.n_misc;
        }
        best_t[slot] = best.t;
        best_b[slot] = ANY ? (occluded ? 1u : 0u) : best.body;
    }
    uint32_t qn = 0;   // warp-uniform: candidates waiting in cq[warp]

    // Evaluates candidates cq[warp][first .. first+count) — one per lane — exactly.
    auto drain = [&](uint32_t first, uint32_t count) {
        bool have = (uint32_t)lane < count;
        uint32_t slot = 0, sph = 0;
        bool hit = false;
        double t = 0.0;
        if (have) {
            uint32_t e = cq[warp][first + lane];
            slot = e & ((1u << kSlotBits) - 1u);
            sph = e >> kSlotBits;
            Ray ray = load_ray(a.q, phys_index(seg_len, a.seg_stride, block_base + slot));
            double4 sp = s.sph[sph];
            hit = sphere_intersect(sp.x, sp.y, sp.z, sp.w, ray, t);
            ++n_exact;
            if (hit && t != t) { ++nan_count; hit = false; }
#ifdef RG_DEBUG_DRAIN
            if (hit && t == 0.0) printf("drain: ray %u slot %u sph %u o=(%.17g,%.17g,%.17g) d=(%.17g,%.17g,%.17g) sp=(%.17g,%.17g,%.17g,%.17g)\n", block_base + slot, slot, sph, ray.o.x, ray.o.y, ray.o.z, ray.d.x, ray.d.y, ray.d.z, sp.x, sp.y, sp.z, sp.w);
#endif
        }
        if (ANY) {
            if (hit && t <= a.tmax[phys_index(seg_len, a.seg_stride, block_base + slot)]) best_b[slot] = 1u;   // benign race: all write 1
        } else {
            const uint32_t body = hit ? s.sph_body[sph] : 0u;
            bool pend = hit;
            while (__any_sync(0xffffffffu, pend)) {      // serialise candidates of the same ray
                if (pend) tag[slot] = (uint8_t)lane;
                __syncwarp();
                if (pend && tag[slot] == (uint8_t)lane) {
                    Nearest cur;
                    cur.t = best_t[slot];
                    cur.body = best_b[slot];
                    cur.offer(t, body);
                    best_t[slot] = cur.t;
                    best_b[slot] = cur.body;
                    pend = false;
                }
                __syncwarp();
            }
        }
    };

    // ---- main loop: stream the cull records through shared memory
    for (uint32_t c = 0; c < nchunks; ++c) {
        const uint32_t st = c & 1u;
        if (tid == 0 && c + 1 < nchunks) {   // prefetch the next chunk into the other stage
            asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
            uint32_t bytes = chunk_records(c + 1) * 16u;
            mbar_expect_tx(&mbar[st ^ 1u], bytes);
            bulk_g2s(&stage[st ^ 1u][0], s.cull2 + (size_t)(c + 1) * kChunkSpheres, bytes, &mbar[st ^ 1u]);
        }
        mbar_wait(&mbar[st], (c >> 1) & 1u);
        const uint32_t cnt = chunk_records(c);
        const uint32_t sph_base = c * kChunkSpheres;
        const float4 *sp = stage[st];
        // Rare path for the group of U records starting at j0: re-run the U*R cull tests (cheaper
        // than keeping U*R flags live in the hot loop), queue the survivors with warp ballot /
        // popc compaction, evaluate them exactly 32 at a time.
        auto survivors = [&](uint32_t j0) {
#pragma unroll
            for (int u = 0; u < U; ++u) {
                const uint32_t sph = sph_base + j0 + u;
                const float4 A = sp[(j0 + u) & ~1u], B = sp[((j0 + u) & ~1u) + 1];
#pragma unroll
                for (int r = 0; r < R; ++r) {
                    const uint32_t slot = r * kTraceThreads + tid;
                    const bool live = (block_base + slot < n_rays) && sph < nsph;
                    const bool rej = cull_reject_half(cr[r], A, B, (j0 + u) & 1);
                    const bool pass = live && !rej;
                    if (a.verify && live && rej) {   // debug: a culled pair must miss exactly
                        Ray ray = load_ray(a.q, phys_index(seg_len, a.seg_stride, block_base + slot));
                        double4 e = s.sph[sph];
                        double t;
                        if (sphere_intersect(e.x, e.y, e.z, e.w, ray, t)) ++unsound;
                    }
                    const uint32_t mask = __ballot_sync(0xffffffffu, pass);
                    if (mask) {
                        if (pass) cq[warp][qn + __popc(mask & lanemask_lt)] = (sph << kSlotBits) | slot;
                        qn += __popc(mask);
                        __syncwarp();
                        if (qn >= 32u) {
                            drain(qn - 32u, 32u);
                            qn -= 32u;
                            __syncwarp();
                        }
                    }
                }
            }
        };
        // Hot loop: the software-pipelined form of k_trace_brute_resident (see there): one reject predicate per group from
        // NaN-propagating maxima, the h values kept in registers for the rare survivor, records addressed by their
        // shared-window address, a group's vote + branch issued behind the next group's FFMA2s.
        auto enqueue = [&](bool pass, uint32_t sph, uint32_t slot) {
            const uint32_t mask = __ballot_sync(0xffffffffu, pass);
            if (mask) {
                if (pass) cq[warp][qn + __popc(mask & lanemask_lt)] = (sph << kSlotBits) | slot;
                qn += __popc(mask);
                __syncwarp();
                if (qn >= 32u) {
                    drain(qn - 32u, 32u);
                    qn -= 32u;
                    __syncwarp();
                }
            }
        };
        auto test_group = [&](const float4 (&sc)[U], float2 (&hh)[R][U / 2]) -> bool {
            bool all_rej = true;
#pragma unroll
            for (int r = 0; r < R; ++r) {
#pragma unroll
                for (int u = 0; u < U; u += 2) {
                    hh[r][u / 2] = cull_h2(cr[r], sc[u], sc[u + 1]);
                    all_rej = all_rej & (max_nan(hh[r][u / 2].x, hh[r][u / 2].y) < cr[r].nthr);
                }
            }
            return !all_rej;
        };
        auto collect = [&](const float2 (&hh)[R][U / 2], uint32_t j) {
#pragma unroll
            for (int r = 0; r < R; ++r) {
                bool pass_r = false;
#pragma unroll
                for (int u = 0; u < U; u += 2) pass_r = pass_r | !(hh[r][u / 2].x < cr[r].nthr) | !(hh[r][u / 2].y < cr[r].nthr);
                if (__any_sync(0xffffffffu, pass_r)) {
                    const uint32_t slot = r * kTraceThreads + tid;
                    const bool live = block_base + slot < n_rays;
#pragma unroll
                    for (int u = 0; u < U; u += 2) {
                        const uint32_t sph = sph_base + j + u;
                        enqueue(live && sph < nsph && !(hh[r][u / 2].x < cr[r].nthr), sph, slot);
                        enqueue(live && sph + 1 < nsph && !(hh[r][u / 2].y < cr[r].nthr), sph + 1, slot);
                    }
                }
            }
        };
        if (a.verify) {   // debug form of the loop: every culled pair is re-tested exactly (survivors())
#pragma unroll 1
            for (uint32_t j = 0; j < cnt; j += U) survivors(j);
        } else {
            uint32_t saddr = smem_u32(sp);
            float4 s0[U], s1[U];
            float2 hA[R][U / 2], hB[R][U / 2];
            bool fB = false;
            uint32_t jB = 0;
#pragma unroll
            for (int u = 0; u < U; ++u) s0[u] = lds128(saddr + 16u * u);
#pragma unroll 1
            for (uint32_t j = 0; j < cnt; j += 2 * U, saddr += 32u * U) {
#pragma unroll
                for (int u = 0; u < U; ++u) s1[u] = lds128(saddr + 16u * (U + u));       // (the stage has 3 kCullPad records of slack)
                const bool fA = test_group(s0, hA);
                if (__any_sync(0xffffffffu, fB)) collect(hB, jB);                        // the previous turn's second group
                fB = false;
                if (j + U < cnt) {
#pragma unroll
                    for (int u = 0; u < U; ++u) s0[u] = lds128(saddr + 16u * (2 * U + u));
                    fB = test_group(s1, hB);
                    jB = j + U;
                }
                if (__any_sync(0xffffffffu, fA)) collect(hA, j);
            }
            if (__any_sync(0xffffffffu, fB)) collect(hB, jB);
        }
        __syncthreads();   // everyone is done with stage[st] before it is refilled
    }
    if (qn) drain(0u, qn);
    __syncwarp();

    // ---- epilogue
#pragma unroll
    for (int r = 0; r < R; ++r) {
        const uint32_t slot = r * kTraceThreads + tid;
        const uint32_t i = block_base + slot;
        if (i < n_rays) {
            const uint32_t pi = phys_index(seg_len, a.seg_stride, i);
            if (ANY) a.out_lit[pi] = best_b[slot] ? 0 : 1;
            else { a.out_t[pi] = best_t[slot]; a.out_body[pi] = best_b[slot]; }
        }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        n_exact += __shfl_xor_sync(0xffffffffu, n_exact, o);
        nan_count += __shfl_xor_sync(0xffffffffu, nan_count, o);
        unsound += __shfl_xor_sync(0xffffffffu, unsound, o);
    }
    if (lane == 0) {
        if (n_exact) atomicAdd(&a.ctr->exact_tests, n_exact);
        if (nan_count) atomicAdd(&a.ctr->err_nan, (unsigned long long)nan_count);
        if (unsound) atomicAdd(&a.ctr->cull_unsound, (unsigned long long)unsound);
    }
}

// ---- the same scan with the WHOLE cull array resident in shared memory ----------------------
// When every sphere's 16-byte cull record fits in one SM's shared memory (<= ~11,000 spheres in
// the 227 KB a CTA may use), the chunk pipeline above is unnecessary — and so is its block-wide
// barrier per chunk, which is where the streaming kernel loses its time on incoherent bounces
// (warps whose rays produce more exact tests arrive late; ncu: barrier = 24 % of the stall
// samples of a deep level, 2.9 % at level 0).  Here one persistent 1024-thread CTA per SM loads the
// array ONCE (bulk async copies on one mbarrier), after which its 32 warps never synchronise with
// each other again: each warp pulls tiles of 32*R rays from a global counter, scans all records,
// evaluates its own survivors and writes its own results.  The arithmetic and the survivor logic
// are the streaming kernel's, so results are identical.
// dynamic shared memory: records (+ slack) | per-warp best_t, best_b, cq, tag
__host__ __device__ inline size_t resident_smem_bytes(uint32_t n_records, int R, int warps) {
    const size_t rec = ((size_t)n_records + kCullPad) * 16;
    const size_t per_warp = (size_t)32 * R * (8 + 4 + 1) + 64 * 4;
    return rec + (size_t)warps * ((per_warp + 15) & ~(size_t)15) + 16;
}

// T threads per CTA (one CTA per SM); PF = software prefetch of the next U records (costs U float4 of registers)
template <bool ANY, int R, int U, int T, bool PF>
__global__ void __launch_bounds__(T, 1)
k_trace_brute_resident(const DScene s, const TraceArgs a, const uint32_t n_records) {
    static_assert(U == 2 || U == 4, "U spheres = U/2 pairs per iteration");
    static_assert(32 * R <= (1 << kSlotBits), "slot bits");
    extern __shared__ __align__(128) unsigned char smem_raw[];
    __shared__ uint64_t mbar;
    float4 *stage = reinterpret_cast<float4 *>(smem_raw);
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    constexpr size_t kPerWarp = (((size_t)32 * R * (8 + 4 + 1) + 64 * 4) + 15) & ~(size_t)15;
    unsigned char *mine = smem_raw + ((size_t)n_records + kCullPad) * 16 + (size_t)warp * kPerWarp;
    double *best_t = reinterpret_cast<double *>(mine);                        // [32 R]
    uint32_t *best_b = reinterpret_cast<uint32_t *>(mine + 32 * R * 8);       // [32 R] nearest: body; ANY: 1 = occluded
    uint32_t *cq = reinterpret_cast<uint32_t *>(mine + 32 * R * 12);          // [64]
    uint8_t *tag = reinterpret_cast<uint8_t *>(mine + 32 * R * 12 + 64 * 4);  // [32 R]

    const uint32_t lanemask_lt = (1u << lane) - 1u;
    const uint32_t nsph = s.n_spheres;
    const uint32_t n_rays = ray_count(a);
    if (n_rays == 0) return;   // an empty level of a device-sized frame: do not even load the records
    const uint32_t seg_len = segment_length(a);
    unsigned long long n_exact = 0;
    unsigned nan_count = 0, unsound = 0;

    if (tid == 0) {
        mbar_init(&mbar, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        const uint32_t total = n_records * 16u;
        mbar_expect_tx(&mbar, total);
        for (uint32_t off = 0; off < total; off += 16384u) {
            const uint32_t bytes = total - off < 16384u ? total - off : 16384u;
            bulk_g2s(reinterpret_cast<unsigned char *>(stage) + off, reinterpret_cast<const unsigned char *>(s.cull2) + off, bytes, &mbar);
        }
    }
    __syncthreads();          // the barrier is initialised before anyone waits on it
    mbar_wait(&mbar, 0u);     // ... and this is the last time the warps of this CTA meet
    const float4 *sp = stage;
    const uint32_t cnt = n_records;

    for (;;) {
        uint32_t tile = 0;
        if (lane == 0) tile = atomicAdd(a.fetch, 1u);
        tile = __shfl_sync(0xffffffffu, tile, 0);
        const uint64_t base64 = (uint64_t)tile * (32u * R);
        if (base64 >= n_rays) break;
        const uint32_t tile_base = (uint32_t)base64;

        // ---- prologue: my R rays; the few non-sphere bodies are tested exactly right here
        CullRay2 cr[R];
#pragma unroll
        for (int r = 0; r < R; ++r) {
            const uint32_t slot = r * 32 + lane;
            const uint32_t i = tile_base + slot;
            const bool active = i < n_rays;
            Ray ray;
            ray.o = d3(0, 0, 0);
            ray.d = d3(0, 0, 0);
            const uint32_t pi = active ? phys_index(seg_len, a.seg_stride, i) : 0u;
            if (active) ray = load_ray(a.q, pi);
            cr[r] = make_cull_ray2(make_cull_ray(s, ray, active));
            Nearest best;
            best.init();
            bool occluded = false;
            if (active) {
                const double tmax = ANY ? a.tmax[pi] : 0.0;
                for (uint32_t m = 0; m < s.n_misc; ++m) {
                    uint32_t b = s.misc_body[m];
                    double t;
                    if (misc_intersect(s, b, ray, t)) {
                        if (t != t) { ++nan_count; continue; }
                        if (ANY) occluded = occluded || (t <= tmax);
                        else best.offer(t, b);
                    }
                }
                n_exact += s.n_misc;
            }
            best_t[slot] = best.t;
            best_b[slot] = ANY ? (occluded ? 1u : 0u) : best.body;
        }
        __syncwarp();
        uint32_t qn = 0;   // warp-uniform: candidates waiting in cq

        // Evaluates candidates cq[first .. first+count) — one per lane — exactly.
        auto drain = [&](uint32_t first, uint32_t count) {
            bool have = (uint32_t)lane < count;
            uint32_t slot = 0, sph = 0;
            bool hit = false;
            double t = 0.0;
            if (have) {
                uint32_t e = cq[first + lane];
                slot = e & ((1u << kSlotBits) - 1u);
                sph = e >> kSlotBits;
                Ray ray = load_ray(a.q, phys_index(seg_len, a.seg_stride, tile_base + slot));
                double4 e4 = s.sph[sph];
                hit = sphere_intersect(e4.x, e4.y, e4.z, e4.w, ray, t);
                ++n_exact;
                if (hit && t != t) { ++nan_count; hit = false; }
            }
            if (ANY) {
                if (hit && t <= a.tmax[phys_index(seg_len, a.seg_stride, tile_base + slot)]) best_b[slot] = 1u;   // benign race: all write 1
            } else {
                const uint32_t body = hit ? s.sph_body[sph] : 0u;
                bool pend = hit;
                while (__any_sync(0xffffffffu, pend)) {      // serialise candidates of the same ray
                    if (pend) tag[slot] = (uint8_t)lane;
                    __syncwarp();
                    if (pend && tag[slot] == (uint8_t)lane) {
                        Nearest cur;
                        cur.t = best_t[slot];
                        cur.body = best_b[slot];
                        cur.offer(t, body);
                        best_t[slot] = cur.t;
                        best_b[slot] = cur.body;
                        pend = false;
                    }
                    __syncwarp();
                }
            }
        };
        // Rare path for the group of U records starting at j0 (see k_trace_brute).
        auto survivors = [&](uint32_t j0) {
#pragma unroll
            for (int u = 0; u < U; ++u) {
                const uint32_t sph = j0 + u;
                const float4 A = sp[(j0 + u) & ~1u], B = sp[((j0 + u) & ~1u) + 1];
#pragma unroll
                for (int r = 0; r < R; ++r) {
                    const uint32_t slot = r * 32 + lane;
                    const bool live = (tile_base + slot < n_rays) && sph < nsph;
                    const bool rej = cull_reject_half(cr[r], A, B, (j0 + u) & 1);
                    const bool pass = live && !rej;
                    if (a.verify && live && rej) {   // debug: a culled pair must miss exactly
                        Ray ray = load_ray(a.q, phys_index(seg_len, a.seg_stride, tile_base + slot));
                        double4 e = s.sph[sph];
                        double t;
                        if (sphere_intersect(e.x, e.y, e.z, e.w, ray, t)) ++unsound;
                    }
                    const uint32_t mask = __ballot_sync(0xffffffffu, pass);
                    if (mask) {
                        if (pass) cq[qn + __popc(mask & lanemask_lt)] = (sph << kSlotBits) | slot;
                        qn += __popc(mask);
                        __syncwarp();
                        if (qn >= 32u) {
                            drain(qn - 32u, 32u);
                            qn -= 32u;
                            __syncwarp();
                        }
                    }
                }
            }
        };
        // Appends the (ray slot, sphere) pairs of the lanes with `pass` to the candidate queue.
        auto enqueue = [&](bool pass, uint32_t sph, uint32_t slot) {
            const uint32_t mask = __ballot_sync(0xffffffffu, pass);
            if (mask) {
                if (pass) cq[qn + __popc(mask & lanemask_lt)] = (sph << kSlotBits) | slot;
                qn += __popc(mask);
                __syncwarp();
                if (qn >= 32u) {
                    drain(qn - 32u, 32u);
                    qn -= 32u;
                    __syncwarp();
                }
            }
        };
        // One group of U records (spheres j .. j+U-1) against my R rays: the h values (kept in registers) and whether
        // every one of them is below its ray's threshold.  both rejected <=> max(h.x, h.y) < nthr; the NaN-propagating
        // max keeps "NaN = test exactly".
        auto test_group = [&](const float4 (&sc)[U], float2 (&hh)[R][U / 2]) -> bool {
            bool all_rej = true;
#pragma unroll
            for (int r = 0; r < R; ++r) {
#pragma unroll
                for (int u = 0; u < U; u += 2) {
                    hh[r][u / 2] = cull_h2(cr[r], sc[u], sc[u + 1]);
                    all_rej = all_rej & (max_nan(hh[r][u / 2].x, hh[r][u / 2].y) < cr[r].nthr);
                }
            }
            return !all_rej;
        };
        // The rare half (8 % of the groups hold a survivor): a ballot per ray and an append for each pair that passed,
        // from the h values still in registers — not a scalar re-run of all U * R tests, which used to be ~20 % of
        // the instructions this kernel issued.
        auto collect = [&](const float2 (&hh)[R][U / 2], uint32_t j) {
#pragma unroll
            for (int r = 0; r < R; ++r) {
                bool pass_r = false;
#pragma unroll
                for (int u = 0; u < U; u += 2) pass_r = pass_r | !(hh[r][u / 2].x < cr[r].nthr) | !(hh[r][u / 2].y < cr[r].nthr);
                if (__any_sync(0xffffffffu, pass_r)) {
                    const uint32_t slot = r * 32 + lane;
                    const bool live = tile_base + slot < n_rays;
#pragma unroll
                    for (int u = 0; u < U; u += 2) {
                        enqueue(live && j + u < nsph && !(hh[r][u / 2].x < cr[r].nthr), j + u, slot);
                        enqueue(live && j + u + 1 < nsph && !(hh[r][u / 2].y < cr[r].nthr), j + u + 1, slot);
                    }
                }
            }
        };
        if (a.verify) {   // debug build of the loop: every culled pair is re-tested exactly (survivors())
#pragma unroll 1
            for (uint32_t j = 0; j < cnt; j += U) survivors(j);
        } else if (PF && U == 2) {
            // Software-pipelined by hand over two register sets: the records of the group after next are loaded
            // before the current one is used (no register copies), and a group's vote + branch are issued after the
            // NEXT group's FFMA2s, so that the compare -> vote -> branch latency never leaves the FMA pipe idle.
            // cnt is a multiple of kCullPad = 4 = 2 U; the loads run up to kCullPad records past the array (slack).
            uint32_t saddr = smem_u32(sp);
            float4 s0[U], s1[U];
            float2 hA[R][U / 2], hB[R][U / 2];
            bool fB = false;
#pragma unroll
            for (int u = 0; u < U; ++u) s0[u] = lds128(saddr + 16u * u);
#pragma unroll 1
            for (uint32_t j = 0; j < cnt; j += 2 * U, saddr += 32u * U) {
#pragma unroll
                for (int u = 0; u < U; ++u) s1[u] = lds128(saddr + 16u * (U + u));
                const bool fA = test_group(s0, hA);
                if (__any_sync(0xffffffffu, fB)) collect(hB, j - U);      // the previous turn's second group
#pragma unroll
                for (int u = 0; u < U; ++u) s0[u] = lds128(saddr + 16u * (2 * U + u));
                fB = test_group(s1, hB);
                if (__any_sync(0xffffffffu, fA)) collect(hA, j);
            }
            if (__any_sync(0xffffffffu, fB)) collect(hB, cnt - U);
        } else {
#pragma unroll 1
            for (uint32_t j = 0; j < cnt; j += U) {
                float4 sc[U];
                float2 hh[R][U / 2];
#pragma unroll
                for (int u = 0; u < U; ++u) sc[u] = sp[j + u];
                if (__any_sync(0xffffffffu, test_group(sc, hh))) collect(hh, j);
            }
        }
        if (qn) drain(0u, qn);
        __syncwarp();

        // ---- epilogue of the tile
#pragma unroll
        for (int r = 0; r < R; ++r) {
            const uint32_t slot = r * 32 + lane;
            const uint32_t i = tile_base + slot;
            if (i < n_rays) {
                const uint32_t pi = phys_index(seg_len, a.seg_stride, i);
                if (ANY) a.out_lit[pi] = best_b[slot] ? 0 : 1;
                else { a.out_t[pi] = best_t[slot]; a.out_body[pi] = best_b[slot]; }
            }
        }
        __syncwarp();
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        n_exact += __shfl_xor_sync(0xffffffffu, n_exact, o);
        nan_count += __shfl_xor_sync(0xffffffffu, nan_count, o);
        unsound += __shfl_xor_sync(0xffffffffu, unsound, o);
    }
    if (lane == 0) {
        if (n_exact) atomicAdd(&a.ctr->exact_tests, n_exact);
        if (nan_count) atomicAdd(&a.ctr->err_nan, (unsigned long long)nan_count);
        if (unsound) atomicAdd(&a.ctr->cull_unsound, (unsigned long long)unsound);
    }
}

}  // namespace rg
