// Per-pixel ray counts of the CPU oracle, for the RG_OPT_SUPERSAMPLE_EDGES tests (test infrastructure only).
//
// The oracle is included verbatim, so every pixel is rendered by its own render_pixel; rgo_render_rows_counts adds
// what rgo_render_rows does not report: the rays each pixel traced, taken as Counters differences around
// render_pixel.  The tests sum them over the refined pixels and the reference rows of a call to predict its counters.
#include "../oracle/raingun_oracle.cpp"

extern "C" {

// rgo_render_rows's arguments plus `counts`: 7 per pixel, row-major over rows [y0, y1): primary, shadow, reflection and
// transmission rays, then the err_nan_distance, err_transmission_none and err_aabb_normal counts.
int rgo_render_rows_counts(const rg_scene_desc *desc, uint32_t width, uint32_t height, uint32_t y0, uint32_t y1, int threads,
                           uint8_t *rgba_out, float *rgb_f32, uint64_t *counts) {
    if (!desc || !rgba_out || !counts) return RG_E_INVALID;
    if (width < height) return RG_E_PORTRAIT;
    if ((uint64_t)width * height > 0xFFFFFFFFull) return RG_E_TOO_LARGE;
    if (y1 > height || y0 > y1) return RG_E_INVALID;
    Scene s;
    s.d = desc;
    s.fov_adjustment = rgo_fov_adjustment(desc->fov);
    s.max_depth = desc->max_recursion_depth;
    s.default_color = {desc->default_color[0], desc->default_color[1], desc->default_color[2]};
    if (threads < 1) threads = 1;
    const uint64_t total = (uint64_t)(y1 - y0) * width;
    std::atomic<uint64_t> next_px{0};
    auto worker = [&]() {
        Counters c;
        for (;;) {
            const uint64_t p0 = next_px.fetch_add(64);
            if (p0 >= total) break;
            const uint64_t p1 = p0 + 64 < total ? p0 + 64 : total;
            for (uint64_t p = p0; p < p1; ++p) {
                const uint32_t x = (uint32_t)(p % width), y = y0 + (uint32_t)(p / width);
                const Counters before = c;
                const Color col = render_pixel(s, x, y, width, height, c);
                rgba_out[4 * p + 0] = f32_as_u8(col.r * 255.0f);
                rgba_out[4 * p + 1] = f32_as_u8(col.g * 255.0f);
                rgba_out[4 * p + 2] = f32_as_u8(col.b * 255.0f);
                rgba_out[4 * p + 3] = 255;
                if (rgb_f32) { rgb_f32[3 * p] = col.r; rgb_f32[3 * p + 1] = col.g; rgb_f32[3 * p + 2] = col.b; }
                uint64_t *o = counts + 7 * p;
                o[0] = c.primary - before.primary;
                o[1] = c.shadow - before.shadow;
                o[2] = c.reflection - before.reflection;
                o[3] = c.transmission - before.transmission;
                o[4] = c.err_nan - before.err_nan;
                o[5] = c.err_trans - before.err_trans;
                o[6] = c.err_aabb - before.err_aabb;
            }
        }
    };
    std::vector<std::thread> pool;
    for (int t = 0; t < threads; ++t) pool.emplace_back(worker);
    for (auto &t : pool) t.join();
    return RG_OK;
}

}  // extern "C"
