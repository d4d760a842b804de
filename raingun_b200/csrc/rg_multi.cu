// rg_multi.cu — one scene on every GPU of the box, behind the same handle.
//
// The reference parallelises INSIDE render_image: a rayon par_iter over the pixels, work-stealing
// across the cores of the machine (rendering.rs:27-35).  The B200 counterpart keeps that inside the
// library too: rg_scene_create(desc, RG_DEVICE_ALL, ...) uploads the scene to every visible GPU and
// starts one host thread per device; rg_render / rg_render_rows / rg_render_stream then cut the image
// into row tiles, every device renders the tiles it owns — plus whatever it claims from the shared
// std::atomic tile counter (work stealing) — and copies its finished rows over ITS OWN PCIe link
// straight to their place in the caller's buffer.  Pixels are independent, so there is no collective
// and nothing is exchanged between the GPUs; `collect` (rendering.rs:34-35) is the D2H copies.
#include <algorithm>
#include <atomic>
#include <chrono>
#include <condition_variable>
#include <cstring>
#include <mutex>
#include <thread>

#include <string>

#include "rg_host.h"

namespace rg {

constexpr uint32_t kTileRowsDefault = 8;
// static ownership: tile t belongs to device t mod N.  With stealing, every kStealEvery-th tile is kept
// back and handed out by the counter, in chunks, to whichever device has finished its own share.
constexpr uint32_t kStealEvery = 16;
constexpr uint32_t kAutoStaticMinTilesPerDevice = 16;

struct MultiJob {
    uint32_t w = 0, h = 0, y0 = 0, y1 = 0;
    uint8_t *out = nullptr;           // host, rows [y0, y1)
    bool out_pinned = false;
    uint32_t tile_rows = kTileRowsDefault;
    std::vector<std::vector<uint32_t>> first;    // per device: the tiles it owns
    std::vector<std::vector<uint32_t>> chunks;   // stealable tail, claimed through `next_chunk`
    std::atomic<uint32_t> next_chunk{0};
};

struct MultiState {
    std::vector<rg_scene *> dev;
    std::vector<std::thread> threads;
    std::mutex m;
    std::condition_variable cv_job, cv_done;
    uint64_t job_seq = 0;
    uint32_t running = 0;
    bool quit = false;
    MultiJob job;
    std::vector<rg_stats> stats;
    std::vector<int> rc;
    std::vector<std::string> err;
    std::vector<uint32_t> claims;      // batches each device rendered in the last call
    int schedule = 0;                  // RG_OPT_SCHEDULE
    uint32_t tile_rows = kTileRowsDefault;
};

// rows of the listed tiles, in list order
static void rows_of_tiles(const MultiJob &j, const std::vector<uint32_t> &tiles, std::vector<uint32_t> &rows) {
    rows.clear();
    for (uint32_t t : tiles) {
        const uint32_t r0 = j.y0 + t * j.tile_rows, r1 = std::min(j.y1, r0 + j.tile_rows);
        for (uint32_t r = r0; r < r1; ++r) rows.push_back(r);
    }
}

// Copies rows that lie compactly (in list order) in device memory to their own places in a host frame
// (`frame` = address of image row 0): runs of adjacent rows travel as one copy each, and a list of
// equal runs at a constant stride — an interleaved static share — as ONE strided copy.
static int copy_rows_to_host(const uint8_t *d_src, const uint32_t *rows, size_t n_rows, uint8_t *frame, size_t row_bytes, cudaStream_t stream) {
    struct Run { uint32_t row; uint32_t count; };
    std::vector<Run> runs;
    for (size_t k = 0; k < n_rows;) {
        size_t e = k + 1;
        while (e < n_rows && rows[e] == rows[e - 1] + 1) ++e;
        runs.push_back({rows[k], (uint32_t)(e - k)});
        k = e;
    }
    size_t r = 0, done_rows = 0;
    if (runs.size() >= 3 && runs[1].row > runs[0].row) {
        const uint32_t stride = runs[1].row - runs[0].row, cnt = runs[0].count;
        size_t full = 1;
        while (full < runs.size() && runs[full].count == cnt && runs[full].row - runs[full - 1].row == stride) ++full;
        if (full >= 3) {
            RG_CUDA(cudaMemcpy2DAsync(frame + (size_t)runs[0].row * row_bytes, (size_t)stride * row_bytes, d_src, (size_t)cnt * row_bytes,
                                      (size_t)cnt * row_bytes, full, cudaMemcpyDeviceToHost, stream));
            r = full;
            done_rows = full * cnt;
        }
    }
    for (; r < runs.size(); ++r) {
        RG_CUDA(cudaMemcpyAsync(frame + (size_t)runs[r].row * row_bytes, d_src + done_rows * row_bytes, (size_t)runs[r].count * row_bytes,
                                cudaMemcpyDeviceToHost, stream));
        done_rows += runs[r].count;
    }
    return RG_OK;
}

// Renders the listed image rows on the scene's device and delivers each at its place in a HOST frame.
int render_rowlist_to_host(rg_scene *sc, uint32_t w, uint32_t h, const uint32_t *rows, uint32_t n_rows, uint8_t *frame, rg_stats *st) {
    if (n_rows == 0) { if (st) std::memset(st, 0, sizeof *st); return RG_OK; }
    const size_t row_bytes = (size_t)w * 4;
    int rc = sc->frame.reserve((size_t)n_rows * row_bytes);
    if (rc) return rc;
    rg_stats local;
    std::memset(&local, 0, sizeof local);
    rc = render_rowlist_device(sc, w, h, rows, n_rows, OutKind::Rgba8, sc->frame.ptr, sc->stream, &local);
    if (rc) return rc;
    if ((rc = copy_rows_to_host(static_cast<const uint8_t *>(sc->frame.ptr), rows, n_rows, frame, row_bytes, sc->stream))) return rc;
    RG_CUDA(cudaStreamSynchronize(sc->stream));
    if (st) *st = local;
    return RG_OK;
}

// One batch on one device of a multi-GPU scene
static int render_tiles_to_host(rg_scene *sc, const MultiJob &j, const std::vector<uint32_t> &tiles, std::vector<uint32_t> &rows,
                                rg_stats *st) {
    rows_of_tiles(j, tiles, rows);
    if (rows.empty()) return RG_OK;
    rg_stats local;
    // j.out holds rows [y0, y1): address of image row 0 = out - y0 rows
    const int rc = render_rowlist_to_host(sc, j.w, j.h, rows.data(), (uint32_t)rows.size(), j.out - (size_t)j.y0 * j.w * 4, &local);
    if (rc) return rc;
    merge_stats(*st, local, false);
    return RG_OK;
}

static void worker(MultiState *ms, uint32_t k) {
    rg_scene *sc = ms->dev[k];
    cudaSetDevice(sc->device);
    std::vector<uint32_t> rows;
    uint64_t seen = 0;
    for (;;) {
        {
            std::unique_lock<std::mutex> lock(ms->m);
            ms->cv_job.wait(lock, [&] { return ms->quit || ms->job_seq != seen; });
            if (ms->quit) return;
            seen = ms->job_seq;
        }
        MultiJob &j = ms->job;
        rg_stats st;
        std::memset(&st, 0, sizeof st);
        uint32_t claims = 0;
        int rc = RG_OK;
        if (!j.first[k].empty()) { rc = render_tiles_to_host(sc, j, j.first[k], rows, &st); ++claims; }
        while (rc == RG_OK) {   // work stealing: an atomic fetch-add, microseconds per claim
            const uint32_t c = j.next_chunk.fetch_add(1, std::memory_order_relaxed);
            if (c >= j.chunks.size()) break;
            rc = render_tiles_to_host(sc, j, j.chunks[c], rows, &st);
            ++claims;
        }
        {
            std::lock_guard<std::mutex> lock(ms->m);
            ms->stats[k] = st;
            ms->rc[k] = rc;
            ms->claims[k] = claims;
            if (rc != RG_OK) ms->err[k] = rg_last_error();
            if (--ms->running == 0) ms->cv_done.notify_all();
        }
    }
}

int multi_create(const rg_scene_desc *desc, const int32_t *devices, uint32_t n_devices, rg_scene **out) {
    *out = nullptr;
    if (n_devices == 0) { set_error("no devices given"); return RG_E_INVALID; }
    MultiState *ms = new MultiState();
    ms->dev.assign(n_devices, nullptr);
    ms->rc.assign(n_devices, RG_OK);
    ms->err.assign(n_devices, std::string());
    ms->stats.resize(n_devices);
    ms->claims.assign(n_devices, 0);
    {   // upload to every device at once (one host thread each)
        std::vector<std::thread> up;
        for (uint32_t k = 0; k < n_devices; ++k)
            up.emplace_back([&, k] {
                ms->rc[k] = rg_scene_create(desc, devices[k], &ms->dev[k]);
                if (ms->rc[k] != RG_OK) ms->err[k] = rg_last_error();
            });
        for (auto &t : up) t.join();
    }
    for (uint32_t k = 0; k < n_devices; ++k)
        if (ms->rc[k] != RG_OK) {
            const int rc = ms->rc[k];
            set_error("device %d: %s", devices[k], ms->err[k].c_str());
            for (auto *c : ms->dev) rg_scene_destroy(c);
            delete ms;
            return rc;
        }
    rg_scene *sc = new rg_scene();
    sc->device = ms->dev[0]->device;
    sc->multi = ms;
    sc->n_bodies = ms->dev[0]->n_bodies;
    sc->scene_max_depth = ms->dev[0]->scene_max_depth;
    for (uint32_t k = 0; k < n_devices; ++k) ms->threads.emplace_back(worker, ms, k);
    *out = sc;
    return RG_OK;
}

void multi_destroy(rg_scene *sc) {
    MultiState *ms = sc->multi;
    {
        std::lock_guard<std::mutex> lock(ms->m);
        ms->quit = true;
    }
    ms->cv_job.notify_all();
    for (auto &t : ms->threads) t.join();
    for (auto *c : ms->dev) rg_scene_destroy(c);
    if (sc->h_frame) { cudaSetDevice(sc->device); cudaFreeHost(sc->h_frame); }
    delete ms;
    delete sc;
}

int multi_set_option(rg_scene *sc, int32_t key, int64_t value) {
    MultiState *ms = sc->multi;
    if (key == RG_OPT_SCHEDULE) {
        if (value < 0 || value > 2) { set_error("bad schedule %lld", (long long)value); return RG_E_INVALID; }
        ms->schedule = (int)value;
        return RG_OK;
    }
    if (key == RG_OPT_TILE_ROWS) {
        if (value < 1 || value > 4096) { set_error("bad tile height %lld", (long long)value); return RG_E_INVALID; }
        ms->tile_rows = (uint32_t)value;
        return RG_OK;
    }
    for (auto *c : ms->dev) {
        const int rc = rg_scene_set_option(c, key, value);
        if (rc) return rc;
    }
    if (key == RG_OPT_SUPERSAMPLE) sc->supersample = (uint32_t)value;   // the handle's own size checks (check_dims)
    return RG_OK;
}

uint32_t multi_device_count(const rg_scene *sc) { return (uint32_t)sc->multi->dev.size(); }

int multi_render_rows(rg_scene *sc, uint32_t w, uint32_t h, uint32_t y0, uint32_t y1, uint8_t *rgba_out, rg_stats *stats) {
    MultiState *ms = sc->multi;
    const auto t0 = std::chrono::steady_clock::now();
    const uint32_t N = (uint32_t)ms->dev.size();
    MultiJob &j = ms->job;
    j.w = w; j.h = h; j.y0 = y0; j.y1 = y1; j.out = rgba_out;
    j.tile_rows = ms->tile_rows;
    const uint32_t rows = y1 - y0, nt = (rows + j.tile_rows - 1) / j.tile_rows;
    j.first.assign(N, {});
    j.chunks.clear();
    j.next_chunk.store(0);
    bool steal = ms->schedule == 2 || (ms->schedule == 0 && nt < kAutoStaticMinTilesPerDevice * N);
    if (N == 1 || nt < 4 * N) steal = N > 1 && nt > N;   // tiny frames: hand every tile out by the counter
    if (N > 1 && steal && nt < 4 * N) {
        for (uint32_t t = 0; t < nt; ++t) j.chunks.push_back({t});
    } else if (steal) {
        std::vector<uint32_t> owned, tail;
        for (uint32_t t = 0; t < nt; ++t) (t % kStealEvery == kStealEvery - 1 ? tail : owned).push_back(t);
        for (size_t i = 0; i < owned.size(); ++i) j.first[i % N].push_back(owned[i]);
        const size_t per = std::max<size_t>(1, (tail.size() + 2 * N - 1) / (2 * N));   // two claims per device on average
        for (size_t i = 0; i < tail.size(); i += per) j.chunks.emplace_back(tail.begin() + (long)i, tail.begin() + (long)std::min(tail.size(), i + per));
    } else {
        for (uint32_t t = 0; t < nt; ++t) j.first[t % N].push_back(t);
    }
    {
        std::lock_guard<std::mutex> lock(ms->m);
        ms->running = N;
        ++ms->job_seq;
    }
    ms->cv_job.notify_all();
    {
        std::unique_lock<std::mutex> lock(ms->m);
        ms->cv_done.wait(lock, [&] { return ms->running == 0; });
    }
    rg_stats total;
    std::memset(&total, 0, sizeof total);
    int rc = RG_OK;
    for (uint32_t k = 0; k < N; ++k) {
        if (ms->rc[k] != RG_OK && rc == RG_OK) {
            rc = ms->rc[k];
            set_error("device %d: %s", ms->dev[k]->device, ms->err[k].c_str());
        }
        merge_stats(total, ms->stats[k], true);   // the devices run concurrently
        if (ms->claims[k]) total.devices_used++;
    }
    total.ms_wall = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count();
    if (stats) *stats = total;
    return rc;
}

}  // namespace rg

// ---- a barrier for the processes of one box (one per GPU) in shared memory ---------------------------------
// The end of a sharded frame needs every rank to know that all rows have landed.  A collective on the GPUs for
// that (an NCCL all-reduce of one word) costs 60-100 us per frame; the ranks have already synchronised their
// own streams when they get here, so a sense-reversing counter in a shared-memory page does it in a few
// microseconds — the "host std::atomic" option of the multi-GPU plan, across processes.
#include <fcntl.h>
#include <sched.h>
#include <sys/mman.h>
#include <unistd.h>

namespace {
struct ShmBarrierPage {
    std::atomic<uint32_t> arrived;
    std::atomic<uint32_t> sense;
    uint32_t parties;
};
struct ShmBarrier {
    ShmBarrierPage *page = nullptr;
    uint32_t local_sense = 0;
    std::string name;
    bool owner = false;
};
}  // namespace

extern "C" {

int rg_shm_barrier_open(const char *name, uint32_t parties, int32_t create, void **handle) {
    if (!name || !handle || parties == 0) { rg::set_error("rg_shm_barrier_open: bad argument"); return RG_E_INVALID; }
    *handle = nullptr;
    static_assert(std::atomic<uint32_t>::is_always_lock_free, "shared-memory atomics must be address-free");
    const int fd = shm_open(name, create ? (O_CREAT | O_RDWR | O_TRUNC) : O_RDWR, 0600);
    if (fd < 0) { rg::set_error("shm_open(%s) failed", name); return RG_E_INVALID; }
    if (create && ftruncate(fd, (off_t)sizeof(ShmBarrierPage)) != 0) { close(fd); rg::set_error("ftruncate failed"); return RG_E_NOMEM; }
    void *p = mmap(nullptr, sizeof(ShmBarrierPage), PROT_READ | PROT_WRITE, MAP_SHARED, fd, 0);
    close(fd);
    if (p == MAP_FAILED) { rg::set_error("mmap of the barrier page failed"); return RG_E_NOMEM; }
    ShmBarrier *b = new ShmBarrier();
    b->page = static_cast<ShmBarrierPage *>(p);
    b->name = name;
    b->owner = create != 0;
    if (create) {   // (a fresh shared-memory object is zero-filled; the creator publishes its name only after this)
        b->page->arrived.store(0);
        b->page->sense.store(0);
        b->page->parties = parties;
    }
    *handle = b;
    return RG_OK;
}

int rg_shm_barrier_wait(void *handle) {
    ShmBarrier *b = static_cast<ShmBarrier *>(handle);
    if (!b || !b->page) { rg::set_error("rg_shm_barrier_wait: bad handle"); return RG_E_INVALID; }
    ShmBarrierPage *pg = b->page;
    const uint32_t my = b->local_sense ^ 1u;
    b->local_sense = my;
    if (pg->arrived.fetch_add(1, std::memory_order_acq_rel) + 1 == pg->parties) {
        pg->arrived.store(0, std::memory_order_relaxed);
        pg->sense.store(my, std::memory_order_release);
        return RG_OK;
    }
    const auto t0 = std::chrono::steady_clock::now();
    for (uint32_t spins = 0; pg->sense.load(std::memory_order_acquire) != my; ++spins) {
        if ((spins & 1023u) == 1023u) {
            sched_yield();
            if (std::chrono::steady_clock::now() - t0 > std::chrono::seconds(120)) {
                rg::set_error("rg_shm_barrier_wait: a rank did not arrive within 120 s");
                return RG_E_CANCELLED;
            }
        }
    }
    return RG_OK;
}

int rg_shm_barrier_close(void *handle) {
    ShmBarrier *b = static_cast<ShmBarrier *>(handle);
    if (!b) return RG_OK;
    if (b->page) munmap(b->page, sizeof(ShmBarrierPage));
    if (b->owner) shm_unlink(b->name.c_str());
    delete b;
    return RG_OK;
}

}  // extern "C"
