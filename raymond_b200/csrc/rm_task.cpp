// rm_task.cpp — render_tiled / TaskHandle / Message over the device-level renderer.
// Reference: src/trace.rs:62-230.  The reference spawns `worker_count` CPU threads that pull
// tiles from a queue and send Tile messages over an mpsc channel; here one driver thread per
// task feeds the GPU and posts the same messages into a single-consumer queue.

#include <algorithm>
#include <cmath>
#include <cstdlib>
#include <cstring>

#include "rm_internal.hpp"

using namespace rm;

// One checkpoint of the render: the whole frame of running sums as it was when the messages were posted.  The
// reference clones a Tile into every message (src/trace.rs:212-218); here the tiles of one checkpoint share one
// frame snapshot and are sliced out of it when a message is delivered.
struct FrameSnapshot {
    rm_vec3* sums = nullptr;        // W * H, row-major: the pinned block the D2H copy landed in (pageable when pinning fails
    bool pinned = false;            // or too much is already held by undelivered checkpoints)
    rm_vec3* mean = nullptr;        // final frame of a multi-device task: sums / sample_count, written by the exchange kernel (pinned)
    bool has_mean = false;
    size_t bytes = 0;
    size_t W = 0;
    FrameSnapshot() = default;
    FrameSnapshot(const FrameSnapshot&) = delete;
    FrameSnapshot& operator=(const FrameSnapshot&) = delete;
    ~FrameSnapshot();
};

struct PendingMessage {
    uint32_t kind;
    size_t sample_count;
    TileRect rect;
    std::shared_ptr<FrameSnapshot> frame;
};

struct rm_task {
    rm_settings settings{};
    rm_gpu_options options{};
    std::vector<rm_renderer*> renderers;     // one per GPU (options.device_count), in rank order
    std::thread driver;
    std::mutex mu;
    std::condition_variable cv;
    std::deque<PendingMessage> messages;
    bool finished = false;          // alive_thread_count == 0   src/trace.rs:74,89
    int status = RM_OK;
    std::string error;
    rm_stats stats{};
    rm_tile_callback callback = nullptr;
    void* callback_user = nullptr;
    bool adaptive = false;          // rm_render_tiled_adaptive with settings
    rm_adaptive_settings adaptive_settings{};
};

namespace {

std::atomic<size_t> g_snapshot_pinned_bytes{0};
constexpr size_t kSnapshotPinnedLimit = (size_t)4 << 30;

std::shared_ptr<FrameSnapshot> new_snapshot(size_t W, size_t H) {
    auto f = std::make_shared<FrameSnapshot>();
    f->W = W;
    f->bytes = std::max<size_t>(W * H, 1) * sizeof(rm_vec3);
    if (g_snapshot_pinned_bytes.load() + f->bytes <= kSnapshotPinnedLimit) f->sums = (rm_vec3*)pinned_acquire(f->bytes);
    f->pinned = f->sums != nullptr;
    if (f->pinned) g_snapshot_pinned_bytes += f->bytes;
    else f->sums = (rm_vec3*)malloc(f->bytes);
    if (!f->sums) throw std::bad_alloc();
    return f;
}

}  // namespace

FrameSnapshot::~FrameSnapshot() {
    if (pinned) { pinned_release(sums); g_snapshot_pinned_bytes -= bytes; }
    else free(sums);
    if (mean) { pinned_release(mean); g_snapshot_pinned_bytes -= bytes; }
}

namespace {

// Tile { sample_count, width, height, left, top, data }: an independent copy the receiver owns
bool make_tile(const PendingMessage& m, rm_tile* out) {
    const TileRect& r = m.rect;
    out->sample_count = m.sample_count;
    out->width = r.width; out->height = r.height; out->left = r.left; out->top = r.top;
    out->data = (rm_vec3*)malloc(std::max<size_t>(r.width * r.height, 1) * sizeof(rm_vec3));
    if (!out->data) return false;
    for (size_t y = 0; y < r.height; y++)
        memcpy(out->data + y * r.width, m.frame->sums + (r.top + y) * m.frame->W + r.left, r.width * sizeof(rm_vec3));
    return true;
}

// `kinds` (optional): one message kind per tile of the layout, 0xff = no message (a tile that finished at an earlier checkpoint)
void post_tiles(rm_task* t, uint32_t kind, size_t sample_count, const std::shared_ptr<FrameSnapshot>& frame, const std::vector<uint8_t>* kinds = nullptr) {
    const size_t W = t->settings.camera_settings.backbuffer_width, H = t->settings.camera_settings.backbuffer_height;
    std::vector<TileRect> tiles = tile_layout(W, H, t->settings.tile_size[0], t->settings.tile_size[1]);
    const int world = t->options.world_size > 1 ? t->options.world_size : 1;
    std::deque<PendingMessage> batch;
    for (size_t i = 0; i < tiles.size(); i++) {
        if (t->options.partition == RM_PARTITION_TILES && (int)(i % (size_t)world) != t->options.rank) continue;
        if (kinds && (*kinds)[i] == 0xff) continue;
        batch.push_back(PendingMessage{kinds ? (uint32_t)(*kinds)[i] : kind, sample_count, tiles[i], frame});
    }
    std::lock_guard<std::mutex> lk(t->mu);
    for (PendingMessage& m : batch) t->messages.push_back(std::move(m));
    t->cv.notify_all();
}

// global sample indices in [begin, end) that rank g of G renders under the sample partition: first, count (stride G)
void sample_share(size_t begin, size_t end, size_t g, size_t G, size_t* first, size_t* count) {
    const size_t f = begin + ((g + G - begin % G) % G);
    *first = f;
    *count = f < end ? (end - f + G - 1) / G : 0;
}

void drive(rm_task* t) {
    const rm_settings& s = t->settings;
    const size_t W = s.camera_settings.backbuffer_width, H = s.camera_settings.backbuffer_height;
    const size_t G = t->renderers.size();                 // GPUs driven by this task
    // a task that is itself one rank of a multi-process job (options.world_size) renders only its share
    const size_t world = G > 1 ? 1 : (t->options.world_size > 1 ? (size_t)t->options.world_size : 1);
    const bool split_samples = world > 1 && t->options.partition == RM_PARTITION_SAMPLES;
    const size_t first = split_samples ? (size_t)t->options.rank : 0;
    const size_t stride = split_samples ? world : 1;
    const size_t total = split_samples ? (s.sample_count > first ? (s.sample_count - first + world - 1) / world : 0) : s.sample_count;
    const bool split_local = G > 1 && t->options.partition == RM_PARTITION_SAMPLES;
    int st = RM_OK;
    Trace trace;
    // adaptive: which tiles still render, and at which checkpoint a tile may first stop
    const size_t n_tiles = tile_layout(W, H, s.tile_size[0], s.tile_size[1]).size();
    std::vector<uint8_t> active(n_tiles, 1);
    bool stopped_early = false;
    const size_t first_stop = std::max<size_t>(t->adaptive_settings.min_samples, 2);
    double* errors = nullptr;
    // every checkpoint's frame of running sums lands in its own snapshot (a pinned block, cached across tasks: D2H at link
    // speed, and the messages slice their tiles straight out of it)
    try {
        // TileProgressed every `samples_per_iteration` passes (src/trace.rs:217-219)
        const size_t chunk = s.samples_per_iteration ? s.samples_per_iteration : (total ? total : 1);
        size_t done = 0;
        while (done < total && st == RM_OK && std::find(active.begin(), active.end(), 1) != active.end()) {
            const size_t n = std::min(chunk, total - done);
            if (G == 1) {
                st = rm_renderer_render(t->renderers[0], first + done * stride, n, stride);
            } else {
                // every GPU gets its share of the samples [done, done + n) (or all of them for its own tiles); launches are
                // asynchronous, so one host thread keeps all devices busy
                for (size_t g = 0; g < G && st == RM_OK; g++) {
                    size_t f = done, c = n;
                    if (split_local) sample_share(done, done + n, g, G, &f, &c);
                    if (c) st = rm_renderer_render(t->renderers[g], f, c, split_local ? G : 1);
                }
            }
            done += n;
            if (st == RM_OK && done < total) {
                std::shared_ptr<FrameSnapshot> frame = new_snapshot(W, H);
                st = reduce_accumulators_to_host(t->renderers.data(), (int)G, frame->sums, frame->pinned);
                if (st == RM_OK && t->adaptive && done >= first_stop) {
                    // TileFinished(done) for every still-active tile whose E_t <= threshold (NaN never is), TileProgressed for the rest
                    if (!errors && !(errors = (double*)pinned_acquire(std::max<size_t>(n_tiles, 1) * sizeof(double)))) throw std::bad_alloc();
                    st = tile_errors_to_host(t->renderers.data(), (int)G, done, errors, n_tiles);
                    std::vector<uint8_t> kinds(n_tiles, 0xff);
                    bool changed = false;
                    for (size_t i = 0; i < n_tiles && st == RM_OK; i++) {
                        if (!active[i]) continue;
                        const bool converged = errors[i] <= t->adaptive_settings.threshold;
                        kinds[i] = converged ? RM_TILE_FINISHED : RM_TILE_PROGRESSED;
                        if (converged) { active[i] = 0; changed = true; }
                    }
                    if (st == RM_OK) post_tiles(t, RM_TILE_PROGRESSED, done, frame, &kinds);
                    for (size_t g = 0; g < G && st == RM_OK && changed; g++) st = rm_renderer_set_active_tiles(t->renderers[g], active.data(), n_tiles);
                    stopped_early = stopped_early || changed;
                } else if (st == RM_OK) {
                    post_tiles(t, RM_TILE_PROGRESSED, done, frame);      // no tile stops before first_stop
                }
            }
        }
        trace.mark("driver: all launches enqueued");
        if (st == RM_OK) {
            std::shared_ptr<FrameSnapshot> frame = new_snapshot(W, H);
            // several devices: the exchange kernel also writes the averaged frame await() hands out (the finalize, fused in)
            if (G > 1 && frame->pinned && t->options.partition == RM_PARTITION_SAMPLES && !stopped_early && g_snapshot_pinned_bytes.load() + frame->bytes <= kSnapshotPinnedLimit) {
                frame->mean = (rm_vec3*)pinned_acquire(frame->bytes);
                if (frame->mean) g_snapshot_pinned_bytes += frame->bytes;
            }
            st = reduce_accumulators_to_host(t->renderers.data(), (int)G, frame->sums, frame->pinned, frame->mean, (double)total, &frame->has_mean);
            trace.mark("driver: devices done, accumulators summed, frame on the host");
            if (st == RM_OK) {                                                     // src/trace.rs:211-212
                for (uint8_t& a : active) a = a ? (uint8_t)RM_TILE_FINISHED : 0xff;
                post_tiles(t, RM_TILE_FINISHED, total, frame, t->adaptive ? &active : nullptr);
            }
            trace.mark("driver: TileFinished messages posted");
        }
    } catch (const std::bad_alloc&) {
        st = fail(RM_ERR_OUT_OF_MEMORY, "out of host memory in the render driver");
    }
    pinned_release(errors);
    rm_stats stats{};
    for (size_t g = 0; g < G; g++) {
        rm_stats one{};
        rm_renderer_stats(t->renderers[g], &one);
        stats.samples += one.samples; stats.rays += one.rays; stats.nonfinite_samples += one.nonfinite_samples;
        stats.kernel_launches += one.kernel_launches; stats.upload_bytes += one.upload_bytes;
        stats.device_ms = std::max(stats.device_ms, one.device_ms);
        stats.upload_ms = std::max(stats.upload_ms, one.upload_ms);
    }
    trace.mark("driver: statistics collected");
    std::lock_guard<std::mutex> lk(t->mu);
    t->stats = stats;
    t->status = st;
    if (st != RM_OK) t->error = rm_last_error();
    t->finished = true;
    t->cv.notify_all();
}

// render_tiled; `adaptive` (optional, validated by the caller) adds per-tile early stopping, for which every share keeps Q
rm_task* create_task(const rm_scene* scene, const rm_settings* settings, const rm_gpu_options* options, const rm_adaptive_settings* adaptive) {
    rm_task* t = new rm_task();
    t->settings = *settings;
    if (options) t->options = *options;
    if (adaptive) {
        t->adaptive = true;
        t->adaptive_settings = *adaptive;
        t->options.flags |= RM_FLAG_MOMENTS;
    }
    const size_t G = t->options.device_count > 1 ? t->options.device_count : 1;
    if (G > 1 && (t->options.world_size > 1 || t->options.stream || t->options.accum_device)) {
        fail(RM_ERR_INVALID_ARGUMENT, "rm_render_tiled: device_count > 1 excludes world_size, stream and accum_device (they describe one device)");
        delete t;
        return nullptr;
    }
    if (G > 1024) {
        fail(RM_ERR_INVALID_ARGUMENT, "rm_render_tiled: device_count > 1024");
        delete t;
        return nullptr;
    }
    // the ordinals this task renders on (the caller's list is only read here; an ordinal may repeat)
    std::vector<int32_t> devices(G);
    for (size_t g = 0; g < G; g++) devices[g] = (t->options.device_list && t->options.device_count >= 1) ? t->options.device_list[g] : t->options.device + (int32_t)g;
    t->options.device_list = nullptr;
    t->options.device = devices[0];
    // Scene upload happens here, before the call returns, so a bad scene or a missing GPU is reported synchronously; the
    // device copies are the snapshot (the caller may destroy `scene`).  One host thread per share creates the share's
    // stream, pixel map, queues and accumulator and then joins the placement of the scene on all devices (rm_scene_group).
    Trace trace;
    t->renderers.assign(G, nullptr);
    std::vector<int> status(G, RM_OK);
    std::vector<std::string> errors(G);
    auto options_for = [&](size_t g) {
        rm_gpu_options o = t->options;
        o.device = devices[g];
        if (G > 1) { o.rank = (int32_t)g; o.world_size = (int32_t)G; }
        o.device_count = 0;
        return o;
    };
    // several shares: the scene image crosses the bus once, in slices, and is gathered over NVLink (rm_scene_group)
    rm_scene_group* group = nullptr;
    if (G > 1) {
        group = rm_scene_group_create(scene, devices.data(), (int)G);
        if (!group) { delete t; return nullptr; }
        trace.mark("rm_render_tiled: host images of the grids ready");
    }
    auto record = [&](size_t g) { status[g] = rm_last_status(); errors[g] = rm_last_error(); };
    auto create = [&](size_t g) {
        rm_gpu_options o = options_for(g);
        if (!group) {
            t->renderers[0] = rm_renderer_create(scene, settings, &o);
            if (!t->renderers[0]) record(0);
            return;
        }
        Trace share_trace;
        rm_renderer* r = rm_renderer_create_unbound(settings, &o);
        if (!r) record(g);
        if (share_trace.on) share_trace.mark(("share " + std::to_string(g) + ": renderer (stream, pixel map, queues, accumulator) ready").c_str());
        rm_device_scene* ds = rm_scene_group_join(group, (int)g);      // every share joins, whatever happened to its renderer
        if (share_trace.on) share_trace.mark(("share " + std::to_string(g) + ": scene slice uploaded, peers' slices gathered").c_str());
        if (!ds && r) record(g);
        if (r && ds) {
            rm_renderer_bind_scene(r, ds, 1);
        } else {
            if (r) rm_renderer_destroy(r);
            if (ds) rm_device_scene_destroy(ds);
            r = nullptr;
        }
        t->renderers[g] = r;
    };
    {
        std::vector<std::thread> pool;
        for (size_t g = 1; g < G; g++) pool.emplace_back(create, g);
        create(0);
        for (std::thread& th : pool) th.join();
    }
    if (group) rm_scene_group_destroy(group);
    trace.mark("rm_render_tiled: scene resident and renderers ready on every device");
    for (size_t g = 0; g < G; g++)
        if (!t->renderers[g]) {
            // report the first share that has an error of its own (a share whose peers failed only knows "another device failed")
            size_t bad = g;
            for (size_t k = 0; k < G; k++)
                if (!t->renderers[k] && status[k] != RM_OK && errors[k].find("another device") == std::string::npos) { bad = k; break; }
            for (rm_renderer* r : t->renderers) rm_renderer_destroy(r);
            fail(status[bad] ? status[bad] : RM_ERR_CUDA, errors[bad]);
            delete t;
            return nullptr;
        }
    t->driver = std::thread(drive, t);
    return t;
}

}  // namespace

extern "C" {

rm_task* rm_render_tiled(const rm_scene* scene, const rm_settings* settings, const rm_gpu_options* options) {
    if (!scene || !settings) { fail(RM_ERR_INVALID_ARGUMENT, "rm_render_tiled: null argument"); return nullptr; }
    if (validate_camera(settings->camera_settings, "rm_render_tiled") != RM_OK) return nullptr;
    return create_task(scene, settings, options, nullptr);
}

rm_task* rm_render_tiled_adaptive(const rm_scene* scene, const rm_settings* settings, const rm_gpu_options* options, const rm_adaptive_settings* adaptive) {
    if (!scene || !settings) { fail(RM_ERR_INVALID_ARGUMENT, "rm_render_tiled_adaptive: null argument"); return nullptr; }
    if (validate_camera(settings->camera_settings, "rm_render_tiled_adaptive") != RM_OK) return nullptr;
    if (adaptive) {
        if (!std::isfinite(adaptive->threshold) || adaptive->threshold <= 0.0) {
            fail(RM_ERR_INVALID_ARGUMENT, "rm_render_tiled_adaptive: threshold must be finite and > 0");
            return nullptr;
        }
        if (settings->samples_per_iteration == 0) {
            fail(RM_ERR_INVALID_ARGUMENT, "rm_render_tiled_adaptive: samples_per_iteration must be > 0 (it is the checkpoint cadence)");
            return nullptr;
        }
        if (options && options->world_size > 1 && options->device_count <= 1) {
            fail(RM_ERR_UNSUPPORTED, "rm_render_tiled_adaptive: one rank of a multi-process job cannot see the other ranks' sums");
            return nullptr;
        }
    }
    return create_task(scene, settings, options, adaptive);
}

int rm_task_poll(rm_task* t, rm_message* out) {
    if (!t || !out) return fail(RM_ERR_INVALID_ARGUMENT, "rm_task_poll: null argument");
    PendingMessage m;
    {
        std::lock_guard<std::mutex> lk(t->mu);
        if (t->messages.empty()) return 0;
        m = std::move(t->messages.front());
        t->messages.pop_front();
    }
    out->kind = m.kind;
    out->reserved = 0;
    if (!make_tile(m, &out->tile)) return fail(RM_ERR_OUT_OF_MEMORY, "out of host memory for a tile");
    return 1;
}

int rm_task_await(rm_task* t, rm_vec3* out) {
    if (!t || !out) return fail(RM_ERR_INVALID_ARGUMENT, "rm_task_await: null argument");
    Trace trace;
    std::unique_lock<std::mutex> lk(t->mu);
    t->cv.wait(lk, [&] { return t->finished; });
    trace.mark("await: render finished");
    if (t->status != RM_OK) return fail(t->status, t->error);
    const size_t W = t->settings.camera_settings.backbuffer_width, H = t->settings.camera_settings.backbuffer_height;
    // drain: TileProgressed messages are skipped, not a stop (the reference breaks at the first one, src/trace.rs:101-103)
    std::vector<PendingMessage> finished;
    while (!t->messages.empty()) {
        if (t->messages.front().kind == RM_TILE_FINISHED) finished.push_back(std::move(t->messages.front()));
        t->messages.pop_front();
    }
    lk.unlock();
    // out[x + left + (y + top) * W] = tile.data[..] / tile.sample_count as f64      src/trace.rs:95-97 — pixels no finished tile
    // covers (another rank's tiles) stay zero; rows are divided by a few host threads
    // every finished tile comes from one snapshot that already holds the averaged frame (multi-device exchange): copy rows
    const FrameSnapshot* whole = nullptr;
    if (!finished.empty() && finished[0].frame->has_mean) {
        size_t covered = 0;
        whole = finished[0].frame.get();
        for (const PendingMessage& m : finished) {
            if (m.frame.get() != whole) { whole = nullptr; break; }
            covered += m.rect.width * m.rect.height;
        }
        if (covered != W * H) whole = nullptr;
    }
    auto rows = [&](size_t y0, size_t y1) {
        if (whole) { memcpy((void*)(out + y0 * W), (const void*)(whole->mean + y0 * W), (y1 - y0) * W * sizeof(rm_vec3)); return; }
        for (size_t y = y0; y < y1; y++) memset((void*)(out + y * W), 0, W * sizeof(rm_vec3));
        for (const PendingMessage& m : finished) {
            const double c = (double)m.sample_count;
            const size_t a = std::max(y0, m.rect.top), b = std::min(y1, m.rect.top + m.rect.height);
            for (size_t y = a; y < b; y++) {
                const rm_vec3* src = m.frame->sums + y * m.frame->W + m.rect.left;
                rm_vec3* dst = out + y * W + m.rect.left;
                for (size_t x = 0; x < m.rect.width; x++) dst[x] = rm_vec3{src[x].x / c, src[x].y / c, src[x].z / c};
            }
        }
    };
    const unsigned hw = std::thread::hardware_concurrency();
    const size_t workers = W * H < ((size_t)1 << 18) ? 1 : std::min<size_t>(hw ? hw : 4, 8);
    std::vector<std::thread> pool;
    for (size_t w = 1; w < workers; w++) pool.emplace_back(rows, H * w / workers, H * (w + 1) / workers);
    rows(0, H / workers);
    for (std::thread& th : pool) th.join();
    trace.mark("await: averaged frame written");
    return RM_OK;
}

int rm_task_set_callback(rm_task* t, rm_tile_callback callback, void* user) {
    if (!t) return fail(RM_ERR_INVALID_ARGUMENT, "rm_task_set_callback: null task");
    std::lock_guard<std::mutex> lk(t->mu);
    t->callback = callback;
    t->callback_user = user;
    return RM_OK;
}

// async_await: hand every queued TileProgressed to the callback; stop at anything else   src/trace.rs:119-134
// (an adaptive task's early TileFinished messages stop it too, as the reference's would)
int rm_task_pump(rm_task* t) {
    if (!t) return fail(RM_ERR_INVALID_ARGUMENT, "rm_task_pump: null task");
    int delivered = 0;
    for (;;) {
        PendingMessage m;
        rm_tile_callback cb;
        void* user;
        {
            std::lock_guard<std::mutex> lk(t->mu);
            if (t->messages.empty() || t->messages.front().kind != RM_TILE_PROGRESSED) break;
            m = std::move(t->messages.front());
            t->messages.pop_front();
            cb = t->callback;
            user = t->callback_user;
        }
        rm_tile tile{};
        if (!make_tile(m, &tile)) return fail(RM_ERR_OUT_OF_MEMORY, "out of host memory for a tile");
        if (cb) cb(&tile, user);
        rm_tile_free(&tile);
        delivered++;
    }
    return delivered;
}

int rm_task_finished(rm_task* t) {
    if (!t) return fail(RM_ERR_INVALID_ARGUMENT, "rm_task_finished: null task");
    std::lock_guard<std::mutex> lk(t->mu);
    return t->finished ? 1 : 0;
}

int rm_task_stats(rm_task* t, rm_stats* out) {
    if (!t || !out) return fail(RM_ERR_INVALID_ARGUMENT, "rm_task_stats: null argument");
    std::unique_lock<std::mutex> lk(t->mu);
    t->cv.wait(lk, [&] { return t->finished; });
    *out = t->stats;
    return t->status;
}

void rm_task_destroy(rm_task* t) {
    if (!t) return;
    if (t->driver.joinable()) t->driver.join();
    for (rm_renderer* r : t->renderers) rm_renderer_destroy(r);
    delete t;
}

}  // extern "C"
