// cli_old.cpp — the reference's one working front-end (cli_old/src/main.rs:35-198) on top of the C ABI.
//
// Builds the GoldDragon scene exactly as cli_old does (scene :45-127, camera/settings :131-150), calls
// render_tiled + await (:152-153), applies the display transform (:157-181), writes output.png (:194-197) and prints
// the total time (:183-188).  With no --mesh the scene is ReflectiveSpheres (the blue sphere cli_old has commented
// out, :56-58).
// --serve PORT is the reference's intended server role (server/src/main.rs:174-192 binds 127.0.0.1:17025 and never renders;
// server/src/protocol.rs:9-14 is the message): listen on 127.0.0.1:PORT, accept one client, and write every Message of the
// render — TileProgressed every --spi samples, then TileFinished — as one JSON text per line ("\r\n", like editor/src/main.js:35).
// --adaptive T [--min-spp N] stops every tile at the first --spi checkpoint where its error estimate is <= T
// (rm_render_tiled_adaptive) and prints the samples actually rendered.
// Compile:  g++ -O2 -std=c++17 -Iinclude examples/cli_old.cpp -Lraymond_b200 -lraymond_cuda -Wl,-rpath,$PWD/raymond_b200 -o cli_old
#include <arpa/inet.h>
#include <netinet/in.h>
#include <sys/socket.h>
#include <unistd.h>

#include <chrono>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <vector>

#include "raymond.h"

static rm_material diffuse(double r, double g, double b, double rough) { rm_material m{}; m.kind = RM_MATERIAL_DIFFUSE; m.a = {r, g, b}; m.p0 = rough; return m; }
static rm_material metal(double r, double g, double b, double rough) { rm_material m{}; m.kind = RM_MATERIAL_METAL; m.a = {r, g, b}; m.p0 = rough; return m; }
static rm_material emission(double e) { rm_material m{}; m.kind = RM_MATERIAL_EMISSION; m.a = {e, e, e}; m.b = {1, 1, 1}; m.p0 = 0.27; m.p1 = 0.0; return m; }

#define CHECK(call) do { if ((call) != RM_OK) { fprintf(stderr, "%s failed: %s\n", #call, rm_last_error()); return 1; } } while (0)

int main(int argc, char** argv) {
    size_t height = 340, width = 340 / 9 * 16, spp = 500;        // cli_old/src/main.rs:131-132,145
    const char* mesh_path = nullptr;
    const char* out_path = "output.png";
    unsigned long long seed = 0;
    unsigned gpus = 1, repeat = 1;
    int serve_port = 0;
    size_t spi = 0;
    double adaptive = 0.0;
    size_t min_spp = 0;
    for (int i = 1; i < argc; i++) {
        if (!strcmp(argv[i], "--mesh") && i + 1 < argc) mesh_path = argv[++i];
        else if (!strcmp(argv[i], "--out") && i + 1 < argc) out_path = argv[++i];
        else if (!strcmp(argv[i], "--width") && i + 1 < argc) width = strtoull(argv[++i], nullptr, 10);
        else if (!strcmp(argv[i], "--height") && i + 1 < argc) height = strtoull(argv[++i], nullptr, 10);
        else if (!strcmp(argv[i], "--spp") && i + 1 < argc) spp = strtoull(argv[++i], nullptr, 10);
        else if (!strcmp(argv[i], "--seed") && i + 1 < argc) seed = strtoull(argv[++i], nullptr, 10);
        else if (!strcmp(argv[i], "--gpus") && i + 1 < argc) gpus = (unsigned)strtoul(argv[++i], nullptr, 10);
        else if (!strcmp(argv[i], "--repeat") && i + 1 < argc) repeat = (unsigned)strtoul(argv[++i], nullptr, 10);
        else if (!strcmp(argv[i], "--serve") && i + 1 < argc) serve_port = atoi(argv[++i]);
        else if (!strcmp(argv[i], "--spi") && i + 1 < argc) spi = strtoull(argv[++i], nullptr, 10);
        else if (!strcmp(argv[i], "--adaptive") && i + 1 < argc) adaptive = strtod(argv[++i], nullptr);
        else if (!strcmp(argv[i], "--min-spp") && i + 1 < argc) min_spp = strtoull(argv[++i], nullptr, 10);
        else {
            fprintf(stderr, "usage: cli_old [--mesh dragon.ply] [--out output.png] [--width W --height H --spp N --seed S --gpus G --repeat R --serve PORT --spi N"
                            " --adaptive T --min-spp N]\n");
            return 2;
        }
    }
    const auto now = std::chrono::steady_clock::now();
    auto lap = [&](const char* what) {       // phase times on stderr (the reference prints only the total)
        fprintf(stderr, "[cli_old] %-28s %.3f s\n", what, std::chrono::duration<double>(std::chrono::steady_clock::now() - now).count());
    };

    rm_scene* scene = rm_scene_create();
    rm_material m = diffuse(1.0, 0.0, 0.0, 0.02);
    CHECK(rm_scene_add_sphere(scene, {-1.0, -0.5, 3.5}, 0.5, &m));                           // :48-55
    if (mesh_path) {
        rm_mesh* mesh = rm_mesh_load_ply(mesh_path);                                          // :60
        if (!mesh) { fprintf(stderr, "load_ply: %s\n", rm_last_error()); return 1; }
        lap("load_ply");
        CHECK(rm_mesh_translate(mesh, {0.0, -0.3, 2.9}));                                     // :61
        int st = RM_OK;
        rm_grid* grid = rm_grid_build(mesh, &st);                                             // :62 AccGrid::build_from_mesh
        rm_mesh_destroy(mesh);
        lap("bake_transform + build grid");
        if (!grid) { fprintf(stderr, "build_from_mesh: %s\n", rm_last_error()); return 1; }
        m = metal(1.0, 1.0, 0.1, 0.15);
        CHECK(rm_scene_add_grid(scene, grid, &m));                                            // :70-75
        rm_grid_release(grid);
    } else {
        m = metal(0.05, 0.25, 1.00, 0.01);
        CHECK(rm_scene_add_sphere(scene, {0.74, -0.25, 3.5}, 0.75, &m));                      // :56-58
    }
    m = diffuse(0.75, 0.75, 0.75, 0.5); CHECK(rm_scene_add_plane(scene, {0, -1, 0}, {0, 1, 0}, &m));      // floor      :77-84
    m = emission(1.5);                  CHECK(rm_scene_add_plane(scene, {0, 2, 0}, {0, -1, 0}, &m));      // ceiling    :85-92
    m = diffuse(1, 1, 1, 0.4);          CHECK(rm_scene_add_plane(scene, {0, 0, -2}, {0, 0, 1}, &m));      // front wall :93-100
    m = diffuse(0, 0, 0, 0.9);          CHECK(rm_scene_add_plane(scene, {0, 0, 5}, {0, 0, -1}, &m));      // back wall  :101-108
    m = diffuse(0, 0, 0, 0.3);          CHECK(rm_scene_add_plane(scene, {-2, 0, 0}, {1, 0, 0}, &m));      // left wall  :109-117
    m = diffuse(0, 0, 0, 0.3);          CHECK(rm_scene_add_plane(scene, {2, 0, 0}, {-1, 0, 0}, &m));      // right wall :118-126

    rm_settings settings{};                                                                   // :134-150
    settings.camera_settings.backbuffer_width = width;
    settings.camera_settings.backbuffer_height = height;
    settings.camera_settings.fov_vert = 55.0;
    settings.camera_settings.position = {0, 0, 0};
    settings.camera_settings.focal_length = 2.5;
    settings.camera_settings.aperture_radius = 0.0;
    settings.sample_count = spp;
    settings.samples_per_iteration = spi;                                                     // TileProgressed every `spi` passes (src/trace.rs:217-219)
    settings.tile_size[0] = 32; settings.tile_size[1] = 32;
    settings.bounce_limit = 5;
    settings.worker_count = 0;
    rm_gpu_options opt{};
    opt.seed = seed;
    opt.device_count = gpus;                 // > 1: the samples are split over that many GPUs of this box

    // --serve: wait for the viewer before rendering (one client, like a render session)
    int client = -1;
    if (serve_port) {
        const int listener = socket(AF_INET, SOCK_STREAM, 0);
        int yes = 1;
        setsockopt(listener, SOL_SOCKET, SO_REUSEADDR, &yes, sizeof(yes));
        sockaddr_in addr{};
        addr.sin_family = AF_INET;
        addr.sin_addr.s_addr = htonl(INADDR_LOOPBACK);                                        // "127.0.0.1:17025", server/src/main.rs:174
        addr.sin_port = htons((uint16_t)serve_port);
        if (listener < 0 || bind(listener, (sockaddr*)&addr, sizeof(addr)) != 0 || listen(listener, 1) != 0) { perror("cli_old --serve"); return 1; }
        fprintf(stderr, "[cli_old] listening on 127.0.0.1:%d\n", serve_port);
        client = accept(listener, nullptr, nullptr);
        close(listener);
        if (client < 0) { perror("accept"); return 1; }
        lap("viewer connected");
    }
    auto send_all = [&](const char* p, size_t n) {
        while (n) {
            const ssize_t w = send(client, p, n, MSG_NOSIGNAL);
            if (w <= 0) return false;
            p += w; n -= (size_t)w;
        }
        return true;
    };

    // --repeat R renders the frame R times in this process: the first one pays CUDA's one-time start-up (a context per GPU)
    std::vector<rm_vec3> render(width * height);
    rm_stats stats{};
    for (unsigned rep = 0; rep < (repeat ? repeat : 1); rep++) {
        const auto r0 = std::chrono::steady_clock::now();
        opt.seed = seed + rep;
        const rm_adaptive_settings adapt{adaptive, min_spp};
        rm_task* task = adaptive != 0.0 ? rm_render_tiled_adaptive(scene, &settings, &opt, &adapt)
                                        : rm_render_tiled(scene, &settings, &opt);                   // :152
        if (!task) { fprintf(stderr, "render_tiled: %s\n", rm_last_error()); return 1; }
        lap("render_tiled returned");
        if (client >= 0) {
            // the intended consumer of TaskHandle::poll (cli/src/main.rs:38-45): every message goes on the wire as it arrives;
            // the frame is assembled from the TileFinished tiles (tile.data / tile.sample_count, src/trace.rs:95)
            std::vector<char> text;
            size_t sent = 0;
            for (;;) {
                rm_message msg{};
                const int got = rm_task_poll(task, &msg);
                if (got < 0) { fprintf(stderr, "poll: %s\n", rm_last_error()); return 1; }
                if (got == 0) {
                    if (rm_task_finished(task)) { if (rm_task_poll(task, &msg) != 1) break; }   // drained after the driver stopped
                    else { usleep(200); continue; }
                }
                const size_t n = rm_message_to_json(&msg, nullptr, 0);
                text.resize(n + 3);
                rm_message_to_json(&msg, text.data(), n + 1);
                text[n] = '\r'; text[n + 1] = '\n';
                if (!send_all(text.data(), n + 2)) { fprintf(stderr, "[cli_old] viewer went away\n"); close(client); client = -1; }
                sent++;
                if (msg.kind == RM_TILE_FINISHED) {
                    const rm_tile& t = msg.tile;
                    const double c = (double)t.sample_count;
                    for (size_t y = 0; y < t.height; y++)
                        for (size_t x = 0; x < t.width; x++) {
                            const rm_vec3 v = t.data[x + y * t.width];
                            render[(x + t.left) + (y + t.top) * width] = {v.x / c, v.y / c, v.z / c};
                        }
                }
                rm_tile_free(&msg.tile);
                if (client < 0) break;
            }
            fprintf(stderr, "[cli_old] %zu messages sent\n", sent);
            if (client < 0) CHECK(rm_task_await(task, render.data()));
        } else {
            CHECK(rm_task_await(task, render.data()));                                        // :153
        }
        lap("await returned");
        rm_task_stats(task, &stats);
        rm_task_destroy(task);
        fprintf(stderr, "[cli_old] frame %u: render_tiled + await %.3f s (device %.1f ms)\n", rep,
                std::chrono::duration<double>(std::chrono::steady_clock::now() - r0).count(), stats.device_ms);
    }
    if (client >= 0) close(client);
    rm_scene_destroy(scene);

    std::vector<uint8_t> export_(width * height * 3);
    CHECK(rm_tonemap_rgb8(render.data(), width * height, 1.0, 2.2, 0, export_.data()));       // :157-181
    lap("tonemap");
    const double secs = std::chrono::duration<double>(std::chrono::steady_clock::now() - now).count();
    printf("Finished render.\nTotal render time: %.3fs\nTotal amount of trace calls: %llu\n", secs, (unsigned long long)stats.rays);   // :183-188
    if (adaptive != 0.0) printf("Samples rendered: %llu of %llu\n", (unsigned long long)stats.samples, (unsigned long long)(width * height * spp));
    CHECK(rm_write_png(out_path, export_.data(), width, height));                             // :194-197
    lap("png written");
    fprintf(stderr, "[cli_old] device time %.1f ms, %llu kernel launches, upload %.1f ms\n", stats.device_ms, (unsigned long long)stats.kernel_launches, stats.upload_ms);
    return 0;
}
