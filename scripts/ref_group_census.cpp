// ref_group_census.cpp — the occupied cells AccGrid::intersects visits, per ray (census tool; built by scripts/ref_group_census.py).
//
// Includes the oracle (oracle/raymond_oracle.cpp) unchanged and adds one walk next to it: `grid_intersects`' loop, statement for
// statement, that records the index of every visited cell holding a reference, up to and including the cell whose list holds the
// answer.  Those are the cells whose lists k_traverse pools.
// Build: g++ -O2 -std=c++17 -fPIC -ffp-contract=off -shared -pthread (the oracle's flags).
#include "../oracle/raymond_oracle.cpp"

namespace {

// AccGrid::intersects (acc_grid.rs:89-185), recording the occupied cells it visits; a ray the reference would panic on records none
void walk_occupied(const AccGrid& g, const Ray& ray, std::vector<uint64_t>& out) {
    double outer_t;
    if (!aabb_intersects(g.mesh.bounding_box, ray, &outer_t)) return;
    V3 outer_hit_position = ray.origin + ray.direction * outer_t;
    V3 start = ray.origin - g.mesh.bounding_box.min;
    int32_t cell[3];
    V3 q = div_ew(start, g.cell_size);
    for (int i = 0; i < 3; i++) if (!cast_i32(q[i], &cell[i])) return;
    if (cell[0] < 0 || cell[1] < 0 || cell[2] < 0) {
        start = outer_hit_position - g.mesh.bounding_box.min;
        q = div_ew(start, g.cell_size);
        for (int i = 0; i < 3; i++) if (!cast_i32(q[i], &cell[i])) return;
    }
    int32_t step[3];
    for (int i = 0; i < 3; i++) if (!cast_i32(signum(ray.direction[i]), &step[i])) return;
    double t_delta_x = (ray.direction.x < 0.0 ? -g.cell_size.x : g.cell_size.x) / ray.direction.x;
    double t_delta_y = (ray.direction.y < 0.0 ? -g.cell_size.y : g.cell_size.y) / ray.direction.y;
    double t_delta_z = (ray.direction.z < 0.0 ? -g.cell_size.z : g.cell_size.z) / ray.direction.z;
    double t_max_x = (((double)(cell[0] + (ray.direction.x < 0.0 ? 0 : 1)) * g.cell_size.x) - start.x) / ray.direction.x;
    double t_max_y = (((double)(cell[1] + (ray.direction.y < 0.0 ? 0 : 1)) * g.cell_size.y) - start.y) / ray.direction.y;
    double t_max_z = (((double)(cell[2] + (ray.direction.z < 0.0 ? 0 : 1)) * g.cell_size.z) - start.z) / ray.direction.z;
    const uint64_t rx = g.resolution[0], ry = g.resolution[1], rz = g.resolution[2];
    for (;;) {
        uint64_t x = (uint64_t)(int64_t)cell[0], y = (uint64_t)(int64_t)cell[1], z = (uint64_t)(int64_t)cell[2];
        uint64_t idx = x + rx * (y + z * rz);
        if (idx >= g.cells.size()) return;
        uint64_t cell_off = g.cells[idx];
        uint64_t count = g.mapping_table[cell_off];
        if (count) out.push_back(idx);
        double closest = 5712515.0;
        bool have = false;
        for (uint64_t i = 1; i <= count; i++) {
            double d;
            if (triangle_intersects(g.mesh.triangles[g.mapping_table[cell_off + i]], ray, &d) && d < closest) { closest = d; have = true; }
        }
        if (have) return;
        if (t_max_x < t_max_y) {
            if (t_max_x < t_max_z) {
                cell[0] += step[0];
                if (cell[0] >= (int32_t)rx || cell[0] < 0) return;
                t_max_x += t_delta_x;
            } else {
                cell[2] += step[2];
                if (cell[2] >= (int32_t)rz || cell[2] < 0) return;
                t_max_z += t_delta_z;
            }
        } else {
            if (t_max_y < t_max_z) {
                cell[1] += step[1];
                if (cell[1] >= (int32_t)ry || cell[1] < 0) return;
                t_max_y += t_delta_y;
            } else {
                cell[2] += step[2];
                if (cell[2] >= (int32_t)rz || cell[2] < 0) return;
                t_max_z += t_delta_z;
            }
        }
    }
}

}  // namespace

extern "C" {

struct rmoc_walk { std::vector<uint64_t> ray, cell; };

// The occupied cells of n rays, on `threads` threads: returns a handle holding (ray index, cell index) pairs in ray order and,
// per ray, in visiting order; *count = number of pairs.
rmoc_walk* rmoc_walk_grid(const rmo_grid* g, const rmo_ray* rays, size_t n, int threads, size_t* count) {
    if (threads < 1) threads = 1;
    std::vector<std::vector<uint64_t>> ray_of((size_t)threads), cells((size_t)threads);
    auto work = [&](int k) {
        const size_t lo = n * (size_t)k / (size_t)threads, hi = n * (size_t)(k + 1) / (size_t)threads;
        std::vector<uint64_t> one;
        for (size_t i = lo; i < hi; i++) {
            one.clear();
            walk_occupied(*g->g, toray(rays[i]), one);
            for (uint64_t c : one) { ray_of[(size_t)k].push_back(i); cells[(size_t)k].push_back(c); }
        }
    };
    std::vector<std::thread> th;
    for (int k = 1; k < threads; k++) th.emplace_back(work, k);
    work(0);
    for (auto& t : th) t.join();
    rmoc_walk* w = new rmoc_walk();
    for (int k = 0; k < threads; k++) {
        w->ray.insert(w->ray.end(), ray_of[(size_t)k].begin(), ray_of[(size_t)k].end());
        w->cell.insert(w->cell.end(), cells[(size_t)k].begin(), cells[(size_t)k].end());
    }
    *count = w->ray.size();
    return w;
}
void rmoc_walk_take(rmoc_walk* w, uint64_t* ray, uint64_t* cell) {
    std::memcpy(ray, w->ray.data(), w->ray.size() * sizeof(uint64_t));
    std::memcpy(cell, w->cell.data(), w->cell.size() * sizeof(uint64_t));
    delete w;
}

}  // extern "C"
