"""Per-tile adaptive sampling against the oracle.

A path's value depends only on (seed, pixel, global sample index), so everything here is predicted from the oracle's per-sample
values (oracle.trace_samples): the second moments Q, the error estimate E_t of include/raymond.h, and the schedule of an
adaptive render — the checkpoint at which every tile stops — together with the sums each TileFinished must carry (the oracle's
render(sample_count = n_t) restricted to the tile).
"""
import ctypes as C
import os
import subprocess
import time

import numpy as np
import pytest

from oracle import oracle as O
from raymond_b200 import api as A
from raymond_b200 import fixtures as F

from test_gpu_nonfinite import SCENES as NONFINITE_SCENES
from util import oracle_scene, product_scene, settings

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

CAM = F.camera(96, 64)
TILE = (16, 16)
SEED = 5
N, SPI, MIN_SPP = 24, 4, 6
SCENES = {"spheres": F.reflective_spheres(), "tube": F.gold_dragon(F.dragon_standin(96, 24))}


def oracle_samples(objs, cam, count, first=0, stride=1, seed=SEED, limit=5):
    """(count, H, W, 3): the value of global sample first + k * stride of every pixel, k = 0 .. count-1."""
    osc = oracle_scene(objs)
    W, H = cam["width"], cam["height"]
    pix = np.arange(W * H, dtype=np.uint32)
    out = np.empty((count, H, W, 3))
    for k in range(count):
        out[k] = O.trace_samples(osc, cam, pix, np.full(W * H, first + k * stride, dtype=np.uint32), seed=seed, bounce_limit=limit).reshape(H, W, 3)
    return out


def running_sums(vals, keep=False):
    """S and Q in sample order, after every sample: (count, H, W, 3) each.  Drop mode leaves non-finite samples out of both."""
    S, Q = np.zeros(vals.shape[1:]), np.zeros(vals.shape[1:])
    Ss, Qs = [], []
    for v in vals:
        w = v if keep else np.where(np.isfinite(v).all(axis=-1, keepdims=True), v, 0.0)
        S = S + w
        Q = Q + w * w
        Ss.append(S)
        Qs.append(Q)
    return np.array(Ss), np.array(Qs)


def tile_errors_np(S, Q, n, layout):
    """E_t exactly as include/raymond.h defines it."""
    m = S / n
    d = Q - S * m
    v = np.where(d < 0.0, 0.0, d) / (n - 1)           # max(., 0) that keeps a NaN
    se2 = v / n
    r = np.sqrt(se2[..., 0] + se2[..., 1] + se2[..., 2]) / (m[..., 0] + m[..., 1] + m[..., 2] + 1e-3)
    return np.array([np.sqrt(np.mean(r[t:t + h, l:l + w] ** 2)) for l, t, w, h in layout])


def assert_close(g, o, what, rel=1e-9):
    """Per element: the same NaN / Inf classes, and finite values within `rel` relative (one element, or 1e-4 of them, left
    as room for a last-ulp libm difference flipping a branch, as in test_gpu_render)."""
    for name, f in (("NaN", np.isnan), ("+Inf", np.isposinf), ("-Inf", np.isneginf)):
        assert np.array_equal(f(g), f(o)), f"{what}: elements differ in being {name}"
    fin = np.isfinite(o)
    err = np.abs(g[fin] - o[fin]) / np.maximum(np.abs(o[fin]), 1e-3)
    bad = int((err > rel).sum())
    assert bad <= max(1, int(1e-4 * err.size)), f"{what}: {bad} of {err.size} elements differ beyond {rel} relative (largest {err.max():.3g})"


def bits(a):
    return np.ascontiguousarray(a).view(np.uint64)


# ---------------------------------------------------------------------------- renderer level


@pytest.mark.parametrize("share", [(0, 8, 1), (1, 5, 2)], ids=["all", "odd_samples"])
@pytest.mark.parametrize("name", list(SCENES))
def test_moments_are_the_oracles(name, share):
    """S is the oracle's render and Q is the sum of squared oracle samples in global sample order, over several batches."""
    objs = SCENES[name]
    first, count, stride = share
    r = A.Renderer(product_scene(objs), settings(CAM, 8, TILE), A.GpuOptions(seed=SEED, batch_spp=3, flags=A.FLAG_MOMENTS))
    r.render(first, count, stride)
    S, Q = r.read_sums(), r.read_moments()
    r.close()
    vals = oracle_samples(objs, CAM, count, first, stride)
    Sn, Qn = running_sums(vals)
    want, _ = O.render(oracle_scene(objs), CAM, count, seed=SEED, first_sample=first, sample_stride=stride)
    assert_close(S, want, f"{name} S")
    assert_close(S, Sn[-1], f"{name} S vs samples")
    assert_close(Q, Qn[-1], f"{name} Q")
    assert (Q > 0).any()


def test_moments_keep_nonfinite():
    """Keep mode: non-finite samples go into Q as into S, so the NaN / Inf classes of both are the oracle's."""
    objs = NONFINITE_SCENES["box"]
    cam, spp = F.camera(64, 48), 4
    r = A.Renderer(product_scene(objs), settings(cam, spp, TILE), A.GpuOptions(seed=3, batch_spp=2, flags=A.FLAG_MOMENTS | A.FLAG_KEEP_NONFINITE))
    r.render(0, spp)
    S, Q = r.read_sums(), r.read_moments()
    r.close()
    Sn, Qn = running_sums(oracle_samples(objs, cam, spp, seed=3), keep=True)
    assert np.isnan(S).any()
    assert_close(S, Sn[-1], "keep S")
    assert_close(Q, Qn[-1], "keep Q")


@pytest.mark.parametrize("keep", [False, True])
def test_default_path_unchanged_by_the_flag(keep):
    """The frame, rays and nonfinite_samples are bit-identical with and without RM_FLAG_MOMENTS."""
    objs = NONFINITE_SCENES["box"] if keep else SCENES["spheres"]
    flags = A.FLAG_KEEP_NONFINITE if keep else 0
    out = []
    for f in (flags, flags | A.FLAG_MOMENTS):
        r = A.Renderer(product_scene(objs), settings(CAM, 6, TILE), A.GpuOptions(seed=SEED, batch_spp=4, flags=f))
        r.render(0, 6)
        out.append((r.read_sums(), r.stats()))
        r.close()
    assert np.array_equal(bits(out[0][0]), bits(out[1][0]))
    for k in ("rays", "nonfinite_samples", "samples"):
        assert out[0][1][k] == out[1][1][k]


def test_moments_need_the_flag():
    r = A.Renderer(product_scene(SCENES["spheres"]), settings(CAM, 2, TILE), A.GpuOptions(seed=SEED))
    with pytest.raises(A.RaymondError) as e:
        r.read_moments()
    assert e.value.status == -10
    r.close()


@pytest.mark.parametrize("share", ["all", "tiles_rank1_of3"])
def test_tile_errors_are_the_definition(share):
    """rm_renderer_tile_errors equals the numpy restatement of E_t on the read-back S and Q; tiles of other shares are NaN."""
    objs = SCENES["spheres"]
    st = settings(CAM, 6, TILE)
    o = A.GpuOptions(seed=SEED, flags=A.FLAG_MOMENTS)
    if share != "all":
        o.partition, o.rank, o.world_size = A.PARTITION_TILES, 1, 3
    r = A.Renderer(product_scene(objs), st, o)
    r.render(0, 6)
    S, Q = r.read_sums(), r.read_moments()
    got = r.tile_errors(6)
    r.close()
    layout = A.tile_layout(st)
    want = tile_errors_np(S, Q, 6, layout)
    owned = np.ones(len(layout), dtype=bool) if share == "all" else (np.arange(len(layout)) % 3 == 1)
    assert np.isnan(got[~owned]).all()
    np.testing.assert_allclose(got[owned], want[owned], rtol=1e-12, atol=0)
    assert (want[owned] > 0).any()


def test_set_active_tiles():
    """Inactive tiles keep their sums bit for bit; active tiles get exactly the full-frame render's sums; NULL restores all."""
    objs = SCENES["tube"]
    st = settings(CAM, 12, TILE)
    layout = A.tile_layout(st)
    mask = (np.arange(len(layout)) % 3) != 0
    part = A.Renderer(product_scene(objs), st, A.GpuOptions(seed=SEED, batch_spp=2, flags=A.FLAG_MOMENTS))
    full = A.Renderer(product_scene(objs), st, A.GpuOptions(seed=SEED, batch_spp=2, flags=A.FLAG_MOMENTS))
    part.render(0, 4)
    before_s, before_q = part.read_sums(), part.read_moments()
    samples_before = part.stats()["samples"]
    part.set_active_tiles(mask)
    part.render(4, 5)
    after_s, after_q = part.read_sums(), part.read_moments()
    full.render(0, 9)
    full_s, full_q = full.read_sums(), full.read_moments()
    active_pixels = 0
    for (l, t, w, h), on in zip(layout, mask):
        sl = (slice(t, t + h), slice(l, l + w))
        if on:
            active_pixels += w * h
            assert np.array_equal(bits(after_s[sl]), bits(full_s[sl])) and np.array_equal(bits(after_q[sl]), bits(full_q[sl]))
        else:
            assert np.array_equal(bits(after_s[sl]), bits(before_s[sl])) and np.array_equal(bits(after_q[sl]), bits(before_q[sl]))
    assert part.stats()["samples"] - samples_before == active_pixels * 5
    part.set_active_tiles(None)
    part.clear()
    part.render(0, 9)
    assert np.array_equal(bits(part.read_sums()), bits(full_s))
    part.close()
    full.close()


# ---------------------------------------------------------------------------- the adaptive task


def checkpoints(n=N, spi=SPI):
    return list(range(spi, n, spi))


def predicted(objs, cam, tau, min_spp=MIN_SPP, n=N, spi=SPI, keep=False, seed=SEED, vals=None, tile=TILE):
    """(n_t per tile, E per checkpoint per tile) from the oracle's samples."""
    st = settings(cam, n, tile, spi=spi)
    layout = A.tile_layout(st)
    if vals is None:
        vals = oracle_samples(objs, cam, n, seed=seed)
    Ss, Qs = running_sums(vals, keep)
    E = {c: tile_errors_np(Ss[c - 1], Qs[c - 1], c, layout) for c in checkpoints(n, spi) if c >= max(min_spp, 2)}
    stop = np.full(len(layout), n)
    for c in sorted(E):
        stop = np.where((stop == n) & (E[c] <= tau), c, stop)
    return stop, E


def pick_threshold(E, n=N):
    """Halfway in log between two neighbouring E values, so that some tiles stop early and some run to the end; the split
    with the most tiles on the smaller side."""
    vals = np.unique(np.concatenate([e[np.isfinite(e) & (e > 0)] for e in E.values()]))
    best, best_tau = -1, None
    for a, b in zip(vals[:-1], vals[1:]):
        if b <= a * (1 + 1e-6):
            continue
        tau = float(np.sqrt(a * b))
        stop = np.full(len(next(iter(E.values()))), n)
        for c in sorted(E):
            stop = np.where((stop == n) & (E[c] <= tau), c, stop)
        side = min(int((stop < n).sum()), int((stop == n).sum()))
        if side > best:
            best, best_tau = side, tau
    return best_tau


def poll_all(task):
    msgs = []
    while True:
        m = task.poll()
        if m is not None:
            msgs.append(m)
            continue
        if task.finished():
            while (m := task.poll()) is not None:
                msgs.append(m)
            return msgs
        time.sleep(0.001)


def expected_sequence(layout, stop, n=N, spi=SPI):
    seq = []
    for c in checkpoints(n, spi):
        for (l, t, w, h), s in zip(layout, stop):
            if s >= c:
                seq.append(("TileFinished" if s == c else "TileProgressed", c, int(l), int(t)))
    seq += [("TileFinished", n, int(l), int(t)) for (l, t, w, h), s in zip(layout, stop) if s == n]
    return seq


def adaptive_options(device_list, partition, flags=0):
    return A.GpuOptions(seed=SEED, device_list=device_list, partition=partition, flags=flags)


SHARES = {"one": (None, A.PARTITION_SAMPLES), "samples2": ([0, 0], A.PARTITION_SAMPLES), "tiles3": ([0, 0, 0], A.PARTITION_TILES)}


@pytest.mark.parametrize("name", list(SCENES))
def test_adaptive_task_follows_the_oracle_schedule(name):
    objs = SCENES[name]
    st = settings(CAM, N, TILE, spi=SPI)
    layout = A.tile_layout(st)
    vals = oracle_samples(objs, CAM, N)
    _, E = predicted(objs, CAM, 1.0, vals=vals)
    tau = pick_threshold(E)
    stop, E = predicted(objs, CAM, tau, vals=vals)
    assert (stop < N).any() and (stop == N).any(), "the threshold must split the tiles"
    for e in E.values():
        assert not (np.abs(e - tau) <= 1e-9 * tau).any(), "a tile's E is too close to the threshold to predict"
    adaptive = A.AdaptiveSettings(tau, MIN_SPP)
    osc = oracle_scene(objs)
    want = {c: O.render(osc, CAM, int(c), seed=SEED, tile_size=TILE)[0] for c in set(stop.tolist())}
    finished_one = None
    for share, (devices, partition) in SHARES.items():
        task = A.render_tiled(product_scene(objs), st, adaptive_options(devices, partition), adaptive)
        msgs = poll_all(task)
        stats = task.stats()
        got_seq = [(m.kind, m.tile.sample_count, m.tile.left, m.tile.top) for m in msgs]
        assert got_seq == expected_sequence(layout, stop), f"{share}: message sequence"
        finished = [m.tile for m in msgs if m.kind == "TileFinished"]
        by_rect = {(t.left, t.top): t for t in finished}
        for (l, t, w, h), s in zip(layout, stop):
            tile = by_rect[(int(l), int(t))]
            assert_close(tile.data, want[s][t:t + h, l:l + w], f"{share}: tile ({l}, {t}) after {s} samples")
        assert stats["samples"] == sum(int(w * h) * int(s) for (l, t, w, h), s in zip(layout, stop))
        if finished_one is None:
            finished_one = by_rect
        else:
            for k, tile in by_rect.items():
                if share == "tiles3":
                    assert np.array_equal(bits(tile.data), bits(finished_one[k].data)), f"{share}: tile {k} differs from one share"
                else:
                    np.testing.assert_allclose(tile.data, finished_one[k].data, rtol=1e-12, atol=1e-300)
        # await: every tile divided by its own count
        frame = A.render_tiled(product_scene(objs), st, adaptive_options(devices, partition), adaptive).await_()
        for (l, t, w, h), s in zip(layout, stop):
            tile = by_rect[(int(l), int(t))]
            assert np.array_equal(bits(frame[t:t + h, l:l + w]), bits(tile.data / float(s))), f"{share}: await of tile ({l}, {t})"


@pytest.mark.parametrize("devices", [None, [0, 0]])
def test_noop_adaptive_settings_are_render_tiled(devices):
    """adaptive=NULL, and min_samples >= sample_count, give the messages and the frame of rm_render_tiled bit for bit."""
    objs = SCENES["spheres"]
    st = settings(CAM, 8, TILE, spi=2)
    o = A.GpuOptions(seed=SEED, device_list=devices)

    def null_adaptive():
        s, oc, scene = st._c(), o._c(), product_scene(objs)       # the scene must outlive the call that snapshots it
        h = A.lib().rm_render_tiled_adaptive(scene._h, C.byref(s), C.byref(oc), None)
        assert h, A.last_error()
        return A.TaskHandle(h, st)

    runs = [lambda: A.render_tiled(product_scene(objs), st, o), null_adaptive,
            lambda: A.render_tiled(product_scene(objs), st, o, A.AdaptiveSettings(1e9, 8))]
    results = []
    for make in runs:
        msgs = poll_all(make())
        frame = make().await_()
        results.append(([(m.kind, m.tile.sample_count, m.tile.left, m.tile.top, bits(m.tile.data).tobytes()) for m in msgs], bits(frame)))
    for seq, frame in results[1:]:
        assert seq == results[0][0]
        assert np.array_equal(frame, results[0][1])


def test_keep_mode_nan_tiles_never_stop_early():
    """With RM_FLAG_KEEP_NONFINITE a tile that holds a NaN pixel has E_t = NaN and renders to the full count, however loose
    the threshold; every other tile stops at the first checkpoint."""
    objs = NONFINITE_SCENES["box"]
    cam, n, spi, seed, tile = F.camera(64, 48), 8, 2, 3, (8, 8)
    st = settings(cam, n, tile, spi=spi)
    layout = A.tile_layout(st)
    vals = oracle_samples(objs, cam, n, seed=seed)
    stop, E = predicted(objs, cam, 1e9, min_spp=2, n=n, spi=spi, keep=True, seed=seed, vals=vals, tile=tile)
    poisoned = np.isnan(E[2])
    assert poisoned.any() and (~poisoned).any()
    assert (stop[poisoned] == n).all() and (stop[~poisoned] == 2).all()
    task = A.render_tiled(product_scene(objs), st, A.GpuOptions(seed=seed, flags=A.FLAG_KEEP_NONFINITE), A.AdaptiveSettings(1e9, 2))
    msgs = poll_all(task)
    assert [(m.kind, m.tile.sample_count, m.tile.left, m.tile.top) for m in msgs] == expected_sequence(layout, stop, n, spi)
    for m in msgs:
        if m.kind == "TileFinished" and m.tile.sample_count == n:
            assert np.isnan(m.tile.data).any()


def test_cli_old_adaptive_twin(tmp_path):
    """cli_old --adaptive writes the PNG of the Python mirror's tonemapped adaptive frame, byte for byte."""
    from PIL import Image
    exe = str(tmp_path / "cli_old")
    lib_dir = os.path.join(ROOT, "raymond_b200")
    subprocess.run(["g++", "-O2", "-std=c++17", "-I", os.path.join(ROOT, "include"), os.path.join(ROOT, "examples", "cli_old.cpp"),
                    "-L", lib_dir, "-lraymond_cuda", f"-Wl,-rpath,{lib_dir}", "-o", exe], check=True)
    W, H, spp, spi, seed, tau, min_spp = 96, 64, 16, 4, 9, 0.05, 4
    out = str(tmp_path / "adaptive.png")
    res = subprocess.run([exe, "--out", out, "--width", str(W), "--height", str(H), "--spp", str(spp), "--spi", str(spi), "--seed", str(seed),
                          "--adaptive", str(tau), "--min-spp", str(min_spp)], check=True, capture_output=True, text=True)
    assert "Samples rendered" in res.stdout
    got = np.asarray(Image.open(out))
    st = A.Settings(A.CameraSettings.from_fixture(F.camera(W, H)), spp, (32, 32), 5, spi)
    task = A.render_tiled(product_scene(F.reflective_spheres()), st, A.GpuOptions(seed=seed), A.AdaptiveSettings(tau, min_spp))
    frame = task.await_()
    stats = task.stats()
    assert np.array_equal(got, A.tonemap(frame))
    assert f"Samples rendered: {stats['samples']} of {W * H * spp}" in res.stdout
