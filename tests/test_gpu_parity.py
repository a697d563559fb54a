"""Parity of the CUDA path (through the C-ABI) against the CPU oracle.

Bar (BASELINE.json north_star): per-point labels bit-exact; terrain-height cells within 1e-5
abs -- these tests demand the stronger bit-exact equality for every layer, every phase.
Oracle = reference semantics at thread_count = 1 (see oracle/gg_oracle.cpp header).
"""
import numpy as np
import pytest

from golden_util import ReferenceRecord, cloud_values
from groundgrid_b200 import capi, synth
from oracle import Oracle

pytestmark = pytest.mark.gpu

LIVE = ("variance", "minGroundHeight", "ground", "groundpatch")
DEAD = ("m2", "meanVariance", "groundCandidates", "planeDist", "maxGroundHeight", "pointsRaw")


def diff_report(name, a, b):
    bad = ~((a == b) | (np.isnan(a) & np.isnan(b)))
    if not bad.any():
        return None
    idx = np.argwhere(bad)
    ex = ", ".join(f"{tuple(i)}: gpu={a[tuple(i)]!r} cpu={b[tuple(i)]!r}" for i in idx[:5])
    return f"{name}: {bad.sum()} cells differ (max abs {np.nanmax(np.abs(a[bad] - b[bad])):.3e}); e.g. {ex}"


def assert_layers_equal(g, o, names, ctx):
    errs = [r for r in (diff_report(n, g.layer(n), o.layer(n)) for n in names) if r]
    assert not errs, f"{ctx}: " + " | ".join(errs)


def make_pair(dim, res, full=True, max_points=140000, **cfg):
    g = capi.GroundGridB200(dim, res, n_slots=1, max_points=max_points, full_layers=full)
    o = Oracle(dim, res)
    if cfg:
        g.set_config(**cfg)
        o.set_config(**cfg)
    return g, o


@pytest.fixture(scope="module")
def scan64():
    scene = synth.make_scene(seed=1234)
    return synth.scan_64(scene, seed=1234)


def test_expected_points_on_device():
    g, o = make_pair(99.0, 0.33)
    assert np.array_equal(g.layer("expectedPoints"), o.expected_points())
    levels, visits, mx = g.spiral_schedule_info()
    assert (levels, visits) == (743, 88504) and mx <= 512


@pytest.mark.parametrize("stage", [1, 2, 3])
def test_single_scan_phase_by_phase(scan64, stage):
    """configs[0]: one synthetic 64-beam scan (~120k pts, flat ground + boxes), N = 300."""
    pts, org = scan64
    g, o = make_pair(99.0, 0.33)
    g.init_map(0.0, 0.0, 0.0)
    o.init_map(0.0, 0.0, 0.0)
    g.run_single(pts, org, 0.0, stop_after=stage)
    o.filter_cloud(pts, org, 0.0, threads=1, stop_after=stage)
    names = ("points",) + LIVE + DEAD
    if stage == 1:  # the reference computes "variance" at the start of patch detection (:323)
        names = tuple(n for n in names if n != "variance")
    assert_layers_equal(g, o, names, f"stage {stage}")


def test_single_scan_labels_and_output_order(scan64):
    pts, org = scan64
    g, o = make_pair(99.0, 0.33)
    g.init_map(0.0, 0.0, 0.0)
    o.init_map(0.0, 0.0, 0.0)
    labels, index, cloud = g.filter_cloud(pts, org, 0.0, want_index=True, want_cloud=True)
    lab_o, idx_o, cloud_o = o.filter_cloud(pts, org, 0.0, threads=1, want_cloud=True)
    assert np.array_equal(labels, lab_o), f"{(labels != lab_o).sum()} labels differ"
    assert np.array_equal(index, idx_o)
    assert cloud.tobytes() == cloud_o.tobytes()
    assert_layers_equal(g, o, ("points",) + LIVE + DEAD, "after full scan")
    assert (labels == 99).sum() > 10000 and (labels == 49).sum() > 50000


def test_stream_with_rolling_prior_outliers_and_yaw():
    """configs[1] shape: a stream with ego motion (map rolls, prior carried), below-ground
    returns (outlier ray-march), pitched base frame (position-dependent seeding)."""
    dim, res = 99.0, 0.33
    g, o = make_pair(dim, res)
    scene = synth.make_scene(seed=77, stream_len=30.0, undulation=0.3)
    rng = np.random.default_rng(5)
    n_out = 0
    for k in range(12):
        (ex, ey), yaw = synth.stream_pose(k, step=1.0)
        ey = 0.4 * k
        pts, org = synth.scan_64(scene, ego_xy=(ex, ey), yaw=yaw, seed=1234 + k)
        if k >= 2:
            idx = rng.choice(len(pts), 400, replace=False)
            pts["z"][idx] -= rng.uniform(0.3, 1.2, 400).astype(np.float32)
        T = synth.base_from_map(ex, ey, yaw, base_z=0.0, pitch=0.01)
        if k == 0:
            g.init_map(ex, ey, 0.0)
            o.init_map(ex, ey, 0.0)
        else:
            mg = g.update_pose(ex, ey, T)
            mo = o.update(ex, ey, T)
            assert int(mg) == mo
            assert np.array_equal(g.position(), o.position())
            assert_layers_equal(g, o, ("ground", "groundpatch"), f"scan {k} after roll")
        labels = g.filter_cloud(pts, org, 0.02 * k)
        lab_o, idx_o, _ = o.filter_cloud(pts, org, 0.02 * k, threads=1)
        assert np.array_equal(labels, lab_o), f"scan {k}: {(labels != lab_o).sum()} labels differ"
        assert_layers_equal(g, o, ("points",) + LIVE + DEAD, f"scan {k}")
        n_out += len(pts) - len(idx_o)
    assert n_out >= 0


def test_odd_cell_count_with_rolls():
    """N = 101 (odd: layers are not 16-byte aligned, the roll kernels take their scalar path; the spiral centre
    cell sits off the geometric centre)."""
    dim, res = 33.33, 0.33
    g, o = make_pair(dim, res)
    assert g.n == 101
    scene = synth.make_scene(seed=41)
    for k in range(4):
        ex, ey = 0.7 * k, -0.45 * k
        pts, org = synth.scan_64(scene, ego_xy=(ex, ey), seed=4100 + k)
        T = synth.base_from_map(ex, ey, 0.0, base_z=0.0, pitch=0.005)
        if k == 0:
            g.init_map(ex, ey, 0.0)
            o.init_map(ex, ey, 0.0)
        else:
            assert int(g.update_pose(ex, ey, T)) == o.update(ex, ey, T)
            assert_layers_equal(g, o, ("ground", "groundpatch"), f"scan {k} after roll")
        labels = g.filter_cloud(pts, org, 0.0)
        lab_o, _, _ = o.filter_cloud(pts, org, 0.0, threads=1)
        assert np.array_equal(labels, lab_o), f"scan {k}: {(labels != lab_o).sum()} labels differ"
        assert_layers_equal(g, o, ("points",) + LIVE, f"scan {k}")


@pytest.mark.parametrize("seed", list(range(10)))
def test_random_geometry_and_config(seed):
    """Seeded random map geometry (odd and even cell counts, 0.2-0.6 m cells), random configuration within sane
    ranges, three scans with rolls, yaw and a pitched base frame, some points pushed below ground (outlier branch)."""
    rng = np.random.default_rng(9000 + seed)
    res = float(np.float32(rng.choice([0.2, 0.25, 0.33, 0.4, 0.5, 0.6])))
    n_target = int(rng.integers(41, 260))
    dim = n_target * res
    cfg = dict(point_count_cell_variance_threshold=int(rng.integers(2, 20)),
               max_ring=int(rng.choice([1024, 60, 48])),
               distance_factor=float(rng.choice([0.0001, 0.0002, 0.0005])),
               minimum_distance_factor=float(rng.choice([0.0005, 0.001, 0.002])),
               miminum_point_height_threshold=float(rng.uniform(0.2, 0.5)),
               minimum_point_height_obstacle_threshold=float(rng.uniform(0.05, 0.2)),
               outlier_tolerance=float(rng.uniform(0.05, 0.2)),
               ground_patch_detection_minimum_point_count_threshold=float(rng.uniform(0.1, 0.5)),
               patch_size_change_distance=float(rng.uniform(5.0, 40.0)),
               occupied_cells_decrease_factor=float(rng.choice([5.0, 3.0, 10.0, 1.5])),
               occupied_cells_point_count_factor=float(rng.choice([20.0, 10.0, 40.0])),
               min_outlier_detection_ground_confidence=float(rng.uniform(0.5, 2.0)))
    full = bool(seed & 1)
    g, o = make_pair(dim, res, full=full, **cfg)
    assert g.n == o.n
    scene = synth.make_scene(seed=9000 + seed, stream_len=15.0, undulation=0.2)
    step = float(rng.uniform(0.3, 2.0))
    for k in range(3):
        ex, ey, yaw = step * k, -0.6 * step * k, 0.02 * k
        pts, org = synth.scan_64(scene, ego_xy=(ex, ey), yaw=yaw, seed=9100 + 10 * seed + k)
        if k:
            idx = rng.choice(len(pts), 300, replace=False)
            pts["z"][idx] -= rng.uniform(0.3, 1.0, 300).astype(np.float32)
        T = synth.base_from_map(ex, ey, yaw, base_z=0.0, pitch=0.008)
        if k == 0:
            g.init_map(ex, ey, 0.0)
            o.init_map(ex, ey, 0.0)
        else:
            assert int(g.update_pose(ex, ey, T)) == o.update(ex, ey, T)
        labels = g.filter_cloud(pts, org, 0.01 * k)
        lab_o, _, _ = o.filter_cloud(pts, org, 0.01 * k, threads=1)
        ctx = f"seed {seed} N {g.n} res {res} scan {k}"
        assert np.array_equal(labels, lab_o), f"{ctx}: {(labels != lab_o).sum()} labels differ"
        assert_layers_equal(g, o, ("points",) + LIVE + (DEAD if full else ()), ctx)


def test_golden_fixtures_on_gpu():
    """The committed vectors of tests/golden/ -- produced by the reference itself (oracle/_ref, tests/golden/
    make_golden.py) -- through the C-ABI: creation, map rolls + seeding, labels, output order and all eleven layers bit
    for bit."""
    import golden_util

    files = golden_util.case_files()
    assert len(files) >= 5
    for path in files:
        case = golden_util.load_case(path)
        g = capi.GroundGridB200(case["dimension"], case["resolution"], n_slots=1, max_points=16384, full_layers=True)
        assert np.array_equal(g.layer("expectedPoints"), case["expected"])
        golden_util.replay(case, g, lambda g, x, y, T: g.update_pose(x, y, T),
                           lambda g, pts, org, bz: g.filter_cloud(pts, org, bz, want_index=True)[:2])
        g.close()


def test_outlier_branch_is_exercised():
    g, o = make_pair(99.0, 0.33)
    scene = synth.make_scene(seed=3)
    g.init_map(0.0, 0.0, 0.0)
    o.init_map(0.0, 0.0, 0.0)
    rng = np.random.default_rng(8)
    n_outliers = 0
    for k in range(3):
        pts, org = synth.scan_64(scene, seed=10 + k)
        if k:
            idx = rng.choice(len(pts), 3000, replace=False)
            pts["z"][idx] -= rng.uniform(0.25, 2.0, 3000).astype(np.float32)
        labels, index, _ = g.filter_cloud(pts, org, 0.0, want_index=True)
        lab_o, idx_o, _ = o.filter_cloud(pts, org, 0.0, threads=1)
        assert np.array_equal(labels, lab_o)
        assert np.array_equal(index, idx_o)
        assert_layers_equal(g, o, ("points",) + LIVE + DEAD, f"outlier scan {k}")
        # outliers = inside points that were neither rasterised nor ignored
        Gp, Cp = o.layer("ground"), o.layer("groundpatch")
        o.filter_cloud(pts, org, 0.0, threads=1, stop_after=1)
        near = ((pts["x"] - org[0]).astype(np.float64) ** 2 + (pts["y"] - org[1]).astype(np.float64) ** 2) < 12.5
        n_outliers += int(o.layer("pointsRaw").sum() - o.layer("points").sum()) - int(near.sum())
        o.set_layer("ground", Gp)
        o.set_layer("groundpatch", Cp)
    assert n_outliers > 100, n_outliers


def test_edge_cases_empty_border_nan_ring():
    g, o = make_pair(99.0, 0.33, max_points=4096)
    g.init_map(0.0, 0.0, 0.0)
    o.init_map(0.0, 0.0, 0.0)
    org = np.array([0.0, 0.0, 1.73], np.float32)
    # empty cloud
    empty = np.zeros(0, synth.POINT_DTYPE)
    labels, index, _ = g.filter_cloud(empty, org, 0.0, want_index=True)
    o.filter_cloud(empty, org, 0.0, threads=1)
    assert len(labels) == 0 and len(index) == 0
    assert_layers_equal(g, o, ("points",) + LIVE + DEAD, "empty cloud")
    n = o.n
    bx, by = o.cell_position(n - 3, 10)
    kx, ky = o.cell_position(n - 4, 10)
    xyz = np.array([[1, 1, 0], [10, 0, 0], [10, 0, 2], [100, 0, 0], [np.nan, 0, 0], [bx, by, 0], [kx, ky, 0], [20, 3, 0],
                    [0, 0, 5], [0.2, 0, 5], [np.inf, 1, 1], [5, -np.inf, 1]], np.float32)
    pts = np.zeros(len(xyz), synth.POINT_DTYPE)
    pts["x"], pts["y"], pts["z"] = xyz[:, 0], xyz[:, 1], xyz[:, 2]
    pts["ring"] = [0, 0, 0, 0, 0, 0, 0, 2000, 0, 0, 0, 0]
    labels, index, cloud = g.filter_cloud(pts, org, 0.0, want_index=True, want_cloud=True)
    lab_o, idx_o, cloud_o = o.filter_cloud(pts, org, 0.0, threads=1, want_cloud=True)
    assert list(labels) == list(lab_o) == [49, 49, 99, 0, 0, 0, 49, 49, 49, 99, 0, 0]
    assert np.array_equal(index, idx_o)
    assert cloud.tobytes() == cloud_o.tobytes()
    assert_layers_equal(g, o, ("points",) + LIVE + DEAD, "edge cases")


def test_points_on_cell_boundaries():
    """Cell index = trunc of an fp64 quotient: points on (and one float ulp around) cell edges must land
    in the oracle's cell (the kernel replaces the division by a guarded reciprocal multiply)."""
    g, o = make_pair(99.0, 0.33, max_points=70000)
    g.init_map(0.0, 0.0, 0.0)
    o.init_map(0.0, 0.0, 0.0)
    n = o.n
    rng = np.random.default_rng(12)
    idx = rng.integers(3, n - 3, (20000, 2))
    ex = np.array([o.cell_position(int(i), 0)[0] for i in range(n)]) + 0.5 * float(np.float32(0.33))   # upper edge of row i
    x = ex[idx[:, 0]].astype(np.float32)
    y = ex[idx[:, 1]].astype(np.float32)
    xs = np.concatenate([x, np.nextafter(x, np.float32(np.inf)), np.nextafter(x, np.float32(-np.inf))])
    ys = np.concatenate([y, np.nextafter(y, np.float32(-np.inf)), np.nextafter(y, np.float32(np.inf))])
    pts = np.zeros(len(xs), synth.POINT_DTYPE)
    pts["x"], pts["y"] = xs, ys
    pts["z"] = rng.uniform(-0.05, 1.0, len(xs)).astype(np.float32)
    org = np.array([0.0, 0.0, 1.73], np.float32)
    for k in range(2):
        a = g.filter_cloud(pts, org, 0.0)
        b, _, _ = o.filter_cloud(pts, org, 0.0, threads=1)
        assert np.array_equal(a, b)
    assert_layers_equal(g, o, ("points",) + LIVE + DEAD, "edge points")


def test_config_change_between_scans(scan64):
    pts, org = scan64
    cfg = dict(max_ring=40, patch_size_change_distance=12.0, occupied_cells_decrease_factor=3.0,
               outlier_tolerance=0.05, point_count_cell_variance_threshold=4, distance_factor=0.0002)
    g, o = make_pair(99.0, 0.33)
    g.init_map(0.0, 0.0, 0.0)
    o.init_map(0.0, 0.0, 0.0)
    a = g.filter_cloud(pts, org, 0.0)
    b, _, _ = o.filter_cloud(pts, org, 0.0, threads=1)
    assert np.array_equal(a, b)
    g.set_config(**cfg)
    o.set_config(**cfg)
    a = g.filter_cloud(pts, org, 0.0)
    b, _, _ = o.filter_cloud(pts, org, 0.0, threads=1)
    assert np.array_equal(a, b)
    assert_layers_equal(g, o, ("points",) + LIVE + DEAD, "after config change")


def test_live_layer_mode_matches_full_mode(scan64):
    """Without GG_FLAG_FULL_LAYERS the dead layers are skipped; everything the algorithm reads is identical."""
    pts, org = scan64
    g, o = make_pair(99.0, 0.33, full=False)
    g.init_map(0.0, 0.0, 0.0)
    o.init_map(0.0, 0.0, 0.0)
    for _ in range(2):
        a = g.filter_cloud(pts, org, 0.0)
        b, _, _ = o.filter_cloud(pts, org, 0.0, threads=1)
        assert np.array_equal(a, b)
    assert_layers_equal(g, o, ("points",) + LIVE, "live layers")
    with pytest.raises(capi.GroundGridError):
        g.layer("m2")


def test_reference_default_geometry_364(scan64):
    pts, org = scan64
    g, o = make_pair(120.0, 0.33)
    assert g.n == o.n == 364
    g.init_map(0.3, -0.2, 0.0)
    o.init_map(0.3, -0.2, 0.0)
    for k in range(2):
        a = g.filter_cloud(pts, org, 0.0)
        b, _, _ = o.filter_cloud(pts, org, 0.0, threads=1)
        assert np.array_equal(a, b)
    assert_layers_equal(g, o, ("points",) + LIVE + DEAD, "N=364")


def test_dense_128_beam_600_grid():
    """configs[2]: ~240k pts, 600 x 600 @ 0.2 m."""
    scene = synth.make_scene(seed=1234)
    pts, org = synth.scan_128(scene, seed=1234)
    g, o = make_pair(120.0, 0.2, max_points=270000)
    assert g.n == o.n == 600
    g.init_map(0.0, 0.0, 0.0)
    o.init_map(0.0, 0.0, 0.0)
    for k in range(2):
        a = g.filter_cloud(pts, org, 0.0)
        b, _, _ = o.filter_cloud(pts, org, 0.0, threads=1)
        assert np.array_equal(a, b), f"{(a != b).sum()} labels differ"
    assert_layers_equal(g, o, ("points",) + LIVE + DEAD, "N=600")


def test_four_lidar_500k():
    """configs[3]: 4-LiDAR fused cloud ~480k pts/frame, N = 364, shared rolling prior over two frames."""
    scene = synth.make_scene(seed=1234)
    g, o = make_pair(120.0, 0.33, max_points=540000)
    g.init_map(0.0, 0.0, 0.0)
    o.init_map(0.0, 0.0, 0.0)
    for k in range(2):
        pts, org = synth.scan_4lidar(scene, seed=1234 + k)
        assert len(pts) > 450000
        a = g.filter_cloud(pts, org, 0.0)
        b, _, _ = o.filter_cloud(pts, org, 0.0, threads=1)
        assert np.array_equal(a, b), f"{(a != b).sum()} labels differ"
    assert_layers_equal(g, o, ("points",) + LIVE + DEAD, "4-lidar")


def test_batched_slots_match_single_and_are_deterministic():
    """configs[4] shape: independent scans in separate slots, one batched call."""
    B = 6
    dim, res = 99.0, 0.33
    g = capi.GroundGridB200(dim, res, n_slots=B, max_points=131072, full_layers=False)
    scans = []
    for b in range(B):
        scene = synth.make_scene(seed=2000 + b)
        scans.append(synth.scan_64(scene, ego_xy=(0.1 * b, -0.2 * b), seed=2000 + b))
        g.init_map(0.1 * b, -0.2 * b, 0.0, slot=b)
    import torch

    hp = [torch.from_numpy(np.ascontiguousarray(p).view(np.uint8).copy()).pin_memory() for p, _ in scans]
    hl = [torch.zeros(len(p), dtype=torch.uint8).pin_memory() for p, _ in scans]
    results = []
    for rep in range(2):
        descs = g.make_descs(list(range(B)), [len(p) for p, _ in scans], [o for _, o in scans], [0.0] * B)
        g.filter_cloud_batch_ptrs(descs, [t.data_ptr() for t in hp], [t.data_ptr() for t in hl])
        results.append([t.numpy().copy() for t in hl])
    for b in range(B):
        o = Oracle(dim, res)
        o.init_map(0.1 * b, -0.2 * b, 0.0)
        for rep in range(2):
            lab_o, _, _ = o.filter_cloud(scans[b][0], scans[b][1], 0.0, threads=1)
            assert np.array_equal(results[rep][b], lab_o), f"slot {b} rep {rep}"
        for name in ("ground", "groundpatch", "variance", "points"):
            r = diff_report(name, g.layer(name, slot=b), o.layer(name))
            assert r is None, f"slot {b}: {r}"
    # determinism: the same inputs through a fresh handle give identical bits
    g2 = capi.GroundGridB200(dim, res, n_slots=B, max_points=131072, full_layers=False)
    for b in range(B):
        g2.init_map(0.1 * b, -0.2 * b, 0.0, slot=b)
    for rep in range(2):
        descs = g2.make_descs(list(range(B)), [len(p) for p, _ in scans], [o for _, o in scans], [0.0] * B)
        g2.filter_cloud_batch_ptrs(descs, [t.data_ptr() for t in hp], [t.data_ptr() for t in hl])
    for b in range(B):
        assert np.array_equal(hl[b].numpy(), results[1][b])
        assert np.array_equal(g2.layer("ground", slot=b), g.layer("ground", slot=b))


@pytest.mark.parametrize("dim,res", [(33.0, 0.33), (99.0, 0.33), (120.0, 0.33)])
def test_batch_of_ten_uses_the_shared_sm_spiral_layout(dim, res):
    """Launches of >= 9 scans run the spiral with time-shared lane threads (small CTAs, several scans per SM);
    fewer scans get one thread per lane.  Both must reproduce the sequential sweep bit for bit."""
    import torch

    B = 10
    g = capi.GroundGridB200(dim, res, n_slots=B, max_points=131072, full_layers=False)
    scans = [synth.scan_64(synth.make_scene(seed=700 + b), ego_xy=(0.05 * b, 0.0), seed=700 + b) for b in range(B)]
    hp = [torch.from_numpy(np.ascontiguousarray(p).view(np.uint8).copy()).pin_memory() for p, _ in scans]
    hl = [torch.zeros(len(p), dtype=torch.uint8).pin_memory() for p, _ in scans]
    for b in range(B):
        g.init_map(0.05 * b, 0.0, 0.0, slot=b)
    got = []
    for rep in range(2):
        descs = g.make_descs(list(range(B)), [len(p) for p, _ in scans], [o for _, o in scans], [0.0] * B)
        g.filter_cloud_batch_ptrs(descs, [t.data_ptr() for t in hp], [t.data_ptr() for t in hl])
        got.append([t.numpy().copy() for t in hl])
    for b in range(B):
        o = Oracle(dim, res)
        o.init_map(0.05 * b, 0.0, 0.0)
        for rep in range(2):
            want, _, _ = o.filter_cloud(scans[b][0], scans[b][1], 0.0, threads=1)
            assert np.array_equal(got[rep][b], want), f"slot {b} rep {rep}"
        for name in ("ground", "groundpatch"):
            r = diff_report(name, g.layer(name, slot=b), o.layer(name))
            assert r is None, f"slot {b}: {r}"
    g.close()


@pytest.mark.parametrize("dim,res", [(33.0, 0.33), (99.0, 0.33), (81.2, 0.4)])
def test_spiral_point_to_point_sync_variant(monkeypatch, dim, res):
    """GG_SPIRAL_ASYNC=1: k_spiral_skew without the CTA barrier per level (progress counters per warp, requirement table
    from gg_host.cpp:build_skew_sync).  Both thread layouts (one scan alone, a batch of ten) against the oracle."""
    import torch

    monkeypatch.setenv("GG_SPIRAL_ASYNC", "1")
    B = 10
    g = capi.GroundGridB200(dim, res, n_slots=B, max_points=131072, full_layers=False)
    scans = [synth.scan_64(synth.make_scene(seed=810 + b), ego_xy=(0.05 * b, 0.0), seed=810 + b) for b in range(B)]
    hp = [torch.from_numpy(np.ascontiguousarray(p).view(np.uint8).copy()).pin_memory() for p, _ in scans]
    hl = [torch.zeros(len(p), dtype=torch.uint8).pin_memory() for p, _ in scans]
    for b in range(B):
        g.init_map(0.05 * b, 0.0, 0.0, slot=b)
    first = g.filter_cloud(scans[0][0], scans[0][1], 0.0, slot=0)      # one scan alone: one thread per lane
    descs = g.make_descs(list(range(B)), [len(p) for p, _ in scans], [o for _, o in scans], [0.0] * B)
    g.filter_cloud_batch_ptrs(descs, [t.data_ptr() for t in hp], [t.data_ptr() for t in hl])   # batch: time-shared lane threads
    for b in range(B):
        o = Oracle(dim, res)
        o.init_map(0.05 * b, 0.0, 0.0)
        if b == 0:   # slot 0 saw its cloud twice: alone, then in the batch
            want, _, _ = o.filter_cloud(scans[0][0], scans[0][1], 0.0, threads=1)
            assert np.array_equal(first, want)
        want, _, _ = o.filter_cloud(scans[b][0], scans[b][1], 0.0, threads=1)
        assert np.array_equal(hl[b].numpy(), want), f"slot {b}"
        for name in ("ground", "groundpatch"):
            r = diff_report(name, g.layer(name, slot=b), o.layer(name))
            assert r is None, f"slot {b}: {r}"
    g.close()


@pytest.mark.parametrize("unit", ["2", "32"])
def test_overlapped_batches_begin_wait(monkeypatch, unit):
    """gg_filter_cloud_batch_begin/_wait: the clouds of step t+1 are packed and copied while the kernels of
    step t still run (two buffer sets); rolls in between; every step's labels and the final layers match."""
    import torch

    monkeypatch.setenv("GG_LAUNCH_UNIT", unit)
    dim, res, B, steps = 99.0, 0.33, 5, 6
    g = capi.GroundGridB200(dim, res, n_slots=B, max_points=131072, full_layers=False)
    scenes = [synth.make_scene(seed=500 + b, stream_len=20.0) for b in range(B)]
    clouds, host, labs = {}, {}, {}
    for k in range(steps):
        for b in range(B):
            p, org = synth.scan_64(scenes[b], ego_xy=(0.9 * k, 0.3 * k * (b - 2)), seed=900 + 10 * k + b)
            clouds[k, b] = (p, org)
            host[k, b] = torch.from_numpy(np.ascontiguousarray(p).view(np.uint8).copy()).pin_memory()
            labs[k, b] = torch.zeros(len(p), dtype=torch.uint8).pin_memory()
    slots = np.arange(B, dtype=np.int32)
    pending = None
    for k in range(steps):
        xy = np.array([[0.9 * k, 0.3 * k * (b - 2)] for b in range(B)])
        Ts = np.stack([synth.base_from_map(x, y).reshape(12) for x, y in xy])
        if k == 0:
            for b in range(B):
                g.init_map(xy[b, 0], xy[b, 1], 0.0, slot=b)
        else:
            g.update_pose_batch(slots, xy, Ts)
        descs = g.make_descs(list(range(B)), [len(clouds[k, b][0]) for b in range(B)], [clouds[k, b][1] for b in range(B)], [0.0] * B)
        ticket = g.filter_cloud_batch_begin(descs, [host[k, b].data_ptr() for b in range(B)], [labs[k, b].data_ptr() for b in range(B)])
        if pending is not None:
            g.filter_cloud_batch_wait(pending)
        pending = ticket
    g.filter_cloud_batch_wait(pending)
    g.synchronize()
    for b in range(B):
        o = Oracle(dim, res)
        for k in range(steps):
            x, y = 0.9 * k, 0.3 * k * (b - 2)
            if k == 0:
                o.init_map(x, y, 0.0)
            else:
                o.update(x, y, synth.base_from_map(x, y))
            want, _, _ = o.filter_cloud(clouds[k, b][0], clouds[k, b][1], 0.0, threads=1)
            assert np.array_equal(labs[k, b].numpy(), want), f"slot {b} step {k}: {(labs[k, b].numpy() != want).sum()} labels differ"
        for name in ("ground", "groundpatch", "variance", "points"):
            r = diff_report(name, g.layer(name, slot=b), o.layer(name))
            assert r is None, f"slot {b}: {r}"
    g.close()


def test_batch_on_a_shuffled_subset_of_slots_with_empty_clouds():
    """Batches need not cover every slot, nor list them in order; a scan may be empty and a label pointer null."""
    import torch

    dim, res, B = 66.0, 0.33, 7
    g = capi.GroundGridB200(dim, res, n_slots=B, max_points=131072, full_layers=False)
    oracles = []
    for b in range(B):
        g.init_map(0.2 * b, 0.0, 0.0, slot=b)
        o = Oracle(dim, res)
        o.init_map(0.2 * b, 0.0, 0.0)
        oracles.append(o)
    empty = np.zeros(0, synth.POINT_DTYPE)
    for rnd, (slots, empties, no_labels) in enumerate([([5, 2, 0, 6], {2}, {0}), ([1, 6, 3, 5, 4], set(), {4}), ([2, 0], {0}, set())]):
        clouds, host, labs = {}, {}, {}
        for b in slots:
            if b in empties:
                clouds[b] = (empty, np.array([0.2 * b, 0.0, 1.73], np.float32))
            else:
                clouds[b] = synth.scan_64(synth.make_scene(seed=800 + b), ego_xy=(0.2 * b, 0.0), seed=800 + 10 * rnd + b)
            p = clouds[b][0]
            host[b] = torch.from_numpy(np.ascontiguousarray(p).view(np.uint8).copy()).pin_memory() if len(p) else None
            labs[b] = torch.full((max(1, len(p)),), 7, dtype=torch.uint8).pin_memory()
        descs = g.make_descs(slots, [len(clouds[b][0]) for b in slots], [clouds[b][1] for b in slots], [0.0] * len(slots))
        g.filter_cloud_batch_ptrs(descs, [host[b].data_ptr() if host[b] is not None else None for b in slots],
                                  [None if b in no_labels else labs[b].data_ptr() for b in slots])
        for b in slots:
            want, _, _ = oracles[b].filter_cloud(clouds[b][0], clouds[b][1], 0.0, threads=1)
            if b in no_labels:
                assert (labs[b].numpy() == 7).all()
            else:
                assert np.array_equal(labs[b].numpy()[:len(want)], want), f"round {rnd} slot {b}"
            for name in ("ground", "groundpatch", "points"):
                r = diff_report(name, g.layer(name, slot=b), oracles[b].layer(name))
                assert r is None, f"round {rnd} slot {b}: {r}"
    g.close()


def test_batch_path_with_and_without_host_packing(monkeypatch):
    import torch

    dim, res, B = 99.0, 0.33, 3
    scans = [synth.scan_64(synth.make_scene(seed=300 + b), seed=300 + b) for b in range(B)]
    hp = [torch.from_numpy(np.ascontiguousarray(p).view(np.uint8).copy()).pin_memory() for p, _ in scans]
    out = {}
    for pack in ("1", "0", "mix"):
        if pack == "mix":      # default: packers and raw 32-byte copies side by side
            monkeypatch.delenv("GG_HOST_PACK", raising=False)
        else:
            monkeypatch.setenv("GG_HOST_PACK", pack)
        g = capi.GroundGridB200(dim, res, n_slots=B, max_points=131072)
        hl = [torch.zeros(len(p), dtype=torch.uint8).pin_memory() for p, _ in scans]
        for b in range(B):
            g.init_map(0.0, 0.0, 0.0, slot=b)
        for rep in range(2):
            descs = g.make_descs(list(range(B)), [len(p) for p, _ in scans], [o for _, o in scans], [0.0] * B)
            g.filter_cloud_batch_ptrs(descs, [t.data_ptr() for t in hp], [t.data_ptr() for t in hl])
        assert (g.host_pack_threads != 0) == (pack != "0")
        n_packed, n_raw, b_packed, b_raw = g.last_batch_transfer()[:4]
        assert n_packed + n_raw == B and (pack != "1" or n_raw == 0) and (pack != "0" or n_packed == 0)
        assert b_raw == sum(32 * len(scans[b][0]) for b in range(B)) if pack == "0" else b_packed + b_raw > 0
        out[pack] = [t.numpy().copy() for t in hl]
        g.close()
    for b in range(B):
        o = Oracle(dim, res)
        o.init_map(0.0, 0.0, 0.0)
        for rep in range(2):
            want, _, _ = o.filter_cloud(scans[b][0], scans[b][1], 0.0, threads=1)
        assert all(np.array_equal(out[k][b], want) for k in ("1", "0", "mix"))


def test_error_codes():
    g = capi.GroundGridB200(33.0, 0.33, n_slots=2, max_points=1024)
    org = np.zeros(3, np.float32)
    pts = np.zeros(4, synth.POINT_DTYPE)
    with pytest.raises(capi.GroundGridError) as e:       # scan before the first odometry: map missing
        g.filter_cloud(pts, org, 0.0)
    assert e.value.code == -3
    g.init_map(0, 0, 0)
    with pytest.raises(capi.GroundGridError) as e:
        g.filter_cloud(np.zeros(5000, synth.POINT_DTYPE), org, 0.0)
    assert e.value.code == -1
    with pytest.raises(capi.GroundGridError) as e:
        g.layer("nonexistent")
    assert e.value.code == -4
    with pytest.raises(capi.GroundGridError) as e:
        g.init_map(0, 0, 0, slot=7)
    assert e.value.code == -1


class CudaPath:
    """The CUDA path, called like the reference: transforms as (quaternion, translation)."""

    def __init__(self, dim, res, max_points):
        self.g = capi.GroundGridB200(dim, res, n_slots=1, max_points=max_points, full_layers=True)
        self.n = self.g.n

    def expected_points(self):
        return self.g.layer("expectedPoints")

    def init_map(self, x, y, z):
        self.g.init_map(x, y, z)

    def update(self, x, y, q, t):
        return self.g.update_pose(x, y, synth.tf2_matrix(q, t))

    def position(self):
        return self.g.position()

    def filter_cloud(self, pts, org, base_z):
        labels, index, _ = self.g.filter_cloud(pts, org, base_z, want_index=True)
        return labels, index

    def layer(self, name):
        return self.g.layer(name)

    def close(self):
        self.g.close()


class Reference:
    """The reference, for recording the scenario (needs oracle/_ref)."""

    def __init__(self, dim, res, max_points):
        from oracle import ref as refmod

        self.r = refmod.Reference(dim, res)
        self.n = self.r.n
        self.expected_points, self.init_map, self.position, self.layer = (self.r.expected_points, self.r.init_map,
                                                                          self.r.position, self.r.layer)

    def update(self, x, y, q, t):
        return bool(self.r.update(x, y, q, t))

    def filter_cloud(self, pts, org, base_z):
        return self.r.filter_cloud(pts, org, base_z)[:2]

    def close(self):
        self.r.close()


REFERENCE_CFGS = {"cfg2_300": (99.0, 0.33, synth.scan_64, 140000), "cfg3_600": (120.0, 0.2, synth.scan_128, 280000),
                  "cfg4_364": (120.0, 0.33, synth.scan_4lidar, 520000)}


def full_size_stream(rec, make, cfg):
    """Three scans with a map roll at one of BASELINE.json's full sizes."""
    dim, res, scan, maxp = REFERENCE_CFGS[cfg]
    m = make(dim, res, maxp)
    rec.check("cells", m.n)
    rec.check("expectedPoints", m.expected_points())
    m.init_map(0.0, 0.0, 0.0)
    scene = synth.make_scene(seed=4321, stream_len=20.0, undulation=0.3)
    rng = np.random.default_rng(17)
    for k in range(3):
        ex, ey, yaw = 1.1 * k, -0.45 * k, 0.01 * k
        pts, org = scan(scene, (ex, ey), yaw, seed=700 + k)
        if k:
            q, t = synth.base_from_map_qt(ex, ey, yaw, 0.0, pitch=0.02)
            rec.check(f"scan {k}: moved", m.update(ex, ey, q, t))
            rec.check(f"scan {k}: position", m.position())
            idx = rng.choice(len(pts), 2000, replace=False)
            pts["z"][idx] -= rng.uniform(0.25, 2.0, 2000).astype(np.float32)
        rec.check(f"scan {k}: input cloud", cloud_values(pts))
        labels, index = m.filter_cloud(pts, org, 0.0)
        rec.check(f"scan {k}: labels", labels)
        rec.check(f"scan {k}: output order", index)
        for n in ("points",) + LIVE + DEAD:
            rec.check(f"scan {k}: layer {n}", m.layer(n))
    m.close()


@pytest.mark.parametrize("cfg", list(REFERENCE_CFGS))
def test_cuda_path_against_the_reference_itself(cfg):
    """The CUDA path against oracle/_ref (the UNMODIFIED reference sources on CPU stand-ins; its answers are stored
    under tests/golden/ref_cuda_*.npz) at BASELINE.json's full sizes: three scans with a map roll, labels / output
    order / every layer bit for bit."""
    rec = ReferenceRecord(f"cuda_{cfg}")
    full_size_stream(rec, CudaPath, cfg)
    rec.finish()
