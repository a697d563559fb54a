"""The oracle port (oracle/gg_oracle.cpp) against the REFERENCE ITSELF (oracle/_ref/libgg_ref.so = the unmodified
reference sources src/GroundSegmentation.cpp + GroundGrid.cpp compiled on CPU stand-ins, oracle/build_ref.py).

This is what pins the oracle: every layer, label, output position and map roll must agree bit for bit at
thread_count = 1 on the BASELINE.json configurations (cfg1/2: 64 beams, 300x300; cfg3: 128 beams, 600x600;
cfg4: four LiDARs ~480k points, 364x364), on rolling streams with outliers, and on random geometries / configs.
Each test is a scenario run once on the reference (tests/golden/make_reference_records.py) and on the port here:
the reference's answers are stored under tests/golden/ref_*.npz (golden_util.ReferenceRecord).
"""
import numpy as np
import pytest

from golden_util import ReferenceRecord, cloud_values
from groundgrid_b200 import synth
from oracle import LAYERS, Oracle
from oracle import ref as refmod


class Port(Oracle):
    """The implementation under test, called like the reference: transforms as (quaternion, translation)."""

    def update(self, x, y, q, t):
        return super().update(x, y, synth.tf2_matrix(q, t))

    def filter_cloud(self, pts, org, base_z):
        return super().filter_cloud(pts, org, base_z, threads=1, want_cloud=True)


class Reference(refmod.Reference):
    """The reference, for recording the scenarios (needs oracle/_ref)."""

    def filter_cloud(self, pts, org, base_z):
        return super().filter_cloud(pts, org, base_z, want_cloud=True)


def check_layers(rec, m, names, ctx):
    for n in names:
        rec.check(f"{ctx}: layer {n}", m.layer(n))


def new_map(rec, make, dim, res, **cfg):
    m = make(dim, res)
    rec.check("cells", m.n)
    if cfg:
        m.set_config(**cfg)
    m.init_map(0.0, 0.0, 0.0)
    check_layers(rec, m, ("points", "ground", "groundpatch", "minGroundHeight", "maxGroundHeight"), "creation")
    return m


def scan(rec, m, pts, org, base_z, ctx):
    rec.check(f"{ctx}: input cloud", cloud_values(pts))
    lab, order, cloud = m.filter_cloud(pts, org, base_z)
    rec.check(f"{ctx}: labels", lab)
    rec.check(f"{ctx}: output order", order)
    rec.check(f"{ctx}: output cloud", cloud_values(cloud))
    check_layers(rec, m, LAYERS, ctx)
    return lab


def push_below_ground(pts, count, seed):
    rng = np.random.default_rng(seed)
    idx = rng.choice(len(pts), count, replace=False)
    pts["z"][idx] -= rng.uniform(0.25, 2.0, count).astype(np.float32)


def expected_points_table(rec, make):
    for dim, res in ((99.0, 0.33), (120.0, 0.33), (120.0, 0.2), (33.0, 0.6)):
        m = make(dim, res)
        rec.check(f"{dim} m @ {res}: cells", m.n)
        rec.check(f"{dim} m @ {res}: expected points", m.expected_points())


def cfg1_cfg2_64_beam_300(rec, make):
    m = new_map(rec, make, 99.0, 0.33)
    scene = synth.make_scene(seed=1234)
    for k in range(3):
        pts, org = synth.scan_64(scene, seed=1234 + k)
        if k == 2:
            push_below_ground(pts, 3000, 5)
        lab = scan(rec, m, pts, org, 0.0, f"cfg2 scan {k}")
    assert (lab == 99).sum() > 10000 and (lab == 49).sum() > 50000


def cfg3_128_beam_600(rec, make):
    m = new_map(rec, make, 120.0, 0.2)
    assert m.n == 600
    scene = synth.make_scene(seed=77)
    for k in range(2):
        pts, org = synth.scan_128(scene, seed=300 + k)
        scan(rec, m, pts, org, 0.0, f"cfg3 scan {k}")


def cfg4_four_lidar_364(rec, make):
    m = new_map(rec, make, 120.0, 0.33)
    assert m.n == 364
    scene = synth.make_scene(seed=99)
    for k in range(2):
        pts, org = synth.scan_4lidar(scene, seed=400 + k)
        assert len(pts) > 450000
        scan(rec, m, pts, org, 0.0, f"cfg4 scan {k}")


def rolling_stream_with_outliers(rec, make):
    m = new_map(rec, make, 99.0, 0.33)
    scene = synth.make_scene(seed=1234, stream_len=30.0, undulation=0.3)
    moved_any = 0
    for k in range(12):
        (ex, ey), yaw = synth.stream_pose(k, step=0.9)
        ey = -0.37 * k
        pts, org = synth.scan_64(scene, (ex, ey), yaw, seed=500 + k, az_steps=1024)
        if k:
            q, t = refmod.base_from_map_qt(ex, ey, yaw, 0.01 * k, pitch=0.02)
            moved = m.update(ex, ey, q, t)
            moved_any += bool(moved)
            rec.check(f"roll {k}: moved", moved)
            rec.check(f"roll {k}: position", m.position())
            check_layers(rec, m, ("ground", "groundpatch"), f"roll {k}")
            push_below_ground(pts, 1500, 600 + k)
        scan(rec, m, pts, org, 0.01 * k, f"stream scan {k}")
    assert moved_any >= 8


def large_jump_clears_the_map(rec, make):
    m = new_map(rec, make, 33.0, 0.33)
    scene = synth.make_scene(seed=10, n_boxes=8, rmin=4.0, rmax=14.0)
    pts, org = synth.lidar_scan(scene, beams=24, az_steps=256, seed=1)
    scan(rec, m, pts, org, 0.0, "before jump")
    q, t = refmod.base_from_map_qt(100.0, -70.0, 0.3, 0.2, pitch=0.01)
    assert m.update(100.0, -70.0, q, t) == 1
    rec.check("jump: position", m.position())
    check_layers(rec, m, ("ground", "groundpatch"), "after jump")


def _draw_geometry(rng):
    return float(rng.integers(24, 70)), float(np.float32(rng.uniform(0.2, 0.6)))


def random_geometry_and_config(rec, make, seed):
    rng = np.random.default_rng(9000 + seed)

    def draws_until_accepted():
        """GroundSegmentation::init takes the map length as size_t: the reference refuses some geometries."""
        probe = np.random.default_rng(9000 + seed)
        for k in range(1, 1000):
            try:
                refmod.Reference(*_draw_geometry(probe))
            except ValueError:
                continue
            return k

    for _ in range(int(rec.given("geometry draws", draws_until_accepted))):
        dim, res = _draw_geometry(rng)
    cfg = dict(point_count_cell_variance_threshold=int(rng.integers(0, 30)), max_ring=int(rng.integers(10, 1024)),
               distance_factor=float(rng.uniform(0.0, 0.001)), minimum_distance_factor=float(rng.uniform(1e-4, 0.002)),
               miminum_point_height_threshold=float(rng.uniform(0.1, 0.6)),
               minimum_point_height_obstacle_threshold=float(rng.uniform(0.02, 0.2)),
               outlier_tolerance=float(rng.uniform(-0.2, 0.3)),
               ground_patch_detection_minimum_point_count_threshold=float(rng.uniform(0.05, 0.8)),
               patch_size_change_distance=float(rng.uniform(3.0, 30.0)),
               occupied_cells_decrease_factor=float(rng.uniform(1.5, 20.0)),
               occupied_cells_point_count_factor=float(rng.uniform(2.0, 40.0)),
               min_outlier_detection_ground_confidence=float(rng.uniform(0.2, 3.0)))
    m = new_map(rec, make, dim, res, **cfg)
    half = 0.5 * dim
    scene = synth.make_scene(seed=seed, n_boxes=10, rmin=3.0, rmax=0.8 * half)
    ex = ey = 0.0
    for k in range(3):
        ex += float(rng.uniform(-1.5, 1.5)) * (k > 0)
        ey += float(rng.uniform(-1.5, 1.5)) * (k > 0)
        yaw = float(rng.uniform(-0.5, 0.5))
        pts, org = synth.lidar_scan(scene, (ex, ey), yaw, beams=32, az_steps=512, seed=seed * 10 + k)
        if k:
            q, t = refmod.base_from_map_qt(ex, ey, yaw, 0.05 * k, pitch=float(rng.uniform(-0.03, 0.03)))
            rec.check(f"scan {k}: moved", m.update(ex, ey, q, t))
            rec.check(f"scan {k}: position", m.position())
            push_below_ground(pts, 400, seed + k)
        scan(rec, m, pts, org, 0.05 * k, f"random {seed} dim {dim} res {res} scan {k}")


def geometry_primitives(rec, make):
    m = new_map(rec, make, 33.0, 0.33)
    rng = np.random.default_rng(4)

    def check(ctx):
        c = m.position()
        xs = np.concatenate([rng.uniform(-20, 20, 400) + c[0], c[0] + 0.5 * 33.0 + np.array([-1e-9, 0.0, 1e-9]),
                             c[0] - 0.5 * 33.0 + np.array([-1e-9, 0.0, 1e-9])])
        ys = np.concatenate([rng.uniform(-20, 20, 400) + c[1], c[1] + rng.uniform(-16, 16, 6)])
        rows = []
        for x, y in zip(xs, ys):
            for fx, fy in ((float(np.float32(x)), float(np.float32(y))), (float(x), float(y))):
                i, j, inside = m.grid_index(fx, fy)
                rows.append((i, j, 1) if inside else (0, 0, 0))   # the index of an outside position is not defined
        rec.check(f"{ctx}: grid_index", np.array(rows))
        ij = rng.integers(0, m.n, (50, 2))
        rec.check(f"{ctx}: cell_position", np.array([m.cell_position(int(i), int(j)) for i, j in ij]))

    check("start")
    q, t = refmod.base_from_map_qt(3.21, -1.77, 0.1, 0.0)
    assert m.update(3.21, -1.77, q, t) == 1
    check("moved")


def single_phase_calls(rec, make):
    m = new_map(rec, make, 33.0, 0.33)
    rng = np.random.default_rng(12)
    G = rng.normal(0.0, 0.5, (m.n, m.n)).astype(np.float32)
    Cf = rng.uniform(0.0, 1.0, (m.n, m.n)).astype(np.float32)
    Cf[rng.uniform(size=Cf.shape) < 0.5] = 0.0
    m.set_layer("ground", G)
    m.set_layer("groundpatch", Cf)
    for x, y in ((5, 7), (48, 49), (49, 49), (1, 1), (97, 97), (60, 12)):
        m.interpolate_cell(x, y)
    check_layers(rec, m, ("ground", "groundpatch"), "interpolate_cell")
    m.spiral(0.25)
    check_layers(rec, m, ("ground", "groundpatch"), "spiral")


SCENARIOS = {
    "expected_points_table": expected_points_table,
    "cfg1_cfg2_64_beam_300": cfg1_cfg2_64_beam_300,
    "cfg3_128_beam_600": cfg3_128_beam_600,
    "cfg4_four_lidar_364": cfg4_four_lidar_364,
    "rolling_stream_with_outliers": rolling_stream_with_outliers,
    "large_jump_clears_the_map": large_jump_clears_the_map,
    **{f"random_geometry_and_config_{s}": (lambda rec, make, s=s: random_geometry_and_config(rec, make, s)) for s in range(8)},
    "geometry_primitives": geometry_primitives,
    "single_phase_calls": single_phase_calls,
}


def against_reference(name):
    rec = ReferenceRecord(name)
    SCENARIOS[name](rec, Port)
    rec.finish()


def test_expected_points_table():
    against_reference("expected_points_table")


def test_cfg1_cfg2_64_beam_300():
    """configs[0]/[1]: ~120 k points, 300 x 300 @ 0.33 m; three scans so that the prior is non-trivial."""
    against_reference("cfg1_cfg2_64_beam_300")


def test_cfg3_128_beam_600():
    """configs[2]: ~240 k points, 600 x 600 @ 0.2 m."""
    against_reference("cfg3_128_beam_600")


def test_cfg4_four_lidar_364():
    """configs[3]: four 64-beam sensors, ~480 k points, the reference's own 364 x 364 map."""
    against_reference("cfg4_four_lidar_364")


def test_rolling_stream_with_outliers():
    """12 scans: ego moves, yaws, the base frame is pitched (position-dependent seeding of exposed cells), points
    pushed below the ground (outlier ray-march against the rolled prior).  Map position, moved flag, the rolled prior and
    every layer after every scan must agree."""
    against_reference("rolling_stream_with_outliers")


def test_large_jump_clears_the_map():
    """A pose jump of more than the map length drops the whole map (grid_map::move -> clearAll + one full region)."""
    against_reference("large_jump_clears_the_map")


@pytest.mark.parametrize("seed", range(8))
def test_random_geometry_and_config(seed):
    """Seeded random geometries (integer map lengths: GroundSegmentation::init takes the dimension as size_t) and
    configurations, two or three scans with a roll in between."""
    against_reference(f"random_geometry_and_config_{seed}")


def test_geometry_primitives_agree():
    """grid_map index <-> position arithmetic of the port (oracle/gridmap_semantics.hpp) against the CPU GridMap the
    reference was compiled with, on random and on edge positions, before and after a move."""
    against_reference("geometry_primitives")


def test_single_phase_calls_agree():
    """interpolate_cell and the whole spiral called on their own (public methods, GroundSegmentation.h:56-62)."""
    against_reference("single_phase_calls")


@pytest.mark.skipif(not refmod.available(), reason="oracle/_ref/libgg_ref.so not built (needs the reference sources)")
def test_reference_threading_as_shipped_runs():
    """thread_count = 8 (the shipped default) is racy and therefore not a parity target; it must still run and label
    nearly everything like the sequential execution (used for the timing baseline)."""
    r1, r8 = refmod.Reference(99.0, 0.33), refmod.Reference(99.0, 0.33)
    r8.set_config(thread_count=8)
    scene = synth.make_scene(seed=1234)
    pts, org = synth.scan_64(scene, seed=1234)
    for r in (r1, r8):
        r.init_map(0.0, 0.0, 0.0)
    l1, _, _ = r1.filter_cloud(pts, org, 0.0)
    l8, _, _ = r8.filter_cloud(pts, org, 0.0)
    assert (l1 != l8).mean() < 0.02
