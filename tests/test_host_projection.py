"""CPU: the map-projection oracle (oracle/projection.py) against a brute-force per-pixel loop, known answers, argument validation of
pagnerf_b200.mapping.project_map and its C ABI entry."""
import numpy as np
import pytest
import torch

from oracle import projection as op


def _camera(cam, ang_deg=(0.0, 0.0)):
    """world -> camera view [4, 4] of a camera at `cam` looking down -z, tilted by ang_deg about x then y (bench.make_cameras)"""
    ax, ay = np.deg2rad(ang_deg)
    Rx = np.array([[1, 0, 0], [0, np.cos(ax), -np.sin(ax)], [0, np.sin(ax), np.cos(ax)]])
    Ry = np.array([[np.cos(ay), 0, np.sin(ay)], [0, 1, 0], [-np.sin(ay), 0, np.cos(ay)]])
    Rcw = Ry @ Rx
    V = np.eye(4)
    V[:3, :3] = Rcw.T
    V[:3, 3] = -Rcw.T @ np.asarray(cam, np.float64)
    return V.astype(np.float32)


def _cloud(seed, P, near):
    """Random points in front of the cameras of _cameras, with the awkward cases: exact duplicates (ties in z and pixel), equal
    depth side by side, points behind the camera, at z == near (camera 0), far off-screen, NaN and inf coordinates."""
    rng = np.random.default_rng(seed)
    f32 = np.float32
    x = rng.uniform(-1, 1, (P, 3)).astype(f32)
    x[:, 2] = rng.uniform(-1, 0.5, P).astype(f32)
    x[5:10] = x[0:5]                                    # duplicates: same z, same pixel, the smaller index wins
    x[10:20, 2] = x[20, 2]                              # equal depth for camera 0 (identity rotation)
    x[20:25, 2] = f32(1.5)                              # behind every camera (cameras at z = 1)
    x[25, 2] = f32(1.0) - f32(near)                     # camera 0: z = -(x_z - 1) computes to exactly near: dropped
    x[26] = [f32(1e30), 0, 0]                           # far off-screen: clamped before the integer conversion
    x[27] = [0, f32(-1e30), -0.5]
    x[28, 0], x[29, 1], x[30, 2], x[31] = np.nan, np.inf, -np.inf, np.nan
    return x


def _cameras(W, H):
    V = np.stack([_camera((0.0, 0.0, 1.0)), _camera((0.2, -0.1, 1.0), (3.0, -2.0)), _camera((-0.3, 0.2, 1.0), (-5.0, 4.0))])
    K = np.array([[0.9 * W, 0.9 * W, W / 2, H / 2], [0.7 * W, 0.8 * W, W / 2 + 0.3, H / 2 - 0.2],
                  [1.3 * W, 1.3 * W, W / 2 - 1.7, H / 2 + 0.4]], np.float32)
    return V, K


@pytest.mark.parametrize("max_radius", [0, 1, 3, 8])
@pytest.mark.parametrize("seed,k,level,H,W", [(0, 2, 2, 9, 13), (1, 1, 3, 12, 10), (2, 4, 1, 7, 16)])
def test_oracle_matches_brute_force(max_radius, seed, k, level, H, W):
    near = 0.0625                                                  # 1 - near is exact: point 25 sits at z == near
    x = _cloud(seed, 70, near)
    V, K = _cameras(W, H)
    point, depth, obj = op.project(x, k, level, V, K, H, W, max_radius, near, component=np.arange(70) % 4 - 1)
    want = op.brute_force(x, k, level, V, K, H, W, max_radius, near)
    assert np.array_equal(point, want)
    assert (point >= 0).any() and (point < 0).any()
    assert not np.isin(point, [20, 21, 22, 23, 24, 25, 26, 27, 28, 29, 30, 31]).any()
    assert not np.isin(point[0], [5, 6, 7, 8, 9]).any()                # ties go to the smaller index (camera 0: exact duplicates)
    hit = point >= 0
    assert np.isinf(depth[~hit]).all() and (depth[hit] > np.float32(near)).all()
    assert np.array_equal(obj, np.where(hit, np.maximum(point, 0) % 4 - 1, -1))
    # depth is the winner's z
    z0 = op.footprints(x, V[0], K[0], op.half_size(k, level), near, max_radius)[0]
    assert np.array_equal(depth[0][hit[0]], z0[point[0][hit[0]]])


def test_clamped_footprints_and_big_focal_lengths():
    """su and sv saturate at max_radius: a near point with a long focal length covers exactly (2R + 1)^2 pixels when it sits on a
    pixel centre; with max_radius = 0 every projected point covers exactly one pixel."""
    V = _camera((0.0, 0.0, 1.0))[None]
    K = np.array([[1000.0, 1000.0, 32.5, 32.5]], np.float32)          # u = 32.5: the centre of pixel 32
    x = np.array([[0, 0, 0.5]], np.float32)                          # z = 0.5, fx h / z = 250 >> R
    for R in (0, 1, 5, 32):
        point, depth, _ = op.project(x, 2, 2, V, K, 65, 65, R, 0.01)
        rows, cols = np.nonzero(point[0] == 0)
        assert rows.min() == 32 - R and rows.max() == 32 + R and cols.min() == 32 - R and cols.max() == 32 + R
        assert (point[0] == 0).sum() == (2 * R + 1) ** 2 and depth[0, 32, 32] == np.float32(0.5)
    rng = np.random.default_rng(3)
    xs = rng.uniform(-0.4, 0.4, (200, 3)).astype(np.float32)
    pairs = op.pixel_pairs(xs, V[0], [60.0, 50.0, 20.0, 15.0], 30, 40, op.half_size(2, 3), 0.01, 0)[0]
    z, u, v, su, sv, ok = op.footprints(xs, V[0], [60.0, 50.0, 20.0, 15.0], op.half_size(2, 3), 0.01, 0)
    on = ok & (u >= 0) & (u < 40) & (v >= 0) & (v < 30)
    assert pairs.size == on.sum() and np.array_equal(np.sort(pairs), np.sort((np.floor(v) * 40 + np.floor(u)).astype(np.int64)[on]))


def test_negative_focal_length_covers_nothing():
    V = _camera((0.0, 0.0, 1.0))[None]
    x = np.random.default_rng(0).uniform(-0.3, 0.3, (50, 3)).astype(np.float32)
    for K in ([-30.0, 30.0, 16.0, 16.0], [30.0, -30.0, 16.0, 16.0]):
        assert (op.project(x, 2, 3, V, np.array([K], np.float32), 32, 32, 4)[0] == -1).all()
        assert (op.brute_force(x, 2, 3, V, np.array([K], np.float32), 32, 32, 4) == -1).all()


def test_known_answers():
    """A point on the optical axis lands on pixel (floor(cx), floor(cy)) with the hand-computed footprint; of two overlapping
    points the nearer one wins."""
    V = np.eye(4, dtype=np.float32)
    V[2, 3] = -1.0                                                    # camera at (0, 0, 1), identity rotation
    K = np.array([[20.0, 12.0, 10.25, 7.75]], np.float32)
    x = np.array([[0.0, 0.0, 0.0]], np.float32)                       # z = 1
    # D = 2 << 2 = 8, h = 0.125: su = 20 * 0.125 = 2.5, sv = 1.5 -> columns 7..12, rows 6..9
    point, depth, _ = op.project(x, 2, 2, V, K, 16, 24, 8)
    want = np.full((16, 24), -1)
    want[6:10, 7:13] = 0
    assert np.array_equal(point[0], want) and (depth[0][want == 0] == 1.0).all() and np.isinf(depth[0][want < 0]).all()
    point, _, _ = op.project(x, 2, 2, V, K, 16, 24, 0)
    assert np.nonzero(point[0] == 0) == (np.array([7]), np.array([10]))
    # a second point at z = 0.5 on the same axis: su = 5, sv = 3 -> columns 5..15, rows 4..10, all nearer
    x2 = np.array([[0.0, 0.0, 0.0], [0.0, 0.0, 0.5]], np.float32)
    point, depth, obj = op.project(x2, 2, 2, V, K, 16, 24, 8, component=np.array([7, -1]))
    want = np.full((16, 24), -1)
    want[4:11, 5:16] = 1
    assert np.array_equal(point[0], want) and (depth[0][want == 1] == 0.5).all() and (obj[0] == -1).all()
    assert np.array_equal(point, op.brute_force(x2, 2, 2, V, K, 16, 24, 8))
    # the far point in front of the near one's rectangle keeps nothing; swap depths and it wins where it covers
    x3 = np.array([[0.0, 0.0, 0.5], [0.0, 0.0, 0.0]], np.float32)
    point, _, obj = op.project(x3, 2, 2, V, K, 16, 24, 8, component=np.array([7, -1]))
    assert np.array_equal(point[0], np.where(want == 1, 0, -1)) and np.array_equal(obj[0], np.where(want == 1, 7, -1))


def test_pixel_convention_matches_the_frame_rays():
    """The pixel a point lands on with max_radius = 0 is the one whose centre ray (bench.make_frame_rays' formula) passes nearest."""
    res, f = 64, 0.9 * 64
    cam = np.array([0.1, -0.05, 0.9])
    V = np.eye(4, dtype=np.float32)
    V[:3, 3] = -cam
    K = np.array([[f, f, res / 2, res / 2]], np.float32)
    rng = np.random.default_rng(5)
    c, r = rng.integers(2, res - 2, 40), rng.integers(2, res - 2, 40)
    fu, fv = rng.uniform(0.1, 0.9, 40), rng.uniform(0.1, 0.9, 40)          # away from the pixel borders
    zc = rng.uniform(0.5, 1.2, 40)
    d = np.stack([(c + fu - res / 2) / f, (r + fv - res / 2) / f, -np.ones(40)], 1)
    x = (cam + d * zc[:, None]).astype(np.float32)
    _, u, v, su, sv, ok = op.footprints(x, V, K[0], op.half_size(2, 7), 0.01, 0)
    assert ok.all() and (su == 0).all() and (sv == 0).all()
    assert np.array_equal(np.floor(u).astype(np.int64), c) and np.array_equal(np.floor(v).astype(np.int64), r)
    point, _, _ = op.project(x, 2, 7, V, K, res, res, 0)
    assert all(point[0, r[i], c[i]] >= 0 for i in range(40))


def _cpu_args(P=10, B=2):
    return dict(pts=torch.zeros(P, 3), samples_per_axis=2, level=3, view=torch.eye(4).repeat(B, 1, 1), intrinsics=torch.ones(B, 4),
                height=8, width=8)


@pytest.mark.parametrize("kwargs,err,match", [
    (dict(samples_per_axis=0), ValueError, "samples_per_axis"), (dict(samples_per_axis=9), ValueError, "samples_per_axis"),
    (dict(samples_per_axis=2.0), ValueError, "samples_per_axis"), (dict(level=-1), ValueError, "level"),
    (dict(level=16), ValueError, "level"), (dict(level=True), ValueError, "level"),
    (dict(pts=torch.zeros(4, 2)), ValueError, "xyz"), (dict(pts=torch.zeros(12)), ValueError, "xyz"),
    (dict(pts=torch.zeros(4, 3, dtype=torch.float64)), TypeError, "xyz"), (dict(pts=np.zeros((4, 3), np.float32)), TypeError, "xyz"),
    (dict(view=torch.eye(4)), ValueError, "view"), (dict(view=torch.zeros(2, 3, 4)), ValueError, "view"),
    (dict(view=torch.eye(4, dtype=torch.float64).repeat(2, 1, 1)), TypeError, "view"),
    (dict(view=torch.zeros(65536, 4, 4)), ValueError, "cameras"),
    (dict(intrinsics=torch.ones(3, 4)), ValueError, "intrinsics"), (dict(intrinsics=torch.ones(2, 3)), ValueError, "intrinsics"),
    (dict(intrinsics=torch.ones(8)), ValueError, "intrinsics"), (dict(intrinsics=torch.ones(2, 4, dtype=torch.float16)), TypeError, "intrinsics"),
    (dict(height=0), ValueError, "height"), (dict(height=16385), ValueError, "height"), (dict(height=8.0), ValueError, "height"),
    (dict(height=True), ValueError, "height"), (dict(width=0), ValueError, "width"), (dict(width=16385), ValueError, "width"),
    (dict(width="8"), ValueError, "width"), (dict(max_radius=-1), ValueError, "max_radius"), (dict(max_radius=33), ValueError, "max_radius"),
    (dict(max_radius=2.0), ValueError, "max_radius"), (dict(max_radius=None), ValueError, "max_radius"),
    (dict(near=0), ValueError, "near"), (dict(near=-0.1), ValueError, "near"), (dict(near=float("nan")), ValueError, "near"),
    (dict(near=float("inf")), ValueError, "near"), (dict(near=1e-50), ValueError, "near"), (dict(near=True), ValueError, "near"),
    (dict(near="0.1"), ValueError, "near"), (dict(near=None), ValueError, "near"),
    (dict(component=torch.zeros(9, dtype=torch.int64)), ValueError, "component"),
    (dict(component=torch.zeros(10, 1, dtype=torch.int64)), ValueError, "component"),
    (dict(component=[0] * 10), ValueError, "component"), (dict(component=torch.zeros(10, dtype=torch.int32)), TypeError, "component")])
def test_argument_validation(kwargs, err, match):
    from pagnerf_b200.mapping import project_map
    args = _cpu_args()
    args.update(kwargs)
    with pytest.raises(err, match=match):
        project_map(**args)


def test_cpu_tensors_are_refused():
    from pagnerf_b200.mapping import PanopticPoints, project_map
    with pytest.raises(RuntimeError, match="CUDA"):
        project_map(**_cpu_args())
    with pytest.raises(RuntimeError, match="CUDA"):
        project_map(**_cpu_args(), max_radius=0, near=1, component=torch.zeros(10, dtype=torch.int64))
    P = 5
    pts = PanopticPoints(torch.zeros(P, 3), torch.zeros(P, 3), torch.zeros(P), torch.zeros(P, dtype=torch.int64), torch.zeros(P),
                         torch.zeros(P, dtype=torch.int64), torch.zeros(P))
    with pytest.raises(RuntimeError, match="CUDA"):
        project_map(**dict(_cpu_args(), pts=pts))


def test_project_entry_point_in_the_header_and_the_library():
    from pagnerf_b200 import _lib
    assert len(_lib.parse_header()["pag_map_project"]) == 16
    assert _lib.KERNELS_PER_CALL["pag_map_project"] == 2
    assert "pag_map_project" in _lib.exported_symbols()
