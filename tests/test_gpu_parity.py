"""GPU parity tests (-m gpu): the CUDA path, called through the C ABI, against the CPU oracle on the same seeded
inputs.  Integer / index / gate results are compared exactly; poses within the north-star tolerance
(1e-4 m / 1e-4 rad)."""
import numpy as np
import pytest

import oracle_lib as orc
import synthetic as syn

pytestmark = pytest.mark.gpu

POSE_TOL_T = 1e-4  # metres   (BASELINE.json north_star)
POSE_TOL_R = 1e-4  # radians


@pytest.fixture(scope="module")
def c1():
    """Config C1: 16-ring x 1024 sweep, 50k-point submap."""
    scene = syn.make_scene()
    traj = syn.trajectory(6)
    surf_map, corner_map = syn.make_submap(scene, 50000)
    cloud, ss, se = syn.make_sweep(scene, traj[4], 16, 1024, seed=4)
    f = orc.extract_cloud(cloud, ss, se)
    cs, _ = orc.voxel_grid(f["corner_points_less_sharp"], 0.2, True)
    sf, _ = orc.voxel_grid(f["surf_points_less_flat"], 0.4, True)
    init = syn.perturb_pose(traj[4], np.random.Generator(np.random.PCG64(11)))
    return dict(scene=scene, truth=traj[4], surf_map=surf_map, corner_map=corner_map, cloud=cloud, ss=ss, se=se, feat=f,
                corner_scan=cs, surf_scan=sf, init=init)


def _rand_cloud(rng, n, lo=-20, hi=20):
    return np.concatenate([rng.uniform(lo, hi, (n, 3)), np.zeros((n, 1))], 1).astype(np.float32)


# ------------------------------------------------------------------------------------------------ kNN
@pytest.mark.parametrize("k", [1, 5, 10])
@pytest.mark.parametrize("cell", [0.25, 0.5, 1.0])
def test_knn_index_exact(ctx, k, cell):
    rng = np.random.default_rng(100 + k)
    m = _rand_cloud(rng, 200000, -10, 10)  # dense: most queries have k neighbours within 1 m
    q = _rand_cloud(rng, 4000, -11, 11)    # some outside the map
    ctx.map_build(2, m, cell)
    idx, sqd = ctx.knn(2, q, k, 1.0)
    ridx, rsqd = orc.knn(m, q, k)
    inside = rsqd < 1.0
    assert np.array_equal(idx[inside], ridx[inside])
    assert np.array_equal(sqd[inside], rsqd[inside])  # bit-exact float distances
    assert np.all(idx[~inside] == -1) and np.all(np.isinf(sqd[~inside]))
    # sortedness / recomputation properties
    ok = idx >= 0
    d = ((m[np.where(ok, idx, 0)][:, :, :3] - q[:, None, :3]) ** 2)
    d2 = (d[..., 0] + d[..., 1]) + d[..., 2]
    assert np.array_equal(d2[ok], sqd[ok])
    assert np.all(np.diff(np.where(ok, sqd, np.float32(3e38)), axis=1) >= 0)


def test_knn_with_pose_and_large_radius(ctx):
    rng = np.random.default_rng(7)
    m = _rand_cloud(rng, 30000, -30, 30)
    q = _rand_cloud(rng, 1000, -5, 5)
    pose = syn.pose7([1, -2, 0.5], syn.quat_from_rpy(0.1, 0.2, 0.3))
    ctx.map_build(3, m, 1.0)
    idx, sqd = ctx.knn(3, q, 1, 25.0, pose7=pose)  # K=1, DISTANCE_SQ_THRESHOLD radius (feature_extract.hpp:155-158)
    qt = orc.associate(q, pose)
    ridx, rsqd = orc.knn(m, qt, 1)
    inside = rsqd < 25.0
    assert inside.mean() > 0.9
    assert np.array_equal(idx[inside], ridx[inside]) and np.array_equal(sqd[inside], rsqd[inside])


def test_knn_tiny_and_empty_maps(ctx):
    m = np.array([[0, 0, 0, 0], [0.5, 0, 0, 0], [0, 0.5, 0, 0]], np.float32)
    ctx.map_build(2, m, 0.5)
    idx, sqd = ctx.knn(2, np.array([[0.1, 0, 0, 0]], np.float32), 5, 1.0)
    assert list(idx[0]) == [0, 1, 2, -1, -1] and np.isinf(sqd[0, 3])
    ctx.map_build(2, np.zeros((0, 4), np.float32), 0.5)
    idx, _ = ctx.knn(2, np.array([[0.1, 0, 0, 0]], np.float32), 5, 1.0)
    assert np.all(idx == -1)
    idx, _ = ctx.knn(2, np.zeros((0, 4), np.float32), 5, 1.0)
    assert idx.shape == (0, 5)


# ------------------------------------------------------------------------------------------------ matching
@pytest.mark.parametrize("kind", ["c", "s"])
def test_match_from_map_exact(ctx, c1, kind):
    slot = 0 if kind == "c" else 1
    map_ = c1["corner_map"] if kind == "c" else c1["surf_map"]
    data = c1["corner_scan"] if kind == "c" else c1["surf_scan"]
    ctx.map_build(slot, map_, 0.5)
    valid, coeffs, nn = ctx.match_from_map(slot, kind, data, c1["init"])
    rvalid, rcoeffs, rnn = orc.match_from_map(kind, map_, data, c1["init"])
    assert rvalid.sum() > 100
    assert np.array_equal(valid, rvalid)                      # identical accept/reject at every gate
    assert np.array_equal(nn[valid], rnn[rvalid])             # identical neighbour sets, same order
    if kind == "s":
        assert np.array_equal(coeffs[valid], rcoeffs[rvalid])  # bit-exact plane (n, d)
    else:
        a, b = coeffs[valid], rcoeffs[rvalid]
        same = np.all(a == b, axis=1)
        swapped = np.all(a[:, [3, 4, 5, 0, 1, 2]] == b, axis=1)  # eigenvector sign is free: [X1;X2] may swap
        assert np.all(same | swapped)
        assert same.mean() > 0.99


def test_match_fov_gate_and_neigh10(ctx, c1, mloam):
    ctx.map_build(1, c1["surf_map"], 0.5)
    ctx.set_params(check_fov=1, n_neigh=10)
    try:
        valid, coeffs, nn = ctx.match_from_map(1, "s", c1["surf_scan"], c1["init"])
        rvalid, rcoeffs, rnn = orc.match_from_map("s", c1["surf_map"], c1["surf_scan"], c1["init"], n_neigh=10, check_fov=True)
        assert 10 < rvalid.sum() < rvalid.shape[0]
        assert np.array_equal(valid, rvalid) and np.array_equal(nn[valid], rnn[rvalid])
        assert np.array_equal(coeffs[valid], rcoeffs[rvalid])
    finally:
        ctx.set_params(check_fov=0, n_neigh=5)


# ------------------------------------------------------------------------------------------------ factors
@pytest.mark.parametrize("kind", [0, 1, 2, 3, 4])
def test_factor_evaluate_matches_oracle(ctx, kind):
    rng = np.random.default_rng(40 + kind)
    n = 257
    pts = rng.normal(size=(n, 3)) * 5
    if kind in (0, 3):
        nrm = rng.normal(size=(n, 3))
        nrm /= np.linalg.norm(nrm, axis=1, keepdims=True)
        coeffs = np.concatenate([nrm, rng.normal(size=(n, 1)), np.zeros((n, 2))], 1)
    else:
        a = rng.normal(size=(n, 3)) * 5
        coeffs = np.concatenate([a, a + rng.normal(size=(n, 3))], 1)
    npar = 3 if kind >= 3 else 1
    x = np.concatenate([syn.pose7(rng.normal(size=3) * 2, rng.normal(size=4)) for _ in range(npar)])
    sinfo = rng.uniform(0.3, 1.0, n) if kind != 2 else None
    res, jac = ctx.factor_evaluate(kind, pts, coeffs, x, sqrt_info=sinfo)
    rows = 3 if kind == 2 else 1
    cols = 21 if kind >= 3 else 7
    for i in range(0, n, 7):
        r, J = orc.factor_eval(kind, pts[i], coeffs[i], 1.0 if sinfo is None else sinfo[i], x)
        assert np.allclose(res[i], r[:rows], rtol=1e-12, atol=1e-12)
        assert np.allclose(jac[i].reshape(-1), J[: rows * cols], rtol=1e-11, atol=1e-11)
    # null-tolerant on jacobians, like Evaluate(param, residuals, nullptr)
    res2, _ = ctx.factor_evaluate(kind, pts, coeffs, x, sqrt_info=sinfo, want_jac=False)
    assert np.array_equal(res, res2)


def test_factor_check_convention_fd(ctx):
    """The reference's check(): forward differences, eps 1e-6, q * deltaQ (lidar_map_factor.hpp:72-120), on the GPU path."""
    rng = np.random.default_rng(5)
    x = syn.pose7([0.3, -1, 2], rng.normal(size=4))
    p = np.array([[1.0, 2.0, -0.5]])
    w = np.array([0.36, 0.48, 0.8])
    coeff = np.array([[*w, 0.7, 0, 0]])
    r, J = ctx.factor_evaluate(0, p, coeff, x)
    for k in range(6):
        d = np.zeros(6)
        d[k] = 1e-6
        rp, _ = ctx.factor_evaluate(0, p, coeff, ctx.pose_plus(x, d), want_jac=False)
        assert abs((rp[0, 0] - r[0, 0]) / 1e-6 - J[0, 0, k]) < 1e-4
    assert J[0, 0, 6] == 0.0


def test_pose_plus_matches_oracle(ctx):
    rng = np.random.default_rng(6)
    for _ in range(10):
        x = syn.pose7(rng.normal(size=3), rng.normal(size=4))
        d = rng.normal(size=6) * 0.1
        V = rng.normal(size=(6, 6))
        assert np.allclose(ctx.pose_plus(x, d), orc.plus(x, d), rtol=0, atol=1e-15)
        assert np.allclose(ctx.pose_plus(x, d, V), orc.plus(x, d, V), rtol=0, atol=1e-15)
    x = syn.pose7([1, 2, 3], [0, 0, 0, 1])
    assert np.array_equal(ctx.pose_plus(x, np.zeros(6)), x)  # Plus(x, 0) = x


def test_normal_equations_match_oracle(ctx, c1):
    # features from the oracle's association so both sides reduce the same rows
    vs, cfs, _ = orc.match_from_map("s", c1["surf_map"], c1["surf_scan"], c1["init"])
    vc, cfc, _ = orc.match_from_map("c", c1["corner_map"], c1["corner_scan"], c1["init"])
    pts = np.concatenate([c1["surf_scan"][vs][:, :3], c1["corner_scan"][vc][:, :3]]).astype(np.float64)
    coeffs = np.concatenate([cfs[vs], cfc[vc]])
    types = np.array([ord("s")] * int(vs.sum()) + [ord("c")] * int(vc.sum()), np.uint8)
    for huber_a in (0.1, 1.0):
        H, g, cost = ctx.normal_equations(types, pts, coeffs, 1.0, huber_a, c1["init"])
        rH, rg, rcost = orc.normal_eq(types, pts, coeffs, 1.0, huber_a, c1["init"])
        assert np.allclose(H, rH, rtol=1e-11, atol=1e-9)
        assert np.allclose(g, rg, rtol=1e-10, atol=1e-10)
        assert abs(cost - rcost) <= 1e-12 * max(1.0, abs(rcost))
        assert np.array_equal(H, H.T)
    # linearity: duplicating the rows doubles H, g, cost
    H2, g2, cost2 = ctx.normal_equations(np.tile(types, 2), np.tile(pts, (2, 1)), np.tile(coeffs, (2, 1)), 1.0, 0.1, c1["init"])
    H1, g1, cost1 = ctx.normal_equations(types, pts, coeffs, 1.0, 0.1, c1["init"])
    assert np.allclose(H2, 2 * H1, rtol=1e-12) and np.allclose(g2, 2 * g1, rtol=1e-11, atol=1e-12) and abs(cost2 - 2 * cost1) < 1e-9


# ------------------------------------------------------------------------------------------------ voxel grid
@pytest.mark.parametrize("leaf,last", [(0.2, False), (0.4, True), (1.0, False)])
def test_voxel_downsample_bit_exact(ctx, c1, leaf, last):
    pts = c1["feat"]["surf_points_less_flat"]
    out = ctx.voxel_downsample(pts, leaf, last)
    ref, ok = orc.voxel_grid(pts, leaf, last)
    assert ok and out.shape == ref.shape
    assert np.array_equal(out.view(np.uint32), ref.view(np.uint32))
    # idempotence-like property: filtering the centroids again never increases the count
    out2 = ctx.voxel_downsample(out, leaf, last)
    assert out2.shape[0] <= out.shape[0]


def test_voxel_downsample_edge_cases(ctx):
    assert ctx.voxel_downsample(np.zeros((0, 4), np.float32), 0.2).shape[0] == 0
    one = np.array([[1.5, -2.5, 3.5, 9.0]], np.float32)
    assert np.array_equal(ctx.voxel_downsample(one, 0.2), one)
    pts = np.array([[0.1, 0.1, 0.1, 1], [0.3, 0.5, 0.7, 3], [np.nan, 0, 0, 0], [1.5, 0.2, 0.2, 5], [0.2, 1.6, 0.1, 7]], np.float32)
    out = ctx.voxel_downsample(pts, 1.0)
    ref, _ = orc.voxel_grid(pts, 1.0)
    assert np.array_equal(out.view(np.uint32), ref.view(np.uint32)) and out.shape[0] == 3
    # index space overflow: "Leaf size is too small" -> input returned unchanged (voxel_grid_covariance_mloam_impl.hpp:92-101)
    big = np.array([[0, 0, 0, 1], [1e6, 1e6, 1e6, 2], [5, 5, 5, 3]], np.float32)
    assert np.array_equal(ctx.voxel_downsample(big, 0.01), big)
    # large random cloud incl. negative coordinates
    rng = np.random.default_rng(8)
    pts = np.concatenate([rng.uniform(-50, 50, (300000, 3)), rng.uniform(0, 64, (300000, 1))], 1).astype(np.float32)
    out = ctx.voxel_downsample(pts, 0.4, True)
    ref, _ = orc.voxel_grid(pts, 0.4, True)
    assert np.array_equal(out.view(np.uint32), ref.view(np.uint32))


# ------------------------------------------------------------------------------------------------ extractCloud
@pytest.mark.parametrize("rings,horizon", [(16, 1024), (64, 2048)])
def test_extract_features_bit_exact(ctx, rings, horizon):
    scene = syn.make_scene()
    pose = syn.trajectory(3)[2]
    cloud, ss, se = syn.make_sweep(scene, pose, rings, horizon, seed=21)
    out = ctx.extract_features(cloud, ss, se)
    ref = orc.extract_cloud(cloud, ss, se)
    curv, label = ctx.extract_debug(cloud.shape[0])
    assert np.array_equal(curv.view(np.uint32)[5:-5], ref["curvature"].view(np.uint32)[5:-5])
    assert np.array_equal(label, ref["label"])
    for k in ("corner_points_sharp", "corner_points_less_sharp", "surf_points_flat", "surf_points_less_flat"):
        assert out[k].shape == ref[k].shape, k
        assert np.array_equal(out[k].view(np.uint32), ref[k].view(np.uint32)), k
    assert out["corner_points_sharp"].shape[0] <= 2 * 6 * rings


def test_extract_ragged_and_short_rings(ctx):
    scene = syn.make_scene()
    cloud, ss, se = syn.make_sweep(scene, syn.trajectory(1)[0], 16, 1024, seed=5)
    # drop points to make rings ragged, including one ring left with < 6 usable points and one empty ring
    ring = cloud[:, 3].astype(int)
    rng = np.random.default_rng(3)
    keep = rng.random(cloud.shape[0]) > 0.3
    keep &= ~((ring == 3) & (np.cumsum(ring == 3) > 14))  # ring 3: 14 points -> end-start = 3 < 6: skipped
    keep &= ring != 7                                      # ring 7: empty
    c2 = np.ascontiguousarray(cloud[keep])
    s2, e2 = syn.scan_info_from_cloud(c2, 16)
    out = ctx.extract_features(c2, s2, e2)
    ref = orc.extract_cloud(c2, s2, e2)
    for k in ("corner_points_sharp", "corner_points_less_sharp", "surf_points_flat", "surf_points_less_flat"):
        assert np.array_equal(out[k].view(np.uint32), ref[k].view(np.uint32)), k
    assert not np.any(out["surf_points_flat"][:, 3].astype(int) == 3)


# ------------------------------------------------------------------------------------------------ scan2map / frame
@pytest.mark.parametrize("outer,inner", [(2, 30), (5, 1), (10, 1)])
def test_scan2map_pose_parity(ctx, c1, outer, inner):
    ctx.map_build(1, c1["surf_map"], 0.5)
    ctx.map_build(0, c1["corner_map"], 0.5)
    ctx.set_params(max_outer=outer, max_inner=inner)
    try:
        pose, st = ctx.scan2map(c1["surf_scan"], c1["corner_scan"], c1["init"])
    finally:
        ctx.set_params(max_outer=2, max_inner=30)
    o = orc.default_opts()
    o[orc.O_MAX_OUTER], o[orc.O_MAX_INNER] = outer, inner
    ref, rst = orc.scan2map(c1["surf_map"], c1["corner_map"], c1["surf_scan"], c1["corner_scan"], c1["init"], o)
    dt, dr = syn.pose_err(pose, ref)
    assert dt <= POSE_TOL_T and dr <= POSE_TOL_R, (dt, dr)
    assert st["ran"] == 1 and st["n_surf"] == int(rst["n_surf"]) and st["n_corner"] == int(rst["n_corner"])
    assert st["lm_iterations"] == int(rst["lm_iterations"])
    assert st["degenerate"] == int(rst["degenerate"])
    assert np.allclose(st["eig"], rst["eig"], rtol=1e-8)
    assert np.allclose(st["H"], rst["H"], rtol=1e-9, atol=1e-7)
    # and it actually localises: closer to the truth than the initial guess
    assert syn.pose_err(pose, c1["truth"])[0] < syn.pose_err(c1["init"], c1["truth"])[0]


def test_scan2map_gates_and_degeneracy(ctx, c1):
    # map-size gate (lidar_mapper_keyframe.cpp:429): pose returned unchanged, ran = 0
    ctx.map_build(1, c1["surf_map"][:40], 0.5)
    ctx.map_build(0, c1["corner_map"], 0.5)
    pose, st = ctx.scan2map(c1["surf_scan"], c1["corner_scan"], c1["init"])
    assert st["ran"] == 0 and np.array_equal(pose, c1["init"])
    # degenerate geometry: a floor-only surf map and no usable corners -> evalDegenracy remaps the update
    floor = c1["surf_map"][np.abs(c1["surf_map"][:, 2]) < 0.05]
    ctx.map_build(1, floor, 0.5)
    far = c1["corner_map"].copy()
    far[:, :3] += 500.0
    ctx.map_build(0, far, 0.5)
    pose, st = ctx.scan2map(c1["surf_scan"], c1["corner_scan"], c1["init"])
    ref, rst = orc.scan2map(floor, far, c1["surf_scan"], c1["corner_scan"], c1["init"])
    assert st["degenerate"] == 1 and int(rst["degenerate"]) == 1 and st["n_corner"] == 0
    dt, dr = syn.pose_err(pose, ref)
    assert dt <= POSE_TOL_T and dr <= POSE_TOL_R, (dt, dr)
    # empty scans
    ctx.map_build(1, c1["surf_map"], 0.5)
    ctx.map_build(0, c1["corner_map"], 0.5)
    pose, st = ctx.scan2map(np.zeros((0, 4), np.float32), np.zeros((0, 4), np.float32), c1["init"])
    assert st["n_surf"] == 0 and st["n_corner"] == 0 and np.allclose(pose, c1["init"])


@pytest.mark.parametrize("outer,inner", [(2, 30), (5, 1)])
def test_frame_pose_parity_c1(ctx, c1, mloam, outer, inner):
    ctx.set_params(max_outer=outer, max_inner=inner, n_scans=16, map_cell=0.5)
    try:
        pose, st = ctx.frame(c1["cloud"], c1["ss"], c1["se"], c1["surf_map"], c1["corner_map"], c1["init"])
    finally:
        ctx.set_params(max_outer=2, max_inner=30, n_scans=64, map_cell=0.0)
    o = orc.default_opts()
    o[orc.O_MAX_OUTER], o[orc.O_MAX_INNER] = outer, inner
    ref, rst = orc.scan2map(c1["surf_map"], c1["corner_map"], c1["surf_scan"], c1["corner_scan"], c1["init"], o)
    assert st["n_surf_in"] == c1["surf_scan"].shape[0] and st["n_corner_in"] == c1["corner_scan"].shape[0]
    assert st["n_surf"] == int(rst["n_surf"]) and st["n_corner"] == int(rst["n_corner"])
    dt, dr = syn.pose_err(pose, ref)
    assert dt <= POSE_TOL_T and dr <= POSE_TOL_R, (dt, dr)


@pytest.mark.parametrize("map_kind", ["uniform", "keyframes"])
def test_frame_c2_full_size(ctx, map_kind):
    """Config C2 at full size: 64 x 2048 sweep, 1M-point submap, 10 GN iterations; pose parity against the oracle
    plus size-independent properties.  Two submaps: area-uniform samples of the scene, and the keyframe-built one of SURVEY 8d
    (30 ray-cast keyframes -> extractCloud -> VoxelGrid 0.2 / 0.4 -> re-sampled with 1 cm jitter: clusters of near-duplicates at
    voxel spacing, which exercises the shell / ball search paths and the keep shortcut's zero-slack case)."""
    scene = syn.make_scene()
    traj = syn.trajectory(8)
    if map_kind == "uniform":
        surf_map, corner_map = syn.make_submap(scene, 1_000_000)
    else:
        surf_map, corner_map, _ = syn.make_submap_keyframes(scene, 1_000_000, orc.extract_cloud, orc.voxel_grid)
    cloud, ss, se = syn.make_sweep(scene, traj[7], 64, 2048, seed=7)
    init = syn.perturb_pose(traj[7], np.random.Generator(np.random.PCG64(17)))
    ctx.set_params(max_outer=10, max_inner=1, n_scans=64, map_cell=0.26 if map_kind == "uniform" else 0.0)  # 0: auto cell per map
    try:
        pose, st = ctx.frame(cloud, ss, se, surf_map, corner_map, init)
        pose_b, st_b = ctx.frame(cloud, ss, se, surf_map, corner_map, init)
    finally:
        ctx.set_params(max_outer=2, max_inner=30, map_cell=0.0)
    assert np.array_equal(pose, pose_b)  # deterministic: no atomics in the reductions
    f = orc.extract_cloud(cloud, ss, se)
    cs, _ = orc.voxel_grid(f["corner_points_less_sharp"], 0.2, True)
    sf, _ = orc.voxel_grid(f["surf_points_less_flat"], 0.4, True)
    assert st["n_surf_in"] == sf.shape[0] and st["n_corner_in"] == cs.shape[0]
    o = orc.default_opts()
    o[orc.O_MAX_OUTER], o[orc.O_MAX_INNER] = 10, 1
    ref, rst = orc.scan2map(surf_map, corner_map, sf, cs, init, o)
    assert st["n_surf"] == int(rst["n_surf"]) and st["n_corner"] == int(rst["n_corner"])
    dt, dr = syn.pose_err(pose, ref)
    assert dt <= POSE_TOL_T and dr <= POSE_TOL_R, (dt, dr)
    et, er = syn.pose_err(pose, traj[7])
    assert et < 0.05 and er < 3e-3


# ------------------------------------------------------------------------------------------------ several LiDARs on one GPU
@pytest.mark.parametrize("n_lidars,rings,horizon,map_pts,outer", [(2, 16, 1024, 100_000, 5), (4, 64, 2048, 5_000_000, 10)])
def test_frame_multi_lidar_one_gpu(ctx, n_lidars, rings, horizon, map_pts, outer):
    """BASELINE config C4 on ONE GPU (4 x 64-ring LiDARs of the RV rig, 5M-point submap, 10 GN iterations) and a small 2-LiDAR
    case: batched extractCloud over all rings, per-LiDAR extrinsic + laser id, merged downsample, one scan2MapOptimization —
    against the oracle's per-LiDAR restatement (orc_frame_multi)."""
    scene = syn.make_scene()
    traj = syn.trajectory(8)
    surf_map, corner_map = syn.make_submap(scene, map_pts)
    cloud, ss, se, ext = syn.make_multi_sweep(scene, traj[6], n_lidars, rings, horizon, seed=21)
    init = syn.perturb_pose(traj[6], np.random.Generator(np.random.PCG64(23)))
    ctx.set_params(max_outer=outer, max_inner=1, n_scans=rings, map_cell=0.25, max_ring_points=horizon)
    ctx.set_lidars(n_lidars, ext)
    try:
        pose, st = ctx.frame(cloud, ss, se, surf_map, corner_map, init)
        pose_b, _ = ctx.frame(cloud, ss, se, surf_map, corner_map, init)
        pose_c, _ = ctx.frame(cloud, ss, se, surf_map, corner_map, init)  # third call replays the captured graph
    finally:
        ctx.set_lidars(1)
        ctx.set_params(max_outer=2, max_inner=30, n_scans=64, map_cell=0.0, max_ring_points=0)
    assert np.array_equal(pose, pose_b) and np.array_equal(pose, pose_c)
    o = orc.default_opts()
    o[orc.O_MAX_OUTER], o[orc.O_MAX_INNER] = outer, 1
    ref, rst = orc.frame_multi(cloud, ss, se, n_lidars, ext, surf_map, corner_map, init, o)
    assert st["n_surf_in"] == rst["n_surf_in"] and st["n_corner_in"] == rst["n_corner_in"]
    assert st["n_surf"] == int(rst["n_surf"]) and st["n_corner"] == int(rst["n_corner"])
    dt, dr = syn.pose_err(pose, ref)
    assert dt <= POSE_TOL_T and dr <= POSE_TOL_R, (dt, dr)
    et, er = syn.pose_err(pose, traj[6])
    assert et < 0.05 and er < 2e-3


def test_extract_128_rings(ctx):
    """C5 geometry: 128 rings x 2048 (elevations -25 .. +15 deg) — extractCloud is ring-count agnostic (feature_extract.cpp:152)."""
    scene = syn.make_scene()
    cloud, ss, se = syn.make_sweep(scene, syn.trajectory(3)[2], 128, 2048, seed=9)
    ctx.set_params(n_scans=128, max_ring_points=2048)
    try:
        got = ctx.extract_features(cloud, ss, se)
    finally:
        ctx.set_params(n_scans=64, max_ring_points=0)
    ref = orc.extract_cloud(cloud, ss, se)
    for k in ("corner_points_sharp", "corner_points_less_sharp", "surf_points_flat", "surf_points_less_flat"):
        assert np.array_equal(got[k], ref[k]), k


# ------------------------------------------------------------------------------------------------ range-image projection (f1a)
@pytest.mark.parametrize("rings,horizon,sweep_h", [(16, 1800, 2048), (32, 2169, 2048), (64, 2048, 2048), (64, 1024, 4096)])
def test_project_cloud_matches_oracle(ctx, rings, horizon, sweep_h):
    """ImageSegmenter::segmentCloud with segment_cloud: 0 (image_segmenter.hpp:88-136, 381-389): pixel of every point, first point of a
    pixel wins, intensity += ring, rows concatenated in input order, ScanInfo — bit-exact on a raw (unordered, noisy, duplicate-carrying)
    cloud; then the reference's chain segmentCloud -> extractCloud (estimator.cpp:258-259) end to end."""
    scene = syn.make_scene()
    cloud, _, _ = syn.make_sweep(scene, syn.trajectory(3)[1], rings if rings != 32 else 64, sweep_h, seed=21)
    rng = np.random.default_rng(rings + horizon)
    raw = cloud.copy()
    raw[:, 3] -= np.floor(raw[:, 3])  # the driver's cloud: intensity carries no ring id yet
    raw[:, :3] += rng.normal(0, 0.01, raw[:, :3].shape).astype(np.float32)
    raw = np.concatenate([raw, raw[rng.integers(0, raw.shape[0], 5000)], np.zeros((3, 4), np.float32), [[0, 0, 2, 0], [np.nan, 1, 1, 0]]]).astype(np.float32)
    raw = np.ascontiguousarray(raw[rng.permutation(raw.shape[0])])
    for roi in (0.5, 0.0):
        got, gs, ge = ctx.project_cloud(raw, rings, horizon, roi)
        ref, rs, re_ = orc.project_cloud(raw, rings, horizon, roi)
        assert got.shape == ref.shape and ref.shape[0] > raw.shape[0] // 8
        assert np.array_equal(gs, rs) and np.array_equal(ge, re_)
        assert np.array_equal(got.view(np.uint32), ref.view(np.uint32))
    if rings == 16:
        # sensor-ordered input (azimuth sweep per ring): the projected cloud feeds extractCloud
        sweep, _, _ = syn.make_sweep(scene, syn.trajectory(3)[1], 16, 1800, seed=4)
        sweep[:, 3] -= np.floor(sweep[:, 3])
        got, gs, ge = ctx.project_cloud(sweep, 16, 1800, 0.5)
        ref, rs, re_ = orc.project_cloud(sweep, 16, 1800, 0.5)
        assert np.array_equal(got.view(np.uint32), ref.view(np.uint32)) and np.array_equal(gs, rs) and np.array_equal(ge, re_)
        ctx.set_params(n_scans=16)
        try:
            f = ctx.extract_features(got, gs, ge)
        finally:
            ctx.set_params(n_scans=64)
        rf = orc.extract_cloud(ref, rs, re_)
        for k in ("corner_points_sharp", "corner_points_less_sharp", "surf_points_flat", "surf_points_less_flat"):
            assert np.array_equal(f[k], rf[k]), k
        assert rf["surf_points_less_flat"].shape[0] > 500
    # empty cloud and an unsupported ring count
    e, es, ee = ctx.project_cloud(np.zeros((0, 4), np.float32), rings, horizon, 0.5)
    assert e.shape[0] == 0 and np.all(es == 5) and np.all(ee == -6)
    with pytest.raises(Exception):
        ctx.project_cloud(raw, 40, horizon, 0.5)


# ------------------------------------------------------------------------------------------------ online extrinsic calibration (C3)
@pytest.mark.parametrize("rings,horizon,map_pts,outer,inner", [(16, 1024, 100_000, 10, 1), (16, 1024, 100_000, 2, 4), (64, 2048, 2_000_000, 10, 1)])
def test_calib_frame_matches_oracle(ctx, rings, horizon, map_pts, outer, inner):
    """12-DoF step [pose_i | ext_cal]: buildCalibMap's association (n_neigh 5 / 10, CHECK_FOV true) + LidarPureOdom rows of the
    reference LiDAR + LidarOnlineCalib rows of the second LiDAR, both groups in one context (one GPU).  The last case is BASELINE
    config C3's size (64-ring sweeps, 2M-point map, 10 iterations)."""
    scene = syn.make_scene()
    cs = syn.make_calib_case(scene, orc.extract_cloud, orc.voxel_grid, rings, horizon, map_pts)
    ctx.map_build(0, cs["corner_map"], 0.25)
    ctx.map_build(1, cs["surf_map"], 0.25)
    pi, ec, st = ctx.calib_frame(cs["surf_ref"], cs["corner_ref"], cs["surf_cal"], cs["corner_cal"], cs["pivot"], cs["pose_i_init"], cs["ext_ref"],
                                 cs["ext_cal_init"], outer, inner)
    rpi, rec, rst = orc.calib_frame(cs["surf_map"], cs["corner_map"], cs["surf_ref"], cs["corner_ref"], cs["surf_cal"], cs["corner_cal"], cs["pivot"],
                                    cs["pose_i_init"], cs["ext_ref"], cs["ext_cal_init"], outer, inner)
    assert st["n_surf"] == rst["rows"] and st["lm_iterations"] == rst["lm_iterations"]
    for got, ref in ((pi, rpi), (ec, rec)):
        dt, dr = syn.pose_err(got, ref)
        assert dt <= POSE_TOL_T and dr <= POSE_TOL_R, (dt, dr)
    # the step does calibrate: the 2 deg error of the initial extrinsic shrinks
    assert syn.pose_err(ec, cs["ext_cal"])[1] < 0.5 * syn.pose_err(cs["ext_cal_init"], cs["ext_cal"])[1]
    # one group at a time (what each rank of the 2-GPU run evaluates) is the 6-DoF sub-problem of that group
    pi_only, ec_same, _ = ctx.calib_frame(cs["surf_ref"], cs["corner_ref"], None, None, cs["pivot"], cs["pose_i_init"], cs["ext_ref"], cs["ext_cal_init"], outer, inner)
    rpi_only, _, _ = orc.calib_frame(cs["surf_map"], cs["corner_map"], cs["surf_ref"], cs["corner_ref"], None, None, cs["pivot"], cs["pose_i_init"],
                                     cs["ext_ref"], cs["ext_cal_init"], outer, inner)
    assert np.allclose(ec_same, cs["ext_cal_init"], atol=1e-12) and max(syn.pose_err(pi_only, rpi_only)) <= POSE_TOL_T
    if rings == 16 and inner == 1:
        # the calibrated LiDAR's OWN local map (buildCalibMap filters it with leaf 0.2, estimator.cpp:1103-1109) in the scan slots
        surf_c, _ = orc.voxel_grid(cs["surf_map"], 0.2, False)
        corner_c, _ = orc.voxel_grid(cs["corner_map"], 0.2, False)
        ctx.map_build(2, corner_c, 0.25)
        ctx.map_build(3, surf_c, 0.25)
        pi2, ec2, st2 = ctx.calib_frame(cs["surf_ref"], cs["corner_ref"], cs["surf_cal"], cs["corner_cal"], cs["pivot"], cs["pose_i_init"], cs["ext_ref"],
                                        cs["ext_cal_init"], outer, inner, own_cal_maps=True)
        rpi2, rec2, rst2 = orc.calib_frame(cs["surf_map"], cs["corner_map"], cs["surf_ref"], cs["corner_ref"], cs["surf_cal"], cs["corner_cal"], cs["pivot"],
                                           cs["pose_i_init"], cs["ext_ref"], cs["ext_cal_init"], outer, inner, surf_map_cal=surf_c, corner_map_cal=corner_c)
        assert st2["n_surf"] == rst2["rows"] and max(syn.pose_err(ec2, rec2) + syn.pose_err(pi2, rpi2)) <= POSE_TOL_T


# ------------------------------------------------------------------------------------------------ odometry node: local map + good features
def test_local_map_build_and_odometry_good_features(ctx):
    """Estimator::buildLocalMap for one LiDAR: window clouds -> pivot frame -> VoxelGrid(leaf formula) -> map slot, then
    Estimator::goodFeatureMatching of a later frame against it (PureOdom pose_i rows for surf, the identity row for corners)."""
    scene = syn.make_scene()
    traj = syn.trajectory(8)
    ext = syn.rig_extrinsics(2)[1]
    pivot = traj[2]
    window = [2, 3, 4, 5]                                        # frames of the window that enter the local map
    leaf = float(0.4 * min(2.0, max(0.75, 1.0 / 192 * float(16 * 2 * 4))))   # estimator.cpp:1194 with N_SCANS 16, 2 LiDARs, WINDOW_SIZE 4
    surf_stack, corner_stack, pose_local = [], [], []
    for i in window:
        c, ss, se = syn.make_sweep(scene, traj[i], 16, 1024, seed=400 + i, lidar_id=1, ext=ext)
        f = orc.extract_cloud(c, ss, se)
        surf_stack.append(orc.voxel_grid(f["surf_points_less_flat"], 0.4, False)[0])     # window-level down-sampling, estimator.cpp:485-496
        corner_stack.append(orc.voxel_grid(f["corner_points_less_sharp"], 0.2, False)[0])
        pose_local.append(syn.pose_mul(syn.pose_inv(pivot), syn.pose_mul(traj[i], ext)))
    for slot, stack in ((1, surf_stack), (0, corner_stack)):
        got = ctx.local_map_build(slot, stack, pose_local, leaf, 0.5)
        ref = orc.local_map_build(stack, pose_local, leaf)
        assert got.shape == ref.shape and np.array_equal(got, ref) and ctx.map_size(slot) == ref.shape[0]
    surf_map, corner_map = orc.local_map_build(surf_stack, pose_local, leaf), orc.local_map_build(corner_stack, pose_local, leaf)
    # frame 6 against the window's local map
    c, ss, se = syn.make_sweep(scene, traj[6], 16, 1024, seed=406, lidar_id=1, ext=ext)
    f = orc.extract_cloud(c, ss, se)
    pose_i = syn.perturb_pose(traj[6], np.random.Generator(np.random.PCG64(9)))
    for kind, slot, scan, mp in (("s", 1, orc.voxel_grid(f["surf_points_less_flat"], 0.4, False)[0], surf_map),
                                 ("c", 0, orc.voxel_grid(f["corner_points_less_sharp"], 0.2, False)[0], corner_map)):
        for ratio in (1.0, 0.4):
            g = ctx.good_features_odom(slot, kind, scan, pivot, pose_i, ext, ratio, 77)
            r = orc.good_features_odom(kind, mp, scan, pivot, pose_i, ext, ratio, 77)
            assert np.array_equal(g["matched"], r["matched"]) and g["matched"].sum() > 50
            assert np.allclose(g["jaco"], r["jaco"], rtol=1e-9, atol=1e-12)
            assert np.array_equal(g["sel"], r["sel"]) and np.allclose(g["H"], r["H"], rtol=1e-9, atol=1e-12)
            if kind == "c":
                assert np.array_equal(g["jaco"][g["matched"]], np.tile([1.0, 0, 0, 0, 0, 0], (int(g["matched"].sum()), 1)))


# ------------------------------------------------------------------------------------------------ submap assembly with uncertainty (f2)
def _uct_case(n_kf=4, n_lasers=2):
    scene = syn.make_scene()
    traj = syn.trajectory(n_kf + 2)
    ext = syn.rig_extrinsics(n_lasers)
    rng = np.random.default_rng(5)
    A = rng.normal(size=(6, 6)) * 0.01
    cov_pose = A @ A.T + np.eye(6) * 1e-5                      # keyframe pose covariance [translation | rotation]
    cov_ext = [np.zeros((6, 6))] + [np.eye(6) * (1e-4 * (l + 1)) for l in range(1, n_lasers)]
    cov_meas = np.eye(3) * 0.0025
    clouds, poses, pcs, ccs = [], [], [], []
    for k in range(n_kf):
        parts = []
        for l in range(n_lasers):
            c, ss, se = syn.make_sweep(scene, traj[k + 1], 16, 512, seed=300 + k, lidar_id=l, ext=ext[l])
            f = orc.extract_cloud(c, ss, se)
            surf_l = orc.associate(f["surf_points_less_flat"], ext[l])   # keyframe features are stored in the base frame, laser id in the intensity
            surf_l[:, 3] = l
            parts.append(surf_l)
        clouds.append(np.ascontiguousarray(np.concatenate(parts)))
        poses.append(traj[k + 1])
        pk, ck = [], []
        for l in range(n_lasers):
            p, cv = orc.compound_pose_cov(traj[k + 1], cov_pose * (1 + 0.3 * k), ext[l], cov_ext[l])
            pk.append(p), ck.append(cv)
        pcs.append(pk), ccs.append(ck)
    return dict(clouds=clouds, poses=np.array(poses), ext=ext, pose_compound=np.array(pcs), cov_compound=np.array(ccs), cov_meas=cov_meas,
                cov_pose=cov_pose, cov_ext=cov_ext)


def test_compound_pose_cov_and_uct_associate(ctx, mloam):
    u = _uct_case()
    # compoundPoseWithCov: host-side algebra of the library vs the oracle restatement
    for l in range(2):
        p, cv = mloam.Context.compound_pose_cov(u["poses"][1], u["cov_pose"], u["ext"][l], u["cov_ext"][l])
        rp, rcv = orc.compound_pose_cov(u["poses"][1], u["cov_pose"], u["ext"][l], u["cov_ext"][l])
        assert np.allclose(p, rp, rtol=0, atol=1e-15) and np.allclose(cv, rcv, rtol=1e-13, atol=1e-18)
    # cloudUCTAssociateToMap: a threshold that drops part of the cloud; points bit-exact, covariances to float rounding
    k = 2
    args = (u["clouds"][k], u["poses"][k], u["ext"], u["pose_compound"][k], u["cov_compound"][k], u["cov_meas"])
    _, _, tr_all = orc.cloud_uct_associate(*args, with_ua=True, trace_threshold=1e9)
    thr = float(np.percentile(tr_all, 70))
    gp, gc, gt = ctx.cloud_uct_associate(*args, with_ua=True, trace_threshold=thr)
    rp, rc, rt = orc.cloud_uct_associate(*args, with_ua=True, trace_threshold=thr)
    assert 0 < rp.shape[0] < u["clouds"][k].shape[0] and gp.shape == rp.shape
    assert np.array_equal(gp, rp)
    assert np.allclose(gc, rc, rtol=2e-6, atol=1e-12) and np.allclose(gt, rt, rtol=2e-6)
    gp0, gc0, _ = ctx.cloud_uct_associate(*args, with_ua=False)
    rp0, rc0, _ = orc.cloud_uct_associate(*args, with_ua=False)
    assert np.array_equal(gp0, rp0) and not gc0.any() and not rc0.any()


def test_voxel_downsample_cov_bit_exact(ctx):
    # the reference's own 4-point example (mloam_test/src/test_pointiwithcov.cpp:23-40): leaf 3, trace threshold 2
    pts = np.array([[0, 0, 0, 0], [1, 0, 0, 0], [0, 1, 0, 0], [1, 1, 0, 0]], np.float32)
    cov6 = np.zeros((4, 6), np.float32)
    cov6[3, 0] = 1
    trace = cov6[:, 0] + cov6[:, 3] + cov6[:, 5]
    gp, gc, gt = ctx.voxel_downsample_cov(pts, cov6, trace, 3.0, 2.0)
    assert gp.shape[0] == 1 and np.allclose(gp[0, :3], [3 / 7, 3 / 7, 0]) and np.isclose(gc[0, 0], 1 / 49)
    # a real merged cloud: bit-exact against the oracle, including voxels whose points are all above the threshold
    u = _uct_case()
    k = 1
    p, c6, tr = orc.cloud_uct_associate(u["clouds"][k], u["poses"][k], u["ext"], u["pose_compound"][k], u["cov_compound"][k], u["cov_meas"], True, 1e9)
    thr = float(np.percentile(tr, 90))
    for leaf in (0.4, 1.0):
        gp, gc, gt = ctx.voxel_downsample_cov(p, c6, tr, leaf, thr)
        rp, rc, rt, ok = orc.voxel_grid_cov(p, c6, tr, leaf, thr)
        assert ok and gp.shape == rp.shape and rp.shape[0] < p.shape[0]
        assert np.array_equal(gp, rp) and np.array_equal(gc, rc) and np.array_equal(gt, rt)


def test_submap_assemble_on_device(ctx):
    """extractSurroundingKeyFrames' data path for one map: 4 keyframes x 2 LiDARs -> cloudUCTAssociateToMap -> merged ->
    VoxelGridCovarianceMLOAM -> map slot; the installed map answers kNN queries like a map built from the oracle's submap."""
    u = _uct_case()
    thr_a, leaf, thr_f = 50.0, 0.4, 50.0
    gp, gc = ctx.submap_assemble(1, u["clouds"], u["poses"], u["ext"], u["pose_compound"], u["cov_compound"], u["cov_meas"], leaf, True, thr_a, thr_f, 0.5)
    mp, mc, mt = [], [], []
    for k in range(len(u["clouds"])):
        p, c6, tr = orc.cloud_uct_associate(u["clouds"][k], u["poses"][k], u["ext"], u["pose_compound"][k], u["cov_compound"][k], u["cov_meas"], True, thr_a)
        mp.append(p), mc.append(c6), mt.append(tr)
    rp, rc, rt, ok = orc.voxel_grid_cov(np.concatenate(mp), np.concatenate(mc), np.concatenate(mt), leaf, thr_f)
    assert ok and gp.shape == rp.shape and np.array_equal(gp, rp)
    assert np.allclose(gc, rc, rtol=1e-5, atol=1e-12)   # covariances enter the merge with float rounding of the device's double sums
    assert ctx.map_size(1) == rp.shape[0]
    q = rp[::7].copy()
    q[:, :3] += 0.05
    idx, sqd = ctx.knn(1, q, 5, 4.0)
    ridx, rsqd = orc.knn(rp, q, 5)
    inside = rsqd < 4.0
    assert np.array_equal(idx[inside], ridx[inside]) and np.array_equal(sqd[inside], rsqd[inside])


# ------------------------------------------------------------------------------------------------ scan-to-scan (tracker)
@pytest.fixture(scope="module")
def two_sweeps():
    scene = syn.make_scene()
    traj = syn.trajectory(4)
    out = {}
    for rings, horizon, key in ((16, 1024, "s16"), (64, 2048, "s64")):
        a, ssa, sea = syn.make_sweep(scene, traj[1], rings, horizon, seed=31)
        b, ssb, seb = syn.make_sweep(scene, traj[2], rings, horizon, seed=32)
        out[key] = dict(fa=orc.extract_cloud(a, ssa, sea), fb=orc.extract_cloud(b, ssb, seb),
                        rel=syn.pose_mul(syn.pose_inv(traj[1]), traj[2]))
    return out


@pytest.mark.parametrize("key", ["s16", "s64"])
@pytest.mark.parametrize("kind", ["c", "s"])
def test_match_from_scan_exact(ctx, two_sweeps, key, kind):
    d = two_sweeps[key]
    scan = d["fa"]["corner_points_less_sharp" if kind == "c" else "surf_points_less_flat"]
    data = d["fb"]["corner_points_sharp" if kind == "c" else "surf_points_flat"]
    guess = syn.pose7([0.05, 0.01, 0.0], syn.quat_from_rpy(0.0, 0.0, 0.005))
    slot = 2 if kind == "c" else 3
    ctx.map_build(slot, scan, 1.3)
    valid, coeffs, nn3 = ctx.match_from_scan(slot, kind, data, guess)
    fidx, rcoeffs = orc.match_from_scan(kind, scan, data, guess)
    assert fidx.shape[0] > 20
    assert np.array_equal(np.nonzero(valid)[0], fidx)      # same features survive, in query order
    assert np.array_equal(coeffs[valid], rcoeffs)          # bit-exact [X_j; X_l] / (w, d)


@pytest.mark.parametrize("key", ["s16", "s64"])
def test_track_cloud_pose_parity(ctx, two_sweeps, key):
    d = two_sweeps[key]
    ident = syn.pose7([0, 0, 0], [0, 0, 0, 1])
    args = (d["fa"]["corner_points_less_sharp"], d["fa"]["surf_points_less_flat"], d["fb"]["corner_points_sharp"],
            d["fb"]["surf_points_flat"], ident)
    pose, st = ctx.track_cloud(*args)
    ref, rst = orc.track_cloud(*args)
    dt, dr = syn.pose_err(pose, ref)
    assert dt <= POSE_TOL_T and dr <= POSE_TOL_R, (dt, dr)
    assert st["n_corner"] == rst["n_corner"] and st["n_surf"] == rst["n_surf"]
    assert st["lm_iterations"] == rst["lm_iterations"]
    et, er = syn.pose_err(pose, d["rel"])
    assert et < 0.05 and er < 5e-3  # recovers the inter-sweep motion


def test_track_cloud_too_few_correspondences(ctx, two_sweeps):
    """< 10 correspondences: both outer iterations are skipped and the initial pose comes back (lidar_tracker.cpp:64-68)."""
    d = two_sweeps["s16"]
    ident = syn.pose7([0.1, 0.2, 0.3], syn.quat_from_rpy(0.01, 0.02, 0.03))
    far = d["fa"]["corner_points_less_sharp"].copy()
    far[:, :3] += 1000.0
    far2 = d["fa"]["surf_points_less_flat"].copy()
    far2[:, :3] += 1000.0
    pose, st = ctx.track_cloud(far, far2, d["fb"]["corner_points_sharp"], d["fb"]["surf_points_flat"], ident)
    ref, rst = orc.track_cloud(far, far2, d["fb"]["corner_points_sharp"], d["fb"]["surf_points_flat"], ident)
    assert st["n_corner"] + st["n_surf"] < 10 and st["lm_iterations"] == 0 == rst["lm_iterations"]
    assert np.allclose(pose, ref, atol=1e-15) and np.allclose(pose, ident, atol=1e-15)


def test_cpp_host_shim_selftest(mloam):
    """The reference-shaped C++ surface (FeatureExtract, MapHandle, PoseLocalParameterization, Lidar*Factor::Evaluate with
    the check() finite-difference convention, scan2MapOptimization) end to end through the C ABI."""
    import os
    import subprocess

    exe = os.path.join(mloam.HERE, "host", "shim_selftest")
    assert os.path.exists(exe), "build() must have produced the host shim self-test"
    out = subprocess.run([exe], capture_output=True, text=True, timeout=300)
    assert out.returncode == 0 and "SHIM_SELFTEST OK" in out.stdout, out.stdout[-3000:] + out.stderr[-1000:]


# ------------------------------------------------------------------------------------------------ odometry rows (1x6 / 1x12)
@pytest.mark.parametrize("free_mask,max_it", [(1, 4), (2, 4), (3, 4), (3, 30)])
def test_odom_solve_matches_oracle(ctx, free_mask, max_it):
    from test_oracle_cpu import _odom_problem

    rng = np.random.default_rng(90 + free_mask)
    xp, xi, xe, types, pts, coeffs = _odom_problem(rng, n=3000)
    d = lambda: syn.pose7(rng.normal(size=3) * 0.02, syn.quat_from_rpy(*(rng.normal(size=3) * 0.004)))
    xi0 = syn.pose_mul(xi, d()) if free_mask & 1 else xi
    xe0 = syn.pose_mul(xe, d()) if free_mask & 2 else xe
    gi, ge, st = ctx.odom_solve(types, pts, coeffs, xp, xi0, xe0, free_mask, max_iterations=max_it)
    oi, oe, rst = orc.odom_solve(types, pts, coeffs, xp, xi0, xe0, free_mask, max_it=max_it)
    assert st["lm_iterations"] == rst["lm_iterations"] and st["termination"] == rst["termination"]
    for a, b in ((gi, oi), (ge, oe)):
        dt, dr = syn.pose_err(a, b)
        assert dt <= POSE_TOL_T and dr <= POSE_TOL_R, (dt, dr)
    assert abs(st["final_cost"] - rst["final_cost"]) <= 1e-9 * max(1.0, rst["final_cost"])
    if not free_mask & 1:
        assert np.array_equal(gi, xi0)
    if not free_mask & 2:
        assert np.array_equal(ge, xe0)


def test_frame_graph_replay_equals_stream_path(mloam, c1):
    """max_inner == 1 frames are replayed from a captured CUDA graph from their third sighting on; the pose staged in pinned
    memory must be re-read on every replay, and results must be bit-identical to the plain stream path."""
    import os

    p = mloam.default_params()
    p.n_scans, p.max_outer, p.max_inner, p.map_cell = 16, 4, 1, 0.5
    rng = np.random.Generator(np.random.PCG64(21))
    inits = [syn.perturb_pose(c1["truth"], rng) for _ in range(5)]
    os.environ["MLOAM_DISABLE_GRAPHS"] = "1"
    try:
        plain = mloam.Context(0, p)
    finally:
        os.environ.pop("MLOAM_DISABLE_GRAPHS")
    ref = [plain.frame(c1["cloud"], c1["ss"], c1["se"], c1["surf_map"], c1["corner_map"], x)[0] for x in inits]
    n_plain = plain.launch_count()
    plain.close()
    g = mloam.Context(0, p)
    out = [g.frame(c1["cloud"], c1["ss"], c1["se"], c1["surf_map"], c1["corner_map"], x) for x in inits]
    for (pose, st), r in zip(out, ref):
        assert np.array_equal(pose, r)
        assert st["ran"] == 1 and st["n_surf"] > 1000
    assert len({tuple(p_) for p_, _ in out}) == len(inits)  # different guesses -> different (re-read) inputs
    assert g.launch_count() == n_plain                       # replayed launches are accounted for
    g.close()


@pytest.mark.parametrize("n_lidars", [1, 2])
@pytest.mark.parametrize("gf", [0, orc.GF_GD])
def test_frame_lookahead_is_exact(mloam, n_lidars, gf):
    """Sweep look-ahead (mloam_frame_set_next / _device): the next sweep is extracted on a side stream while the current frame is
    solved.  A sequence of frames must give bit-identical poses and statistics with and without announcements — through the host
    API and the device API, on the stream path and from replayed graphs, when an announcement is NOT followed by that sweep, and
    with the map rebuilt on some frames only (the keyframe cadence)."""
    import torch

    scene = syn.make_scene()
    traj = syn.trajectory(8)
    surf_map, corner_map = syn.make_submap(scene, 200_000)
    p = mloam.default_params()
    p.n_scans, p.max_outer, p.max_inner, p.map_cell, p.max_ring_points = 16, 4, 1, 0.0, 1024
    p.gf_method, p.gf_ratio = gf, 0.5
    rng = np.random.Generator(np.random.PCG64(5))
    sweeps = []
    for k in range(4):
        if n_lidars == 1:
            cloud, ss, se = syn.make_sweep(scene, traj[2 + k], 16, 1024, seed=30 + k)
            ext = None
        else:
            cloud, ss, se, ext = syn.make_multi_sweep(scene, traj[2 + k], n_lidars, 16, 1024, seed=30 + k)
        sweeps.append(dict(cloud=np.ascontiguousarray(cloud, np.float32), ss=np.ascontiguousarray(ss, np.int32), se=np.ascontiguousarray(se, np.int32),
                           init=syn.perturb_pose(traj[2 + k], rng)))
    order = [0, 1, 2, 3, 0, 1, 2, 3, 0, 1, 2, 3, 1, 3]  # the last two break the announced order
    rebuild = [k % 3 == 0 for k in range(len(order))]

    def new_ctx():
        c = mloam.Context(0, p)
        if n_lidars > 1:
            c.set_lidars(n_lidars, ext)
        return c

    def run_host(c, announce):
        out = []
        for i, k in enumerate(order):
            s = sweeps[k]
            if announce:
                nk = (k + 1) % 4  # what a sequential reader would announce; wrong for the last two frames of `order`
                c.frame_set_next(sweeps[nk]["cloud"], sweeps[nk]["ss"], sweeps[nk]["se"])
            pose, st = c.frame(s["cloud"], s["ss"], s["se"], surf_map, corner_map, s["init"], rebuild[i])
            out.append((pose, st["n_surf"], st["n_corner"], st["n_surf_in"], st["n_corner_in"], st["final_cost"]))
        return out

    plain = new_ctx()
    ref = run_host(plain, False)
    l_plain = plain.launch_count()
    plain.close()
    ahead = new_ctx()
    got = run_host(ahead, True)
    ahead.close()
    for a, b in zip(got, ref):
        assert np.array_equal(a[0], b[0]) and a[1:] == b[1:]
    assert ref[0][1] > 500 and l_plain > 0
    # device API: sweeps and maps resident, announcements by device pointer
    dev = torch.device("cuda", 0)
    d_s = [dict(cloud=torch.from_numpy(s["cloud"]).to(dev), ss=torch.from_numpy(s["ss"]).to(dev), se=torch.from_numpy(s["se"]).to(dev)) for s in sweeps]
    d_sm, d_cm = torch.from_numpy(surf_map).to(dev), torch.from_numpy(corner_map).to(dev)
    c = new_ctx()
    got_d = []
    for i, k in enumerate(order):
        nk = (k + 1) % 4
        c.frame_set_next_device(d_s[nk]["cloud"].data_ptr(), sweeps[nk]["cloud"].shape[0], d_s[nk]["ss"].data_ptr(), d_s[nk]["se"].data_ptr(), sweeps[nk]["ss"].shape[0])
        pose, st = c.frame_device(d_s[k]["cloud"].data_ptr(), sweeps[k]["cloud"].shape[0], d_s[k]["ss"].data_ptr(), d_s[k]["se"].data_ptr(), sweeps[k]["ss"].shape[0],
                                  d_sm.data_ptr(), surf_map.shape[0], d_cm.data_ptr(), corner_map.shape[0], sweeps[k]["init"], rebuild[i])
        got_d.append((pose, st["n_surf"], st["n_corner"], st["n_surf_in"], st["n_corner_in"], st["final_cost"]))
    c.close()
    for a, b in zip(got_d, ref):
        assert np.array_equal(a[0], b[0]) and a[1:] == b[1:]


@pytest.mark.parametrize("outer,inner,guess", [(6, 1, 0.0), (3, 4, 0.0), (4, 1, 0.6)])
@pytest.mark.parametrize("switch,off,on", [("MLOAM_DISABLE_SEEDS", "1", "0"), ("MLOAM_FUSE_ITER", "0", "1")], ids=["seeds", "fuse_iter"])
def test_seeded_reassociation_is_exact(mloam, c1, switch, off, on, outer, inner, guess):
    """From the second re-association on, the kNN is seeded with the previous neighbour lists and unchanged lists keep
    their fit.  That is an exact shortcut: poses, match counts and the Hessian must be BIT-identical to the blind
    search — also when the pose moves a lot between iterations (a poor initial guess).  The same holds for the fused
    evaluation (fit inside the first evaluation, both evaluations of an LM iteration in one launch) against one launch
    per step."""
    import os

    p = mloam.default_params()
    p.max_outer, p.max_inner, p.map_cell = outer, inner, 0.5
    init = np.array(c1["init"], dtype=np.float64)
    init[:3] += guess
    res = []
    for value in (off, on):
        os.environ[switch] = value
        try:
            cx = mloam.Context(0, p)
        finally:
            os.environ.pop(switch)
        cx.map_build(1, c1["surf_map"], 0.5)
        cx.map_build(0, c1["corner_map"], 0.5)
        res.append(cx.scan2map(c1["surf_scan"], c1["corner_scan"], init))
        cx.close()
    (pa, sa), (pb, sb) = res
    assert np.array_equal(pa, pb)
    assert sa["n_surf"] == sb["n_surf"] and sa["n_corner"] == sb["n_corner"] and sa["n_surf"] > 500
    assert sa["lm_iterations"] == sb["lm_iterations"]
    assert np.array_equal(np.asarray(sa["H"]), np.asarray(sb["H"])) and sa["final_cost"] == sb["final_cost"]


# ------------------------------------------------------------------------------------------------ uncertainty-aware mapping
def test_point_uncertainty_and_scan2map_ua(ctx, c1):
    rng = np.random.default_rng(12)
    ext = syn.pose7([0.3, -0.2, 0.1], syn.quat_from_rpy(0.02, -0.01, 0.5))
    A = rng.normal(size=(6, 6)) * 0.01
    cov_pose = A @ A.T + np.diag([1e-4] * 3 + [1e-5] * 3)
    cov_meas = np.diag([0.0025, 0.0025, 0.0025])
    pts = c1["surf_scan"]
    cov6 = ctx.point_uncertainty(pts, ext, cov_pose, cov_meas)
    ref6 = orc.point_uncertainty(pts, ext, cov_pose, cov_meas)
    assert np.allclose(cov6, ref6, rtol=2e-6, atol=1e-9)
    assert np.all(cov6[:, [0, 3, 5]] > 0)
    # known answer: zero pose covariance -> cov = R COV_MEASUREMENT R^T = 0.0025 I for an isotropic measurement covariance
    iso = ctx.point_uncertainty(pts[:16], ext, np.zeros((6, 6)), cov_meas)
    assert np.allclose(iso[:, [0, 3, 5]], 0.0025, rtol=1e-6) and np.allclose(iso[:, [1, 2, 4]], 0.0, atol=1e-9)
    # weighted solve: distance-dependent covariances (far points weigh less), both factor types
    sc = ctx.point_uncertainty(c1["surf_scan"], ext, cov_pose * 40, cov_meas)
    cc = ctx.point_uncertainty(c1["corner_scan"], ext, cov_pose * 40, cov_meas)
    tr = sc[:, 0] + sc[:, 3] + sc[:, 5]
    assert (np.sqrt(1 / tr) < 3).mean() > 0.2  # a good share of the weights is below the clamp
    ctx.map_build(1, c1["surf_map"], 0.5)
    ctx.map_build(0, c1["corner_map"], 0.5)
    pose, st = ctx.scan2map_ua(c1["surf_scan"], sc, c1["corner_scan"], cc, c1["init"])
    ref, rst = orc.scan2map_ua(c1["surf_map"], c1["corner_map"], c1["surf_scan"], sc, c1["corner_scan"], cc, c1["init"])
    dt, dr = syn.pose_err(pose, ref)
    assert dt <= POSE_TOL_T and dr <= POSE_TOL_R, (dt, dr)
    assert st["n_surf"] == rst["n_surf"] and st["lm_iterations"] == rst["lm_iterations"]
    plain, _ = ctx.scan2map(c1["surf_scan"], c1["corner_scan"], c1["init"])
    assert not np.allclose(pose, plain, atol=1e-9)  # the weights matter


# ------------------------------------------------------------------------------------------------ good-feature selection (a23)
@pytest.mark.parametrize("kind", ["s", "c"])
@pytest.mark.parametrize("method,ratio", [(orc.GF_WO, 1.0), (orc.GF_RND, 0.2), (orc.GF_FPS, 0.2), (orc.GF_GD, 0.2), (orc.GF_GD, 0.05),
                                          (orc.GF_GD, 0.8)])
def test_good_feature_selection_matches_oracle(ctx, c1, kind, method, ratio):
    """goodFeatureMatching with the explicit seed: same matched set, Jacobian rows to 1e-9, and the SAME features in the SAME
    selection order as the oracle restatement of the reference's loops (rnd / fps / stochastic greedy)."""
    slot = 1 if kind == "s" else 0
    ctx.map_build(1, c1["surf_map"], 0.5)
    ctx.map_build(0, c1["corner_map"], 0.5)
    scan = c1["surf_scan"] if kind == "s" else c1["corner_scan"]
    mp = c1["surf_map"] if kind == "s" else c1["corner_map"]
    for seed in (3, 12345):
        out = ctx.good_features(slot, kind, scan, c1["init"], method, ratio, seed)
        ref = orc.good_features(kind, mp, scan, c1["init"], method, ratio, seed)
        assert np.array_equal(out["matched"], ref["matched"])
        assert np.allclose(out["jaco"], ref["jaco"], rtol=1e-9, atol=1e-11)
        assert np.array_equal(out["sel"], ref["sel"]), (method, ratio, seed, out["sel"][:10], ref["sel"][:10])
        assert np.allclose(out["H"], ref["H"], rtol=1e-9, atol=1e-12)
        assert len(set(out["sel"].tolist())) == len(out["sel"]) and out["matched"][out["sel"]].all()
        if method != orc.GF_WO:
            assert len(out["sel"]) <= int(scan.shape[0] * ratio)


def test_good_feature_greedy_beats_random_and_handles_edges(ctx, c1):
    ctx.map_build(1, c1["surf_map"], 0.5)
    scan = c1["surf_scan"]
    ld = {}
    for name, m in (("rnd", orc.GF_RND), ("gd", orc.GF_GD)):
        vals = []
        for seed in range(4):
            out = ctx.good_features(1, "s", scan, c1["init"], m, 0.1, seed)
            vals.append(np.linalg.slogdet(out["H"])[1])
        ld[name] = np.mean(vals)
    assert ld["gd"] > ld["rnd"]  # the point of the method: more information from the same number of features
    # ratio 0 -> nothing selected, H = 1e-6 I; empty scan
    out = ctx.good_features(1, "s", scan, c1["init"], orc.GF_GD, 0.0, 1)
    assert len(out["sel"]) == 0 and np.allclose(out["H"], 1e-6 * np.eye(6))
    out = ctx.good_features(1, "s", np.zeros((0, 4), np.float32), c1["init"], orc.GF_FPS, 0.5, 1)
    assert len(out["sel"]) == 0
    # a scan with no map support at all: nothing matches, every method terminates with an empty selection
    far = scan.copy()
    far[:, :3] += 1000.0
    for m in (orc.GF_RND, orc.GF_FPS, orc.GF_GD):
        assert len(ctx.good_features(1, "s", far, c1["init"], m, 0.3, 5)["sel"]) == 0


@pytest.mark.parametrize("method", [orc.GF_RND, orc.GF_FPS, orc.GF_GD])
def test_scan2map_with_good_feature_selection(ctx, c1, method):
    """scan2MapOptimization with FLAGS_gf_method != wo_gf (lidar_mapper_keyframe.cpp:474-560): every outer iteration selects
    gf_ratio of the features per set on the device and solves on those.  Same selected counts and pose as the oracle."""
    ctx.map_build(1, c1["surf_map"], 0.5)
    ctx.map_build(0, c1["corner_map"], 0.5)
    ctx.set_params(max_outer=3, max_inner=4, gf_method=method, gf_ratio=0.3, gf_seed=5)
    try:
        pose, st = ctx.scan2map(c1["surf_scan"], c1["corner_scan"], c1["init"])
    finally:
        ctx.set_params(max_outer=2, max_inner=30, gf_method=0, gf_ratio=1.0, gf_seed=0)
    o = orc.default_opts()
    o[orc.O_MAX_OUTER], o[orc.O_MAX_INNER] = 3, 4
    o[orc.O_GF_METHOD], o[orc.O_GF_RATIO], o[orc.O_GF_SEED] = method, 0.3, 5
    ref, rst = orc.scan2map(c1["surf_map"], c1["corner_map"], c1["surf_scan"], c1["corner_scan"], c1["init"], o)
    assert st["n_surf"] == int(rst["n_surf"]) and st["n_corner"] == int(rst["n_corner"])
    assert 0 < st["n_surf"] <= int(0.3 * c1["surf_scan"].shape[0])
    dt, dr = syn.pose_err(pose, ref)
    assert dt <= POSE_TOL_T and dr <= POSE_TOL_R, (dt, dr)
    assert syn.pose_err(pose, c1["truth"])[0] < syn.pose_err(c1["init"], c1["truth"])[0]


# ------------------------------------------------------------------------------------------------ committed golden fixtures
def _golden(name):
    import os

    return np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", name))


def test_golden_reference_nanoflann_knn(ctx):
    """GPU kNN against the answers of the reference's own kd-tree (tests/golden/knn_nanoflann.npz, generated from
    /root/reference's nanoflann.hpp by tests/golden/make_golden.py): indices and float distances, exactly."""
    g = _golden("knn_nanoflann.npz")
    ctx.map_build(2, g["map"], 0.5)
    for k in (1, 5, 10):
        idx, sqd = ctx.knn(2, g["query"], k, 1.0)
        inside = g[f"sqd{k}"] < 1.0
        assert inside.sum() > 100
        assert np.array_equal(idx[inside], g[f"idx{k}"][inside]) and np.array_equal(sqd[inside], g[f"sqd{k}"][inside])
        assert np.all(idx[~inside] == -1)


def test_golden_oracle_vectors_on_gpu(ctx):
    """The whole path against the committed oracle vectors (no oracle call): feature sets and voxel filters bit-exact,
    match decisions and neighbour sets exact, good-feature selection exact, pose within the north-star tolerance."""
    g = _golden("oracle_small.npz")
    out = ctx.extract_features(g["cloud"], g["ss"], g["se"])
    for key, name in (("corner_points_sharp", "sharp"), ("corner_points_less_sharp", "less_sharp"), ("surf_points_flat", "flat"),
                      ("surf_points_less_flat", "less_flat")):
        assert np.array_equal(out[key].view(np.uint32), g[name].view(np.uint32)), key
    assert np.array_equal(ctx.voxel_downsample(g["less_sharp"], 0.2, True).view(np.uint32), g["corner_ds"].view(np.uint32))
    assert np.array_equal(ctx.voxel_downsample(g["less_flat"], 0.4, True).view(np.uint32), g["surf_ds"].view(np.uint32))
    ctx.map_build(1, g["surf_map"], 0.5)
    ctx.map_build(0, g["corner_map"], 0.5)
    valid, coeffs, nn = ctx.match_from_map(1, "s", g["surf_ds"], g["init"])
    assert np.array_equal(valid, g["surf_valid"]) and np.array_equal(nn[valid], g["surf_nn"][g["surf_valid"]])
    assert np.array_equal(coeffs[valid], g["surf_coeff"][g["surf_valid"]])
    valid, _, nn = ctx.match_from_map(0, "c", g["corner_ds"], g["init"])
    assert np.array_equal(valid, g["corner_valid"]) and np.array_equal(nn[valid], g["corner_nn"][g["corner_valid"]])
    gf = ctx.good_features(1, "s", g["surf_ds"], g["init"], orc.GF_GD, 0.25, 11)
    assert np.array_equal(gf["sel"], g["gf_sel"]) and np.allclose(gf["H"], g["gf_H"], rtol=1e-9)
    ctx.set_params(max_outer=3, max_inner=4)
    try:
        pose, st = ctx.scan2map(g["surf_ds"], g["corner_ds"], g["init"])
    finally:
        ctx.set_params(max_outer=2, max_inner=30)
    dt, dr = syn.pose_err(pose, g["pose"])
    assert dt <= POSE_TOL_T and dr <= POSE_TOL_R and st["n_surf"] == int(g["n_surf"]) and st["n_corner"] == int(g["n_corner"])


def test_bench_dump_outputs_repeat(tmp_path):
    """bench.py --dump-outputs: two runs with the same arguments write the same float64 arrays of the last timed step (seeded
    inputs, deterministic path), far below 64 MB, and the result line reports the requested number of timed steps."""
    import json
    import os
    import subprocess
    import sys

    bench = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "bench.py")
    runs = []
    for name in ("a", "b"):
        d = tmp_path / name
        out = subprocess.run([sys.executable, bench, "--steps", "3", "--warmup", "0", "--no-cpu-baseline", "--no-c4", "--dump-outputs", str(d)],
                             capture_output=True, text=True, timeout=900)
        assert out.returncode == 0, out.stdout[-2000:] + out.stderr[-2000:]
        assert json.loads(out.stdout.strip().splitlines()[-1])["steps"] == 3
        runs.append({f: np.load(d / f) for f in sorted(os.listdir(d))})
    a, b = runs
    assert sorted(a) == sorted(b) and "pose.npy" in a and "H.npy" in a
    for f in a:
        assert a[f].dtype == np.float64 and np.array_equal(a[f], b[f]), f
    assert sum(x.nbytes for x in a.values()) <= 64 << 20
    assert a["ran.npy"] == 1 and a["n_surf.npy"] > 1000
