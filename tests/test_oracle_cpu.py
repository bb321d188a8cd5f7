"""CPU tests: the oracle against analytic known answers, brute force and the reference's own kd-tree
(its answers stored under tests/golden/ by make_golden.py).  The reference ships no golden
vectors for this path (SURVEY.md §4), so known answers are derived analytically with the conventions of the
reference's check() printers (eps 1e-6, right-multiplied deltaQ; lidar_map_factor.hpp:72-120)."""
import math
import os

import numpy as np
import pytest

import oracle_lib as orc
import synthetic as syn


def rand_pose(rng):
    q = rng.normal(size=4)
    return syn.pose7(rng.normal(size=3) * 3, q)


def knn_uniform_case():
    """Seeded 20k-point map and 500 queries; tests/golden/knn_nanoflann_uniform.npz holds the reference kd-tree's answers on them."""
    rng = np.random.default_rng(1)
    m = np.concatenate([rng.uniform(-20, 20, (20000, 3)), np.zeros((20000, 1))], 1).astype(np.float32)
    q = np.concatenate([rng.uniform(-20, 20, (500, 3)), np.zeros((500, 1))], 1).astype(np.float32)
    return m, q


def test_knn_tree_vs_brute_and_reference_nanoflann():
    m, q = knn_uniform_case()
    g = np.load(os.path.join(GOLDEN, "knn_nanoflann_uniform.npz"))
    assert np.array_equal(q, g["query"]), "the seeded inputs no longer match the stored reference answers"
    for k in (1, 5, 10):
        i_t, d_t = orc.knn(m, q, k)
        i_b, d_b = orc.knn(m, q, k, brute=True)
        assert np.array_equal(i_t, i_b) and np.array_equal(d_t, d_b)
        # the reference's vendored nanoflann on the same map and queries (stored by tests/golden/make_golden.py)
        assert np.array_equal(d_t, g[f"sqd{k}"])
        assert np.array_equal(i_t, g[f"idx{k}"])


def test_knn_small_map_missing_slots():
    m = np.array([[0, 0, 0, 0], [1, 0, 0, 0], [0, 2, 0, 0]], np.float32)
    q = np.array([[0.1, 0, 0, 0]], np.float32)
    idx, sqd = orc.knn(m, q, 5)
    assert list(idx[0]) == [0, 1, 2, -1, -1]
    assert np.isinf(sqd[0, 3])


def test_eig3f_known():
    # diag + rotation: eigenvalues known
    rng = np.random.default_rng(2)
    for _ in range(50):
        R = syn.quat_to_mat(rand_pose(rng)[3:])
        lam = np.sort(rng.uniform(0.01, 5, 3))
        A = (R @ np.diag(lam) @ R.T).astype(np.float32)
        w, V = orc.eig3f(A)
        assert np.allclose(w, lam, rtol=2e-5, atol=1e-6)
        assert np.allclose(np.abs(V.T @ R), np.eye(3), atol=2e-3)
        assert np.allclose(V.T @ V, np.eye(3), atol=1e-5)


def test_lsq_plane_known():
    rng = np.random.default_rng(3)
    for _ in range(50):
        n = rng.normal(size=3)
        n /= np.linalg.norm(n)
        d = rng.uniform(1, 20)
        # points on plane n.x + d = 0
        B = np.linalg.svd(n[None, :])[2][1:]
        P = (-d * n)[None, :] + rng.uniform(-1, 1, (5, 2)) @ B
        ok, sol = orc.lsq_plane(P.astype(np.float32))
        assert ok
        # A sol = -1  ->  sol = n/d
        assert np.allclose(sol, n / d, rtol=2e-3, atol=1e-5)
        ref = np.linalg.lstsq(P.astype(np.float32).astype(np.float64), -np.ones(5), rcond=None)[0]
        assert np.allclose(sol, ref, rtol=5e-3, atol=1e-5)
    ok, _ = orc.lsq_plane(np.zeros((5, 3), np.float32))
    assert not ok


def test_voxel_grid_hand_placed():
    # 4 points, leaf 1: two share a voxel (mean), two alone; output ascending voxel index
    pts = np.array([[0.1, 0.1, 0.1, 1], [0.3, 0.5, 0.7, 3], [1.5, 0.2, 0.2, 5], [0.2, 1.6, 0.1, 7]], np.float32)
    out, ok = orc.voxel_grid(pts, 1.0)
    assert ok and out.shape[0] == 3
    assert np.allclose(out[0], [0.2, 0.3, 0.4, 2.0], atol=1e-6)
    assert np.allclose(out[1], pts[2]) and np.allclose(out[2], pts[3])
    out2, _ = orc.voxel_grid(pts, 1.0, intensity_last=True)
    assert out2[0, 3] == 3.0  # VoxelGridCovarianceMLOAM keeps the last point's intensity
    # the 4-point example of mloam_test/src/test_pointiwithcov.cpp:23-40 (leaf 3): all four in one voxel
    pts = np.array([[0, 0, 0, 0], [1, 0, 0, 0], [0, 1, 0, 0], [1, 1, 0, 0]], np.float32)
    out, _ = orc.voxel_grid(pts, 3.0)
    assert out.shape[0] == 1 and np.allclose(out[0, :3], [0.5, 0.5, 0])
    # empty and overflow edge cases
    out, ok = orc.voxel_grid(np.zeros((0, 4), np.float32), 0.2)
    assert ok and out.shape[0] == 0
    big = np.array([[0, 0, 0, 0], [1e6, 1e6, 1e6, 0]], np.float32)
    out, ok = orc.voxel_grid(big, 0.01)
    assert (not ok) and out.shape[0] == 2  # "Leaf size is too small": input copied


@pytest.mark.parametrize("kind", [orc.F_PLANE, orc.F_EDGE, orc.F_EDGE_VEC])
def test_single_pose_factor_jacobians_fd(kind):
    """Analytic Jacobian vs forward differences, exactly the reference's check() convention."""
    rng = np.random.default_rng(10 + kind)
    eps = 1e-6
    for _ in range(20):
        x = rand_pose(rng)
        p = rng.normal(size=3) * 5
        if kind == orc.F_PLANE:
            n = rng.normal(size=3)
            n /= np.linalg.norm(n)
            coeff = np.array([*n, rng.normal()])
        else:
            a = rng.normal(size=3) * 5
            coeff = np.array([*a, *(a + rng.normal(size=3))])
        s = 0.7 if kind != orc.F_EDGE_VEC else 1.0
        r, J = orc.factor_eval(kind, p, coeff, s, x)
        rows = 3 if kind == orc.F_EDGE_VEC else 1
        J = J[: rows * 7].reshape(rows, 7)
        assert np.all(J[:, 6] == 0)
        for k in range(6):
            d = np.zeros(6)
            d[k] = eps
            xp = orc.plus(x, d)  # t += d ; q = q * deltaQ(d)
            rp, _ = orc.factor_eval(kind, p, coeff, s, xp, want_jac=False)
            num = (rp[:rows] - r[:rows]) / eps
            assert np.allclose(num, J[:, k], rtol=1e-4, atol=2e-4), (kind, k, num, J[:, k])


def test_plane_residual_zero_on_plane_and_edge_distance():
    x = syn.pose7([1, 2, 3], syn.quat_from_rpy(0.1, -0.2, 0.3))
    R = syn.quat_to_mat(x[3:])
    p = np.array([0.5, -1.0, 2.0])
    pw = R @ p + x[:3]
    n = np.array([0.0, 0.6, 0.8])
    r, _ = orc.factor_eval(orc.F_PLANE, p, [*n, -n @ pw], 1.0, x)
    assert abs(r[0]) < 1e-12
    # line through pw + (0,0,1)*t shifted by 0.3 in x: distance 0.3
    a = pw + np.array([0.3, 0, 1.0])
    b = pw + np.array([0.3, 0, -1.0])
    r, _ = orc.factor_eval(orc.F_EDGE, p, [*a, *b], 1.0, x)
    assert abs(r[0] - 0.3) < 1e-12
    rv, _ = orc.factor_eval(orc.F_EDGE_VEC, p, [*a, *b], 1.0, x)
    assert abs(np.linalg.norm(rv) - 0.3) < 1e-12


@pytest.mark.parametrize("kind", [orc.F_ODOM_PLANE, orc.F_ODOM_EDGE])
def test_odom_factor_chain_and_jacobians(kind):
    """Three-pose chain: residual equals the single-pose factor at the composed pose; the pose_i block and the
    translation part of the ext block match forward differences.  The ext ROTATION block is the reference's own
    closed form ([R_e p]x instead of R_e [p]x, lidar_pure_odom_factor.hpp:94-95,273-275) and the pivot block
    (:67-70,247-249) are kept verbatim, inconsistencies included (SURVEY.md §7 "quirks"), so they are not
    compared with finite differences."""
    rng = np.random.default_rng(30 + kind)
    eps = 1e-6
    for _ in range(10):
        xp, xi, xe = rand_pose(rng), rand_pose(rng), rand_pose(rng)
        p = rng.normal(size=3) * 4
        if kind == orc.F_ODOM_PLANE:
            n = rng.normal(size=3)
            n /= np.linalg.norm(n)
            coeff = np.array([*n, rng.normal(), 0, 0])
            single = orc.F_PLANE
        else:
            a = rng.normal(size=3) * 5
            coeff = np.array([*a, *(a + rng.normal(size=3))])
            single = orc.F_EDGE
        x = np.concatenate([xp, xi, xe])
        r, J = orc.factor_eval(kind, p, coeff, 1.0, x)
        comp = syn.pose_mul(syn.pose_mul(syn.pose_inv(xp), xi), xe)
        r1, _ = orc.factor_eval(single, p, coeff, 1.0, comp)
        assert abs(r[0] - r1[0]) < 1e-9
        J = J[:21].reshape(3, 7)
        for blk in (1, 2):
            for k in range(6 if blk == 1 else 3):
                d = np.zeros(6)
                d[k] = eps
                xx = x.copy()
                xx[blk * 7:(blk + 1) * 7] = orc.plus(x[blk * 7:(blk + 1) * 7], d)
                rp, _ = orc.factor_eval(kind, p, coeff, 1.0, xx, want_jac=False)
                num = (rp[0] - r[0]) / eps
                assert abs(num - J[blk, k]) < 5e-4 * max(1.0, abs(num)), (kind, blk, k, num, J[blk, k])


def test_plus_and_huber_and_sqrt_info():
    x = syn.pose7([1, 2, 3], syn.quat_from_rpy(0.3, 0.2, 0.1))
    assert np.allclose(orc.plus(x, np.zeros(6)), x, atol=1e-15)
    d = np.array([0.1, -0.2, 0.3, 0.01, 0.02, -0.03])
    out = orc.plus(x, d)
    assert np.allclose(out[:3], x[:3] + d[:3])
    q = syn.quat_mul(x[3:], np.array([*(d[3:] / 2), 1.0]))
    assert np.allclose(out[3:], q / np.linalg.norm(q))
    V = np.diag([1, 1, 0, 1, 1, 1.0])  # degenerate z translation is not updated
    assert orc.plus(x, d, V)[2] == x[2]
    assert np.allclose(orc.huber(0.1, 0.005), [0.005, 1.0])
    s = 0.04
    assert np.allclose(orc.huber(0.1, s), [2 * 0.1 * math.sqrt(s) - 0.01, 0.1 / math.sqrt(s)])
    assert orc.lib().orc_map_sqrt_info(0.0075) == 1.0  # sqrt(1/0.0075)=11.5 >= 3 -> 1
    assert abs(orc.lib().orc_map_sqrt_info(1.0) - 1.0 / 3.0) < 1e-15


def test_eval_degeneracy_remap():
    rng = np.random.default_rng(5)
    Q = np.linalg.qr(rng.normal(size=(6, 6)))[0]
    lam = np.array([5.0, 50.0, 500.0, 1e3, 1e4, 1e5])
    H = Q @ np.diag(lam) @ Q.T
    V, eig, deg = orc.eval_degeneracy(H, 100.0)
    assert deg and np.allclose(eig, lam, rtol=1e-9)
    # V_update projects out the two weakest eigen-directions
    assert np.allclose(V @ Q[:, 0], 0, atol=1e-9) and np.allclose(V @ Q[:, 1], 0, atol=1e-9)
    assert np.allclose(V @ Q[:, 3], Q[:, 3], atol=1e-9)
    V, eig, deg = orc.eval_degeneracy(H, 1.0)
    assert (not deg) and np.allclose(V, np.eye(6))


def test_extract_cloud_structure():
    scene = syn.make_scene()
    pose = syn.trajectory(1)[0]
    cloud, ss, se = syn.make_sweep(scene, pose, 16, 1024, seed=0)
    f = orc.extract_cloud(cloud, ss, se)
    ns = 16
    assert f["corner_points_sharp"].shape[0] <= 2 * 6 * ns
    assert f["corner_points_less_sharp"].shape[0] <= 20 * 6 * ns
    assert f["surf_points_flat"].shape[0] <= 4 * 6 * ns
    lab = f["label"]
    assert (lab == 2).sum() == f["corner_points_sharp"].shape[0]
    assert ((lab == 2) | (lab == 1)).sum() == f["corner_points_less_sharp"].shape[0]
    assert (lab == -1).sum() == f["surf_points_flat"].shape[0]
    # curvature known answer: collinear equally spaced points have zero curvature
    line = np.zeros((40, 4), np.float32)
    line[:, 0] = np.arange(40) * 0.5
    g = orc.extract_cloud(line, np.array([5], np.int32), np.array([34], np.int32))
    assert np.all(g["curvature"][5:35] == 0)
    assert g["corner_points_sharp"].shape[0] == 0 and g["surf_points_flat"].shape[0] == 6 * 4
    # short ring (< 6 usable points) is skipped (feature_extract.cpp:155)
    g = orc.extract_cloud(line[:16], np.array([5], np.int32), np.array([10], np.int32))
    assert sum(g[k].shape[0] for k in ("corner_points_sharp", "surf_points_flat", "surf_points_less_flat")) == 0


def test_scan2map_converges_and_schedules_agree():
    scene = syn.make_scene()
    traj = syn.trajectory(4)
    surf_map, corner_map = syn.make_submap(scene, 50000)
    cloud, ss, se = syn.make_sweep(scene, traj[3], 16, 1024, seed=3)
    f = orc.extract_cloud(cloud, ss, se)
    cs, _ = orc.voxel_grid(f["corner_points_less_sharp"], 0.2, True)
    sf, _ = orc.voxel_grid(f["surf_points_less_flat"], 0.4, True)
    init = syn.perturb_pose(traj[3], np.random.Generator(np.random.PCG64(9)))
    out, st = orc.scan2map(surf_map, corner_map, sf, cs, init)
    assert st["ran"] == 1 and st["n_surf"] > 1000 and st["n_corner"] > 50
    dt, dr = syn.pose_err(out, traj[3])
    dt0, dr0 = syn.pose_err(init, traj[3])
    assert dt < 0.01 and dr < 1e-3 and dt < dt0
    o = orc.default_opts()
    o[orc.O_MAX_OUTER], o[orc.O_MAX_INNER] = 5, 1  # north-star schedule: re-associate every GN iteration
    out2, _ = orc.scan2map(surf_map, corner_map, sf, cs, init, o)
    d2 = syn.pose_err(out, out2)
    assert d2[0] < 2e-3 and d2[1] < 2e-4
    # map-size gate (lidar_mapper_keyframe.cpp:429)
    out3, st3 = orc.scan2map(surf_map[:40], corner_map, sf, cs, init)
    assert st3["ran"] == 0 and np.array_equal(out3, init)


def test_track_cloud_recovers_motion():
    scene = syn.make_scene()
    traj = syn.trajectory(3)
    a, ssa, sea = syn.make_sweep(scene, traj[0], 16, 1024, seed=0)
    b, ssb, seb = syn.make_sweep(scene, traj[1], 16, 1024, seed=1)
    fa, fb = orc.extract_cloud(a, ssa, sea), orc.extract_cloud(b, ssb, seb)
    rel = syn.pose_mul(syn.pose_inv(traj[0]), traj[1])
    out, st = orc.track_cloud(fa["corner_points_less_sharp"], fa["surf_points_less_flat"], fb["corner_points_sharp"],
                              fb["surf_points_flat"], syn.pose7([0, 0, 0], [0, 0, 0, 1]))
    assert st["n_corner"] + st["n_surf"] >= 10
    dt, dr = syn.pose_err(out, rel)
    assert dt < 0.05 and dr < 5e-3


def _odom_problem(rng, n=400):
    """Features consistent with a 3-pose chain: planes/lines through the chained point, plus noise."""
    xp, xi, xe = (rand_pose(rng) for _ in range(3))
    comp = syn.pose_mul(syn.pose_mul(syn.pose_inv(xp), xi), xe)
    R = syn.quat_to_mat(comp[3:])
    pts = rng.normal(size=(n, 3)) * 6
    types = np.array([ord("s") if k % 3 else ord("c") for k in range(n)], np.uint8)
    coeffs = np.zeros((n, 6))
    for k in range(n):
        lp = R @ pts[k] + comp[:3]
        if types[k] == ord("s"):
            nrm = rng.normal(size=3)
            nrm /= np.linalg.norm(nrm)
            coeffs[k, :4] = [*nrm, -nrm @ lp + rng.normal() * 0.01]
        else:
            d = rng.normal(size=3)
            d /= np.linalg.norm(d)
            off = np.cross(d, rng.normal(size=3)) * 0.01
            coeffs[k] = [*(lp + off + 0.1 * d), *(lp + off - 0.1 * d)]
    # float-valued like the reference's PointPlaneFeature (built from float clouds)
    return xp, xi, xe, types, pts.astype(np.float32).astype(np.float64), coeffs.astype(np.float32).astype(np.float64)


@pytest.mark.parametrize("free_mask", [1, 2, 3])
def test_odom_solve_recovers_perturbed_blocks(free_mask):
    rng = np.random.default_rng(70 + free_mask)
    xp, xi, xe, types, pts, coeffs = _odom_problem(rng)
    d = lambda: syn.pose7(rng.normal(size=3) * 0.02, syn.quat_from_rpy(*(rng.normal(size=3) * 0.004)))
    xi0 = syn.pose_mul(xi, d()) if free_mask & 1 else xi
    xe0 = syn.pose_mul(xe, d()) if free_mask & 2 else xe
    oi, oe, st = orc.odom_solve(types, pts, coeffs, xp, xi0, xe0, free_mask, max_it=30)
    assert st["lm_iterations"] >= 2
    if not free_mask & 1:
        assert np.array_equal(oi, xi0)
    if not free_mask & 2:
        assert np.array_equal(oe, xe0)
    # the composed pivot<-sensor transform is what the residuals constrain
    c_true = syn.pose_mul(syn.pose_mul(syn.pose_inv(xp), xi), xe)
    c_est = syn.pose_mul(syn.pose_mul(syn.pose_inv(xp), oi), oe)
    c_ini = syn.pose_mul(syn.pose_mul(syn.pose_inv(xp), xi0), xe0)
    assert syn.pose_err(c_est, c_true)[0] < 0.25 * syn.pose_err(c_ini, c_true)[0]


def test_good_feature_selection_oracle_properties():
    """orc_gf.hpp: selection sizes, determinism per seed, no duplicates, only matched features, greedy > random in log det."""
    rng = np.random.default_rng(5)
    n = 600
    matched = rng.random(n) < 0.7
    jaco = rng.normal(size=(n, 6)) * matched[:, None]
    xyz = np.concatenate([rng.uniform(-20, 20, (n, 3)), np.zeros((n, 1))], 1).astype(np.float32)
    sel_all, H_all = orc.gf_select(orc.GF_WO, 1.0, 1, matched, jaco, xyz)
    assert np.array_equal(sel_all, np.flatnonzero(matched))
    assert np.allclose(H_all, 1e-6 * np.eye(6) + jaco.T @ jaco)
    ld = {}
    for name, m in (("rnd", orc.GF_RND), ("fps", orc.GF_FPS), ("gd", orc.GF_GD)):
        s1, H1 = orc.gf_select(m, 0.2, 42, matched, jaco, xyz)
        s2, H2 = orc.gf_select(m, 0.2, 42, matched, jaco, xyz)
        s3, _ = orc.gf_select(m, 0.2, 43, matched, jaco, xyz)
        assert np.array_equal(s1, s2) and np.array_equal(H1, H2) and not np.array_equal(s1, s3)
        assert len(s1) == int(n * 0.2) and len(set(s1.tolist())) == len(s1) and matched[s1].all()
        ld[name] = np.linalg.slogdet(H1)[1]
        if m != orc.GF_FPS:  # fps never adds its start point to H (reference quirk, lidar_mapper.h:375-379)
            assert np.allclose(H1, 1e-6 * np.eye(6) + jaco[s1].T @ jaco[s1])
    assert ld["gd"] > ld["rnd"]
    # nothing matched: every method terminates empty
    none = np.zeros(n, bool)
    for m in (orc.GF_RND, orc.GF_FPS, orc.GF_GD):
        assert len(orc.gf_select(m, 0.3, 1, none, np.zeros((n, 6)), xyz)[0]) == 0


# ------------------------------------------------------------------------------------------------ committed golden fixtures
GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def test_golden_reference_nanoflann_pins_oracle_knn():
    """tests/golden/knn_nanoflann.npz holds the answers of the REFERENCE's own kd-tree (nanoflann.hpp compiled in place,
    see make_golden.py): the oracle's kNN must reproduce indices and float distances exactly — also on hosts without
    /root/reference."""
    g = np.load(os.path.join(GOLDEN, "knn_nanoflann.npz"))
    for k in (1, 5, 10):
        idx, sqd = orc.knn(g["map"], g["query"], k)
        assert np.array_equal(idx, g[f"idx{k}"]) and np.array_equal(sqd, g[f"sqd{k}"])


def test_golden_oracle_regression_vectors():
    """The oracle reproduces its committed outputs bit for bit (guards the checker itself against accidental change)."""
    g = np.load(os.path.join(GOLDEN, "oracle_small.npz"))
    f = orc.extract_cloud(g["cloud"], g["ss"], g["se"])
    for key, name in (("corner_points_sharp", "sharp"), ("corner_points_less_sharp", "less_sharp"), ("surf_points_flat", "flat"),
                      ("surf_points_less_flat", "less_flat")):
        assert np.array_equal(f[key].view(np.uint32), g[name].view(np.uint32)), key
    cs, _ = orc.voxel_grid(g["less_sharp"], 0.2, True)
    sf, _ = orc.voxel_grid(g["less_flat"], 0.4, True)
    assert np.array_equal(cs.view(np.uint32), g["corner_ds"].view(np.uint32)) and np.array_equal(sf.view(np.uint32), g["surf_ds"].view(np.uint32))
    vs, cfs, nns = orc.match_from_map("s", g["surf_map"], g["surf_ds"], g["init"])
    assert np.array_equal(vs, g["surf_valid"]) and np.array_equal(nns, g["surf_nn"]) and np.array_equal(cfs, g["surf_coeff"])
    o = orc.default_opts()
    o[orc.O_MAX_OUTER], o[orc.O_MAX_INNER] = 3, 4
    pose, st = orc.scan2map(g["surf_map"], g["corner_map"], g["surf_ds"], g["corner_ds"], g["init"], o)
    assert np.array_equal(pose, g["pose"]) and int(st["n_surf"]) == int(g["n_surf"]) and int(st["n_corner"]) == int(g["n_corner"])
    gf = orc.good_features("s", g["surf_map"], g["surf_ds"], g["init"], orc.GF_GD, 0.25, 11)
    assert np.array_equal(gf["sel"], g["gf_sel"])


def test_solver_restatement_converges_to_independent_optimum():
    """The ceres::Solve restatement (orc_solver.hpp) + the factor restatements against an INDEPENDENT solver: with the
    correspondences of one association fixed, scipy's trust-region least squares with the Huber loss minimises the same
    objective (ceres::HuberLoss(a): rho(s) = s | 2a sqrt(s) - a^2  ==  scipy loss='huber', f_scale=a) written directly
    in numpy.  Both must land on the same pose."""
    from scipy.optimize import least_squares
    from scipy.spatial.transform import Rotation

    scene = syn.make_scene()
    traj = syn.trajectory(6)
    surf_map, corner_map = syn.make_submap(scene, 30000)
    cloud, ss, se = syn.make_sweep(scene, traj[4], 16, 512, seed=21)
    f = orc.extract_cloud(cloud, ss, se)
    cs, _ = orc.voxel_grid(f["corner_points_less_sharp"], 0.2, True)
    sf, _ = orc.voxel_grid(f["surf_points_less_flat"], 0.4, True)
    init = syn.perturb_pose(traj[4], np.random.Generator(np.random.PCG64(2)))
    o = orc.default_opts()
    o[orc.O_MAX_OUTER], o[orc.O_MAX_INNER] = 1, 60  # one association, LM to convergence
    pose, st = orc.scan2map(surf_map, corner_map, sf, cs, init, o)
    assert st["n_surf"] > 300 and st["n_corner"] > 50

    vs, cfs, _ = orc.match_from_map("s", surf_map, sf, init)
    vc, cfc, _ = orc.match_from_map("c", corner_map, cs, init)
    ps, ws, ds = sf[vs][:, :3].astype(np.float64), cfs[vs][:, :3], cfs[vs][:, 3]
    pc, la, lb = cs[vc][:, :3].astype(np.float64), cfc[vc][:, :3], cfc[vc][:, 3:6]
    sinfo = orc.map_sqrt_info(0.0075)
    t0, R0 = init[:3], Rotation.from_quat(init[3:7])  # x, y, z, w

    def residuals(x):
        R = (R0 * Rotation.from_rotvec(x[3:6])).as_matrix()
        t = t0 + x[:3]
        rs = sinfo * (np.einsum("ij,ij->i", ws, ps @ R.T + t) + ds)            # plane: s (w.(Rp+t) + d)
        lp = pc @ R.T + t
        rc = sinfo * np.linalg.norm(np.cross(lp - la, lp - lb), axis=1) / np.linalg.norm(la - lb, axis=1)  # edge: s |..x..| / |a-b|
        return np.concatenate([rs, rc])

    sol = least_squares(residuals, np.zeros(6), loss="huber", f_scale=0.1, xtol=1e-14, ftol=1e-14, gtol=1e-14, max_nfev=400)
    R_ref = (R0 * Rotation.from_rotvec(sol.x[3:6]))
    pose_ref = np.concatenate([t0 + sol.x[:3], R_ref.as_quat()])
    dt, dr = syn.pose_err(pose, pose_ref)
    # Ceres' default function tolerance (1e-6 relative cost change) stops the LM a few 1e-5 m short of the exact optimum
    assert dt < 1e-4 and dr < 1e-4, (dt, dr)
    assert dt < 0.05 * syn.pose_err(init, pose_ref)[0]
    # and the objective value agrees: 1/2 sum rho
    r = residuals(sol.x)
    rho = np.where(np.abs(r) <= 0.1, r * r, 2 * 0.1 * np.abs(r) - 0.01)
    assert abs(0.5 * rho.sum() - st["final_cost"]) < 1e-6 * max(1.0, st["final_cost"])


# ------------------------------------------------------------------------------------------------ round-2 restatements: known answers
def _skew(v):
    return np.array([[0, -v[2], v[1]], [v[2], 0, -v[0]], [-v[1], v[0], 0]], float)


def _se3_exp(xi):
    """exp of [rho | phi] (translation first, as associate_uct.hpp's pose covariances) -> (R, t)."""
    rho, phi = xi[:3], xi[3:]
    th = np.linalg.norm(phi)
    K = _skew(phi)
    if th < 1e-12:
        return np.eye(3) + K, rho + 0.5 * K @ rho
    R = np.eye(3) + np.sin(th) / th * K + (1 - np.cos(th)) / th ** 2 * K @ K
    J = np.eye(3) + (1 - np.cos(th)) / th ** 2 * K + (th - np.sin(th)) / th ** 3 * K @ K
    return R, J @ rho


def _rand_spd(rng, scale):
    A = rng.normal(size=(6, 6))
    return scale * (A @ A.T + 0.5 * np.eye(6))


def test_compound_pose_with_cov_first_order_and_identities():
    """compoundPoseWithCov (associate_uct.hpp:9-88): the pose is the product; for small covariances the result tends to the first-order
    propagation cov1 + Ad(T1) cov2 Ad(T1)^T (written here independently, [translation | rotation] ordering); the 4th-order terms are
    O(cov^2); compounding with an exactly known identity is the identity."""
    rng = np.random.default_rng(3)
    p1 = syn.pose7([1.0, -2.0, 0.5], syn.quat_from_rpy(0.1, -0.2, 0.7))
    p2 = syn.pose7([0.3, 0.2, -0.1], syn.quat_from_rpy(-0.05, 0.15, -0.4))
    R1, t1 = syn.quat_to_mat(p1[3:]), p1[:3]
    Ad = np.zeros((6, 6))
    Ad[:3, :3], Ad[:3, 3:], Ad[3:, 3:] = R1, _skew(t1) @ R1, R1
    for scale, tol in ((1e-9, 1e-6), (1e-4, 2e-3)):
        c1, c2 = _rand_spd(rng, scale), _rand_spd(rng, scale)
        pc, cc = orc.compound_pose_cov(p1, c1, p2, c2)
        assert max(syn.pose_err(pc, syn.pose_mul(p1, p2))) < 1e-12
        first = c1 + Ad @ c2 @ Ad.T
        assert np.allclose(cc, cc.T, atol=1e-18) and np.all(np.linalg.eigvalsh(cc) > 0)
        assert np.linalg.norm(cc - first) / np.linalg.norm(first) < tol
    ident = syn.pose7([0, 0, 0], [0, 0, 0, 1])
    c1 = _rand_spd(rng, 1e-3)
    pc, cc = orc.compound_pose_cov(p1, c1, ident, np.zeros((6, 6)))
    assert np.allclose(pc, p1) and np.allclose(cc, c1, rtol=0, atol=1e-15)
    # Monte-Carlo: T = exp(xi1^) T1 exp(xi2^) T2 with xi ~ N(0, cov); the compounded covariance is that of log(T * inv(T1 T2))
    c1, c2 = _rand_spd(rng, 2e-4), _rand_spd(rng, 2e-4)
    _, cc = orc.compound_pose_cov(p1, c1, p2, c2)
    L1, L2 = np.linalg.cholesky(c1), np.linalg.cholesky(c2)
    R2, t2 = syn.quat_to_mat(p2[3:]), p2[:3]
    Rm, tm = R1 @ R2, R1 @ t2 + t1
    n = 20000
    xs = np.zeros((n, 6))
    for i in range(n):
        Ra, ta = _se3_exp(L1 @ rng.normal(size=6))
        Rb, tb = _se3_exp(L2 @ rng.normal(size=6))
        Rl, tl = Ra @ R1, Ra @ t1 + ta          # exp(xi1) T1
        Rr, tr = Rb @ R2, Rb @ t2 + tb          # exp(xi2) T2
        R, t = Rl @ Rr, Rl @ tr + tl
        dR, dt = R @ Rm.T, t - R @ Rm.T @ tm    # T * inv(mean)
        phi = 0.5 * np.array([dR[2, 1] - dR[1, 2], dR[0, 2] - dR[2, 0], dR[1, 0] - dR[0, 1]])  # small angles: log ~ vee of the skew part
        xs[i] = np.concatenate([dt - 0.5 * np.cross(phi, dt), phi])
    mc = xs.T @ xs / n
    assert np.linalg.norm(mc - cc) / np.linalg.norm(cc) < 0.06


def test_point_uncertainty_is_the_propagated_jacobian():
    """evalPointUncertainty (associate_uct.hpp:164-215): cov = G blockdiag(cov_pose, cov_meas) G^T with G = [I | -(Rp+t)^ | R]; G is
    checked here against numerical derivatives of y = exp(xi^) T (p + d)."""
    rng = np.random.default_rng(4)
    pose = syn.pose7([2.0, -1.0, 0.3], syn.quat_from_rpy(0.2, 0.1, -0.9))
    R, t = syn.quat_to_mat(pose[3:]), pose[:3]
    pts = np.concatenate([rng.uniform(-20, 20, (50, 3)), np.zeros((50, 1))], 1).astype(np.float32)
    cov_pose, cm = _rand_spd(rng, 1e-3), np.diag([0.0025, 0.0025, 0.0025])
    got = orc.point_uncertainty(pts, pose, cov_pose, cm)
    for i in (0, 7, 49):
        p = pts[i, :3].astype(float)

        def f(xi, d):
            Re, te = _se3_exp(xi)
            return Re @ (R @ (p + d) + t) + te

        G = np.zeros((3, 9))
        h = 1e-6
        for k in range(6):
            e = np.zeros(6)
            e[k] = h
            G[:, k] = (f(e, np.zeros(3)) - f(-e, np.zeros(3))) / (2 * h)
        for k in range(3):
            e = np.zeros(3)
            e[k] = h
            G[:, 6 + k] = (f(np.zeros(6), e) - f(np.zeros(6), -e)) / (2 * h)
        S = np.zeros((9, 9))
        S[:6, :6], S[6:, 6:] = cov_pose, cm
        Cn = G @ S @ G.T
        want = np.array([Cn[0, 0], Cn[0, 1], Cn[0, 2], Cn[1, 1], Cn[1, 2], Cn[2, 2]])
        assert np.allclose(got[i], want, rtol=2e-4, atol=1e-7), (got[i], want)


def test_voxel_grid_cov_hand_computed_merge():
    """VoxelGridCovarianceMLOAM<PointIWithCov> merge (voxel_grid_covariance_mloam_impl.hpp:293-333): weight w = threshold - trace,
    centroid = sum(w x) / sum(w), covariance = sum(w^2 C) / sum(w)^2, intensity of the heaviest point, points with |trace| >= threshold
    skipped; voxels come out in index order (x fastest)."""
    thr = 1.0
    pts = np.array([[0.10, 0.10, 0.10, 5.0], [0.30, 0.20, 0.10, 7.0], [0.20, 0.30, 0.30, 9.0],   # voxel (0,0,0) at leaf 0.5
                    [0.70, 0.10, 0.10, 1.0],                                                   # voxel (1,0,0)
                    [0.10, 0.10, 0.60, 2.0], [0.20, 0.20, 0.70, 3.0]], np.float32)             # voxel (0,0,1); the second one is over the threshold
    tr = np.array([0.2, 0.5, 0.8, 0.1, 0.4, 1.5], np.float32)
    c6 = np.zeros((6, 6), np.float32)
    c6[:, 0], c6[:, 3], c6[:, 5] = tr / 2, tr / 4, tr / 4   # xx, yy, zz; trace = tr
    c6[:, 1] = 0.01
    op, oc, ot, ok = orc.voxel_grid_cov(pts, c6, tr, 0.5, thr)
    assert ok and op.shape[0] == 3
    w = thr - tr[:3]
    mu = (w[:, None] * pts[:3, :3]).sum(0) / w.sum()
    assert np.allclose(op[0, :3], mu, atol=1e-6) and op[0, 3] == 5.0          # heaviest point: the first (w = 0.8)
    assert np.allclose(oc[0], (w[:, None] ** 2 * c6[:3]).sum(0) / w.sum() ** 2, atol=1e-7)
    assert np.isclose(ot[0], oc[0, 0] + oc[0, 3] + oc[0, 5])
    assert np.allclose(op[1], pts[3]) and np.allclose(oc[1], c6[3], atol=1e-7)  # single point: w cancels
    assert np.allclose(op[2], pts[4]) and np.allclose(oc[2], c6[4], atol=1e-7)  # the over-threshold point is ignored
    # a voxel whose points are ALL over the threshold still emits a point: weight_total falls back to 1 -> zero centroid (reference :326)
    op2, oc2, ot2, _ = orc.voxel_grid_cov(pts[5:6], c6[5:6], tr[5:6], 0.5, thr)
    assert op2.shape[0] == 1 and np.all(op2[0, :3] == 0) and ot2[0] == 0


def test_project_cloud_known_pixels():
    """ImageSegmenter::projectCloud (image_segmenter.hpp:88-136) + ring order + ScanInfo (:381-389) on points with known pixels."""
    H = 1800
    res = 360.0 / H

    def pt(elev_deg, az_deg, r=10.0, w=0.25):
        e, a = np.deg2rad(elev_deg), np.deg2rad(az_deg)  # azimuth measured as atan2(x, y)
        return [r * np.cos(e) * np.sin(a), r * np.cos(e) * np.cos(a), r * np.sin(e), w]

    # VLP-16: row = int((elev + 15.1) / 2): ring elevations -15, -13, ... ; column = -round((az - 90) / res) + H/2 (wrapped)
    cloud = np.array([pt(-15, 90), pt(-13, 90), pt(15, 90),            # rows 0, 1, 15 at column H/2
                      pt(-15, 90 - 10 * res), pt(-15, 90 + 10 * res),    # columns H/2 + 10, H/2 - 10
                      pt(-15, 90.02),                                    # same pixel as the first point: dropped (first wins)
                      pt(-15, 90, r=0.3),                                # inside ROI_RANGE 0.5: dropped
                      pt(-17.5, 90), pt(17.5, 90),                       # below row 0 / above row 15: dropped
                      pt(-13, -100)], np.float32)                        # az -100 deg: column H/2 + 950 -> wraps to 50
    pix = orc.project_pixels(cloud, 16, H, 0.5)
    assert list(pix[:5]) == [0 * H + H // 2, 1 * H + H // 2, 15 * H + H // 2, H // 2 + 10, H // 2 - 10]
    assert pix[5] == pix[0] and list(pix[6:9]) == [-1, -1, -1] and pix[9] == 1 * H + 50
    out, ss, se = orc.project_cloud(cloud, 16, H, 0.5)
    # ring order: row 0 (points 0, 3, 4 in input order), row 1 (points 1, 9), row 15 (point 2); intensity += row
    assert out.shape[0] == 6
    assert np.array_equal(out[:, :3], cloud[[0, 3, 4, 1, 9, 2], :3])
    assert np.allclose(out[:, 3], [0.25, 0.25, 0.25, 1.25, 1.25, 15.25])
    assert list(ss[:3]) == [5, 8, 10] and list(se[:3]) == [-3, -1, -1] and ss[15] == 10 and se[15] == 0
    # HDL-64E: row = int((2 - elev) * 3 + 0.5) down to -8.83 deg, then 32 + int((-8.83 - elev) * 2 + 0.5); rows above 50 are dropped
    c64 = np.array([pt(2, 90), pt(0, 90), pt(-8.5, 90), pt(-9.0, 90), pt(-17.83, 90), pt(-18.5, 90), pt(2.2, 90), pt(-24.5, 90)], np.float32)
    rows = orc.project_pixels(c64, 64, 2048, 0.5)
    assert list(rows // 2048 * (rows >= 0) + (rows < 0) * -1) == [0, 6, 32, 32, 50, -1, -1, -1]
    # 32 rings: ang_res_y = 41.33 / 31, bottom 30.67
    r32 = orc.project_pixels(np.array([pt(-30.67 + 41.33 / 31 * (k + 0.5), 45) for k in range(32)], np.float32), 32, 2169, 0.5)
    assert list(r32 // 2169) == list(range(32))


def test_frame_multi_reduces_to_frame_and_local_map_build_to_its_parts():
    """One LiDAR with an identity extrinsic through the rig path gives the single-LiDAR frame; buildLocalMap's map half equals
    transform (PCL float matrix) + concatenation + VoxelGrid done by hand."""
    scene = syn.make_scene()
    traj = syn.trajectory(6)
    surf_map, corner_map = syn.make_submap(scene, 50000)
    cloud, ss, se = syn.make_sweep(scene, traj[3], 16, 1024, seed=8)
    init = syn.perturb_pose(traj[3], np.random.Generator(np.random.PCG64(2)))
    o = orc.default_opts()
    o[orc.O_MAX_OUTER], o[orc.O_MAX_INNER] = 3, 1
    a, sa = orc.frame(cloud, ss, se, surf_map, corner_map, init, o)
    ident = np.array([[0, 0, 0, 0, 0, 0, 1.0]])
    b, sb = orc.frame_multi(cloud, ss, se, 1, ident, surf_map, corner_map, init, o)
    assert max(syn.pose_err(a, b)) < 1e-12 and int(sa["n_surf"]) == int(sb["n_surf"]) and int(sa["n_corner"]) == int(sb["n_corner"])
    # two LiDARs: the second one's features enter through its extrinsic — the frame still lands on the truth
    cl2, ss2, se2, ext = syn.make_multi_sweep(scene, traj[3], 2, 16, 1024, seed=8)
    c, sc = orc.frame_multi(cl2, ss2, se2, 2, ext, surf_map, corner_map, init, o)
    et, er = syn.pose_err(c, traj[3])
    assert et < 0.05 and er < 3e-3 and int(sc["n_surf"]) > int(sb["n_surf"])
    # local map: three window clouds brought to the pivot frame and filtered
    f = orc.extract_cloud(cloud, ss, se)["surf_points_less_flat"]
    poses = np.stack([syn.pose7([0.1 * k, 0.05 * k, 0.0], syn.quat_from_rpy(0, 0, 0.02 * k)) for k in range(3)])
    got = orc.local_map_build([f, f[::2], f[::3]], poses, 0.4)
    parts = []
    for cl, p in zip([f, f[::2], f[::3]], poses):
        M = np.eye(4, dtype=np.float32)
        M[:3, :3], M[:3, 3] = syn.quat_to_mat(p[3:]).astype(np.float32), p[:3].astype(np.float32)
        q = cl.copy()
        x, y, z = cl[:, 0], cl[:, 1], cl[:, 2]
        for r in range(3):  # pcl::transformPointCloud: float, m(r,0) x + m(r,1) y + m(r,2) z + m(r,3)
            q[:, r] = M[r, 0] * x + M[r, 1] * y + M[r, 2] * z + M[r, 3]
        parts.append(q)
    want, _ = orc.voxel_grid(np.concatenate(parts), 0.4, False)
    assert got.shape == want.shape and np.allclose(got, want, atol=2e-5)


def test_calib_frame_oracle_reduces_the_extrinsic_error():
    """The 12-DoF step [pose_i | ext_cal] (buildCalibMap association + LidarPureOdom rows of the reference LiDAR + LidarOnlineCalib rows of
    the second one, estimator.cpp:687-848,1067-1156): from a 2 deg / 5 cm wrong extrinsic the step moves towards the true one; with the
    second LiDAR's rows absent the extrinsic block does not move; the row count is the number of gated matches of both groups."""
    scene = syn.make_scene()
    cs = syn.make_calib_case(scene, orc.extract_cloud, orc.voxel_grid, 16, 1024, 100_000)
    e0 = syn.pose_err(cs["ext_cal_init"], cs["ext_cal"])
    pi, ec, st = orc.calib_frame(cs["surf_map"], cs["corner_map"], cs["surf_ref"], cs["corner_ref"], cs["surf_cal"], cs["corner_cal"], cs["pivot"],
                                 cs["pose_i_init"], cs["ext_ref"], cs["ext_cal_init"], 10, 1)
    e1 = syn.pose_err(ec, cs["ext_cal"])
    assert e0[1] > 0.03 and e1[1] < 0.5 * e0[1] and e1[0] < e0[0]
    assert st["rows"] > 1000 and st["lm_iterations"] >= 5
    pi_only, ec_same, st_only = orc.calib_frame(cs["surf_map"], cs["corner_map"], cs["surf_ref"], cs["corner_ref"], None, None, cs["pivot"],
                                                cs["pose_i_init"], cs["ext_ref"], cs["ext_cal_init"], 10, 1)
    assert np.allclose(ec_same, cs["ext_cal_init"], atol=1e-12) and 0 < st_only["rows"] < st["rows"]
