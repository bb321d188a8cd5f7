#!/usr/bin/env python
"""Generate the committed golden fixtures of tests/golden/ (run in the build container, where /root/reference exists).

    python tests/golden/make_golden.py

knn_nanoflann.npz   REFERENCE-DERIVED: neighbour indices and float squared distances returned by the reference's own
                    kd-tree (nanoflann.hpp vendored at /root/reference/mloam_loop/include/mloam_loop/scan_context/,
                    compiled in place into oracle/_ref/libref_knn.so) on a seeded map / query set.  This is the one
                    piece of the hot path whose reference code builds here; the fixture carries its answers to the GPU
                    box, where /root/reference does not exist.
oracle_small.npz    ORACLE-DERIVED regression vectors (the reference ships no golden vectors for this path — SURVEY.md §4;
                    DESIGN.md §2 "parity unpinned"): a seeded 16 x 512 sweep + 20k-point submap with the oracle's feature
                    sets, voxel filters, match results, good-feature selection and scan2map pose.  They pin the oracle
                    against accidental change (CPU suite) and give the GPU suite fixed targets that do not depend on the
                    oracle being rebuilt identically on the GPU box.
"""
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
import oracle_lib as orc  # noqa: E402
import synthetic as syn  # noqa: E402


def small_case():
    scene = syn.make_scene()
    traj = syn.trajectory(5)
    surf_map, corner_map = syn.make_submap(scene, 20000)
    cloud, ss, se = syn.make_sweep(scene, traj[3], 16, 512, seed=9)
    init = syn.perturb_pose(traj[3], np.random.Generator(np.random.PCG64(3)))
    return surf_map, corner_map, cloud, ss, se, init


def knn_uniform():
    """knn_nanoflann_uniform.npz: the reference kd-tree's answers on test_oracle_cpu.knn_uniform_case() (the map is re-made from its seed)."""
    from test_oracle_cpu import knn_uniform_case
    m, q = knn_uniform_case()
    out = {"query": q}
    for k in (1, 5, 10):
        out[f"idx{k}"], out[f"sqd{k}"] = orc.ref_knn(m, q, k)
    np.savez_compressed(os.path.join(HERE, "knn_nanoflann_uniform.npz"), **out)


def main():
    # ---- reference nanoflann
    assert orc.ref_lib() is not None, "oracle/_ref/libref_knn.so missing: run `make -C oracle ref` where the reference sources are"
    rng = np.random.default_rng(2024)
    m = np.concatenate([rng.uniform(-8, 8, (6000, 3)), np.zeros((6000, 1))], 1).astype(np.float32)
    q = np.concatenate([rng.uniform(-8.5, 8.5, (300, 3)), np.zeros((300, 1))], 1).astype(np.float32)
    out = {"map": m, "query": q}
    for k in (1, 5, 10):
        idx, sqd = orc.ref_knn(m, q, k)
        out[f"idx{k}"], out[f"sqd{k}"] = idx, sqd
    np.savez_compressed(os.path.join(HERE, "knn_nanoflann.npz"), **out)
    knn_uniform()

    # ---- oracle regression vectors
    surf_map, corner_map, cloud, ss, se, init = small_case()
    f = orc.extract_cloud(cloud, ss, se)
    cs, _ = orc.voxel_grid(f["corner_points_less_sharp"], 0.2, True)
    sf, _ = orc.voxel_grid(f["surf_points_less_flat"], 0.4, True)
    vs, cfs, nns = orc.match_from_map("s", surf_map, sf, init)
    vc, cfc, nnc = orc.match_from_map("c", corner_map, cs, init)
    o = orc.default_opts()
    o[orc.O_MAX_OUTER], o[orc.O_MAX_INNER] = 3, 4
    pose, st = orc.scan2map(surf_map, corner_map, sf, cs, init, o)
    gf = orc.good_features("s", surf_map, sf, init, orc.GF_GD, 0.25, 11)
    np.savez_compressed(
        os.path.join(HERE, "oracle_small.npz"), surf_map=surf_map, corner_map=corner_map, cloud=cloud, ss=ss, se=se, init=init,
        sharp=f["corner_points_sharp"], less_sharp=f["corner_points_less_sharp"], flat=f["surf_points_flat"], less_flat=f["surf_points_less_flat"],
        corner_ds=cs, surf_ds=sf, surf_valid=vs, surf_coeff=cfs, surf_nn=nns, corner_valid=vc, corner_nn=nnc, pose=pose,
        n_surf=int(st["n_surf"]), n_corner=int(st["n_corner"]), lm_iterations=int(st["lm_iterations"]), gf_sel=gf["sel"], gf_H=gf["H"])
    # ---- workload cache: voxel-filtered keyframe features of the §8d submap (synthetic.keyframe_map_features); ~30 s of ray casting
    import synthetic as syn
    surf_f, corner_f = syn.keyframe_map_features(syn.make_scene(), orc.extract_cloud, orc.voxel_grid, use_cache=False)
    np.savez_compressed(os.path.join(HERE, "submap_keyframes_filtered.npz"), surf=surf_f, corner=corner_f, tag=f"{syn.SEED}_30_64x2048")
    for name in ("knn_nanoflann.npz", "knn_nanoflann_uniform.npz", "oracle_small.npz", "submap_keyframes_filtered.npz"):
        print(name, os.path.getsize(os.path.join(HERE, name)), "bytes")


if __name__ == "__main__":
    main()
