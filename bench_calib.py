"""bench_calib.py — the C3 workload of bench.py (BASELINE.json configs[2]): 2 LiDARs, 64 x 2048 sweeps, 2M-point local map,
12-DoF online extrinsic calibration.  A step is one calibration step of Estimator::optimizeMap with ESTIMATE_EXTRINSIC == 1
(mloam_calib_frame): upload of the two LiDARs' window-level features, GN_ITERS x (buildCalibMap association of both groups +
residuals / Jacobians + 12x12 normal equations + LM step), local maps uploaded + rebuilt on keyframe steps.
--gpus 2: rank 0 holds the reference LiDAR's features, rank 1 the calibrated LiDAR's; one ncclAllReduce of the packed 12x12 normal
equations (92 doubles) per LM evaluation.  --gpus 1: both groups in one context."""
from __future__ import annotations

import os
import statistics
import time

import numpy as np


def _oracle_fn(name):
    def f(*a, **k):
        import oracle_lib as orc
        return getattr(orc, name)(*a, **k)
    return f


def make_calib_workload(syn, cfg, n_cases, map_kind):
    from bench import make_submap
    scene = syn.make_scene()
    surf_w, corner_w, info = make_submap(syn, scene, cfg["map_points"], map_kind)
    cases = [syn.make_calib_case(scene, _oracle_fn("extract_cloud"), _oracle_fn("voxel_grid"), cfg["rings"], cfg["horizon"], cfg["map_points"],
                                 seed=31 + 7 * k, submap=(surf_w, corner_w)) for k in range(n_cases)]
    return cases, info


def cpu_calib_arm(orc, cfg, cases, steps, time_cap_s=None):
    ref_tree = orc.use_ref_tree(True)
    times, last = [], None
    try:
        for k in range(steps):
            cs = cases[k % len(cases)]
            t = time.perf_counter()
            last = orc.calib_frame(cs["surf_map"], cs["corner_map"], cs["surf_ref"], cs["corner_ref"], cs["surf_cal"], cs["corner_cal"], cs["pivot"],
                                   cs["pose_i_init"], cs["ext_ref"], cs["ext_cal_init"], cfg["gn_iters"], 1)
            times.append(time.perf_counter() - t)
            if time_cap_s is not None and sum(times) > time_cap_s:
                break
    finally:
        orc.use_ref_tree(False)
    return len(times) / sum(times), times, last, ("reference nanoflann (oracle/_ref/libref_knn.so)" if ref_tree else "oracle restatement")


def gpu_measure_calib(m, syn, torch, dist, cfg_name, cfg, args, rank, local_rank, world, steps, warmup, n_frames):
    from bench import ClockSampler
    p = m.default_params()
    p.n_scans, p.map_cell, p.max_ring_points = cfg["rings"], args.map_cell, cfg["horizon"]
    ctx = m.Context(local_rank, p)
    exchange = None
    if world > 1:
        uid = [m.Context.comm_unique_id() if rank == 0 else None]
        dist.broadcast_object_list(uid, src=0)
        ctx.comm_init(world, rank, uid[0])
        exchange = "ncclAllReduce of the packed 12x12 normal equations (92 doubles) per LM evaluation"
        dist.barrier()
    cases, map_info = make_calib_workload(syn, cfg, n_frames, args.map)
    KF = max(1, args.keyframe_every)
    dev = torch.device("cuda", local_rank)
    flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device=dev)
    stream = torch.cuda.Stream(device=dev)
    ctx.set_stream(stream.cuda_stream)

    def step(k, rebuild):
        cs = cases[k % len(cases)]
        if rebuild:
            ctx.map_build(0, cs["corner_map"], args.map_cell)
            ctx.map_build(1, cs["surf_map"], args.map_cell)
        ref = (cs["surf_ref"], cs["corner_ref"]) if (world == 1 or rank == 0) else (None, None)
        cal = (cs["surf_cal"], cs["corner_cal"]) if (world == 1 or rank == 1) else (None, None)
        return ctx.calib_frame(ref[0], ref[1], cal[0], cal[1], cs["pivot"], cs["pose_i_init"], cs["ext_ref"], cs["ext_cal_init"], cfg["gn_iters"], 1)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    sampler = ClockSampler(local_rank)
    sampler.start()
    sampler.wait_first()
    for k in range(max(warmup, 3)):
        step(k, True)
    barrier()
    sampler.mark()
    launches0 = ctx.launch_count()
    evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
    last = None
    with torch.cuda.stream(stream):
        for k in range(steps):
            flush.fill_(k & 0xFF)
            if world > 1:
                dist.barrier()
            evs[k][0].record(stream)
            last = step(k, k % KF == 0)
            evs[k][1].record(stream)
    barrier()
    clocks = sampler.stop()
    ms_steps = [a.elapsed_time(b) for a, b in evs]
    srt = sorted(ms_steps)
    t_max = sum(ms_steps) / 1e3
    if world > 1:
        tt = torch.tensor([t_max], dtype=torch.float64, device=dev)
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        t_max = float(tt.item())
    L = cfg["lidars"]
    # e2e: wall clock around the same host-buffer calls (this API takes host features; the maps are uploaded on keyframe steps)
    barrier()
    t0 = time.perf_counter()
    for k in range(steps):
        step(k, k % KF == 0)
    torch.cuda.synchronize()
    t_e2e = time.perf_counter() - t0
    if world > 1:
        tt = torch.tensor([t_e2e], dtype=torch.float64, device=dev)
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        t_e2e = float(tt.item())
    cs0 = cases[0]
    feat_bytes = int(sum(cs0[k].nbytes for k in ("surf_ref", "corner_ref", "surf_cal", "corner_cal")) / max(1, world)) + 28 * 8
    map_bytes = int(cs0["surf_map"].nbytes + cs0["corner_map"].nbytes)
    n_kf = len(range(0, steps, KF))
    res = dict(step_stats={"min": srt[0], "median": srt[len(srt) // 2], "p90": srt[int(0.9 * (len(srt) - 1))], "max": srt[-1]},
               keyframe_ms=statistics.mean(ms_steps[0::KF]), regular_ms=(statistics.mean([x for i, x in enumerate(ms_steps) if i % KF]) if KF > 1 and steps > 1 else None),
               clocks=clocks, launches=int(ctx.launch_count() - launches0), exchange=exchange, exchange_timeouts=0,
               features_per_step=float(sum(cs0[k].shape[0] for k in ("surf_ref", "corner_ref", "surf_cal", "corner_cal"))),
               t_max=t_max, value=L * steps / t_max, k_last=(steps - 1) % len(cases), last_pose=last[0], last_ext=last[1], last_stats=last[2],
               wl={"map_info": map_info, "cases": cases},
               e2e={"value": L * steps / t_e2e, "unit": "frames/s", "h2d_bytes_per_step": int(feat_bytes + map_bytes * n_kf / steps), "d2h_bytes_per_step": 2000,
                    "steps": steps, "h2d_detail": {"features_every_step": feat_bytes, "local_maps_on_keyframe_steps": map_bytes, "keyframe_steps": n_kf}})
    if rank == 0:
        import oracle_lib as orc
        cs = cases[res["k_last"]]
        rpi, rec, rst = orc.calib_frame(cs["surf_map"], cs["corner_map"], cs["surf_ref"], cs["corner_ref"], cs["surf_cal"], cs["corner_cal"], cs["pivot"],
                                        cs["pose_i_init"], cs["ext_ref"], cs["ext_cal_init"], cfg["gn_iters"], 1)
        dtp, drp = syn.pose_err(last[0], rpi)
        dte, dre = syn.pose_err(last[1], rec)
        res["parity"] = {"m": max(dtp, dte), "rad": max(drp, dre), "pose_i": {"m": dtp, "rad": drp}, "ext_cal": {"m": dte, "rad": dre},
                         "rows_gpu": last[2]["n_surf"], "rows_oracle": rst["rows"], "ext_err_vs_truth_rad": syn.pose_err(last[1], cs["ext_cal"])[1],
                         "ext_err_initial_rad": syn.pose_err(cs["ext_cal_init"], cs["ext_cal"])[1]}
    ctx.close()
    return res
